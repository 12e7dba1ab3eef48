"""Scenarios for per-asset / per-env tick sizes (MarketEnv::new(start_time, tick_sizes, step_size, trading),
crates/step_sim/src/market_env.rs:73-90: each asset's OrderBook has its own tick, create_order raises PriceError against
it, orderbook.rs:367-383, and its level-2 record puts the levels at its own tick offsets, orderbook.rs:229-264).

`m` exposes `MarketEnv(seed, start_time, tick_sizes, step_size, trading)` whose objects have the Rust method names plus
`history(asset)` (the asset's level-2 records), so the same hand-worked numbers are asserted against the CPU oracle and
the CUDA path.  Sides are booleans (True = Bid) and order ids `(asset, id)` tuples."""
import numpy as np
import pytest

MAX_PRICE = 2**32 - 1
BID, ASK = True, False


def l2_record(trade_vol, bid, ask, ask_vol, bid_vol, bids=(), asks=()):
    """A 45-word level-2 record (step_sim_numpy.rs:351-368); `bids` / `asks`: (vol, n_orders) of levels 0, 1, ..."""
    r = [trade_vol, bid, ask, ask_vol, bid_vol] + [0] * 40
    for i, (v, n) in enumerate(bids):
        r[5 + 4 * i], r[6 + 4 * i] = v, n
    for i, (v, n) in enumerate(asks):
        r[7 + 4 * i], r[8 + 4 * i] = v, n
    return np.array(r, dtype=np.uint32)


def market_env_tick_known_answers(m):
    """Ticks [1, 2, 5]: price 11 is refused on assets 1 and 2 only, a refused call creates no id, and each asset's
    level-2 record steps by its own tick (an empty level in between stays in the record)."""
    env = m.MarketEnv(0, 0, [1, 2, 5], 1000)
    for a in (1, 2):
        with pytest.raises(ValueError):
            env.place_order(a, BID, 10, 0, 11)
    assert env.place_order(0, BID, 10, 0, 11) == (0, 0)
    assert env.place_order(1, ASK, 5, 0, 20) == (1, 0)   # the refused calls above created nothing
    assert env.place_order(1, ASK, 6, 0, 22) == (1, 1)
    assert env.place_order(1, ASK, 7, 0, 26) == (1, 2)
    with pytest.raises(ValueError):
        env.place_order(2, BID, 3, 0, 52)
    assert [env.place_order(2, BID, v, 0, p) for p, v in ((50, 3), (45, 4), (35, 2))] == [(2, 0), (2, 1), (2, 2)]
    assert [env.place_order(2, ASK, v, 0, p) for p, v in ((60, 1), (65, 9))] == [(2, 3), (2, 4)]
    env.step()
    assert env.bid_asks() == [(11, MAX_PRICE), (0, 20), (50, 60)]
    assert np.array_equal(env.history(0)[-1], l2_record(0, 11, MAX_PRICE, 0, 10, bids=[(10, 1)]))
    # asset 1 (tick 2): ask levels 20, 22, 24 (empty), 26
    assert np.array_equal(env.history(1)[-1], l2_record(0, 0, 20, 18, 0, asks=[(5, 1), (6, 1), (0, 0), (7, 1)]))
    # asset 2 (tick 5): bid levels 50, 45, 40 (empty), 35; ask levels 60, 65
    assert np.array_equal(env.history(2)[-1], l2_record(0, 50, 60, 10, 9, bids=[(3, 1), (4, 1), (0, 0), (2, 1)], asks=[(1, 1), (9, 1)]))
    # a market buy of 3 takes 1 @ 60 and 2 of 9 @ 65 on asset 2 only
    env.place_order(2, BID, 3, 0, None)
    env.step()
    assert env.bid_asks() == [(11, MAX_PRICE), (0, 20), (50, 65)]
    assert np.array_equal(env.history(2)[-1], l2_record(3, 50, 65, 7, 9, bids=[(3, 1), (4, 1), (0, 0), (2, 1)], asks=[(7, 1)]))
    assert np.array_equal(env.history(1)[-1], l2_record(0, 0, 20, 18, 0, asks=[(5, 1), (6, 1), (0, 0), (7, 1)]))


ALL_KNOWN = [market_env_tick_known_answers]


def grid_price(rng, tick, center=600, half=12):
    """A price on `tick`'s grid within `half` ticks of `center`."""
    return int(rng.integers(center // tick - half, center // tick + half + 1)) * tick


def drive_markets(rng, envs, ticks, n_steps, n_markets=1, p_off=0.05):
    """Feed identical random MarketEnv instructions to every object in `envs` (place_order / cancel_order /
    modify_order taking `market=`, and step).  Limit prices are drawn on each asset's grid; with probability `p_off` a
    NEW row is priced off its asset's grid instead, and every env must refuse it.  Returns the number of refusals."""
    n_assets = len(ticks)
    ids = [[[] for _ in range(n_assets)] for _ in range(n_markets)]
    n_off = 0
    for _ in range(n_steps):
        for mk in range(n_markets):
            for _ in range(int(rng.integers(0, 25))):
                a = int(rng.integers(n_assets))
                t = ticks[a]
                u = rng.random()
                if u < 0.6 or not ids[mk][a]:
                    bid, vol, trader = bool(rng.random() < 0.5), int(rng.integers(1, 40)), int(rng.integers(100))
                    if t > 1 and rng.random() < p_off:
                        bad = grid_price(rng, t) + 1 + int(rng.integers(t - 1))
                        for e in envs:
                            with pytest.raises(ValueError):
                                e.place_order(a, bid, vol, trader, bad, market=mk)
                        n_off += 1
                        continue
                    price = None if rng.random() < 0.08 else grid_price(rng, t)
                    got = {e.place_order(a, bid, vol, trader, price, market=mk) for e in envs}
                    assert len(got) == 1
                    ids[mk][a].append(got.pop()[1])
                elif u < 0.8:
                    i = ids[mk][a][int(rng.integers(len(ids[mk][a])))]
                    for e in envs:
                        e.cancel_order((a, i), market=mk)
                else:
                    i = ids[mk][a][int(rng.integers(len(ids[mk][a])))]
                    p = None if rng.random() < 0.3 else grid_price(rng, t)
                    v = None if (p is not None and rng.random() < 0.3) else int(rng.integers(1, 40))
                    for e in envs:
                        e.modify_order((a, i), p, v, market=mk)
        for e in envs:
            e.step()
    return n_off


class OracleMarkets:
    """`n_markets` oracle MarketEnvs behind the batched interface (market k shuffles with seed + k)."""

    def __init__(self, oracle, seed, ticks, n_markets, step_size):
        self.m = [oracle.MarketEnv(seed + k, 0, list(ticks), step_size) for k in range(n_markets)]

    def place_order(self, a, bid, vol, trader, price, market=0): return self.m[market].place_order(a, bid, vol, trader, price)
    def cancel_order(self, oid, market=0): self.m[market].cancel_order(oid)
    def modify_order(self, oid, p, v, market=0): self.m[market].modify_order(oid, p, v)

    def step(self):
        for x in self.m:
            x.step()


def env_rows(rng, tick, n_orders):
    """One env's random Env-mode rows for a step: (action, bid, vol, trader, price, order_id, flags) tuples, limit prices
    on `tick`'s grid; `n_orders`: ids issued so far (the rows' NEW ids follow in order)."""
    from bourse_b200 import abi   # (constants only: no library call)
    rows = []
    for _ in range(int(rng.integers(0, 12))):
        u = rng.random()
        if u < 0.6 or not n_orders:
            market = rng.random() < 0.08
            rows.append((abi.ACT_NEW, int(rng.random() < 0.5), int(rng.integers(1, 40)), int(rng.integers(100)),
                         0 if market else grid_price(rng, tick), 0, abi.F_MARKET if market else abi.F_HAS_PRICE))
            n_orders += 1
        elif u < 0.8:
            rows.append((abi.ACT_CANCEL, 0, 0, 0, 0, int(rng.integers(n_orders)), 0))
        else:
            rows.append((abi.ACT_MODIFY, 0, int(rng.integers(1, 40)), 0, grid_price(rng, tick), int(rng.integers(n_orders)),
                         abi.F_HAS_PRICE | abi.F_HAS_VOL))
    return rows, n_orders


def apply_rows_oracle(o, rows):
    """The same rows on an oracle StepEnv."""
    from bourse_b200 import abi
    for act, bid, vol, trader, price, oid, flags in rows:
        if act == abi.ACT_NEW:
            o.place_order(bool(bid), vol, trader, None if flags & abi.F_MARKET else price)
        elif act == abi.ACT_CANCEL:
            o.cancel_order(oid)
        else:
            o.modify_order(oid, price, vol)
