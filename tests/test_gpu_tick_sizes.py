"""GPU suite for per-book tick sizes (bb_set_tick_sizes; MarketEnv::new(start_time, tick_sizes, ...),
market_env.rs:73-90): mixed-tick markets and per-env batched handles bit-exact against the oracle on the paged, dense and
deep engines, in-kernel market agents on mixed ticks, VectorEnv with per-env ticks, and the call's argument checks."""
import types

import numpy as np
import pytest

from bourse_b200 import abi, core, gym, market, workloads

from . import scenarios_ticks as st

pytestmark = pytest.mark.gpu

ERR_GRANULE, ERR_PRICE = 0x20, 0x200


class _GpuMarketEnv(market.MarketEnv):
    def history(self, asset, market=0): return self.get_level_2_data_history(asset, market)


@pytest.mark.parametrize("kw", [dict(), dict(price_window=(0, 256), live_cap=128)], ids=["paged", "dense"])
def test_known_answers_mixed_ticks(kw):
    def env(*a, **k): return _GpuMarketEnv(*a, max_orders=1024, max_trades=1024, max_queue=64, **kw, **k)
    for scenario in st.ALL_KNOWN:
        scenario(types.SimpleNamespace(MarketEnv=env))
    e = env(0, 0, [1, 2, 5], 1000)
    with pytest.raises(ValueError, match="tick-size 5"):   # the message names the asset's own tick
        e.place_order(2, True, 1, 0, 12)
    assert list(e._env.tick_sizes) == [1, 2, 5]


HANDLES = [([1, 2, 5], dict(pages_smem=32, pages_total=32)),                        # gcd 1: FAST engine
           ([2, 4, 6], dict(pages_smem=8, pages_total=64)),                         # gcd 2: generic paged engine, HBM pages
           ([1, 2, 5], dict(price_window=(500, 700), live_cap=254))]                # dense engine


@pytest.mark.parametrize("ticks,kw", HANDLES, ids=["fast_1_2_5", "paged_2_4_6", "dense_1_2_5"])
def test_random_mixed_tick_markets_bit_exact(oracle, ticks, kw):
    n_markets, n_steps, seed = 4, 60, 31
    g = market.MarketEnv(seed, 0, ticks, 10_000, n_markets=n_markets, max_orders=4096, max_trades=8192, max_queue=128, **kw)
    assert g.tick_size == int(np.gcd.reduce(ticks)) and list(g._env.tick_sizes) == ticks * n_markets
    o = st.OracleMarkets(oracle, seed, ticks, n_markets, 10_000)
    n_off = st.drive_markets(np.random.default_rng(8), [g, o], ticks, n_steps, n_markets)
    assert n_off > 10
    assert not g.env_errors().any(), g.env_errors()
    n_tr = 0
    for mk in range(n_markets):
        assert g.bid_asks(mk) == o.m[mk].bid_asks()
        for a in range(len(ticks)):
            assert np.array_equal(g.get_level_2_data_history(a, mk), o.m[mk].history(a)), (mk, a)
            assert g.get_trades(a, mk) == o.m[mk].get_trades(a), (mk, a)
            assert g.get_orders(a, mk) == o.m[mk].get_orders(a), (mk, a)
            n_tr += len(o.m[mk].get_trades(a))
    assert n_tr > 500


MOM = market.MomentumParams(tick_size=1, p_cancel=0.1, trade_vol=10, decay=1.0, demand=5.0, scale=0.5, order_ratio=1.0,
                            price_dist_mu=0.0, price_dist_sigma=1.0)
NOISE = market.NoiseAgentParams(tick_size=1, p_limit=0.3, p_market=0.1, p_cancel=0.2, trade_vol=7, price_dist_mu=0.5,
                                price_dist_sigma=0.8)


def mixed_tick_agents(ticks, noise=True):
    """Random, Momentum and Noise twins whose group ticks are multiples of their asset's tick.  noise=False: the dense
    window population (no noise traders, momentum traders send market orders only)."""
    n = len(ticks)
    out = [market.RandomMarketAgents(a, 40 - 5 * a, (40, 60), (10, 20), t * (1 + a % 2), 0.7) for a, t in enumerate(ticks)]
    out.append(market.MomentumMarketAgent(100, 12, n - 1, MOM._replace(tick_size=2 * ticks[-1], order_ratio=1.0 if noise else 0.0)))
    if noise:
        out.append(market.NoiseMarketAgent(1, 200, 9, NOISE._replace(tick_size=ticks[1])))
    out.append(market.RandomMarketAgents(n - 1, 17, (10, 90), (50, 70), ticks[-1], 0.3))
    return out


@pytest.mark.parametrize("ticks", [[1, 2], [1, 2, 5, 3]], ids=["2_assets", "4_assets"])
@pytest.mark.parametrize("kw", [dict(pages_smem=16, pages_total=64), dict(price_window=(0, 1024), live_cap=254)], ids=["paged", "dense"])
def test_market_agents_mixed_ticks_bit_exact(oracle, ticks, kw):
    n_markets, seed, n_steps = 3, 2024, 30
    g = market.MarketEnv(0, 0, ticks, 100_000, n_markets=n_markets, max_orders=8192, max_trades=8192, max_queue=128, **kw)
    agents = mixed_tick_agents(ticks, noise="price_window" not in kw)
    market.market_sim_runner(g, agents, seed, n_steps)
    assert not g.env_errors().any(), g.env_errors()
    n_tr = 0
    for mk in range(n_markets):
        o = oracle.MarketEnv(0, 0, ticks, 100_000)
        o.set_groups([a.group for a in agents], [a.asset for a in agents])
        o.run_agents(n_steps, seed, market_id=mk)
        for a in range(len(ticks)):
            assert np.array_equal(g.get_level_2_data_history(a, mk), o.history(a)), (mk, a)
            assert g.get_trades(a, mk) == o.get_trades(a), (mk, a)
            assert g.get_orders(a, mk) == o.get_orders(a), (mk, a)
            n_tr += len(o.get_trades(a))
    assert n_tr > 500


def test_momentum_off_its_books_tick_flags_that_asset_only():
    """A Momentum group with tick 3 trading a tick-2 asset: its limit prices are multiples of 3, so some are not on the
    book's grid (the reference unwraps a PriceError): ERR_GRANULE on that asset's books, nothing on the other's."""
    n_markets = 3
    g = market.MarketEnv(0, 0, [1, 2], 100_000, n_markets=n_markets, max_orders=8192, max_trades=8192, max_queue=128,
                         pages_smem=16, pages_total=64)
    agents = [market.RandomMarketAgents(0, 40, (40, 60), (10, 20), 1, 0.7), market.RandomMarketAgents(1, 40, (40, 60), (10, 20), 2, 0.7),
              market.MomentumMarketAgent(100, 12, 1, MOM._replace(tick_size=3))]
    market.market_sim_runner(g, agents, 5, 30)
    err = g.env_errors()
    assert (err[0::2] == 0).all(), err
    assert ((err[1::2] & ERR_GRANULE) != 0).all(), err


ENV_KW = [dict(pages_smem=32, pages_total=32), dict(price_window=(400, 800), live_cap=254)]


@pytest.mark.parametrize("kw", ENV_KW, ids=["paged", "dense"])
def test_batched_env_per_env_ticks_bit_exact(oracle, kw):
    """8 envs with ticks 1..8, a host-queued random Env-mode stream against one oracle StepEnv per env."""
    n, seed, ticks = 8, 3, list(range(1, 9))
    e = core.BatchedEnv(n, seed, 0, ticks, 1000, obs_words=abi.OBS_L2, max_orders=4096, max_trades=8192, max_steps=64,
                        max_queue=64, **kw)
    assert list(e.tick_sizes) == ticks and e.tick_size == 1
    oracles = [oracle.StepEnv(seed + k, 0, ticks[k], 1000) for k in range(n)]
    rng, n_ord = np.random.default_rng(11), [0] * n
    for step in range(40):
        rows, envs = [], []
        for k in range(n):
            r, n_ord[k] = st.env_rows(rng, ticks[k], n_ord[k])
            st.apply_rows_oracle(oracles[k], r)
            rows += r
            envs += [k] * len(r)
        if rows:
            a = np.array(rows, dtype=np.uint64)
            e.submit(a[:, 0].astype(np.uint32), a[:, 1].astype(np.uint8), a[:, 2], a[:, 3], a[:, 4], a[:, 5], env=envs,
                     flags=a[:, 6].astype(np.uint32))
        if step % 7 == 3:   # an off-tick limit order names the env's own tick and queues nothing
            k = int(rng.integers(1, n))
            with pytest.raises(ValueError, match=f"tick-size {ticks[k]}$"):
                e.submit([abi.ACT_NEW], side=[1], vol=[1], trader=[0], price=[ticks[k] * 70 + 1], env=[k])
        e.step()
        for o in oracles:
            o.step()
    assert not e.env_errors().any(), e.env_errors()
    l2 = e.level_2_data()
    n_tr = 0
    for k, o in enumerate(oracles):
        assert np.array_equal(e.history(k), o._history()), k
        assert e.get_orders(k) == o.get_orders() and e.get_trades(k) == o.get_trades(), k
        assert np.array_equal(e.book_level_2(k), o._l2()) and np.array_equal(l2[k], o._l2()), k
        n_tr += len(o.get_trades())
    assert n_tr > 100


def test_deep_replay_per_env_ticks(oracle):
    """Deep-engine replay with emit records on books with ticks 1 and 2, against oracle OrderBook.replay."""
    n, window = 6000, (1792, 2304)
    streams = [workloads.replay_stream(n, 40 + t, tick_size=t, mid_ticks=2048 // t, trading_windows=False) for t in (1, 2)]
    e = core.BatchedEnv(2, 5, 0, [1, 2], 1000, obs_words=abi.OBS_L2, max_orders=n + 64, max_trades=4 * n + 64,
                        max_steps=n // 32 + 64, max_queue=32, price_window=window, deep_chunks=n // 8 + 2 * (window[1] - window[0]) + 64)
    e.replay(np.concatenate(streams), np.array([0, n, 2 * n], dtype=np.uint64))
    assert not e.env_errors().any(), e.env_errors()
    for k, t in enumerate((1, 2)):
        ob = oracle.OrderBook(0, t)
        obs = ob.replay(streams[k], obs_cap=n)
        assert len(obs) > 50
        assert np.array_equal(e.history(k), obs), k
        assert e.get_orders(k) == ob.get_orders() and e.get_trades(k) == ob.get_trades(), k
        assert list(e.book_level_1(k)) == ob._l1() and np.array_equal(e.book_level_2(k), ob.level_2_data()), k


def test_vector_env_per_env_ticks(oracle):
    n, rows, seed, ticks = 4, 6, 9, [1, 2, 3, 4]
    v = gym.VectorEnv(n, rows, seed, 0, ticks, 1000, max_orders=1024, max_trades=2048, max_steps=32)
    v.reset()
    oracles = [oracle.StepEnvNumpy(seed + k, 0, ticks[k], 1000) for k in range(n)]
    rng, n_ord = np.random.default_rng(4), [0] * n
    for _ in range(30):
        op = np.zeros((n, rows), np.uint32)
        bid, vol, price, oid = (np.zeros((n, rows), np.uint32) for _ in range(4))
        for k in range(n):
            for r in range(rows):
                u = rng.random()
                if u < 0.6 or not n_ord[k]:
                    op[k, r], bid[k, r], vol[k, r] = abi.OP_NEW, rng.random() < 0.5, rng.integers(1, 30)
                    price[k, r] = st.grid_price(rng, ticks[k])
                    n_ord[k] += 1
                elif u < 0.85:
                    op[k, r], oid[k, r] = abi.OP_CANCEL, rng.integers(n_ord[k])
            act = np.where(op[k] == abi.OP_NEW, 1, np.where(op[k] == abi.OP_CANCEL, 2, 0))
            oracles[k].submit_instructions((act, bid[k].astype(bool), vol[k], np.ones(rows, np.uint32), price[k], oid[k]))
            oracles[k].step()
        obs, _ = v.step(gym.pack_actions(op, bid=bid, vol=vol, price=price, order_id=oid, trader=1))
        obs = obs.numpy()
        for k in range(n):
            assert np.array_equal(obs[k], oracles[k].level_2_data()), k
    v.check_errors()
    # 6 is on the grids of ticks 1, 2 and 3 but not 4: only env 3 refuses it
    op = np.zeros((n, rows), np.uint32)
    op[:, 0] = abi.OP_NEW
    v.step(gym.pack_actions(op, bid=1, vol=1, price=6, trader=1))
    err = v.env.env_errors()
    assert err[3] & ERR_PRICE and not err[:3].any(), err
    v.close()


def test_set_tick_sizes_argument_checks():
    e = core.BatchedEnv(4, 0, 0, 1, 1000, max_orders=256, max_trades=256, max_steps=16, max_queue=16)
    lib = e._lib
    assert lib.bb_set_tick_sizes(e._h, None, 4) == abi.BB_EINVAL
    with pytest.raises(ValueError, match="n must be"):
        e.set_tick_sizes([1, 2, 3])
    with pytest.raises(ValueError, match="is 0"):
        e.set_tick_sizes([1, 0, 1, 1])
    e.set_tick_sizes([1, 2, 3, 4])
    # an env with queued transactions, then one with orders: refused, the ticks unchanged
    e.submit([abi.ACT_NEW], side=[1], vol=[5], trader=[0], price=[30], env=[2])
    with pytest.raises(ValueError, match="orders or queued"):
        e.set_tick_sizes([1, 1, 1, 1])
    e.step()
    with pytest.raises(ValueError, match="orders or queued"):
        e.set_tick_sizes([1, 1, 1, 1])
    assert list(e.tick_sizes) == [1, 2, 3, 4]
    with pytest.raises(ValueError, match="tick-size 3"):
        e.submit([abi.ACT_NEW], side=[1], vol=[5], trader=[0], price=[31], env=[2])
    # the ticks survive reset()
    e.reset()
    with pytest.raises(ValueError, match="tick-size 4"):
        e.submit([abi.ACT_NEW], side=[1], vol=[5], trader=[0], price=[6], env=[3])
    e.submit([abi.ACT_NEW] * 2, side=[1, 0], vol=[5, 3], trader=[0, 0], price=[8, 12], env=[3, 3])
    e.step()
    assert np.array_equal(e.book_level_2(3), st.l2_record(0, 8, 12, 3, 5, bids=[(5, 1)], asks=[(3, 1)]))
    e.close()
    # a tick that is not a multiple of the price granule
    g = core.BatchedEnv(2, 0, 0, 2, 1000, price_granule=2, max_orders=64, max_trades=64, max_steps=8, max_queue=8)
    with pytest.raises(ValueError, match="granule"):
        g.set_tick_sizes([2, 3])
    g.set_tick_sizes([4, 6])
    g.close()
    # a market handle takes one tick per asset, or one per book
    m = core.BatchedEnv(6, 0, 0, 1, 1000, assets=3, max_orders=64, max_trades=64, max_steps=8, max_queue=8)
    m.set_tick_sizes([1, 2, 5])
    assert list(m.tick_sizes) == [1, 2, 5] * 2
    with pytest.raises(ValueError, match="n must be"):
        m.set_tick_sizes([1, 2])
    m.set_tick_sizes([1, 2, 5, 3, 2, 1])
    m.close()


def _run_pair(groups, obs_words, **kw):
    out = []
    for call in (False, True):
        e = core.BatchedEnv(8, 0, 0, 1, 1_000_000, obs_words=obs_words, max_orders=4096, max_trades=8192, max_steps=32,
                            max_queue=128, **kw)
        if call:
            e.set_tick_sizes([1] * 8)
        e.set_agents(groups)
        e.run_agents(32, 101)
        out.append((e.history_all(32), [e.get_trades(k) for k in range(8)], e.level_2_data(), e.env_errors()))
        e.close()
    return out


@pytest.mark.parametrize("pop", ["c3", "momentum"])
def test_uniform_ticks_through_the_call_change_nothing(pop):
    if pop == "c3":
        groups = workloads.c3_groups()
        a, b = _run_pair(groups, abi.OBS_L1, **core.dense_kwargs_for(groups))
    else:
        groups = [core.random_group(40, (40, 60), (10, 20), 2, 0.7),
                  core.momentum_group(100, 12, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0)]
        a, b = _run_pair(groups, abi.OBS_L2)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    assert sum(len(t) for t in a[1]) > 100
