"""GPU suite for the device-resident market step (bb_step_device_market, gym.MarketVectorEnv): per market, the rows of a
step do exactly what MarketEnv::place_order / cancel_order / modify_order in row order and then MarketEnv::step(rng) do
(crates/step_sim/src/market_env.rs:108-121, 163-219).  Everything is checked against oracle.MarketEnv, and against a twin
handle driven through the host path (MarketEnv.submit + step)."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, market

pytestmark = pytest.mark.gpu

ERR_CAP_QUEUE, ERR_TIME_ORDER, ERR_PRICE, ERR_ROW_OP = 0x08, 0x100, 0x200, 0x400
ENGINES = {
    "fast": dict(pages_smem=32, pages_total=32),
    "paged": dict(pages_smem=8, pages_total=64),
    "dense": dict(price_window=(0, 256)),
    "dense_l": dict(price_window=(0, 512), live_cap=254),
}
TICKS = {2: [1, 2], 3: [1, 2, 3], 5: [1, 2, 3, 1, 2], 8: [1, 2, 3, 1, 2, 1, 3, 2]}


def random_block(rng, ticks, issued, rows, off_tick=True, bad_asset=False):
    """One market's action rows for a step (packed, host) with mixed limit / market NEWs, cancels and modifies of ids
    already issued (or issued earlier in the block), no-ops and, optionally, off-tick limit prices and rows naming no asset.
    `issued[a]` counts the ids of asset a's book and is advanced by the block's on-tick NEWs."""
    A = len(ticks)
    cols = {k: np.zeros(rows, np.int64) for k in ("op", "asset", "bid", "vol", "trader", "price", "oid", "mkt", "hp", "hv")}
    bad_row = int(rng.integers(rows)) if bad_asset else -1
    for r in range(rows):
        a = int(rng.integers(A))
        u = rng.random()
        c = {"asset": a, "vol": int(rng.integers(1, 30)), "trader": int(rng.integers(1000)), "bid": int(rng.random() < 0.5)}
        if r == bad_row:   # a NEW naming an asset the market does not have
            c["op"], c["asset"], c["price"] = abi.OP_NEW, A + int(rng.integers(3)), ticks[0] * 40
        elif u < 0.08:
            c["op"] = abi.OP_NOOP
        elif u < 0.6 or issued[a] == 0:
            c["op"] = abi.OP_NEW
            if rng.random() < 0.1:
                c["mkt"] = 1
            else:
                c["price"] = ticks[a] * int(rng.integers(30 // ticks[a] + 10, 150 // ticks[a] - 10))
                if off_tick and ticks[a] > 1 and rng.random() < 0.08:
                    c["price"] += 1
            if c.get("mkt") or c["price"] % ticks[a] == 0:
                issued[a] += 1
        elif u < 0.8:
            c["op"], c["oid"] = abi.OP_CANCEL, int(rng.integers(issued[a]))
        else:
            c["op"], c["oid"] = abi.OP_MODIFY, int(rng.integers(issued[a]))
            c["hp"], c["hv"] = int(rng.random() < 0.5), int(rng.random() < 0.7)
            c["price"] = ticks[a] * int(rng.integers(30 // ticks[a] + 10, 150 // ticks[a] - 10))
        for k, v in c.items():
            cols[k][r] = v
    return gym.pack_actions(cols["op"], bid=cols["bid"], vol=cols["vol"], trader=cols["trader"], price=cols["price"],
                            order_id=cols["oid"], market=cols["mkt"], has_price=cols["hp"], has_vol=cols["hv"], asset=cols["asset"])


def oracle_rows(o, blk):
    """The block through one oracle MarketEnv, then one step.  Returns (ids, assets whose place_order raised, row-op rows)."""
    ids, bad, row_op = [], set(), 0
    for x in blk:
        op, a = int(x["op_flags"]) & 0xFF, int(x["aux"])
        i = abi.NO_ID
        if a >= o.n_assets:
            row_op += 1
        elif op == abi.OP_NEW:
            price = None if x["op_flags"] & abi.F_MARKET else int(x["price"])
            try:
                i = o.place_order(a, bool(x["op_flags"] & abi.F_BID), int(x["vol"]), int(x["trader"]), price)[1]
            except ValueError:
                bad.add(a)
        elif op == abi.OP_CANCEL:
            o.cancel_order((a, int(x["order_id"])))
        elif op == abi.OP_MODIFY:
            f = int(x["op_flags"])
            o.modify_order((a, int(x["order_id"])), int(x["price"]) if f & abi.F_HAS_PRICE else None,
                           int(x["vol"]) if f & abi.F_HAS_VOL else None)
        ids.append(i)
    o.step()
    return ids, bad, row_op


def assert_books_equal(env, mk, A, o):
    for a in range(A):
        b = mk * A + a
        assert np.array_equal(env.history(b), o.history(a)), (mk, a)
        assert env.get_orders(b) == o.get_orders(a), (mk, a)
        assert env.get_trades(b) == o.get_trades(a), (mk, a)
    assert [tuple(int(x) for x in env.book_level_1(mk * A + a)[:2]) for a in range(A)] == o.bid_asks(), mk
    assert env.time(mk * A) == o.time(), mk


def run_against_oracle(oracle, v, seeds, ticks, n_steps, rng, rows, off_tick=True, bad_asset=False):
    """Drive a MarketVectorEnv and one oracle market per market with the same random blocks; per step the ids and the
    observation must match.  Returns the oracles, the assets whose oracle place_order raised per market, row-op counts."""
    A, n_markets = len(ticks), v.n_markets
    oracles = [oracle.MarketEnv(s, 0, ticks, 1000) for s in seeds]
    issued = [[0] * A for _ in range(n_markets)]
    bad, row_op = [set() for _ in range(n_markets)], [0] * n_markets
    for _ in range(n_steps):
        blk = np.stack([random_block(rng, ticks, issued[mk], rows, off_tick, bad_asset and rng.random() < 0.3) for mk in range(n_markets)])
        obs, ids = v.step(blk)
        obs, ids = obs.numpy(), ids.numpy()
        for mk in range(n_markets):
            want, b, r = oracle_rows(oracles[mk], blk[mk])
            bad[mk] |= b
            row_op[mk] += r
            assert list(ids[mk]) == want, mk
            for a in range(A):
                assert np.array_equal(obs[mk, a], oracles[mk].history(a)[-1]), (mk, a)
    return oracles, bad, row_op


@pytest.mark.parametrize("engine", list(ENGINES))
@pytest.mark.parametrize("A", [2, 3, 5, 8])
def test_random_blocks_bit_exact(oracle, engine, A):
    """Mixed NEW (limit, market, off-tick), CANCEL, MODIFY and no-op rows, and now and then a row naming no asset, on 2-8
    assets; 5 and 8 go past the in-kernel market agents' 4-asset limit."""
    ticks, n_markets, n_steps, seed = TICKS[A], 6, 32, 11
    rows = 4 * A
    v = gym.MarketVectorEnv(n_markets, rows, seed, 0, ticks, 1000, max_orders=4096, max_trades=8192, max_steps=64, **ENGINES[engine])
    v.reset()
    oracles, bad, row_op = run_against_oracle(oracle, v, [seed + m for m in range(n_markets)], ticks, n_steps,
                                              np.random.default_rng(A * 7 + len(engine)), rows, bad_asset=True)
    n_tr = 0
    for mk in range(n_markets):
        assert_books_equal(v.env, mk, A, oracles[mk])
        n_tr += sum(len(oracles[mk].get_trades(a)) for a in range(A))
    assert n_tr > 100
    err = v.env.env_errors().reshape(n_markets, A)
    want = np.array([[(ERR_PRICE if a in bad[mk] else 0) | (ERR_ROW_OP if a == 0 and row_op[mk] else 0) for a in range(A)]
                     for mk in range(n_markets)])
    assert np.array_equal(err, want), (err, want)
    assert sum(len(b) for b in bad) > 0 and sum(row_op) > 0
    v.close()


def _host_submit(m, blocks, A):
    """The rows of every market through MarketEnv.submit (market by market, row order kept), no-op rows left out."""
    rows = [(mk, x) for mk, blk in enumerate(blocks) for x in blk if int(x["op_flags"]) & 0xFF != abi.OP_NOOP]
    ids = np.full((len(blocks), max(len(b) for b in blocks)), abi.NO_ID, np.uint64)
    if not rows:
        return ids
    f = np.array([int(x["op_flags"]) for _, x in rows], np.uint32)
    op = f & 0xFF
    flags = np.where(op == abi.OP_NEW, np.where(f & abi.F_MARKET, abi.F_MARKET, abi.F_HAS_PRICE), f & (abi.F_HAS_PRICE | abi.F_HAS_VOL))
    out = m.submit(op, [int(x["aux"]) for _, x in rows], side=(f & abi.F_BID) != 0, vol=[int(x["vol"]) for _, x in rows],
                   trader=[int(x["trader"]) for _, x in rows], price=[int(x["price"]) for _, x in rows],
                   order_id=[int(x["order_id"]) for _, x in rows], market=[mk for mk, _ in rows], flags=flags.astype(np.uint32))
    k = 0
    for mk, blk in enumerate(blocks):
        for r, x in enumerate(blk):
            if int(x["op_flags"]) & 0xFF != abi.OP_NOOP:
                ids[mk, r] = out[k]
                k += 1
    return ids


@pytest.mark.parametrize("engine", list(ENGINES))
def test_twin_handle_host_path_equivalence(engine):
    """The same rows through MarketEnv.submit + step on a twin handle give identical ids, books, trades, history and error
    words.  On the dense engines a short step_size makes some books receive more events than step_size, so the time-order
    flag is raised by both paths on the same books."""
    ticks, n_markets, rows, seed = [1, 2, 3], 8, 12, 5
    step = 6 if engine.startswith("dense") else 1000
    kw = dict(max_orders=4096, max_trades=8192, max_steps=64, **ENGINES[engine])
    v = gym.MarketVectorEnv(n_markets, rows, seed, 0, ticks, step, **kw)
    m = market.MarketEnv(seed, 0, ticks, step, n_markets=n_markets, **kw)
    v.reset()
    rng = np.random.default_rng(3)
    issued = [[0] * 3 for _ in range(n_markets)]
    for s in range(30):
        blocks = [random_block(rng, ticks, issued[mk], rows, off_tick=False) for mk in range(n_markets)]
        _, ids = v.step(np.stack(blocks))
        want = _host_submit(m, blocks, 3)
        try:
            m.step()
        except MemoryError:   # (the host path reports the device's time-order flags at once; the words stay set)
            assert engine.startswith("dense")
        assert np.array_equal(ids.numpy(), want), s
    for b in range(3 * n_markets):
        assert np.array_equal(v.env.history(b), m._env.history(b)), b
        assert v.env.get_orders(b) == m._env.get_orders(b), b
        assert v.env.get_trades(b) == m._env.get_trades(b), b
    err_v, err_m = v.env.env_errors(), m.env_errors()
    assert np.array_equal(err_v, err_m), (err_v, err_m)
    if engine.startswith("dense"):
        assert (err_v & ERR_TIME_ORDER).any() and not (err_v & np.uint32(0xFFFFFFFF ^ ERR_TIME_ORDER)).any(), err_v
    else:
        assert not err_v.any(), err_v
    v.close()
    m._env.close()


def test_twin_handle_queue_overflow_flags():
    """A market whose every book's share exceeds max_queue: both paths flag BB_ERR_CAP_QUEUE on every book of that market
    and nowhere else.  (What runs differs by design: the host path applies each book's first max_queue events, the device
    path drops the market's whole step.)"""
    ticks, n_markets, rows = [1, 2], 3, 10
    kw = dict(max_orders=1024, max_trades=1024, max_steps=16, max_queue=4, pages_smem=32, pages_total=32)
    d = market.MarketEnv(1, 0, ticks, 1000, n_markets=n_markets, **kw)   # driven through bb_step_device_market
    m = market.MarketEnv(1, 0, ticks, 1000, n_markets=n_markets, **kw)
    blocks = []
    for mk in range(n_markets):
        n = rows if mk == 1 else 6   # market 1: 10 rows, 5 per asset > max_queue 4; the others 6 rows, within both limits
        blocks.append(gym.pack_actions(np.full(n, abi.OP_NEW), bid=np.arange(n) % 4 < 2, vol=5, trader=1, price=40, asset=np.arange(n) % 2))
    flat = np.concatenate(blocks)
    offs_h = np.concatenate([[0], np.cumsum([len(x) for x in blocks])]).astype(np.uint64)
    acts, offs = gym.DeviceArray(d._env, flat.shape, gym.ACTION_DTYPE), gym.DeviceArray(d._env, offs_h.shape, np.uint64)
    acts.copy_from_host(flat)
    offs.copy_from_host(offs_h)
    d._env.step_device_market(acts.ptr, offs.ptr, len(flat))
    _host_submit(m, blocks, 2)
    with pytest.raises(MemoryError):
        m.step()
    err_v, err_m = d.env_errors(), m.env_errors()
    assert np.array_equal(err_v, err_m) and list(err_v) == [0, 0, ERR_CAP_QUEUE, ERR_CAP_QUEUE, 0, 0], (err_v, err_m)
    assert d.get_orders(0, 1) == [] and d.time(1) == 1000   # the device path ran market 1's step with none of its rows
    acts.free(); offs.free()
    d._env.close()
    m._env.close()


def test_oracle_keyed_runner_leaves_the_market_stream_alone(oracle):
    """The oracle's keyed market runner shuffles with Philox only: after it, a market's own Xoroshiro stream is where it
    was, as on the GPU (whose in-kernel market agents never touch the books' copies of it).  The same 6 orders placed into
    a fresh market and into one that ran 4 keyed agent steps land at the same positions of their step's shuffled queue."""
    agents = [market.RandomMarketAgents(0, 30, (40, 60), (10, 20), 1, 0.8), market.RandomMarketAgents(1, 30, (40, 60), (10, 20), 2, 0.8)]
    offsets = []
    for run in (0, 4):
        o = oracle.MarketEnv(9, 0, [1, 2], 1000)
        o.set_groups([a.group for a in agents], [a.asset for a in agents])
        if run:
            o.run_agents(run, 77, market_id=0, keyed=True)
            assert o.n_instructions() > 50
        t0 = o.time()
        for k in range(6):
            o.place_order(0, k % 2 == 0, 1, 9000 + k, 1000 + k)   # far from the agents' prices: these rest
        o.step()
        by_trader = {x[7]: x[2] - t0 for x in o.get_orders(0) if x[7] >= 9000}
        offsets.append([by_trader[9000 + k] for k in range(6)])
    assert offsets[0] == offsets[1] and sorted(offsets[0]) == list(range(6)), offsets


@pytest.mark.parametrize("engine", ["fast", "dense"])
def test_interleaving_host_device_and_agent_steps(oracle, engine):
    """One handle alternates device steps, host-path steps and in-kernel market agents; the shuffle streams hand over in
    both directions and across a reset.  The oracle's keyed runner counts only its own steps in the Philox key while the
    GPU counts every step, so the active population runs first in each epoch; later agent launches use a quiet population
    (activity 0), which queues nothing and is one plain step on the oracle's side."""
    ticks, n_markets, rows, seed, aseed = [1, 2, 3], 4, 9, 21, 99
    A = len(ticks)
    m = market.MarketEnv(seed, 0, ticks, 1000, n_markets=n_markets, max_orders=8192, max_trades=8192, max_steps=128,
                         max_queue=128, **ENGINES[engine])
    env = m._env
    ids_d = gym.DeviceArray(env, (n_markets, rows), np.uint64)
    acts_d = gym.DeviceArray(env, (n_markets, rows), gym.ACTION_DTYPE)
    offs_d = gym.DeviceArray(env, (n_markets + 1,), np.uint64)
    offs_d.copy_from_host(np.arange(n_markets + 1, dtype=np.uint64) * np.uint64(rows))
    active = [market.RandomMarketAgents(a, 25, (40, 60), (5, 15), ticks[a], 0.6) for a in range(A)]
    quiet = [market.RandomMarketAgents(0, 4, (40, 60), (5, 15), 1, 0.0)]
    rng = np.random.default_rng(4)

    def epoch(plan):
        os_ = [oracle.MarketEnv(seed + mk, 0, ticks, 1000) for mk in range(n_markets)]
        for o in os_:
            o.set_groups([a.group for a in active], [a.asset for a in active])
        issued = [[len(os_[mk].get_orders(a)) for a in range(A)] for mk in range(n_markets)]
        for what in plan:
            if what == "agents":
                m.set_agents(active)
                m.run_agents(3, aseed)
                for mk, o in enumerate(os_):
                    o.run_agents(3, aseed, market_id=mk, keyed=True)
                issued = [[len(os_[mk].get_orders(a)) for a in range(A)] for mk in range(n_markets)]
                m.set_agents(quiet)
            elif what == "quiet":
                m.run_agents(2, aseed)
                for o in os_:
                    o.step(); o.step()
            else:
                blocks = [random_block(rng, ticks, issued[mk], rows, off_tick=False) for mk in range(n_markets)]
                if what == "device":
                    acts_d.copy_from_host(np.stack(blocks))
                    env.step_device_market(acts_d.ptr, offs_d.ptr, n_markets * rows, ids_d.ptr)
                    got = ids_d.numpy()
                else:
                    got = _host_submit(m, blocks, A)
                    m.step()
                for mk, o in enumerate(os_):
                    want, _, _ = oracle_rows(o, blocks[mk])
                    assert list(got[mk]) == want, (what, mk)
        for mk, o in enumerate(os_):
            assert_books_equal(env, mk, A, o)
        assert not env.env_errors().any()

    epoch(["agents", "device", "host", "device", "device", "host", "host", "quiet", "device", "quiet", "host", "device"])
    env.reset()
    epoch(["device", "host", "quiet", "device", "host"])
    env.reset()
    epoch(["host", "device", "quiet", "host"])
    for a in (ids_d, acts_d, offs_d):
        a.free()
    env.close()


def test_sharding_env_id_base():
    """With env_id_base != 0 market m shuffles with seed + env_id_base / assets + m, as bb_step does: a shard equals the
    same markets cut out of a larger handle."""
    ticks, rows, A = [1, 2, 3], 9, 3
    kw = dict(max_orders=2048, max_trades=4096, max_steps=32, pages_smem=32, pages_total=32)
    full = gym.MarketVectorEnv(6, rows, 4, 0, ticks, 1000, **kw)
    shard = gym.MarketVectorEnv(3, rows, 4, 0, ticks, 1000, env_id_base=3 * A, **kw)
    full.reset(); shard.reset()
    rng = np.random.default_rng(1)
    issued = [[0] * A for _ in range(6)]
    for _ in range(20):
        blk = np.stack([random_block(rng, ticks, issued[mk], rows, off_tick=False) for mk in range(6)])
        _, ids_f = full.step(blk)
        _, ids_s = shard.step(blk[3:])
        assert np.array_equal(ids_f.numpy()[3:], ids_s.numpy())
    for b in range(3 * A):
        assert np.array_equal(full.env.history(9 + b), shard.env.history(b)), b
        assert full.env.get_trades(9 + b) == shard.env.get_trades(b), b
    assert sum(len(shard.env.get_trades(b)) for b in range(9)) > 20
    full.close(); shard.close()


def test_sharding_against_oracle(oracle):
    ticks, rows, A = [1, 2], 6, 2
    v = gym.MarketVectorEnv(4, rows, 4, 0, ticks, 1000, env_id_base=5 * A, max_orders=2048, max_trades=4096, max_steps=32,
                            price_window=(0, 256))
    v.reset()
    oracles, _, _ = run_against_oracle(oracle, v, [4 + 5 + m for m in range(4)], ticks, 20, np.random.default_rng(2), rows,
                                       off_tick=False)
    for mk in range(4):
        assert_books_equal(v.env, mk, A, oracles[mk])
    v.close()


def test_market_step_inside_a_cuda_graph(oracle):
    """A captured MarketVectorEnv.step replayed K times equals K eager steps on a twin and the oracle.  Capture right after
    a host bb_step that shuffled is refused (the books' copies of the streams are stale); one eager device step fixes it."""
    import torch

    ticks, n_markets, rows, k = [1, 2, 3], 16, 6, 5
    A = len(ticks)
    kw = dict(max_orders=1024, max_trades=2048, max_steps=32)
    a, b = gym.MarketVectorEnv(n_markets, rows, 2, 0, ticks, 1000, **kw), gym.MarketVectorEnv(n_markets, rows, 2, 0, ticks, 1000, **kw)
    stream = torch.cuda.Stream()
    a.env.set_stream(stream.cuda_stream)
    a.reset(); b.reset()
    acts = torch.zeros((n_markets, rows, 8), dtype=torch.int32, device="cuda")
    rng = np.random.default_rng(0)
    blocks = []

    def fill():
        op = np.full((n_markets, rows), abi.OP_NEW, np.uint32)
        asset = rng.integers(0, A, (n_markets, rows))
        price = np.array(ticks)[asset] * rng.integers(18, 22, (n_markets, rows))
        blk = gym.pack_actions(op, bid=rng.random((n_markets, rows)) < 0.5, vol=rng.integers(1, 20, (n_markets, rows)),
                               price=price, trader=3, asset=asset)
        blocks.append(blk)
        acts.copy_(torch.from_numpy(blk.view(np.int32).reshape(n_markets, rows, 8)))
        torch.cuda.synchronize()

    fill()
    with torch.cuda.stream(stream):
        a.step(acts)                       # warm-up outside the capture (attribute / occupancy queries happen here)
    stream.synchronize()
    b.step(acts); b.env.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        a.step(acts)
    for _ in range(k):
        fill()
        g.replay()
        torch.cuda.synchronize()
        b.step(acts); b.env.synchronize()
        assert np.array_equal(a.obs.numpy(), b.obs.numpy()) and np.array_equal(a.ids.numpy(), b.ids.numpy())
    assert len(blocks) == k + 1
    for mk in (0, 7, 15):
        o = oracle.MarketEnv(2 + mk, 0, ticks, 1000)
        for blk in blocks:
            oracle_rows(o, blk[mk])
        assert_books_equal(a.env, mk, A, o)
        assert_books_equal(b.env, mk, A, o)
    assert sum(len(a.env.get_trades(x)) for x in range(A * n_markets)) > 50
    # a host step that shuffles (two rows in market 0) leaves the device copies behind: capture is refused, nothing recorded
    a.env.submit([abi.ACT_NEW, abi.ACT_NEW], side=[1, 0], vol=[1, 1], trader=[5, 5], price=[10, 200], env=[0, 1],
                 flags=[abi.F_HAS_PRICE, abi.F_HAS_PRICE])
    a.env.step()
    g2 = torch.cuda.CUDAGraph()
    with pytest.raises(ValueError, match="outside the capture"):
        with torch.cuda.graph(g2, stream=stream):
            a.step(acts)
    # one eager device step brings them up to date; capture works again and continues the stream bb_step left
    o = oracle.MarketEnv(2, 0, ticks, 1000)
    for blk in blocks:
        oracle_rows(o, blk[0])
    o.place_order(0, True, 1, 5, 10); o.place_order(1, False, 1, 5, 200); o.step()
    fill()
    with torch.cuda.stream(stream):
        a.step(acts)
    stream.synchronize()
    oracle_rows(o, blocks[-1][0])
    g3 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g3, stream=stream):
        a.step(acts)
    for _ in range(2):
        fill()
        g3.replay()
        torch.cuda.synchronize()
        oracle_rows(o, blocks[-1][0])
    assert_books_equal(a.env, 0, A, o)
    a.close(); b.close()


def test_edges_bad_asset_overlong_and_empty_slices(oracle):
    """aux >= assets: BB_ERR_ROW_OP on book 0 and BB_NO_ID; a slice longer than assets * max_queue: BB_ERR_CAP_QUEUE on
    every book of that market, nothing applied, time advanced; an empty slice: the books still step."""
    ticks, A = [1, 2], 2
    env = core.BatchedEnv(4 * A, 3, 0, 1, 1000, assets=A, max_orders=256, max_trades=256, max_steps=16, max_queue=4,
                          pages_smem=32, pages_total=32)
    env.set_tick_sizes(ticks)
    # market 0: 3 rows, one of them naming asset 7; market 1: 9 rows (> 2 * 4); market 2: empty; market 3: 2 rows
    rows = [gym.pack_actions([abi.OP_NEW, abi.OP_NEW, abi.OP_NEW], bid=[1, 0, 1], vol=5, trader=1, price=[40, 60, 40], asset=[0, 7, 1]),
            gym.pack_actions(np.full(9, abi.OP_NEW), bid=np.arange(9) % 2, vol=5, trader=1, price=40, asset=np.arange(9) % 2),
            gym.pack_actions(np.zeros(0, np.uint32)),
            gym.pack_actions([abi.OP_NEW, abi.OP_NEW], bid=[1, 0], vol=5, trader=1, price=[50, 50], asset=[1, 1])]
    flat = np.concatenate(rows)
    offs = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.uint64)
    d_rows, d_offs = gym.DeviceArray(env, flat.shape, gym.ACTION_DTYPE), gym.DeviceArray(env, offs.shape, np.uint64)
    d_ids, d_obs = gym.DeviceArray(env, flat.shape, np.uint64), gym.DeviceArray(env, (4 * A, 45), np.uint32)
    d_rows.copy_from_host(flat); d_offs.copy_from_host(offs)
    env.step_device_market(d_rows.ptr, d_offs.ptr, len(flat), d_ids.ptr, d_obs.ptr)
    ids = d_ids.numpy()
    N = abi.NO_ID
    assert list(ids) == [0, N, 0] + [N] * 9 + [0, 1], ids
    err = env.env_errors()
    assert list(err) == [ERR_ROW_OP, 0, ERR_CAP_QUEUE, ERR_CAP_QUEUE, 0, 0, 0, 0], err
    for b in range(4 * A):
        assert env.time(b) == 1000 and env.n_steps(b) == 1, b
    assert [env.n_orders(b) for b in range(8)] == [1, 1, 0, 0, 0, 0, 0, 2]
    obs = d_obs.numpy()
    for mk, blk in ((0, rows[0]), (2, rows[2]), (3, rows[3])):
        o = oracle.MarketEnv(3 + mk, 0, ticks, 1000)
        oracle_rows(o, [x for x in blk if x["aux"] < A])
        for a in range(A):
            assert np.array_equal(obs[mk * A + a], o.history(a)[-1]) and np.array_equal(env.history(mk * A + a), o.history(a))
    # the over-long market stepped with nothing applied
    assert env.get_orders(2) == [] and env.get_orders(3) == []
    for a in (d_rows, d_offs, d_ids, d_obs):
        a.free()
    env.close()


def test_argument_refusals():
    A = 2
    m = core.BatchedEnv(2 * A, 0, 0, 1, 1000, assets=A, max_orders=64, max_trades=64, max_steps=8, pages_smem=32, pages_total=32)
    offs = gym.DeviceArray(m, (3,), np.uint64)
    offs.copy_from_host(np.zeros(3, np.uint64))
    with pytest.raises(ValueError, match="null argument"):
        m.step_device_market(0, 0, 0)
    with pytest.raises(ValueError, match="null argument"):
        m.step_device_market(0, offs.ptr, 4)
    m.submit([abi.ACT_NEW], side=[1], vol=[1], price=[10], env=[1])
    with pytest.raises(ValueError, match="host-queued instructions pending"):
        m.step_device_market(0, offs.ptr, 0)
    m.step()
    m.step_device_market(0, offs.ptr, 0)   # rows: none; every book steps
    m.synchronize()
    assert [m.n_steps(b) for b in range(4)] == [2, 2, 2, 2]
    offs.free()
    m.close()
    single = core.BatchedEnv(4, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8)
    o1 = gym.DeviceArray(single, (5,), np.uint64)
    o1.copy_from_host(np.zeros(5, np.uint64))
    with pytest.raises(ValueError, match="bb_step_device"):
        single.step_device_market(0, o1.ptr, 0)
    o1.free()
    single.close()
    deep = core.BatchedEnv(2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8, price_window=(0, 256), deep_chunks=64)
    o2 = gym.DeviceArray(deep, (3,), np.uint64)
    o2.copy_from_host(np.zeros(3, np.uint64))
    with pytest.raises(ValueError):
        deep.step_device_market(0, o2.ptr, 0)
    o2.free()
    deep.close()
    with pytest.raises(ValueError, match="use VectorEnv"):
        gym.MarketVectorEnv(4, 2, 0, 0, [1], 1000)


def test_zero_copy_torch_and_history_ring(oracle):
    """Actions as a torch device tensor, observations and ids viewed in torch without a copy, and a loop running well past
    max_steps (the history is a scratch ring) still matching the oracle step by step."""
    import torch

    ticks, n_markets, rows, A = [2, 3], 3, 4, 2
    v = gym.MarketVectorEnv(n_markets, rows, 8, 0, ticks, 1000, max_orders=4096, max_trades=4096, max_steps=4, price_window=(0, 256))
    v.reset()
    obs_t, ids_t = torch.from_dlpack(v.obs), torch.from_dlpack(v.ids)
    assert obs_t.data_ptr() == v.obs.ptr and ids_t.data_ptr() == v.ids.ptr and tuple(obs_t.shape) == (n_markets, A, 45)
    oracles = [oracle.MarketEnv(8 + mk, 0, ticks, 1000) for mk in range(n_markets)]
    rng = np.random.default_rng(6)
    issued = [[0] * A for _ in range(n_markets)]
    for s in range(11):
        blk = np.stack([random_block(rng, ticks, issued[mk], rows, off_tick=False) for mk in range(n_markets)])
        acts = torch.from_numpy(blk.view(np.int32).reshape(n_markets, rows, 8)).cuda()
        torch.cuda.synchronize()
        v.step(acts)
        torch.cuda.synchronize()
        got_obs, got_ids = obs_t.cpu().numpy().view(np.uint32), ids_t.cpu().numpy().view(np.uint64)
        for mk in range(n_markets):
            want, _, _ = oracle_rows(oracles[mk], blk[mk])
            assert list(got_ids[mk]) == want, (s, mk)
            for a in range(A):
                assert np.array_equal(got_obs[mk, a], oracles[mk].history(a)[-1]), (s, mk, a)
    assert v.env.n_steps(0) == 3   # 11 steps through a 4-record ring: cleared after steps 4 and 8
    for mk in range(n_markets):
        for a in range(A):
            assert np.array_equal(v.env.history(mk * A + a), oracles[mk].history(a)[-3:])
    v.check_errors()
    v.close()
