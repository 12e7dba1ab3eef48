"""GPU suite for the device-resident order and trade reads (bb_orders_device / bb_trades_device, VectorEnv / MarketVectorEnv
.orders() / .trades()): the reference's get_orders()[id] / order_status(id) and the trades get_trades() gained since the last
read (rust/src/types.rs:4-31), batched over every env.  Checked after every step against the oracle's order table and trade
log, and against the host reads bb_orders / bb_trades."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import market_split_oracle as mks
from .test_gpu_market_agents_rows import ENGINES as MARKET_ENGINES
from .test_gpu_market_agents_rows import TICKS, learner_block, mixed_agents, oracle_market, oracle_rows, random_agents

pytestmark = pytest.mark.gpu

ERR_CAP_ORDERS, ERR_CAP_TRADES, ERR_BAD_ID, ERR_ROW_OP = 0x01, 0x02, 0x10, 0x400
ENGINES = {   # C3 prices are 20 .. 178
    "fast": dict(),
    "paged": dict(pages_smem=4, pages_total=16),
    "dense": dict(price_window=(20, 180), live_cap=128),
    "dense_l": dict(price_window=(20, 180), live_cap=254),
}
NONE_ROW = (False, abi.STATUS_NONE, 0, 0, 0, 0, 0, 0)


def host(cols):
    return {k: v.numpy() for k, v in cols.items()}


def order_row(c, *idx):
    """One query's output as the first eight fields of a PyOrder tuple (side, status, arr, end, vol, start_vol, price, trader)."""
    return (bool(c["side_is_bid"][idx]), int(c["status"][idx]), int(c["arr_time"][idx]), int(c["end_time"][idx]), int(c["vol"][idx]),
            int(c["start_vol"][idx]), int(c["price"][idx]), int(c["trader"][idx]))


def trade_rows(c, n, *book):
    """The first n slots of one book's trade window as PyTrade tuples (t, side, price, vol, active_id, passive_id)."""
    return [(int(c["t"][book + (i,)]), bool(c["side_is_bid"][book + (i,)]), int(c["price"][book + (i,)]), int(c["vol"][book + (i,)]),
             int(c["active_id"][book + (i,)]), int(c["passive_id"][book + (i,)])) for i in range(n)]


def assert_padding(c, n, *book):
    """Slots n .. cap of a window: NO_ID ids and zeros elsewhere."""
    assert (c["active_id"][book][n:] == abi.NO_ID).all() and (c["passive_id"][book][n:] == abi.NO_ID).all()
    for k in ("t", "side_is_bid", "price", "vol"):
        assert not c[k][book][n:].any(), k


def padded(lists, width, fill):
    out = np.full((len(lists), width), fill, np.uint64)
    for i, x in enumerate(lists):
        out[i, :len(x)] = x
    return out


@pytest.mark.parametrize("engine", list(ENGINES))
def test_vector_env_reads_equal_the_oracle_every_step(oracle, engine):
    """VectorEnv with the C3 population: after every step, orders() of every id the learner holds equals the oracle's
    get_orders()[id], and trades(cap) equals the entries the oracle's get_trades() gained; at the end the windows make up
    the whole log."""
    groups = workloads.c3_groups()
    n_envs, rows, n_steps, seed, cap = 16, 3, 25, 91, 256
    v = gym.VectorEnv(n_envs, rows, 0, 0, 1, 1_000_000, agents=groups, agent_seed=seed, max_orders=8192, max_trades=8192,
                      max_steps=64, max_queue=160, **ENGINES[engine])
    orcs = [oracle.StepEnv(0, 0, 1, 1_000_000) for _ in range(n_envs)]
    for o in orcs:
        o.set_groups(groups)
    v.reset()
    rng = np.random.default_rng(len(engine))
    mine = [[] for _ in range(n_envs)]
    seen = [[] for _ in range(n_envs)]
    for s in range(n_steps):
        op = np.zeros((n_envs, rows), np.uint32)
        cols = {k: np.zeros((n_envs, rows), np.uint64) for k in ("bid", "vol", "trader", "price", "order_id", "market")}
        for e in range(n_envs):
            for r in range(rows):
                u = rng.random()
                if u < 0.15:
                    continue
                if u < 0.45 or not mine[e]:   # (few resting learner orders: the dense engine holds 128 per book)
                    op[e, r] = abi.OP_NEW
                    cols["bid"][e, r], cols["vol"][e, r] = rng.random() < 0.5, rng.integers(1, 30)
                    cols["trader"][e, r], cols["market"][e, r] = 500 + r, rng.random() < 0.3
                    cols["price"][e, r] = 2 * rng.integers(44, 57)
                else:
                    op[e, r] = abi.OP_CANCEL
                    cols["order_id"][e, r] = mine[e][rng.integers(len(mine[e]))]
        _, ids = v.step(gym.pack_actions(op, **cols))
        ids = ids.numpy()
        for e, o in enumerate(orcs):
            o.agents_update(seed, e)
            n0 = len(mine[e])
            for r in range(rows):
                if op[e, r] == abi.OP_NEW:
                    mine[e].append(o.place_order(bool(cols["bid"][e, r]), int(cols["vol"][e, r]), int(cols["trader"][e, r]),
                                                 None if cols["market"][e, r] else int(cols["price"][e, r])))
                elif op[e, r] == abi.OP_CANCEL:
                    o.cancel_order(int(cols["order_id"][e, r]))
            o.step_keyed(seed, e)
            assert [i for i in ids[e] if i != abi.NO_ID] == mine[e][n0:], (s, e)
        got = host(v.orders(padded(mine, rows * n_steps, abi.NO_ID)))
        tc, count = v.trades(cap)
        tc, count = host(tc), count.numpy()
        for e, o in enumerate(orcs):
            want_o = o.get_orders()
            for j in range(rows * n_steps):
                assert order_row(got, e, j) == (want_o[mine[e][j]][:8] if j < len(mine[e]) else NONE_ROW), (s, e, j)
            new = o.get_trades()[len(seen[e]):]
            assert count[e] == len(new) <= cap, (s, e)
            assert trade_rows(tc, len(new), e) == new, (s, e)
            assert_padding(tc, len(new), e)
            seen[e] += new
    v.check_errors()
    for e, o in enumerate(orcs):
        assert seen[e] == o.get_trades() == v.env.get_trades(e), e
    assert any(t[4] in mine[e] or t[5] in mine[e] for e in range(n_envs) for t in seen[e])   # the learner traded
    v.close()


MARKET_CASES = [("fast", 2, "mixed"), ("dense", 3, "random"), ("dense_l", 4, "random"), ("paged", 4, "mixed"), ("fast", 3, None),
                ("dense", 2, None)]


@pytest.mark.parametrize("engine,A,pop", MARKET_CASES, ids=[f"{e}-{A}-{p or 'rows_only'}" for e, A, p in MARKET_CASES])
def test_market_vector_env_reads_equal_the_oracle_every_step(oracle, engine, A, pop):
    """MarketVectorEnv with per-asset ticks, with the market agent populations of test_gpu_market_agents_rows and without
    agents: after every step orders(ids, assets) of every (asset, id) the learner holds equals the oracle's
    get_orders(asset)[id], and trades(cap)[m, a] equals the entries asset a's get_trades() gained."""
    ticks, n_markets, rows, n_steps, seed, cap = TICKS[A], 6, 6, 25, 0xB0A5, 256
    agents = None if pop is None else random_agents(A) if pop == "random" else mixed_agents(A)
    kw = dict(max_orders=8192, max_trades=16384, max_steps=64, max_queue=128, **MARKET_ENGINES[engine])
    if agents:
        v = gym.MarketVectorEnv(n_markets, rows, 0, 0, ticks, 1000, agents=agents, agent_seed=seed, **kw)
        orcs = [oracle_market(oracle, agents, ticks, 1000) for _ in range(n_markets)]
    else:
        v = gym.MarketVectorEnv(n_markets, rows, 7, 0, ticks, 1000, **kw)
        orcs = [oracle.MarketEnv(7 + mk, 0, ticks, 1000) for mk in range(n_markets)]
    v.reset()
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    seen = [[[] for _ in range(A)] for _ in range(n_markets)]
    rng = np.random.default_rng(A * 7 + len(engine))
    width = rows * n_steps
    for s in range(n_steps):
        blk = np.stack([learner_block(rng, ticks, mine[mk], rows) for mk in range(n_markets)])
        _, ids = v.step(blk)
        ids = ids.numpy()
        for mk, o in enumerate(orcs):
            if agents:
                mks.agents_update(o, seed, mk)
            assert list(ids[mk]) == oracle_rows(o, blk[mk], mine[mk]), (s, mk)
            mks.step_keyed(o, seed, mk) if agents else o.step()
        held = [[(a, i) for a in range(A) for i in mine[mk][a]] for mk in range(n_markets)]
        q_ids = padded([[i for _, i in h] for h in held], width, abi.NO_ID)
        q_assets = padded([[a for a, _ in h] for h in held], width, 0).astype(np.uint32)
        got = host(v.orders(q_ids, q_assets))
        tc, count = v.trades(cap)
        tc, count = host(tc), count.numpy()
        assert tc["t"].shape == (n_markets, A, cap) and count.shape == (n_markets, A)
        for mk, o in enumerate(orcs):
            for j in range(width):
                want = o.get_orders(held[mk][j][0])[held[mk][j][1]][:8] if j < len(held[mk]) else NONE_ROW
                assert order_row(got, mk, j) == want, (s, mk, j)
            for a in range(A):
                new = o.get_trades(a)[len(seen[mk][a]):]
                assert count[mk, a] == len(new) <= cap, (s, mk, a)
                assert trade_rows(tc, len(new), mk, a) == new, (s, mk, a)
                assert_padding(tc, len(new), mk, a)
                seen[mk][a] += new
    v.check_errors()
    for mk, o in enumerate(orcs):
        for a in range(A):
            assert seen[mk][a] == o.get_trades(a) == v.env.get_trades(mk * A + a), (mk, a)
    assert sum(len(x) for m in seen for x in m) > 100
    v.close()


def test_small_cap_continues_where_the_last_call_stopped():
    """A cap smaller than a step's trades: count > cap, and the following calls hand out the rest in order — no duplicate,
    no gap — so the concatenated windows equal the host read of the whole log."""
    n_envs, cap = 8, 3
    v = gym.VectorEnv(n_envs, 1, 0, 0, 1, 1_000_000, agents=workloads.c3_groups(), agent_seed=4, max_orders=4096, max_trades=4096,
                      max_steps=64, max_queue=128)
    v.reset()
    noop = gym.pack_actions(np.zeros((n_envs, 1), np.uint32))
    got = [[] for _ in range(n_envs)]
    over = False
    for s in range(12):
        v.step(noop)
        tc, count = v.trades(cap)
        tc, count = host(tc), count.numpy()
        over |= bool((count > cap).any())
        for e in range(n_envs):
            got[e] += trade_rows(tc, min(int(count[e]), cap), e)
            assert_padding(tc, min(int(count[e]), cap), e)
    assert over
    while True:   # drain
        tc, count = v.trades(cap)
        tc, count = host(tc), count.numpy()
        for e in range(n_envs):
            got[e] += trade_rows(tc, min(int(count[e]), cap), e)
        if (count <= cap).all():
            break
    assert not v.trades(cap)[1].numpy().any()
    for e in range(n_envs):
        assert got[e] == v.env.get_trades(e) and len(got[e]) > 3 * cap, e
    v.close()


def test_full_trade_log(oracle):
    """With a tiny max_trades the log overflows: the windows equal the first max_trades entries of the oracle's log, the count
    stops there, BB_ERR_CAP_TRADES is set on exactly the books that overflowed, and their neighbours' windows stay exact
    (nothing past a book's log is read)."""
    n_envs, rows, max_trades, cap = 6, 4, 24, 5
    v = gym.VectorEnv(n_envs, rows, 3, 0, 1, 1000, max_orders=1024, max_trades=max_trades, max_steps=64)
    orcs = [oracle.StepEnv(3 + e, 0, 1, 1000) for e in range(n_envs)]
    v.reset()
    rng = np.random.default_rng(2)
    got = [[] for _ in range(n_envs)]
    for s in range(20):
        bid = rng.random((n_envs, rows)) < 0.5
        vol = rng.integers(1, 10, (n_envs, rows))
        price = 50 + rng.integers(-2, 3, (n_envs, rows))
        price[1::2] = np.where(bid[1::2], 40, 60)   # odd envs never cross: few trades, they stay inside the log
        price[1::2, 0] = np.where(bid[1::2, 0] & (s % 5 == 0), 60, price[1::2, 0])
        v.step(gym.pack_actions(np.full((n_envs, rows), abi.OP_NEW, np.uint32), bid=bid, vol=vol, price=price, trader=1))
        for e, o in enumerate(orcs):
            for r in range(rows):
                o.place_order(bool(bid[e, r]), int(vol[e, r]), 1, int(price[e, r]))
            o.step()
        tc, count = v.trades(cap)
        tc, count = host(tc), count.numpy()
        for e in range(n_envs):
            logged = min(len(orcs[e].get_trades()), max_trades)
            assert count[e] == logged - len(got[e]), (s, e)
            got[e] += trade_rows(tc, min(int(count[e]), cap), e)
            assert_padding(tc, min(int(count[e]), cap), e)
    while v.trades(cap)[1].numpy().any():
        pass
    err = v.env.env_errors()
    full = 0
    for e, o in enumerate(orcs):
        want = o.get_trades()
        # (the drain above advanced the cursors: read the whole log again from a fresh cursor)
        assert got[e] == want[:len(got[e])], e
        overflowed = len(want) > max_trades
        full += overflowed
        assert (err[e] == ERR_CAP_TRADES) if overflowed else (err[e] == 0), (e, err[e])
        assert v.env.get_trades(e) == want[:max_trades], e
    assert 0 < full < n_envs
    # a fresh cursor reads each whole log: exactly min(trades, max_trades) entries
    import torch
    cursor = torch.zeros(n_envs, dtype=torch.int32, device="cuda")
    count = torch.zeros(n_envs, dtype=torch.int32, device="cuda")
    cols = {k: torch.zeros((n_envs, 64), dtype=torch.int64, device="cuda") for k in ("t", "active_id", "passive_id")}
    v.env.trades_device(cursor.data_ptr(), 64, count.data_ptr(), t=cols["t"].data_ptr(), active_id=cols["active_id"].data_ptr(),
                        passive_id=cols["passive_id"].data_ptr())
    torch.cuda.synchronize()
    for e, o in enumerate(orcs):
        n = min(len(o.get_trades()), max_trades)
        assert int(count[e]) == int(cursor[e]) == n, e
        assert [(int(cols["t"][e, i]), int(cols["active_id"][e, i]), int(cols["passive_id"][e, i])) for i in range(n)] == \
               [(t[0], t[4], t[5]) for t in o.get_trades()[:n]], e
        assert (cols["active_id"][e, n:] == -1).all()
    v.close()


def test_error_bits():
    """NO_ID queries: STATUS_NONE and zeros, no error.  A bad id: BB_ERR_BAD_ID on exactly its book.  A bad asset: BB_ERR_ROW_OP
    on book 0 of its market.  No other book's error word changes."""
    v = gym.VectorEnv(4, 2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8)
    v.reset()
    v.step(gym.pack_actions(np.full((4, 2), abi.OP_NEW, np.uint32), bid=[[1, 0]] * 4, vol=5, price=[[40, 60]] * 4, trader=3))
    got = host(v.orders(np.full((4, 3), abi.NO_ID, np.uint64)))
    assert all(order_row(got, e, j) == NONE_ROW for e in range(4) for j in range(3))
    assert not v.env.env_errors().any()
    q = np.array([[0, 1], [1, abi.NO_ID], [2, 0], [1, 64]], np.uint64)   # envs 2 and 3: ids 2 and 64 not issued
    got = host(v.orders(q))
    for e in range(4):
        want = v.env.get_orders(e)
        assert [w[:2] for w in want] == [(True, 1), (False, 1)]   # both resting (status Active)
        for j in range(2):
            assert order_row(got, e, j) == (want[q[e, j]][:8] if q[e, j] < 2 else NONE_ROW), (e, j)
    assert list(v.env.env_errors()) == [0, 0, ERR_BAD_ID, ERR_BAD_ID]
    with pytest.raises(RuntimeError):
        v.check_errors()
    v.close()
    A, n_markets = 2, 3
    m = gym.MarketVectorEnv(n_markets, 2, 0, 0, [1, 2], 1000, max_orders=64, max_trades=64, max_steps=8)
    m.reset()
    m.step(gym.pack_actions(np.full((n_markets, 2), abi.OP_NEW, np.uint32), bid=1, vol=5, price=40, trader=3, asset=[[0, 1]] * n_markets))
    q_ids = np.array([[0, abi.NO_ID], [0, 0], [1, 0]], np.uint64)
    q_assets = np.array([[1, 9], [5, 1], [1, 0]], np.uint32)   # market 0: NO_ID with a bad asset is no error
    got = host(m.orders(q_ids, q_assets))
    assert order_row(got, 0, 0)[:2] == (True, 1) and order_row(got, 0, 1) == NONE_ROW
    assert order_row(got, 1, 0) == NONE_ROW and order_row(got, 1, 1)[:2] == (True, 1)
    assert order_row(got, 2, 0) == NONE_ROW and order_row(got, 2, 1)[:2] == (True, 1)
    assert list(m.env.env_errors()) == [0, 0, ERR_ROW_OP, 0, 0, ERR_BAD_ID]
    m.close()
    # an order table that overflowed: ids keep being handed out past max_orders (BB_ERR_CAP_ORDERS), those have no record
    o = gym.VectorEnv(2, 6, 0, 0, 1, 1000, max_orders=4, max_trades=64, max_steps=8)
    o.reset()
    op = np.zeros((2, 6), np.uint32)
    op[0] = abi.OP_NEW
    o.step(gym.pack_actions(op, bid=1, vol=5, price=40, trader=3))
    assert o.env.n_orders(0) == 6 and list(o.env.env_errors()) == [ERR_CAP_ORDERS, 0]
    o.env.clear_errors()
    got = host(o.orders(np.array([[3, 4, 5], [abi.NO_ID] * 3], np.uint64)))
    assert order_row(got, 0, 0) == o.env.get_orders(0)[3][:8] and order_row(got, 0, 1) == order_row(got, 0, 2) == NONE_ROW
    assert list(o.env.env_errors()) == [ERR_BAD_ID, 0]
    o.close()


def test_cursor_reset_and_past_the_log():
    """reset() zeroes the env's cursor; a raw call with a cursor past the log returns count 0 and leaves the cursor alone."""
    import torch
    v = gym.VectorEnv(2, 2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8)
    blk = gym.pack_actions(np.full((2, 2), abi.OP_NEW, np.uint32), bid=[[1, 0]] * 2, vol=5, price=50, trader=3)
    v.reset()
    v.step(blk)
    first = host(v.trades(4)[0])
    assert list(v.trades(4)[1].numpy()) == [0, 0]
    v.reset()
    v.step(blk)
    cols, count = v.trades(4)
    assert list(count.numpy()) == [1, 1] and host(cols)["active_id"].tolist() == first["active_id"].tolist()
    cursor = torch.tensor([1, 7], dtype=torch.int32, device="cuda")
    count = torch.full((2,), 99, dtype=torch.int32, device="cuda")
    vol = torch.full((2, 4), 5, dtype=torch.int32, device="cuda")
    v.env.trades_device(cursor.data_ptr(), 4, count.data_ptr(), vol=vol.data_ptr())
    torch.cuda.synchronize()
    assert cursor.tolist() == [1, 7] and count.tolist() == [0, 0] and not vol.any()
    v.close()


def test_deep_engine_reads_equal_the_host_reads():
    """After bb_replay_device of C5-style streams on a deep handle, bb_orders_device / bb_trades_device equal bb_orders /
    bb_trades for sampled ids and the whole logs."""
    import torch
    n_rest, n_steps, per_step, n_books = 6000, 4, 800, 3
    streams = [workloads.c5_stream(n_rest, n_steps, per_step, seed=60 + i, mid_ticks=3000, depth_ticks=256) for i in range(n_books)]
    n = len(streams[0])
    env = core.BatchedEnv(n_books, 5, 0, 1, 1000, max_orders=n + 64, max_trades=4 * n, max_steps=64, max_queue=32,
                          price_window=(2688, 3328), deep_chunks=n // 8 + 1400)
    d_instrs = torch.from_numpy(np.concatenate(streams).view(np.uint8)).cuda()
    d_offs = torch.from_numpy((np.arange(n_books + 1, dtype=np.uint64) * n).view(np.int64)).cuda()
    torch.cuda.synchronize()
    env.replay_device(d_instrs.data_ptr(), d_offs.data_ptr())
    env.synchronize()
    assert not env.env_errors().any()
    rng = np.random.default_rng(0)
    k = 512
    q = np.stack([rng.choice(env.n_orders(b), k, replace=False) for b in range(n_books)]).astype(np.int64)
    d_q = torch.from_numpy(q).cuda()
    names = [c for c, _ in gym.ORDER_COLUMNS]
    out = {c: torch.zeros((n_books, k), dtype=torch.uint8 if dt == np.uint8 else torch.int64 if dt == np.uint64 else torch.int32,
                          device="cuda") for c, dt in gym.ORDER_COLUMNS}
    env.orders_device(d_q.data_ptr(), 0, k, **{c: out[c].data_ptr() for c in names})
    total = max(env.n_trades(b) for b in range(n_books))
    cursor = torch.zeros(n_books, dtype=torch.int32, device="cuda")
    count = torch.zeros(n_books, dtype=torch.int32, device="cuda")
    tr = {c: torch.zeros((n_books, total), dtype=torch.uint8 if dt == np.uint8 else torch.int64 if dt == np.uint64 else torch.int32,
                         device="cuda") for c, dt in gym.TRADE_COLUMNS}
    env.trades_device(cursor.data_ptr(), total, count.data_ptr(), **{c: tr[c].data_ptr() for c in tr})
    torch.cuda.synchronize()
    for b in range(n_books):
        ho, ht = env.orders_arrays(b), env.trades_arrays(b)
        for c, hc in zip(names, ("side", "status", "arr_time", "end_time", "vol", "start_vol", "price", "trader")):
            want = ho[hc][q[b]]
            assert np.array_equal(out[c][b].cpu().numpy().astype(want.dtype), want), (b, c)
        nt = len(ht["t"])
        assert nt > 500 and int(count[b]) == int(cursor[b]) == nt
        for c, hc in (("t", "t"), ("side_is_bid", "side"), ("price", "price"), ("vol", "vol"), ("active_id", "active"),
                      ("passive_id", "passive")):
            assert np.array_equal(tr[c][b, :nt].cpu().numpy().astype(ht[hc].dtype), ht[hc]), (b, c)
    env.close()


def _graph_twins(make, fill, read, k):
    """Capture step + orders + trades of `a` into a CUDA graph and replay it k times; `b` runs the same eagerly.  Every
    replay's outputs must equal the eager twin's."""
    import torch
    a, b = make(), make()
    stream = torch.cuda.Stream()
    a.env.set_stream(stream.cuda_stream)
    a.reset(); b.reset()
    fill()
    with torch.cuda.stream(stream):
        read(a)                           # warm-up outside the capture: allocates the read outputs
    stream.synchronize()
    ref = read(b); b.env.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        out = read(a)
    traded = 0
    for _ in range(k):
        fill()
        g.replay()
        torch.cuda.synchronize()
        ref = read(b); b.env.synchronize()
        for x, y in zip(out, ref):
            for c in x:
                assert np.array_equal(x[c].numpy(), y[c].numpy()), c
        traded += int(ref[2]["count"].numpy().sum())
    assert traded > 0
    a.close(); b.close()


def test_reads_inside_a_cuda_graph():
    """VectorEnv and MarketVectorEnv without agents: step + orders + trades captured with torch.cuda.graph and replayed."""
    import torch
    rng = np.random.default_rng(3)
    n_envs, rows = 64, 3
    acts = torch.zeros((n_envs, rows, 8), dtype=torch.int32, device="cuda")

    def fill():
        blk = gym.pack_actions(np.full((n_envs, rows), abi.OP_NEW, np.uint32), bid=rng.random((n_envs, rows)) < 0.5,
                               vol=rng.integers(1, 20, (n_envs, rows)), price=rng.integers(45, 56, (n_envs, rows)), trader=3)
        acts.copy_(torch.from_numpy(blk.view(np.int32).reshape(n_envs, rows, 8)))
        torch.cuda.synchronize()

    def read(v):
        _, ids = v.step(acts)
        tc, count = v.trades(16)
        return v.orders(ids), tc, {"count": count}

    _graph_twins(lambda: gym.VectorEnv(n_envs, rows, 2, 0, 1, 1000, max_orders=512, max_trades=1024, max_steps=32), fill, read, 5)
    n_markets, A = 16, 3
    macts = torch.zeros((n_markets, rows, 8), dtype=torch.int32, device="cuda")
    assets = torch.zeros((n_markets, rows), dtype=torch.int32, device="cuda")

    def mfill():
        a = rng.integers(0, A, (n_markets, rows))
        blk = gym.pack_actions(np.full((n_markets, rows), abi.OP_NEW, np.uint32), bid=rng.random((n_markets, rows)) < 0.5,
                               vol=rng.integers(1, 20, (n_markets, rows)), price=6 * rng.integers(8, 11, (n_markets, rows)), trader=3,
                               asset=a)
        macts.copy_(torch.from_numpy(blk.view(np.int32).reshape(n_markets, rows, 8)))
        assets.copy_(torch.from_numpy(a.astype(np.int32)))
        torch.cuda.synchronize()

    def mread(v):
        _, ids = v.step(macts)
        tc, count = v.trades(16)
        return v.orders(ids, assets), tc, {"count": count}

    _graph_twins(lambda: gym.MarketVectorEnv(n_markets, rows, 2, 0, [1, 2, 3], 1000, max_orders=512, max_trades=1024, max_steps=32),
                 mfill, mread, 5)


def test_refusals():
    e = core.BatchedEnv(2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8, max_queue=16)
    p = e.device_alloc(64)
    with pytest.raises(ValueError, match="null"):
        e.orders_device(0, 0, 1)
    with pytest.raises(ValueError, match="must be NULL"):
        e.orders_device(p, p, 1)
    with pytest.raises(ValueError, match="null"):
        e.trades_device(0, 4)
    e.submit([abi.ACT_NEW], [1], [1], [0], [10], env=[1])
    with pytest.raises(ValueError, match="pending"):
        e.orders_device(p, 0, 1)
    with pytest.raises(ValueError, match="pending"):
        e.trades_device(p, 4)
    e.device_free(p)
    e.close()
    m = core.BatchedEnv(4, 0, 0, 1, 1000, assets=2, max_orders=64, max_trades=64, max_steps=8, max_queue=16)
    p = m.device_alloc(64)
    with pytest.raises(ValueError, match="required"):
        m.orders_device(p, 0, 1)
    m.device_free(p)
    m.close()
    z = core.BatchedEnv(2, 0, 0, 1, 1000, max_orders=64, max_trades=0, max_steps=8, max_queue=16)
    p = z.device_alloc(64)
    with pytest.raises(ValueError, match="max_trades == 0"):
        z.trades_device(p, 4)
    z.device_free(p)
    z.close()
    v = gym.VectorEnv(2, 2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8)
    with pytest.raises(ValueError, match="shape"):
        v.orders(np.zeros((3, 2), np.uint64))

    class DLPackOnly:   # a producer without __cuda_array_interface__: its shape and element type are checked too
        def __init__(self, t): self.t = t
        def __dlpack__(self, stream=None): return self.t.__dlpack__()
        def __dlpack_device__(self): return self.t.__dlpack_device__()

    import torch
    for bad in (torch.zeros((2, 4), dtype=torch.int32, device="cuda"), torch.zeros(8, dtype=torch.int64, device="cuda"),
                torch.zeros((2, 2), dtype=torch.float64, device="cuda")):
        with pytest.raises(ValueError, match="8-byte integers"):
            v.orders(DLPackOnly(bad))
    got = host(v.orders(DLPackOnly(torch.full((2, 3), -1, dtype=torch.int64, device="cuda"))))   # -1 == NO_ID
    assert all(order_row(got, e, j) == NONE_ROW for e in range(2) for j in range(3))
    v.close()


def test_fills_example():
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "vector_env_fills_torch.py")], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    assert "device fills match the host reads" in out.stdout and "'error_envs': 0" in out.stdout
