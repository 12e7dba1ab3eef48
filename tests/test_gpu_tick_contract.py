"""GPU suite for the tick-size contract on every order path, against the oracle.  The reference checks a limit price
against its book's tick in create_order (orderbook.rs:367-383); its agents unwrap that PriceError and panic, and its
replay stops at it.  Here:
- in-kernel agents that draw an off-tick price flag exactly the envs whose oracle run raised (ERR_GRANULE), at the
  step it raised in, and every other env stays bit-exact;
- bb_replay refuses a stream with an off-tick limit NEW before it changes anything;
- per-env ticks on every agent, row and replay path are bit-exact when everything is on the grid."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import scenarios_ticks as st

pytestmark = pytest.mark.gpu

ERR_GRANULE, ERR_PRICE = 0x20, 0x200
CAPS = dict(max_orders=4096, max_trades=8192, max_steps=64, max_queue=128)

# engine -> (price granule u, keywords); the agent populations of scenarios_ticks quote on multiples of u
ENGINES = {"fast": (1, dict(pages_smem=32, pages_total=32)),
           "paged": (2, dict(pages_smem=8, pages_total=64)),                 # generic paged engine, HBM pages
           "dense": (1, dict(price_window=(0, 256), live_cap=254)),
           "dense_l": (1, dict(price_window=(0, 1024), live_cap=254))}
CASES = [(eng, pop) for eng in ENGINES for pop in st.OFFGRID_POPS if not (pop == "noise" and eng.startswith("dense"))]


def _oracle_env(oracle, groups, tick, env_id, n_steps):
    """(oracle env, index of the step whose agent update raised, or None)."""
    o = oracle.StepEnvNumpy(0, 0, tick, st.STEP)
    o.set_groups(groups)
    try:
        o.run_agents(n_steps, st.SEED, env_id=env_id)
        return o, None
    except ValueError:
        return o, len(o._history())


def _check_book(hist, trades, orders, err, o_hist, o_trades, o_orders, fail, err_want):
    """A book that ran on: bit-exact when its oracle did not raise; else the records and trades before the failing step."""
    if fail is None:
        assert err == 0, hex(err)
        assert np.array_equal(hist, o_hist) and trades == o_trades and orders == o_orders
    else:
        assert err == err_want, hex(err)
        assert np.array_equal(hist[:fail], o_hist)
        assert [t for t in trades if t[0] < fail * st.STEP] == o_trades


def _single(eng, pop, ticks):
    u, kw = ENGINES[eng]
    groups = st.offgrid_groups(core, pop, u, eng.startswith("dense"))
    e = core.BatchedEnv(len(ticks), 0, 0, [u * t for t in ticks], st.STEP, obs_words=abi.OBS_L2, **CAPS, **kw)
    e.set_agents(groups)
    return e, groups, [u * t for t in ticks]


@pytest.mark.parametrize("eng,pop", CASES)
def test_offgrid_agents_single_asset(oracle, eng, pop):
    e, groups, ticks = _single(eng, pop, [1, 2, 4, 2, 4, 2, 1])
    e.run_agents(st.N_STEPS, st.SEED)
    err = e.env_errors()
    fails = []
    for k, t in enumerate(ticks):
        o, f = _oracle_env(oracle, groups, t, k, st.N_STEPS)
        _check_book(e.history(k), e.get_trades(k), e.get_orders(k), int(err[k]), o._history(), o.get_trades(), o.get_orders(),
                    f, ERR_GRANULE)
        fails.append(f)
    assert fails[0] is None and fails[-1] is None and any(f is not None and f > 0 for f in fails), fails
    e.close()


@pytest.mark.parametrize("mode", ["split", "to_host"])
@pytest.mark.parametrize("eng", ["fast", "dense"])
def test_offgrid_agents_split_and_streamed(oracle, eng, mode):
    """Two launches: an env is flagged after the first exactly when its oracle raised in a step the first launch ran.
    Streamed to host: the streamed records are the handle's own."""
    e, groups, ticks = _single(eng, "random", [1, 2, 4, 2, 4, 2, 1])
    n1 = 5
    outs = [o_f for o_f in (_oracle_env(oracle, groups, t, k, st.N_STEPS) for k, t in enumerate(ticks))]
    if mode == "split":
        e.run_agents(n1, st.SEED)
        err1 = e.env_errors()
        assert [bool(x) for x in err1] == [f is not None and f < n1 for _, f in outs], (err1, [f for _, f in outs])
        e.run_agents(st.N_STEPS - n1, st.SEED)
        hist = [e.history(k) for k in range(len(ticks))]
    else:
        out = e.run_agents_to_host(st.N_STEPS, st.SEED, chunk_steps=8)
        hist = [out[k] for k in range(len(ticks))]
        for k in range(len(ticks)):
            assert np.array_equal(hist[k], e.history(k))
    err = e.env_errors()
    for k, (o, f) in enumerate(outs):
        _check_book(hist[k], e.get_trades(k), e.get_orders(k), int(err[k]), o._history(), o.get_trades(), o.get_orders(), f,
                    ERR_GRANULE)
    assert any(f is not None and f >= n1 for _, f in outs) or mode == "to_host"
    e.close()


@pytest.mark.parametrize("eng,pop", CASES)
def test_offgrid_agents_markets(oracle, eng, pop):
    """Market twins on ticks [u, 2u]: the off-grid group trades asset 1, so a market whose oracle raised has ERR_GRANULE on
    its asset-1 book only; both its books match the oracle up to the failing step."""
    u, kw = ENGINES[eng]
    n_markets, ticks = 6, st.market_ticks(u)
    groups, assets = st.offgrid_market_groups(core, pop, u, eng.startswith("dense"))
    e = core.BatchedEnv(2 * n_markets, 0, 0, ticks * n_markets, st.STEP, obs_words=abi.OBS_L2, assets=2, **CAPS, **kw)
    e.set_agents(groups, assets)
    e.run_agents(st.N_STEPS, st.SEED)
    err = e.env_errors()
    fails = []
    for mk in range(n_markets):
        o = oracle.MarketEnv(0, 0, ticks, st.STEP)
        o.set_groups(groups, assets)
        try:
            o.run_agents(st.N_STEPS, st.SEED, market_id=mk)
            f = None
        except ValueError:
            f = len(o.history(0))
        fails.append(f)
        for a in range(2):
            b = 2 * mk + a
            _check_book(e.history(b), e.get_trades(b), e.get_orders(b), int(err[b]), o.history(a), o.get_trades(a),
                        o.get_orders(a), f, ERR_GRANULE if a == 1 else 0)
    assert any(f is not None and f > 0 for f in fails), fails
    e.close()


def test_offgrid_background_agents_vector_env(oracle):
    """VectorEnv steps with background agents (bb_run_agents_with_rows): the same flags and records as the oracle."""
    ticks = [1, 2, 4, 2, 4, 2]
    groups = st.offgrid_groups(core, "momentum", 1)
    v = gym.VectorEnv(len(ticks), 2, 0, 0, ticks, st.STEP, agents=groups, agent_seed=st.SEED, max_orders=4096, max_trades=8192,
                      max_steps=64, max_queue=160)
    v.reset()
    noop = gym.pack_actions(np.zeros((len(ticks), 2), np.uint32))
    for _ in range(st.N_STEPS):
        v.step(noop)
    err = v.env.env_errors()
    fails = []
    for k, t in enumerate(ticks):
        o, f = _oracle_env(oracle, groups, t, k, st.N_STEPS)
        _check_book(v.env.history(k), v.env.get_trades(k), v.env.get_orders(k), int(err[k]), o._history(), o.get_trades(),
                    o.get_orders(), f, ERR_GRANULE)
        fails.append(f)
    assert fails[0] is None and any(f is not None and f > 0 for f in fails), fails
    v.close()


# ---- bb_replay: an off-tick limit NEW is refused before anything is applied
REPLAY = {"fast": (1, dict(pages_smem=32, pages_total=32)),
          "paged_res": (1, dict(pages_smem=64, pages_total=64)),             # generic geometry, every page on chip
          "paged": (2, dict(pages_smem=8, pages_total=64)),
          "dense": (1, dict(price_window=(256, 800), live_cap=254)),
          "deep": (1, dict(price_window=(256, 800)))}


def _replay_streams(u, ticks, n):
    """One C2-style stream per env on its tick; market NEWs carry off-tick prices and price MODIFYs go off the env's tick
    (never off the granule u), which the reference accepts: neither is checked by create_order."""
    out = []
    for k, t in enumerate(ticks):
        s = workloads.replay_stream(n, 60 + k, tick_size=t, mid_ticks=512 // t, half_width=128 // t, trading_windows=False)
        op = s["op_flags"] & 0xFF
        off = ((op == abi.OP_NEW) & ((s["op_flags"] & abi.F_MARKET) != 0)) | ((op == abi.OP_MODIFY) & ((s["op_flags"] & abi.F_HAS_PRICE) != 0))
        s["price"][off] += u
        out.append(s)
    return out


@pytest.mark.parametrize("eng", list(REPLAY))
def test_replay_refuses_off_tick_new_and_changes_nothing(oracle, eng):
    u, kw = REPLAY[eng]
    ticks, n, n0 = [u, 2 * u, 3 * u], 1500, 500
    streams = _replay_streams(u, ticks, n)
    if eng == "deep":
        kw = dict(kw, deep_chunks=n // 8 + 2 * 544 + 64)
    e = core.BatchedEnv(3, 0, 0, ticks, 1000, obs_words=abi.OBS_L2, max_orders=n + 64, max_trades=4 * n + 64, max_steps=n // 32 + 64,
                        max_queue=32, **kw)

    def replay(parts):
        e.replay(np.concatenate(parts), np.cumsum([0] + [len(p) for p in parts]).astype(np.uint64))

    replay([s[:n0] for s in streams])
    before = [(e.history(k), e.get_orders(k), e.get_trades(k), e.book_level_2(k)) for k in range(3)]
    assert sum(len(b[1]) for b in before) > 500
    # env 1's rest with one limit NEW one granule off its tick inserted at row 100
    bad = streams[1][n0:n0 + 1].copy()
    bad["op_flags"], bad["price"] = abi.OP_NEW | abi.F_BID, ticks[1] * 250 + u
    rest = [s[n0:] for s in streams]
    with pytest.raises(ValueError, match=f"env 1 row {n - n0 + 100}: Price {ticks[1] * 250 + u} was not a multiple of tick-size {ticks[1]}"):
        replay([rest[0], np.concatenate([rest[1][:100], bad, rest[1][100:]]), rest[2]])
    for k in range(3):
        h, o, t, l2 = before[k]
        assert np.array_equal(e.history(k), h) and e.get_orders(k) == o and e.get_trades(k) == t
        assert np.array_equal(e.book_level_2(k), l2)
    replay(rest)
    assert not e.env_errors().any(), e.env_errors()
    for k, t in enumerate(ticks):
        ob = oracle.OrderBook(0, t)
        obs = ob.replay(streams[k], obs_cap=n)
        assert np.array_equal(e.history(k), obs), k
        assert e.get_orders(k) == ob.get_orders() and e.get_trades(k) == ob.get_trades(), k
        assert np.array_equal(e.book_level_2(k), ob.level_2_data()), k
    e.close()


# ---- on-grid per-env ticks: bit-exact against one oracle env per book
ONGRID = {"dense": (1, dict(price_window=(232, 488), live_cap=254)),
          "dense_l": (1, dict(price_window=(0, 1024), live_cap=254)),
          "fast": (1, dict(pages_smem=32, pages_total=32)),
          "paged": (2, dict(pages_smem=8, pages_total=64)),
          "momentum": (1, dict(pages_smem=32, pages_total=32))}


@pytest.mark.parametrize("eng", list(ONGRID))
def test_ongrid_per_env_ticks_agents_bit_exact(oracle, eng):
    u, kw = ONGRID[eng]
    ticks = [u * t for t in (1, 2, 3, 4, 6, 12)]
    groups = [core.random_group(40, (20, 40), (10, 20), 12 * u, 0.7), core.random_group(30, (21, 38), (1, 9), 12 * u, 0.5)]
    if eng == "momentum":
        groups.append(core.momentum_group(100, 12, 12, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0))
    e = core.BatchedEnv(len(ticks), 0, 0, ticks, st.STEP, obs_words=abi.OBS_L2, **CAPS, **kw)
    e.set_agents(groups)
    e.run_agents(st.N_STEPS, st.SEED)
    assert not e.env_errors().any(), e.env_errors()
    n_tr = 0
    for k, t in enumerate(ticks):
        o, f = _oracle_env(oracle, groups, t, k, st.N_STEPS)
        assert f is None
        assert np.array_equal(e.history(k), o._history()), k
        assert e.get_trades(k) == o.get_trades() and e.get_orders(k) == o.get_orders(), k
        n_tr += len(o.get_trades())
    assert n_tr > 500
    e.close()


def test_ongrid_per_env_ticks_agents_with_rows(oracle):
    """bb_run_agents_with_rows on per-env ticks: background agents plus the caller's NEW / CANCEL rows on each env's grid."""
    ticks, rows = [1, 2, 3, 4], 3
    groups = [core.random_group(40, (20, 40), (10, 20), 12, 0.7)]
    v = gym.VectorEnv(len(ticks), rows, 0, 0, ticks, st.STEP, agents=groups, agent_seed=st.SEED, max_orders=4096, max_trades=8192,
                      max_steps=64, max_queue=160)
    orcs = [oracle.StepEnv(0, 0, t, st.STEP) for t in ticks]
    for o in orcs:
        o.set_groups(groups)
    v.reset()
    rng, mine = np.random.default_rng(3), [[] for _ in ticks]
    for s in range(30):
        op = np.zeros((len(ticks), rows), np.uint32)
        cols = {c: np.zeros((len(ticks), rows), np.uint64) for c in ("bid", "vol", "trader", "price", "order_id")}
        for k, t in enumerate(ticks):
            for r in range(rows):
                if rng.random() < 0.7 or not mine[k]:
                    op[k, r] = abi.OP_NEW
                    cols["bid"][k, r], cols["vol"][k, r], cols["trader"][k, r] = rng.random() < 0.5, rng.integers(1, 30), 500 + r
                    cols["price"][k, r] = t * rng.integers(240 // t, 480 // t)
                else:
                    op[k, r] = abi.OP_CANCEL
                    cols["order_id"][k, r] = mine[k][rng.integers(len(mine[k]))]
        obs, ids = v.step(gym.pack_actions(op, **cols))
        obs, ids = obs.numpy(), ids.numpy()
        for k, o in enumerate(orcs):
            o.agents_update(st.SEED, k)
            for r in range(rows):
                if op[k, r] == abi.OP_NEW:
                    oid = o.place_order(bool(cols["bid"][k, r]), int(cols["vol"][k, r]), int(cols["trader"][k, r]), int(cols["price"][k, r]))
                    assert ids[k, r] == oid, (s, k, r)
                    mine[k].append(oid)
                else:
                    o.cancel_order(int(cols["order_id"][k, r]))
            o.step_keyed(st.SEED, k)
            assert np.array_equal(obs[k], o.level_2_data_array()), (s, k)
    v.check_errors()
    for k, o in enumerate(orcs):
        assert v.env.get_trades(k) == o.get_trades() and v.env.get_orders(k) == o.get_orders(), k
        assert np.array_equal(v.env.history(k), o._history()), k
    v.close()


def test_deepw_compact_per_env_ticks(oracle):
    """300 deep books (more than two per SM: k_deepw's compact instantiation) on ticks cycling [1, 2, 3]."""
    n_books, n, window = 300, 600, (256, 800)
    ticks = [1 + k % 3 for k in range(n_books)]
    streams = [workloads.replay_stream(n, 900 + k, tick_size=t, mid_ticks=512 // t, half_width=96 // t, emit_every=32,
                                       trading_windows=False) for k, t in enumerate(ticks)]
    e = core.BatchedEnv(n_books, 0, 0, ticks, 1000, obs_words=abi.OBS_L2, max_orders=n + 64, max_trades=4 * n + 64,
                        max_steps=n // 32 + 8, max_queue=32, price_window=window, deep_chunks=n // 8 + 2 * 544 + 64)
    e.replay(np.concatenate(streams), np.arange(n_books + 1, dtype=np.uint64) * np.uint64(n))
    assert not e.env_errors().any(), e.env_errors()
    n_tr = 0
    for k, t in enumerate(ticks):
        ob = oracle.OrderBook(0, t)
        obs = ob.replay(streams[k], obs_cap=n)
        assert np.array_equal(e.history(k), obs), k
        assert e.get_orders(k) == ob.get_orders() and e.get_trades(k) == ob.get_trades(), k
        n_tr += len(ob.get_trades())
    assert n_tr > 10 * n_books
    e.close()


def test_step_device_continues_after_a_dropped_row(oracle):
    """bb_step_device drops an off-tick NEW row (ERR_PRICE) without consuming an id; the env then runs on exactly as an
    oracle env that never saw the row."""
    ticks, rows, n_steps, bad_step = [1, 2, 3, 4], 4, 24, 8
    v = gym.VectorEnv(len(ticks), rows, 0, 0, ticks, 1000, max_orders=1024, max_trades=2048, max_steps=64)
    v.reset()
    orcs = [oracle.StepEnvNumpy(k, 0, t, 1000) for k, t in enumerate(ticks)]
    rng, n_ord = np.random.default_rng(5), [0] * len(ticks)
    for s in range(n_steps):
        op = np.zeros((len(ticks), rows), np.uint32)
        bid, vol, price, oid = (np.zeros((len(ticks), rows), np.uint32) for _ in range(4))
        for k, t in enumerate(ticks):
            for r in range(rows):
                if rng.random() < 0.7 or not n_ord[k] or (s == bad_step and k == 3):   # (no cancel of the dropped row's id)
                    op[k, r], bid[k, r], vol[k, r] = abi.OP_NEW, rng.random() < 0.5, rng.integers(1, 30)
                    price[k, r] = st.grid_price(rng, t)
                    n_ord[k] += 1
                else:
                    op[k, r], oid[k, r] = abi.OP_CANCEL, rng.integers(n_ord[k])
        want = []
        for k in range(len(ticks)):
            keep = np.ones(rows, bool)
            if s == bad_step and k == 3:   # row 1 of env 3 goes one off its tick: dropped, the next NEW takes its id
                assert op[k, 1] == abi.OP_NEW
                price[k, 1] += 1
                keep[1] = False
                n_ord[k] -= 1
            act = np.where(op[k] == abi.OP_NEW, 1, np.where(op[k] == abi.OP_CANCEL, 2, 0))
            ids = np.full(rows, abi.NO_ID, np.uint64)
            ids[keep] = orcs[k].submit_instructions((act[keep], bid[k][keep].astype(bool), vol[k][keep], np.ones(keep.sum(), np.uint32),
                                                     price[k][keep], oid[k][keep]))
            orcs[k].step()
            want.append(ids)
        obs, ids = v.step(gym.pack_actions(op, bid=bid, vol=vol, price=price, order_id=oid, trader=1))
        obs, ids = obs.numpy(), ids.numpy()
        for k in range(len(ticks)):
            assert np.array_equal(ids[k], want[k]), (s, k)
            assert np.array_equal(obs[k], orcs[k].level_2_data()), (s, k)
    err = v.env.env_errors()
    assert list(err) == [0, 0, 0, ERR_PRICE], err
    for k, o in enumerate(orcs):
        assert np.array_equal(v.env.history(k), o._history()) and v.env.get_trades(k) == o.get_trades(), k
        assert v.env.get_orders(k) == o.get_orders(), k
    v.close()
