"""GPU suite: background agents on the deep-book engine (bb_run_agents / bb_run_agents_with_rows on a deep handle:
k_env_agents_stage + k_deepw<.., ENV>, and gym.VectorEnv(agents=..., deep_chunks=...)).  Every env is compared bit for bit
with an oracle StepEnv run with the same groups: run_agents(..., keyed=True), or agents_update + place_order / cancel_order
+ step_keyed where the env also takes rows.  Deep books are preloaded by replaying a C5 stream into the device book and,
through the oracle's book replay, into the oracle env's book."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import episode_reset_oracle as ers
from .test_gpu_deep_env import closed, oracle_replay

pytestmark = pytest.mark.gpu

MID = 10_000
WINDOW = (9728, 10368)   # 640 levels around the C5 mid
STEP = 1000
ERR_CAP_PAGES, ERR_CAP_QUEUE, ERR_GRANULE, ERR_TIME_ORDER, ERR_ROW_OP = 0x4, 0x8, 0x20, 0x100, 0x400
ASEED = 101
SAME_SLICE = 0xFFFFFFFF


def deep_env(n_envs, seed=0, tick=1, n_orders=1 << 14, max_steps=256, max_queue=256, step_size=STEP, window=WINDOW, **kw):
    return core.BatchedEnv(n_envs, seed, 0, tick, step_size, max_orders=n_orders, max_trades=4 * n_orders, max_steps=max_steps,
                           max_queue=max_queue, price_window=window, deep_chunks=n_orders // 8 + 2 * (window[1] - window[0]) + 64,
                           **kw)


def background(noise=True, momentum=True):
    """C3 re-centred on the C5 mid, plus a Noise group and a Momentum group quoting around the book's mid."""
    g = workloads.c3_groups_around(MID)
    if noise:
        g.append(core.noise_group(100, 10, 1, 0.5, 0.05, 0.1, 5, 1.5, 0.6))
    if momentum:
        g.append(core.momentum_group(200, 20, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0))
    return g


def c5_preload(n_resting, seed, depth=256):
    return closed(workloads.c5_stream(n_resting, 1, 200, seed=seed, mid_ticks=MID, depth_ticks=depth))


def assert_same(env, o, e, skip=0):
    """Order table, trade log and history equal the oracle's; `skip`: oracle records before the env's first (a restored
    book's history starts empty)."""
    assert env.get_orders(e) == o.get_orders(), e
    assert env.get_trades(e) == o.get_trades(), e
    assert np.array_equal(env.history(e), o._history()[skip:]), e


def random_rows(rng, n_envs, rows, orcs):
    """NEW (limit around the mid, some market), CANCEL of any id issued so far (the agents' included) or of an id this slice
    creates, and no-op rows."""
    a = np.zeros((n_envs, rows), dtype=gym.ACTION_DTYPE)
    for e in range(n_envs):
        issued, made = len(orcs[e].get_orders()), 0
        for r in range(rows):
            u = rng.random()
            if u < 0.15:
                continue
            x = a[e, r]
            if u < 0.65 or issued == 0:
                bid = rng.random() < 0.5
                mkt = rng.random() < 0.1
                x["op_flags"] = abi.OP_NEW | (abi.F_BID if bid else 0) | (abi.F_MARKET if mkt else 0)
                x["price"] = 0 if mkt else MID + int(rng.integers(-20, 21))
                x["vol"], x["trader"] = int(rng.integers(1, 40)), 600 + r
                made += 1
            else:
                x["op_flags"] = abi.OP_CANCEL
                if made and rng.random() < 0.3:   # an id this slice creates: resolved in step_and_check, after the agents' ids
                    x["order_id"] = SAME_SLICE
                else:
                    x["order_id"] = int(rng.integers(0, issued))
    return a


@pytest.mark.parametrize("n_envs", [4, 300], ids=["roomy", "compact"])
def test_run_agents_on_fresh_books(oracle, n_envs):
    """C3 re-centred on the window on fresh deep books: two launches split unevenly, then run_agents_to_host; histories,
    order tables, trade logs and error bits equal the oracle's keyed runs."""
    groups = workloads.c3_groups_around(MID)
    env = deep_env(n_envs, seed=5)
    env.set_agents(groups)
    env.run_agents(11, ASEED)
    env.run_agents(19, ASEED)
    out = env.run_agents_to_host(9, ASEED)
    check = range(n_envs) if n_envs < 10 else range(0, n_envs, 23)
    for e in check:
        o = oracle.StepEnv(5 + e, 0, 1, STEP)
        o.set_groups(groups)
        o.run_agents(39, ASEED, env_id=e, keyed=True)
        assert_same(env, o, e)
        assert np.array_equal(out[e], o._history()[30:]), e
    assert not env.env_errors().any()
    assert min(len(env.get_trades(e)) for e in check) > 50
    env.close()


def test_cross_engine_parity():
    """The same population, seed and steps on the deep engine and on the FAST engine: identical histories, order tables and
    trade logs.  An odd max_queue (what VectorEnv picks for an odd number of rows) on both: the shuffle's draw array stays
    aligned."""
    groups = workloads.c3_groups_around(MID)
    n_envs = 8
    deep = deep_env(n_envs, seed=3, max_queue=201)
    fast = core.BatchedEnv(n_envs, 3, 0, 1, STEP, max_orders=1 << 14, max_trades=1 << 16, max_steps=256, max_queue=201)
    for env in (deep, fast):
        env.set_agents(groups)
        env.run_agents(17, ASEED)
        env.run_agents(8, ASEED)
    for e in range(n_envs):
        assert deep.get_orders(e) == fast.get_orders(e), e
        assert deep.get_trades(e) == fast.get_trades(e), e
        assert np.array_equal(deep.history(e), fast.history(e)), e
    assert not deep.env_errors().any() and not fast.env_errors().any()
    deep.close(), fast.close()


def step_and_check(v, orcs, rng, n_steps, seed, keys=None, reads=False, seen=None):
    """Random rows on every env for n_steps; ids and observations per step equal each env's oracle."""
    n_envs, rows = v.n_envs, v.rows
    for s in range(n_steps):
        a = random_rows(rng, n_envs, rows, orcs)
        want = []
        for e in range(n_envs):   # the oracle first: same-slice cancels name the id of the slice's latest NEW before them
            # (or of its first NEW, created later), which follows the ids the agents' update took
            o, k = orcs[e], seed ^ (0 if keys is None else int(keys[e]))
            o.agents_update(k, e)
            base = len(o.get_orders())
            news = 0
            for r in range(rows):
                x = a[e, r]
                of = int(x["op_flags"])
                if of & 0xFF == abi.OP_NEW:
                    news += 1
                elif of & 0xFF == abi.OP_CANCEL and int(x["order_id"]) == SAME_SLICE:
                    x["order_id"] = base + max(news - 1, 0)
            ids = np.full(rows, abi.NO_ID, np.uint64)
            for r in range(rows):
                x = a[e, r]
                of = int(x["op_flags"])
                if of & 0xFF == abi.OP_NEW:
                    ids[r] = o.place_order(bool(of & abi.F_BID), int(x["vol"]), int(x["trader"]), None if of & abi.F_MARKET else int(x["price"]))
                elif of & 0xFF == abi.OP_CANCEL:
                    o.cancel_order(int(x["order_id"]))
            o.step_keyed(k, e)
            want.append(ids)
        obs, ids = v.step(a)
        if reads:
            got = v.orders(ids)
            tcols, count = v.trades(4096)
            st, vol, pr = (got[c].numpy() for c in ("status", "vol", "price"))
            tc = {c: x.numpy() for c, x in tcols.items()}
            cnt = count.numpy()
        obs, ids = obs.numpy(), ids.numpy()
        for e in range(n_envs):
            assert np.array_equal(ids[e], want[e]), (s, e)
            assert np.array_equal(obs[e], orcs[e].level_2_data_array()), (s, e)
            if reads:
                table = orcs[e].get_orders()
                for r in range(rows):
                    if want[e][r] != abi.NO_ID:
                        o = table[int(want[e][r])]
                        assert (st[e, r], vol[e, r], pr[e, r]) == (o[1], o[4], o[6]), (s, e, r)
                n = int(cnt[e])
                assert n <= 4096
                seen[e] += [(int(tc["t"][e, i]), bool(tc["side_is_bid"][e, i]), int(tc["price"][e, i]), int(tc["vol"][e, i]),
                             int(tc["active_id"][e, i]), int(tc["passive_id"][e, i])) for i in range(n)]
                assert seen[e] == orcs[e].get_trades(), (s, e)


def preloaded_vector(n_envs, rows, seed, groups, n_rest=3000, **kw):
    v = gym.VectorEnv(n_envs, rows, seed, 0, 1, STEP, agents=groups, agent_seed=ASEED, max_orders=1 << 14, max_trades=1 << 16,
                      max_steps=256, price_window=WINDOW, deep_chunks=(1 << 14) // 8 + 2 * (WINDOW[1] - WINDOW[0]) + 64, **kw)
    v.reset()
    orcs = [oracle_env(seed + e, groups) for e in range(n_envs)]
    streams = [c5_preload(n_rest, 40 + e) for e in range(n_envs)]
    v.env.replay(np.concatenate(streams), np.cumsum([0] + [len(s) for s in streams]).astype(np.uint64))
    for o, s in zip(orcs, streams):
        oracle_replay(o, s)
    return v, orcs


def oracle_env(seed, groups):
    from oracle import oracle as orc   # (the `oracle` fixture has built it)
    o = orc.StepEnv(seed, 0, 1, STEP)
    o.set_groups(groups)
    return o


def test_vector_env_on_c5_books(oracle):
    """VectorEnv(agents=..., deep_chunks=...) on C5-preloaded books: RandomAgents, Noise and Momentum groups, and random NEW /
    CANCEL / no-op rows (cancels of the agents' ids and of ids the same slice creates); ids and observations at every step,
    the orders() / trades() reads, and the whole books at the end."""
    groups = background()
    v, orcs = preloaded_vector(4, 8, 21, groups)
    seen = [[] for _ in range(4)]
    step_and_check(v, orcs, np.random.default_rng(3), 16, ASEED, reads=True, seen=seen)
    for e in range(4):
        assert_same(v.env, orcs[e], e)
    v.check_errors()
    assert min(len(o.get_trades()) for o in orcs) > 100
    # the learner's orders (trader ids 600..) traded with the agents' (RandomAgents < 100, Noise 100.., Momentum 200..)
    table = orcs[0].get_orders()
    kinds = {(table[t[4]][7] >= 600, table[t[5]][7] >= 600) for t in orcs[0].get_trades()[200:]}
    assert (True, False) in kinds or (False, True) in kinds
    v.close()


def test_reset_with_and_without_seeds(oracle):
    """reset(mask, seeds) with the envs' creation seeds makes them equal to fresh envs (held agent orders and Momentum / Noise
    state are reset with the book); an unseeded reset continues the agents' step counter."""
    groups = background(momentum=False) + [core.momentum_group(200, 20, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0)]
    n_envs, rows, seed = 6, 4, 9
    v, orcs = preloaded_vector(n_envs, rows, seed, groups, n_rest=1500)
    rng = np.random.default_rng(11)
    step_and_check(v, orcs, rng, 6, ASEED)
    # seeded: the creation seeds; books go empty, so preload them again (device and oracle) before stepping
    mask = np.array([1, 0, 1, 0, 0, 1], bool)
    v.reset(mask, np.arange(seed, seed + n_envs, dtype=np.uint64))
    streams = []
    for e in range(n_envs):
        if mask[e]:
            ers.sim_reset(orcs[e], 0, seed=seed + e)
            streams.append(c5_preload(1500, 40 + e))
            oracle_replay(orcs[e], streams[-1])
        else:
            streams.append(np.zeros(0, dtype=abi.INSTR_DTYPE))
    v.env.replay(np.concatenate(streams), np.cumsum([0] + [len(s) for s in streams]).astype(np.uint64))
    step_and_check(v, orcs, rng, 6, ASEED)
    # unseeded: the step counter continues (other agent draws than a fresh env's)
    mask2 = np.array([0, 1, 0, 0, 1, 0], bool)
    v.reset(mask2)
    for e in np.flatnonzero(mask2):
        ers.sim_reset(orcs[e], 0)
    streams = [c5_preload(1500, 70 + e) if mask2[e] else np.zeros(0, dtype=abi.INSTR_DTYPE) for e in range(n_envs)]
    v.env.replay(np.concatenate(streams), np.cumsum([0] + [len(s) for s in streams]).astype(np.uint64))
    for e in np.flatnonzero(mask2):
        oracle_replay(orcs[e], streams[e])
    step_and_check(v, orcs, rng, 6, ASEED)
    for e in range(n_envs):
        assert_same(v.env, orcs[e], e)
    v.check_errors()
    v.close()


def test_restore_warmed_book_and_agent_keys(oracle):
    """A C5 book warmed up by agent steps in env 0, saved and restored into every env: each continues as its oracle (the
    slot's agent state and step counter, its own env id); then per-env agent keys match the oracle run with seed ^ key."""
    groups = background()
    n_envs, rows, seed = 12, 4, 2
    v = gym.VectorEnv(n_envs, rows, seed, 0, 1, STEP, agents=groups, agent_seed=ASEED, max_orders=1 << 14, max_trades=1 << 16,
                      max_steps=256, price_window=WINDOW, deep_chunks=(1 << 14) // 8 + 2 * (WINDOW[1] - WINDOW[0]) + 64)
    v.reset()
    stream = c5_preload(3000, 77)
    v.env.replay(np.concatenate([stream] * n_envs), np.arange(n_envs + 1, dtype=np.uint64) * np.uint64(len(stream)))
    v.env.run_agents(7, ASEED)   # (env 0 is the one saved)
    store = v.snapshots(1)
    v.save(store, np.array([0], np.uint32))
    v.restore(store, np.zeros(n_envs, np.uint32))
    orcs = []
    for e in range(n_envs):
        o = oracle_env(seed, groups)
        oracle_replay(o, stream)
        o.run_agents(7, ASEED, env_id=0, keyed=True)
        orcs.append(o)
    step_and_check(v, orcs, np.random.default_rng(4), 6, ASEED)
    for e in range(n_envs):
        assert_same(v.env, orcs[e], e, skip=7)
    keys = np.arange(1, n_envs + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    v.set_agent_params(keys=keys)
    step_and_check(v, orcs, np.random.default_rng(5), 6, ASEED, keys=keys)
    for e in range(n_envs):
        assert_same(v.env, orcs[e], e, skip=7)
    v.check_errors()
    v.close()


def test_refusals_and_flags(oracle):
    # an out-of-window RandomAgents range is refused; the previous population stays
    groups = workloads.c3_groups_around(MID)
    env = deep_env(2, seed=1)
    env.set_agents(groups)
    with pytest.raises(ValueError, match="deep-book engine"):
        env.set_agents(workloads.c3_groups())
    with pytest.raises(ValueError, match="deep-book engine"):
        env.set_agents(workloads.c3_groups_around(WINDOW[1] - 60))
    env.run_agents(5, ASEED)
    for e in range(2):
        o = oracle_env(1 + e, groups)
        o.run_agents(5, ASEED, env_id=e, keyed=True)
        assert_same(env, o, e)
    # max_steps exhausted, stream capture
    small = deep_env(2, max_steps=8)
    small.set_agents(groups)
    small.run_agents(8, ASEED)
    with pytest.raises(MemoryError, match="max_steps"):
        small.run_agents(1, ASEED)
    small.close()
    import torch
    st = torch.cuda.Stream()
    env.set_stream(st.cuda_stream)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(ValueError, match="cannot be captured"):
        with torch.cuda.graph(g, stream=st):
            env.run_agents(1, ASEED, sync=False)
    env.close()


def test_modify_rows_and_time_order():
    """A MODIFY row is dropped with BB_ERR_ROW_OP; step_size < max_queue flags BB_ERR_TIME_ORDER."""
    v = gym.VectorEnv(2, 2, 0, 0, 1, STEP, agents=workloads.c3_groups_around(MID), agent_seed=1, max_orders=4096, max_trades=4096,
                      max_steps=8, price_window=WINDOW, deep_chunks=4096)
    v.reset()
    v.step(gym.pack_actions(np.array([[abi.OP_MODIFY, abi.OP_NOOP], [abi.OP_NOOP, abi.OP_NOOP]], np.uint32), order_id=0, price=MID, vol=1))
    err = v.env.env_errors()
    assert err[0] == ERR_ROW_OP and err[1] == 0, [hex(x) for x in err]
    v.close()
    env = deep_env(3, step_size=4)
    env.set_agents(workloads.c3_groups_around(MID))
    env.run_agents(12, ASEED)
    assert all(x & ERR_TIME_ORDER for x in env.env_errors()), [hex(x) for x in env.env_errors()]
    env.close()


def test_noise_leaving_a_narrow_window(oracle):
    """A Noise group with a wide price distribution on a window of 128 levels: the envs whose oracle places a limit order
    outside the window are flagged BB_ERR_CAP_PAGES; every other env stays exact."""
    window = (MID - 64, MID + 64)
    groups = [core.noise_group(100, 10, 1, 0.5, 0.02, 0.1, 5, 1.5, 1.0)]
    n_envs, n_steps = 16, 30
    env = deep_env(n_envs, seed=7, window=window)
    env.set_agents(groups)
    streams = [closed(workloads.c5_stream(400, 1, 50, seed=90 + e, mid_ticks=MID, depth_ticks=40)) for e in range(n_envs)]
    env.replay(np.concatenate(streams), np.cumsum([0] + [len(s) for s in streams]).astype(np.uint64))
    env.run_agents(n_steps, ASEED)
    err = env.env_errors()
    left = []
    for e in range(n_envs):
        o = oracle_env(7 + e, groups)
        oracle_replay(o, streams[e])
        o.run_agents(n_steps, ASEED, env_id=e, keyed=True)
        out = any(not window[0] <= x[6] < window[1] for x in o.get_orders() if x[6] not in (0, 0xFFFFFFFF))
        left.append(out)
        if out:
            assert err[e] & ERR_CAP_PAGES, e
        else:
            assert err[e] == 0, (e, hex(err[e]))
            assert_same(env, o, e)
    assert any(left) and not all(left), left
    env.close()


def test_off_tick_random_agents(oracle):
    """Per-env ticks 1, 2 and 4 under a RandomAgents group of tick size 2: the tick-4 envs are flagged ERR_GRANULE at the
    step the oracle raises; the others stay exact."""
    groups = workloads.c3_groups_around(MID)
    ticks = [1, 2, 4, 4]
    env = deep_env(4, seed=3, tick=ticks)
    env.set_agents(groups)
    env.run_agents(10, ASEED)
    err = env.env_errors()
    for e, t in enumerate(ticks):
        o = oracle.StepEnv(3 + e, 0, t, STEP)
        o.set_groups(groups)
        raised = False
        try:
            o.run_agents(10, ASEED, env_id=e, keyed=True)
        except ValueError:
            raised = True
        assert raised == (t == 4), e
        if raised:
            assert err[e] & ERR_GRANULE, (e, hex(err[e]))
        else:
            assert err[e] == 0, (e, hex(err[e]))
            assert_same(env, o, e)
    env.close()
