"""Per-unit background-agent parameters and Philox keys (bb_set_agent_params_device, VectorEnv / MarketVectorEnv
.set_agent_params), bit for bit against one oracle env or market per unit.  Each oracle unit is built with that unit's own
groups and runs with seed ^ key; a change mid-run is restated with tests/agent_params_oracle.py, which overwrites a group's
parameters in place."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import market_split_oracle as mks
from .agent_params_oracle import market_set_group, sim_set_group
from .test_agent_params_cpu import _noise_groups, _varied
from .test_gpu_market_agents_rows import TICKS, learner_block, mixed_agents, oracle_rows, random_agents

pytestmark = pytest.mark.gpu

STEP = 1_000_000
SEED = 0x1234_5678_9ABC
POPS = {"c3": workloads.c3_groups, "c4": workloads.c4_groups, "noise": _noise_groups}


def _engine_kw(engine, groups):
    if engine == "paged":
        return dict(pages_smem=8, pages_total=64)
    if engine == "fast":
        return dict(pages_smem=32, pages_total=32)
    kw = core.dense_kwargs_for(groups)   # the window of the declared population holds every unit's narrower ranges
    assert kw
    return kw if engine == "dense" else dict(kw, live_cap=254)   # dense_l: the large size class


def _rows(groups, units, seed):
    rng = np.random.default_rng(seed)
    return np.array([_varied(groups, rng) for _ in range(units)], dtype=abi.GROUP_DTYPE)


def _keys(units, seed):
    k = np.random.default_rng(seed).integers(0, 2**63, units, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    k[::3] = 0   # a third of the units keep the launch's seed
    return k


class _Dev:
    """A host array copied into device memory of a BatchedEnv."""

    def __init__(self, env, a):
        a = np.ascontiguousarray(a)
        self.env, self.ptr = env, env.device_alloc(max(a.nbytes, 1))
        env.memcpy(self.ptr, a.ctypes.data, a.nbytes, 1)

    def free(self):
        self.env.device_free(self.ptr)


def _set(env, params=None, keys=None, mask=None):
    bufs = [None if x is None else _Dev(env, x) for x in (params, keys, mask)]
    env.set_agent_params_device(*(0 if b is None else b.ptr for b in bufs))
    env.synchronize()
    for b in bufs:
        if b is not None:
            b.free()


def _oracle_env(oracle, groups):
    o = oracle.StepEnv(0, 0, 1, STEP)
    o.set_groups(list(groups))
    return o


def _assert_env(env, e, o, obs_words=45):
    assert np.array_equal(env.history(e), o._history()[:, :obs_words]), e
    assert env.get_orders(e) == o.get_orders(), e
    assert env.get_trades(e) == o.get_trades(), e


def _batched(n, groups, engine, **kw):
    env = core.BatchedEnv(n, 0, 0, 1, STEP, max_orders=8192, max_trades=16384, max_steps=96, max_queue=256, **_engine_kw(engine, groups), **kw)
    env.set_agents(groups)
    return env


CASES = [(e, p) for e in ("paged", "fast") for p in POPS] + [(e, "c3") for e in ("dense", "dense_l")]


@pytest.mark.parametrize("engine,pop", CASES, ids=[f"{e}-{p}" for e, p in CASES])
def test_run_agents_with_per_env_params_and_keys(oracle, engine, pop):
    groups, n, n_steps = POPS[pop](), 12, 40
    rows, keys = _rows(groups, n, 11), _keys(n, 12)
    env = _batched(n, groups, engine)
    _set(env, rows, keys)
    env.run_agents(n_steps, SEED)
    for e in range(n):
        o = _oracle_env(oracle, rows[e])
        o.run_agents(n_steps, SEED ^ int(keys[e]), env_id=e, keyed=True)
        _assert_env(env, e, o)
    assert not env.env_errors().any()
    assert sum(len(env.get_trades(e)) for e in range(n)) > 0
    env.close()


def _learner_rows(rng, n, rows, mine):
    op = np.zeros((n, rows), np.uint32)
    cols = {k: np.zeros((n, rows), np.uint64) for k in ("bid", "vol", "trader", "price", "order_id", "market")}
    for e in range(n):
        for r in range(rows):
            u = rng.random()
            if u < 0.2:
                continue
            if u < 0.75 or not mine[e]:
                op[e, r] = abi.OP_NEW
                cols["bid"][e, r], cols["vol"][e, r] = rng.random() < 0.5, rng.integers(1, 30)
                cols["trader"][e, r], cols["market"][e, r] = 500 + r, rng.random() < 0.1
                cols["price"][e, r] = 2 * rng.integers(40, 61)
            else:
                op[e, r] = abi.OP_CANCEL
                cols["order_id"][e, r] = mine[e][rng.integers(len(mine[e]))]
    return op, cols


def _oracle_rows(o, op, cols, e, mine):
    want = np.full(op.shape[1], abi.NO_ID, np.uint64)
    for r in range(op.shape[1]):
        if op[e, r] == abi.OP_NEW:
            want[r] = o.place_order(bool(cols["bid"][e, r]), int(cols["vol"][e, r]), int(cols["trader"][e, r]),
                                    None if cols["market"][e, r] else int(cols["price"][e, r]))
            mine[e].append(int(want[r]))
        elif op[e, r] == abi.OP_CANCEL:
            o.cancel_order(int(cols["order_id"][e, r]))
    return want


@pytest.mark.parametrize("engine,pop", [("fast", "c3"), ("fast", "c4"), ("paged", "noise"), ("dense", "c3"), ("dense_l", "c3")])
def test_vector_env_rows_with_per_env_params(oracle, engine, pop):
    """VectorEnv(agents=...) with learner rows: per env, the oracle's agents_update (that env's groups, seed ^ key) + the
    rows + keyed step."""
    groups, n, rows_per, n_steps, seed = POPS[pop](), 16, 4, 20, 77
    kw = _engine_kw(engine, groups)
    if engine == "dense":   # the learner's resting orders need slots beyond the agents' (the small class holds 128)
        kw["live_cap"], rows_per = 128, 2
    v = gym.VectorEnv(n, rows_per, 0, 0, 1, STEP, agents=groups, agent_seed=seed, max_orders=8192, max_trades=8192,
                      max_steps=64, max_queue=200, **kw)
    p = v.agent_params()
    assert p.shape == (n, len(groups)) and p.dtype == abi.GROUP_DTYPE
    p[:] = _rows(groups, n, 21)
    keys = _keys(n, 22)
    v.reset()
    v.set_agent_params(p, keys=keys)
    orcs = [_oracle_env(oracle, p[e]) for e in range(n)]
    mine = [[] for _ in range(n)]
    rng = np.random.default_rng(5)
    for s in range(n_steps):
        op, cols = _learner_rows(rng, n, rows_per, mine)
        obs, ids = v.step(gym.pack_actions(op, **cols))
        obs, ids = obs.numpy(), ids.numpy()
        for e, o in enumerate(orcs):
            o.agents_update(seed ^ int(keys[e]), e)
            want = _oracle_rows(o, op, cols, e, mine)
            o.step_keyed(seed ^ int(keys[e]), e)
            assert np.array_equal(ids[e], want), (s, e)
            assert np.array_equal(obs[e], o.level_2_data_array()), (s, e)
    v.check_errors()
    for e in range(0, n, 3):
        _assert_env(v.env, e, orcs[e])
    v.close()


@pytest.mark.parametrize("engine,pop", [("fast", "c4"), ("paged", "noise"), ("dense", "c3")])
def test_masked_change_mid_run(oracle, engine, pop):
    """After k steps a subset of envs takes new parameters and keys: those match the oracle with sim_set_group at step k;
    the others are bit-identical to a twin handle that never made the call."""
    groups, n, k, m = POPS[pop](), 12, 15, 25
    env, twin = _batched(n, groups, engine), _batched(n, groups, engine)
    env.run_agents(k, SEED)
    twin.run_agents(k, SEED)
    rows, keys = _rows(groups, n, 31), _keys(n, 32)
    mask = (np.arange(n) % 3 == 1).astype(np.uint8)
    _set(env, rows, keys, mask)
    env.run_agents(m, SEED)
    twin.run_agents(m, SEED)
    for e in range(n):
        if mask[e]:
            o = _oracle_env(oracle, groups)
            o.run_agents(k, SEED, env_id=e, keyed=True)
            for gi in range(len(groups)):
                sim_set_group(o, gi, rows[e][gi])
            o.run_agents(m, SEED ^ int(keys[e]), env_id=e, keyed=True)
            _assert_env(env, e, o)
        else:
            assert np.array_equal(env.history(e), twin.history(e)) and env.get_orders(e) == twin.get_orders(e), e
            assert env.get_trades(e) == twin.get_trades(e), e
    env.close()
    twin.close()


@pytest.mark.parametrize("engine,pop", [("fast", "c4"), ("paged", "c3"), ("dense", "c3"), ("fast", "noise")])
def test_declared_rows_and_zero_keys_equal_the_shared_path(engine, pop):
    """Rows equal to the declared groups and zero keys: the per-unit variants compute exactly what the shared ones do."""
    groups, n = POPS[pop](), 10
    env, twin = _batched(n, groups, engine), _batched(n, groups, engine)
    _set(env, np.array([groups] * n, dtype=abi.GROUP_DTYPE), np.zeros(n, np.uint64))
    for h in (env, twin):
        h.run_agents(30, SEED)
    for e in range(n):
        assert np.array_equal(env.history(e), twin.history(e)) and env.get_orders(e) == twin.get_orders(e), e
        assert env.get_trades(e) == twin.get_trades(e), e
    env.close()
    twin.close()


def test_keys_make_reproducible_distinct_episodes_and_survive_resets(oracle):
    """reset(mask, seeds) + keys: an episode replays under its key and differs under another; reset(), reset(mask) and
    restore keep parameters and keys; set_agents drops them."""
    groups, n, steps = workloads.c4_groups(), 6, 12
    noop = np.zeros((n, 1), dtype=gym.ACTION_DTYPE)
    v = gym.VectorEnv(n, 1, 100, 0, 1, STEP, agents=groups, agent_seed=SEED, max_orders=8192, max_trades=8192, max_steps=256,
                      max_queue=200)
    p = v.agent_params()
    p[:] = _rows(groups, n, 41)
    keys = np.array([5, 6, 5, 0, 9, 11], np.uint64)
    v.reset()
    v.set_agent_params(p, keys=keys)

    def episode(unit):
        for _ in range(steps):
            v.step(noop)
        return v.env.history(unit)[-steps:].copy()

    first = episode(0)
    one = np.zeros(n, np.uint8)
    one[0] = 1
    creation = np.array([100 + u for u in range(n)], np.uint64)
    v.reset(one, creation)
    assert np.array_equal(episode(0), first)                        # same seed, same key: the same episode
    v.set_agent_params(keys=np.full(n, 77, np.uint64), mask=one)
    v.reset(one, creation)
    other = episode(0)
    assert not np.array_equal(other, first)                          # another key: another episode
    v.set_agent_params(keys=keys, mask=one)
    v.reset(one, creation)
    assert np.array_equal(episode(0), first)                         # its key again: the first episode again
    # the oracle's keyed run with seed ^ key (no rows), from a seeded reset
    o = _oracle_env(oracle, p[0])
    o.run_agents(steps, SEED ^ 5, env_id=0, keyed=True)
    assert np.array_equal(first[:, :45], o._history()[-steps:])
    # reset() and restore keep parameters and keys: a full reset replays every unit's first episode
    v.reset()
    base = [None] * n
    for _ in range(steps):
        v.step(noop)
    base = [v.env.history(u)[-steps:].copy() for u in range(n)]
    store = v.snapshots(n)
    v.reset()
    v.save(store)
    for _ in range(steps):
        v.step(noop)
    assert all(np.array_equal(v.env.history(u)[-steps:], base[u]) for u in range(n))
    v.restore(store, np.arange(n, dtype=np.uint32))
    for _ in range(steps):
        v.step(noop)
    assert all(np.array_equal(v.env.history(u)[-steps:], base[u]) for u in range(n))
    v.check_errors()
    # set_agents drops both tables: results equal a fresh handle's
    v.env.set_agents(groups)
    v.reset()
    fresh = gym.VectorEnv(n, 1, 100, 0, 1, STEP, agents=groups, agent_seed=SEED, max_orders=8192, max_trades=8192, max_steps=256,
                          max_queue=200)
    fresh.reset()
    for _ in range(steps):
        v.step(noop)
        fresh.step(noop)
    for u in range(n):
        assert np.array_equal(v.env.history(u)[-steps:], fresh.env.history(u)[-steps:]), u
    v.close()
    fresh.close()


MARKET_CASES = [("fast", 2, "random"), ("fast", 4, "mixed"), ("dense", 3, "random"), ("dense", 4, "random"), ("paged", 3, "mixed")]


def _market_rows(agents, n_markets, seed):
    rng = np.random.default_rng(seed)
    return np.array([_varied([a.group for a in agents], rng) for _ in range(n_markets)], dtype=abi.GROUP_DTYPE)


@pytest.mark.parametrize("engine,A,pop", MARKET_CASES, ids=[f"{e}-{A}-{p}" for e, A, p in MARKET_CASES])
def test_market_vector_env_per_market_params(oracle, engine, A, pop):
    ticks, n_markets, rows_per, n_steps, seed = TICKS[A], 8, 6, 20, 0xB0A5
    agents = random_agents(A) if pop == "random" else mixed_agents(A)
    kw = dict(price_window=(0, 256), live_cap=254) if engine == "dense" else _engine_kw(engine, [])
    v = gym.MarketVectorEnv(n_markets, rows_per, 0, 0, ticks, 1000, agents=agents, agent_seed=seed, max_orders=8192,
                            max_trades=16384, max_steps=64, max_queue=128, **kw)
    p = v.agent_params()
    p[:] = _market_rows(agents, n_markets, 51)
    keys = _keys(n_markets, 52)
    v.reset()
    v.set_agent_params(p, keys=keys)
    orcs = []
    for mk in range(n_markets):
        o = oracle.MarketEnv(0, 0, ticks, 1000)
        o.set_groups(list(p[mk]), [a.asset for a in agents])
        orcs.append(o)
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    rng = np.random.default_rng(A + len(engine))
    for s in range(n_steps):
        blk = np.stack([learner_block(rng, ticks, mine[mk], rows_per) for mk in range(n_markets)])
        obs, ids = v.step(blk)
        obs, ids = obs.numpy(), ids.numpy()
        for mk, o in enumerate(orcs):
            mks.agents_update(o, seed ^ int(keys[mk]), mk)
            want = oracle_rows(o, blk[mk], mine[mk])
            mks.step_keyed(o, seed ^ int(keys[mk]), mk)
            assert list(ids[mk]) == want, (s, mk)
            for a in range(A):
                assert np.array_equal(obs[mk, a], o.history(a)[-1]), (s, mk, a)
    v.check_errors()
    # a masked change of two markets' groups mid-run, then plain agent launches
    rows2 = _market_rows(agents, n_markets, 53)
    mask = np.zeros(n_markets, np.uint8)
    mask[[1, n_markets - 1]] = 1
    v.set_agent_params(rows2, mask=mask)
    v.env.run_agents(5, seed)
    for mk in (0, 1, n_markets - 1):
        o = orcs[mk]
        if mask[mk]:
            for gi in range(len(agents)):
                market_set_group(o, gi, rows2[mk][gi])
        o.run_agents(5, seed ^ int(keys[mk]), market_id=mk, keyed=True)
        for a in range(A):
            b = mk * A + a
            assert np.array_equal(v.env.history(b), o.history(a)), (mk, a)
            assert v.env.get_orders(b) == o.get_orders(a) and v.env.get_trades(b) == o.get_trades(a), (mk, a)
    assert not v.env.env_errors().any()
    v.close()


def _bad_records(groups):
    """(group index, record) pairs, one per way a record can leave the declared population."""
    out = []

    def bad(gi, **f):
        r = groups[gi].copy()
        for k, x in f.items():
            r[k] = x
        out.append((gi, r))
    ri = next(i for i, g in enumerate(groups) if int(g["kind"]) == abi.GROUP_RANDOM)
    mi = next(i for i, g in enumerate(groups) if int(g["kind"]) != abi.GROUP_RANDOM)
    g, m = groups[ri], groups[mi]
    bad(ri, kind=abi.GROUP_NOISE)
    bad(ri, n_agents=int(g["n_agents"]) - 1)
    bad(ri, tick_size=int(g["tick_size"]) + 1)
    bad(ri, tick_lo=int(g["tick_lo"]) - 1)
    bad(ri, tick_hi=int(g["tick_hi"]) + 1)
    bad(ri, tick_lo=int(g["tick_lo"]) + 3, tick_hi=int(g["tick_lo"]) + 3)   # empty range
    bad(ri, vol_lo=int(g["vol_lo"]) - 1)
    bad(ri, vol_hi=int(g["vol_hi"]) + 1)
    bad(ri, vol_lo=int(g["vol_lo"]) + 2, vol_hi=int(g["vol_lo"]) + 2)
    bad(mi, kind=abi.GROUP_RANDOM)
    bad(mi, n_agents=int(m["n_agents"]) + 1)
    bad(mi, tick_size=int(m["tick_size"]) + 1)
    bad(mi, tick_lo=int(m["tick_lo"]) + 1)   # agent_id_start
    bad(mi, vol_hi=int(m["vol_hi"]) + 2)     # live-list capacity
    return out


def test_invalid_rows_flag_their_unit_and_change_nothing(oracle):
    groups = workloads.c4_groups()
    bads = _bad_records(groups)
    n = 2 * len(bads)
    env = _batched(n, groups, "fast")
    first, first_keys = _rows(groups, n, 61), _keys(n, 62) | np.uint64(1)
    _set(env, first, first_keys)
    env.run_agents(10, SEED)
    rows, keys = _rows(groups, n, 63), _keys(n, 64) | np.uint64(2)
    for j, (gi, r) in enumerate(bads):   # even units: one invalid record each; odd units: valid rows
        rows[2 * j][gi] = r
    _set(env, rows, keys)
    err = env.env_errors()
    assert list(np.flatnonzero(err)) == list(range(0, n, 2))
    assert all(int(x) == abi.ERR_PARAMS for x in err[::2])
    env.run_agents(10, SEED)
    for e in range(n):
        o = _oracle_env(oracle, first[e])
        o.run_agents(10, SEED ^ int(first_keys[e]), env_id=e, keyed=True)
        if e % 2:
            for gi in range(len(groups)):
                sim_set_group(o, gi, rows[e][gi])
            o.run_agents(10, SEED ^ int(keys[e]), env_id=e, keyed=True)
        else:   # the refused unit keeps its parameters and key
            o.run_agents(10, SEED ^ int(first_keys[e]), env_id=e, keyed=True)
        _assert_env(env, e, o)
    env.close()


def test_invalid_market_row_flags_every_book_of_the_market():
    A, n_markets = 3, 4
    agents = random_agents(A)
    v = gym.MarketVectorEnv(n_markets, 2, 0, 0, TICKS[A], 1000, agents=agents, max_orders=4096, max_trades=4096, max_steps=16,
                            max_queue=128)
    p = v.agent_params()
    p["tick_hi"][2, 1] += 1
    v.set_agent_params(p)
    err = v.env.env_errors().reshape(n_markets, A)
    assert (err[2] == abi.ERR_PARAMS).all() and not np.delete(err, 2, axis=0).any()
    with pytest.raises(RuntimeError, match="0x2000"):
        v.check_errors()
    v.close()


def test_refusals():
    groups = workloads.c3_groups()
    plain = core.BatchedEnv(4, 0, 0, 1, STEP, max_orders=256, max_trades=256, max_steps=8, max_queue=64)
    d = _Dev(plain, np.zeros(4, np.uint64))
    with pytest.raises(ValueError, match="has not been called"):   # no population
        plain.set_agent_params_device(0, d.ptr, 0)
    plain.set_agents(groups)
    with pytest.raises(ValueError, match="both NULL"):
        plain.set_agent_params_device(0, 0, d.ptr)
    d.free()
    plain.close()
    deep = core.BatchedEnv(1, 0, 0, 1, 1000, obs_words=abi.OBS_L2, max_orders=1024, max_trades=1024, max_steps=8, max_queue=32,
                           price_window=(2816, 3200), deep_chunks=2048)
    d = _Dev(deep, np.zeros(1, np.uint64))
    with pytest.raises(ValueError, match="has not been called"):
        deep.set_agent_params_device(0, d.ptr, 0)
    d.free()
    deep.close()
    v = gym.VectorEnv(4, 1, 0, 0, 1, STEP, max_orders=64, max_trades=64, max_steps=8)
    with pytest.raises(ValueError, match="no background agents"):
        v.set_agent_params(keys=np.zeros(4, np.uint64))
    v.close()


def test_torch_device_inputs_zero_copy(oracle):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("torch sees no GPU")
    groups, n, steps = workloads.c3_groups(), 8, 15
    v = gym.VectorEnv(n, 1, 0, 0, 1, STEP, agents=groups, agent_seed=SEED, max_orders=4096, max_trades=4096, max_steps=64,
                      max_queue=220)
    p = v.agent_params()
    p[:] = _rows(groups, n, 71)
    # domain randomisation drawn on the device: per-env activity rates written into the record bytes
    rates = torch.rand(n, device="cuda") * 0.8 + 0.1
    params = torch.from_numpy(p.view(np.uint8).reshape(n, -1).copy()).cuda()
    rate_off = abi.GROUP_DTYPE.fields["rate"][1]
    params.view(n, len(groups), 80)[:, 0, rate_off:rate_off + 4] = rates.view(torch.uint8).view(n, 4)
    keys = torch.arange(1, n + 1, device="cuda", dtype=torch.int64) * 1000003
    mask = torch.ones(n, device="cuda", dtype=torch.bool)
    v.reset()
    v.set_agent_params(params, keys=keys, mask=mask)
    torch.cuda.synchronize()
    p["rate"][:, 0] = rates.cpu().numpy()
    noop = torch.zeros(n, 32, dtype=torch.uint8, device="cuda")
    for _ in range(steps):
        v.step(noop)
    v.check_errors()
    for e in range(n):
        o = _oracle_env(oracle, p[e])
        o.run_agents(steps, SEED ^ (1000003 * (e + 1)), env_id=e, keyed=True)
        _assert_env(v.env, e, o)
    v.close()
