"""GPU suite for the per-env reset of the device-resident loops (bb_reset_device, VectorEnv / MarketVectorEnv.reset(mask,
seeds)): the units a mask selects return to a fresh book, with their random streams continued (no seeds) or re-seeded, and
every other unit is untouched.  Everything is checked against the oracle's envs reset the same way
(tests/episode_reset_oracle.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from bourse_b200 import abi, core, gym, market, workloads

from . import episode_reset_oracle as ers
from . import market_split_oracle as mks
from .test_gpu_gym import _oracle_step, _random_actions
from .test_gpu_market_agents_rows import TICKS as AGENT_TICKS
from .test_gpu_market_agents_rows import learner_block, mixed_agents, oracle_market, random_agents
from .test_gpu_market_agents_rows import oracle_rows as agent_rows
from .test_gpu_market_device import TICKS, _host_submit, assert_books_equal, oracle_rows, random_block

pytestmark = pytest.mark.gpu

ENGINES = {
    "paged": dict(pages_smem=8, pages_total=64),
    "fast": dict(pages_smem=32, pages_total=32),
    "dense": dict(price_window=(0, 256), live_cap=254),
}


class DLPackOnly:   # a producer without __cuda_array_interface__
    def __init__(self, t): self.t = t
    def __dlpack__(self, stream=None): return self.t.__dlpack__()
    def __dlpack_device__(self): return self.t.__dlpack_device__()


def _mask_as(kind, mask):
    """The same boolean mask as a numpy bool / uint8 array, a torch bool / uint8 tensor or a DLPack-only bool tensor."""
    import torch
    if kind == "np_bool":
        return mask
    if kind == "np_u8":
        return mask.astype(np.uint8)
    t = torch.from_numpy(mask).cuda()
    if kind == "torch_u8":
        t = t.to(torch.uint8)
    torch.cuda.synchronize()
    return DLPackOnly(t) if kind == "dlpack_bool" else t


def _seeds_as(seeds, on_device):
    import torch
    if not on_device:
        return seeds
    t = torch.from_numpy(seeds.view(np.int64)).cuda()
    torch.cuda.synchronize()
    return t


def _random_reset(rng, units, creation):
    """A random subset, unseeded or with seeds (about half of them the units' creation seeds), in a random array type."""
    mask = rng.random(units) < 0.25
    seeds = None
    if rng.random() < 0.5:
        seeds = np.where(rng.random(units) < 0.5, creation, rng.integers(0, 2**63, units).astype(np.uint64))
    kind = ["np_bool", "np_u8", "torch_bool", "torch_u8", "dlpack_bool"][int(rng.integers(5))]
    return mask, seeds, _mask_as(kind, mask), None if seeds is None else _seeds_as(seeds, kind != "np_bool")


def _trade_rows(cols, count, e, cap):
    c = {k: v.numpy() for k, v in cols.items()}
    n = min(int(count.numpy()[e]), cap)
    return [(int(c["t"][e, i]), bool(c["side_is_bid"][e, i]), int(c["price"][e, i]), int(c["vol"][e, i]), int(c["active_id"][e, i]),
             int(c["passive_id"][e, i])) for i in range(n)]


@pytest.mark.parametrize("engine,tick", [("paged", 1), ("paged", 2), ("fast", 1), ("dense", 1)], ids=["paged_t1", "paged_t2", "fast", "dense"])
def test_vector_env_masked_resets_match_the_oracle(oracle, engine, tick):
    """Random rows, and at random steps a random subset reset: ids, observations (the rows reset returns included), order
    and trade reads bit-exact at every step; orders, trades and history of every env at the end; error bits per env."""
    n_envs, rows, n_steps, seed, cap = 40, 7, 36, 11, 64
    rng = np.random.default_rng(21 + tick + len(engine))
    v = gym.VectorEnv(n_envs, rows, seed, 0, tick, 1000, max_orders=1024, max_trades=4096, max_steps=64, **ENGINES[engine])
    orcs = [oracle.StepEnv(seed + e, 0, tick, 1000) for e in range(n_envs)]
    creation = seed + np.arange(n_envs, dtype=np.uint64)
    issued = np.zeros(n_envs, np.int64)
    flagged = np.zeros(n_envs, bool)
    seen = [[] for _ in range(n_envs)]   # every trade trades() reported since the env's last reset
    prev = v.reset().numpy()
    n_reset = n_seeded = 0
    for s in range(n_steps):
        op, cols = _random_actions(rng, n_envs, rows, issued, tick)
        obs, ids = v.step(gym.pack_actions(op, **cols))
        got = v.orders(ids)
        tcols, count = v.trades(cap)
        obs, ids = obs.numpy(), ids.numpy()
        st, vol, pr = (got[k].numpy() for k in ("status", "vol", "price"))
        for e in range(n_envs):
            want, bad = _oracle_step(orcs[e], op, cols, e, rows)
            flagged[e] |= bad
            assert np.array_equal(ids[e], want), (s, e)
            assert np.array_equal(obs[e], orcs[e].level_2_data_array()), (s, e)
            table = orcs[e].get_orders()
            for r in range(rows):
                if want[r] != abi.NO_ID:
                    o = table[int(want[r])]
                    assert (st[e, r], vol[e, r], pr[e, r]) == (o[1], o[4], o[6]), (s, e, r)
            seen[e] += _trade_rows(tcols, count, e, cap)
            assert seen[e] == orcs[e].get_trades(), (s, e)
            issued[e] = len(table)
        prev = obs
        if s % 3 == 2 or rng.random() < 0.3:
            mask, seeds, m_arg, s_arg = _random_reset(rng, n_envs, creation)
            out = v.reset(m_arg, s_arg).numpy()
            for e in range(n_envs):
                if mask[e]:
                    ers.sim_reset(orcs[e], 0, seed=None if seeds is None else int(seeds[e]))
                    issued[e], flagged[e], seen[e] = 0, False, []
                    assert np.array_equal(out[e], orcs[e].level_2_data_array()), (s, e)
                else:
                    assert np.array_equal(out[e], prev[e]), (s, e)
            n_reset += int(mask.sum())
            n_seeded += int(mask.sum()) if seeds is not None else 0
            prev = out
    assert n_reset > 20 and 0 < n_seeded < n_reset
    for e in range(n_envs):
        assert v.env.get_trades(e) == orcs[e].get_trades() and v.env.get_orders(e) == orcs[e].get_orders(), e
        assert np.array_equal(v.env.history(e), orcs[e]._history()), e
    err = v.env.env_errors()
    assert np.array_equal((err & 0x200) != 0, flagged) and not (err & ~np.uint32(0x200)).any()
    v.close()


@pytest.mark.parametrize("engine", ["paged", "fast", "dense"])
def test_creation_seed_replays_episode_one(engine):
    """An env reset with its creation seed replays episode 1 bit for bit under the same rows; the envs not reset go on."""
    n_envs, rows, seed, steps = 16, 5, 3, 12
    rng = np.random.default_rng(4)
    v = gym.VectorEnv(n_envs, rows, seed, 0, 1, 1000, max_orders=1024, max_trades=4096, max_steps=64, **ENGINES[engine])
    v.reset()
    blocks = [gym.pack_actions(np.full((n_envs, rows), abi.OP_NEW, np.uint32), bid=rng.random((n_envs, rows)) < 0.5,
                               vol=rng.integers(1, 20, (n_envs, rows)), price=rng.integers(45, 56, (n_envs, rows)), trader=3)
              for _ in range(steps)]
    first = [tuple(x.numpy() for x in v.step(b)) for b in blocks]
    trades1 = [v.env.get_trades(e) for e in range(n_envs)]
    mask = np.arange(n_envs) % 2 == 0
    v.reset(mask, seed + np.arange(n_envs, dtype=np.uint64))
    for s, b in enumerate(blocks):
        obs, ids = (x.numpy() for x in v.step(b))
        assert np.array_equal(obs[mask], first[s][0][mask]) and np.array_equal(ids[mask], first[s][1][mask]), s
        assert not np.array_equal(ids[~mask], first[s][1][~mask])   # the others kept counting ids
    for e in range(n_envs):
        if mask[e]:
            assert v.env.get_trades(e) == trades1[e] and v.env.n_steps(e) == steps
        else:
            assert len(v.env.get_trades(e)) >= len(trades1[e]) and v.env.n_steps(e) == 2 * steps
    assert sum(len(t) for t in trades1) > 0
    v.close()


@pytest.mark.parametrize("kw,groups_name", [(dict(price_window=(20, 180), live_cap=254), "c3"), (dict(), "c3"), (dict(), "c4")],
                         ids=["dense_c3", "fast_c3", "fast_c4"])
def test_vector_env_resets_with_background_agents(oracle, kw, groups_name):
    """With built-in agents: an unseeded reset continues the Philox step counter (fresh agent draws), a seeded one restarts
    it; per step and env equal to the oracle's agents_update + rows + step_keyed with the same resets."""
    groups = workloads.c3_groups() if groups_name == "c3" else workloads.c4_groups()
    n_envs, rows, n_steps, seed = 24, 4, 30, 77
    rng = np.random.default_rng(9)
    v = gym.VectorEnv(n_envs, rows, 0, 0, 1, 1_000_000, agents=groups, agent_seed=seed, max_orders=8192, max_trades=8192,
                      max_steps=64, max_queue=160, **kw)
    orcs = [oracle.StepEnv(0, 0, 1, 1_000_000) for _ in range(n_envs)]
    for o in orcs:
        o.set_groups(groups)
    v.reset()
    mine = [[] for _ in range(n_envs)]
    kinds = set()
    for s in range(n_steps):
        op = np.zeros((n_envs, rows), np.uint32)
        cols = {k: np.zeros((n_envs, rows), np.uint64) for k in ("bid", "vol", "trader", "price", "order_id", "market")}
        for e in range(n_envs):
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
        obs, ids = v.step(gym.pack_actions(op, **cols))
        obs, ids = obs.numpy(), ids.numpy()
        for e, o in enumerate(orcs):
            o.agents_update(seed, e)
            want = np.full(rows, abi.NO_ID, np.uint64)
            for r in range(rows):
                if op[e, r] == abi.OP_NEW:
                    want[r] = o.place_order(bool(cols["bid"][e, r]), int(cols["vol"][e, r]), int(cols["trader"][e, r]),
                                            None if cols["market"][e, r] else int(cols["price"][e, r]))
                    mine[e].append(int(want[r]))
                elif op[e, r] == abi.OP_CANCEL:
                    o.cancel_order(int(cols["order_id"][e, r]))
            o.step_keyed(seed, e)
            assert np.array_equal(ids[e], want), (s, e)
            assert np.array_equal(obs[e], o.level_2_data_array()), (s, e)
        if s % 4 == 3:
            mask = rng.random(n_envs) < 0.3
            seeded = s % 8 == 7
            seeds = rng.integers(0, 2**63, n_envs).astype(np.uint64) if seeded else None
            out = v.reset(_mask_as("torch_bool", mask), seeds).numpy()
            for e in np.flatnonzero(mask):
                ers.sim_reset(orcs[e], 0, seed=int(seeds[e]) if seeded else None)
                mine[e] = []
                assert np.array_equal(out[e], orcs[e].level_2_data_array())
            kinds.add(seeded)
    assert kinds == {False, True}
    v.check_errors()
    for e in range(n_envs):
        assert v.env.get_trades(e) == orcs[e].get_trades() and v.env.get_orders(e) == orcs[e].get_orders(), e
        assert np.array_equal(v.env.history(e), orcs[e]._history()), e
    v.close()


MARKET_CASES = [("fast", 2, None), ("paged", 3, None), ("dense", 5, None), ("fast", 2, "mixed"), ("dense", 4, "random")]


@pytest.mark.parametrize("engine,A,pop", MARKET_CASES, ids=[f"{e}-{A}-{p or 'rows_only'}" for e, A, p in MARKET_CASES])
def test_market_vector_env_masked_resets_match_the_oracle(oracle, engine, A, pop):
    """Per-market masks on MarketVectorEnv, rows only and against market agents: every book of a reset market starts again,
    ids, observations and the trades reads bit-exact against oracle.MarketEnv reset the same way."""
    ticks, n_markets, seed, aseed, n_steps, cap = (TICKS if pop is None else AGENT_TICKS)[A], 8, 31, 0xB0A5, 28, 128
    agents = None if pop is None else random_agents(A) if pop == "random" else mixed_agents(A)
    rows = 4 * A if agents is None else 6
    kw = dict(max_orders=8192, max_trades=16384, max_steps=64, **ENGINES[engine])
    if agents:
        kw["max_queue"] = 128
    v = gym.MarketVectorEnv(n_markets, rows, seed, 0, ticks, 1000, agents=agents, agent_seed=aseed, **kw)
    v.reset()
    if agents:
        orcs = [oracle_market(oracle, agents, ticks, 1000) for _ in range(n_markets)]
    else:
        orcs = [oracle.MarketEnv(seed + m, 0, ticks, 1000) for m in range(n_markets)]
    creation = seed + np.arange(n_markets, dtype=np.uint64)
    issued = [[0] * A for _ in range(n_markets)]
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    seen = [[[] for _ in range(A)] for _ in range(n_markets)]
    rng = np.random.default_rng(A * 13 + len(engine))
    n_reset = 0
    for s in range(n_steps):
        if agents:
            blk = np.stack([learner_block(rng, ticks, mine[mk], rows) for mk in range(n_markets)])
        else:
            blk = np.stack([random_block(rng, ticks, issued[mk], rows, off_tick=False) for mk in range(n_markets)])
        obs, ids = v.step(blk)
        tcols, count = v.trades(cap)
        tc = {k: x.numpy() for k, x in tcols.items()}
        cnt = count.numpy()
        obs, ids = obs.numpy(), ids.numpy()
        for mk, o in enumerate(orcs):
            if agents:
                mks.agents_update(o, aseed, mk)
                want = agent_rows(o, blk[mk], mine[mk])
                mks.step_keyed(o, aseed, mk)
            else:
                want = oracle_rows(o, blk[mk])[0]
            assert list(ids[mk]) == want, (s, mk)
            for a in range(A):
                assert np.array_equal(obs[mk, a], o.history(a)[-1]), (s, mk, a)
                n = min(int(cnt[mk, a]), cap)
                seen[mk][a] += [(int(tc["t"][mk, a, i]), bool(tc["side_is_bid"][mk, a, i]), int(tc["price"][mk, a, i]),
                                 int(tc["vol"][mk, a, i]), int(tc["active_id"][mk, a, i]), int(tc["passive_id"][mk, a, i])) for i in range(n)]
                assert seen[mk][a] == o.get_trades(a), (s, mk, a)
                issued[mk][a] = len(o.get_orders(a))
        if s % 3 == 1:
            mask = rng.random(n_markets) < 0.35
            seeds = np.where(rng.random(n_markets) < 0.5, creation, rng.integers(0, 2**63, n_markets).astype(np.uint64)) \
                if s % 6 == 4 else None
            out = v.reset(_mask_as("torch_u8" if s % 2 else "np_bool", mask), seeds).numpy()
            for mk in range(n_markets):
                if mask[mk]:
                    ers.market_reset(orcs[mk], 0, seed=None if seeds is None else int(seeds[mk]))
                    mine[mk], seen[mk], issued[mk] = [[] for _ in range(A)], [[] for _ in range(A)], [0] * A
                    assert all(np.array_equal(out[mk, a], _fresh_record()) for a in range(A)), (s, mk)
                else:
                    assert np.array_equal(out[mk], obs[mk]), (s, mk)
            n_reset += int(mask.sum())
    assert n_reset > 5
    v.check_errors()
    for mk, o in enumerate(orcs):
        assert_books_equal(v.env, mk, A, o)
    v.close()


def _fresh_record():
    r = np.zeros(45, np.uint32)
    r[2] = 0xFFFFFFFF
    return r


def test_market_seeded_reset_after_host_steps(oracle):
    """Host-path bb_step (the markets' streams advance on the host), then a seeded reset of some markets, then device steps
    and host steps again, and an unseeded reset in between: every market equals its oracle throughout."""
    ticks, n_markets, rows, seed = [1, 2, 3], 4, 9, 21
    A = len(ticks)
    m = market.MarketEnv(seed, 0, ticks, 1000, n_markets=n_markets, max_orders=8192, max_trades=8192, max_steps=128, max_queue=128,
                         **ENGINES["fast"])
    env = m._env
    ids_d = gym.DeviceArray(env, (n_markets, rows), np.uint64)
    acts_d = gym.DeviceArray(env, (n_markets, rows), gym.ACTION_DTYPE)
    offs_d = gym.DeviceArray(env, (n_markets + 1,), np.uint64)
    offs_d.copy_from_host(np.arange(n_markets + 1, dtype=np.uint64) * np.uint64(rows))
    mask_d = gym.DeviceArray(env, (n_markets,), np.uint8)
    seeds_d = gym.DeviceArray(env, (n_markets,), np.uint64)
    os_ = [oracle.MarketEnv(seed + mk, 0, ticks, 1000) for mk in range(n_markets)]
    rng = np.random.default_rng(6)
    for what in ["host", "host", "seeded", "device", "host", "unseeded", "device", "host", "seeded", "host", "device"]:
        if what in ("seeded", "unseeded"):
            mask = rng.random(n_markets) < 0.5
            mask[0] = True
            seeds = rng.integers(0, 2**63, n_markets).astype(np.uint64)
            mask_d.copy_from_host(mask.astype(np.uint8))
            seeds_d.copy_from_host(seeds)
            env.reset_device(mask_d.ptr, seeds_d.ptr if what == "seeded" else 0)
            for mk in np.flatnonzero(mask):
                ers.market_reset(os_[mk], 0, seed=int(seeds[mk]) if what == "seeded" else None)
            continue
        issued = [[len(os_[mk].get_orders(a)) for a in range(A)] for mk in range(n_markets)]
        blocks = [random_block(rng, ticks, issued[mk], rows, off_tick=False) for mk in range(n_markets)]
        if what == "device":
            acts_d.copy_from_host(np.stack(blocks))
            env.step_device_market(acts_d.ptr, offs_d.ptr, n_markets * rows, ids_d.ptr)
            got = ids_d.numpy()
        else:
            got = _host_submit(m, blocks, A)
            m.step()
        for mk, o in enumerate(os_):
            want = oracle_rows(o, blocks[mk])[0]
            assert list(got[mk]) == want, (what, mk)
    for mk, o in enumerate(os_):
        assert_books_equal(env, mk, A, o)
    assert sum(len(os_[mk].get_trades(a)) for mk in range(n_markets) for a in range(A)) > 0
    assert not env.env_errors().any()
    for a in (ids_d, acts_d, offs_d, mask_d, seeds_d):
        a.free()
    env.close()


def _policy_actions(torch, obs_i32, t_ep, rows, n_units, assets=0):
    """A deterministic device policy: NEW rows whose side, volume and price depend on the observation and the episode step."""
    n = obs_i32.shape[0]
    flat = obs_i32.reshape(n, -1).to(torch.int64)
    r = torch.arange(rows, device="cuda").unsqueeze(0)
    e = torch.arange(n, device="cuda").unsqueeze(1)
    ep = t_ep.unsqueeze(1)
    bid = (ep + e + r) % 2
    vol = 1 + (flat[:, :1] + r) % 20
    price = 45 + (flat[:, 4:5] + 3 * ep + 5 * r + e) % 11
    a = torch.zeros((n, rows, 8), dtype=torch.int64, device="cuda")
    a[:, :, 2] = abi.OP_NEW + bid * abi.F_BID
    a[:, :, 4] = 6 * (price - 37) if assets else price   # (markets: multiples of 6, on every asset's tick)
    a[:, :, 5] = vol
    a[:, :, 6] = 3
    if assets:
        a[:, :, 7] = (e + r) % assets
    return a.to(torch.int32)


@pytest.mark.parametrize("kind", ["vector", "market"])
def test_step_and_reset_inside_a_cuda_graph(kind):
    """{policy; step; done = per-env horizon reached; reset(done)} captured once and replayed 3 x max_steps times equals the
    same loop run eagerly on a twin; the VectorEnv loop resets unseeded, the MarketVectorEnv loop with the creation seeds.
    No history clear is needed: every book restarts its history at its own horizon <= max_steps."""
    import torch
    max_steps, rows, seed = 8, 3, 5
    if kind == "vector":
        n = 64
        make = lambda: gym.VectorEnv(n, rows, seed, 0, 1, 1000, max_orders=512, max_trades=1024, max_steps=max_steps)
        seeds = None
    else:
        n, A = 32, 3
        make = lambda: gym.MarketVectorEnv(n, rows, seed, 0, [1, 2, 3], 1000, max_orders=512, max_trades=1024, max_steps=max_steps)
        seeds = torch.from_numpy((seed + np.arange(n)).astype(np.int64)).cuda()
    horizon = torch.from_numpy(np.random.default_rng(2).integers(3, max_steps + 1, n)).cuda()
    twins = []
    for _ in range(2):
        v = make()
        s = torch.cuda.Stream()
        v.env.set_stream(s.cuda_stream)
        v.reset()
        obs_t = torch.as_tensor(v.obs, device="cuda").view(torch.int32)
        st = dict(v=v, s=s, obs=obs_t, t=torch.zeros(n, dtype=torch.int64, device="cuda"), acts=None, done=None, episodes=0)
        twins.append(st)
    torch.cuda.synchronize()

    def body(st):
        st["acts"] = _policy_actions(torch, st["obs"], st["t"], rows, n, 0 if kind == "vector" else 3)
        st["v"].step(st["acts"])
        st["t"] += 1
        st["done"] = st["t"] >= horizon
        st["t"].masked_fill_(st["done"], 0)
        st["v"].reset(st["done"], seeds)

    a, b = twins
    with torch.cuda.stream(a["s"]):   # warm-up outside the capture (attribute / occupancy queries happen here)
        body(a)
    with torch.cuda.stream(b["s"]):
        body(b)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=a["s"]):
        body(a)
    done_total = 0
    for it in range(3 * max_steps):
        g.replay()
        with torch.cuda.stream(b["s"]):
            body(b)
        torch.cuda.synchronize()
        assert np.array_equal(a["v"].obs.numpy(), b["v"].obs.numpy()) and np.array_equal(a["v"].ids.numpy(), b["v"].ids.numpy()), it
        assert torch.equal(a["t"], b["t"]), it
        done_total += int(b["done"].sum())
    assert done_total > n
    for e in range(0, b["v"].env.n_envs, 7):
        assert a["v"].env.get_trades(e) == b["v"].env.get_trades(e) and a["v"].env.get_orders(e) == b["v"].env.get_orders(e)
        assert a["v"].env.n_steps(e) <= max_steps
    assert not a["v"].env.env_errors().any()
    assert sum(len(a["v"].env.get_trades(e)) for e in range(b["v"].env.n_envs)) > 0
    # a seeded market reset right after a host-side bb_step cannot be captured (the streams must first reach the device)
    if kind == "market":
        m = market.MarketEnv(0, 0, [1, 2], 1000, n_markets=2, max_orders=64, max_trades=64, max_steps=8, max_queue=16)
        m.submit([abi.ACT_NEW, abi.ACT_NEW], [0, 0], side=[True, False], vol=[1, 2], trader=[1, 1], price=[50, 50], market=[0, 0])
        m.step()
        s2 = torch.cuda.Stream()
        m._env.set_stream(s2.cuda_stream)
        mask, sd = torch.ones(2, dtype=torch.uint8, device="cuda"), torch.zeros(2, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        g2 = torch.cuda.CUDAGraph()
        with pytest.raises(ValueError, match="bb_step"):
            with torch.cuda.graph(g2, stream=s2):
                m._env.reset_device(mask.data_ptr(), sd.data_ptr())
        m._env.reset_device(mask.data_ptr(), sd.data_ptr())   # outside a capture it goes through
        m._env.synchronize()
        m._env.close()
    a["v"].close(); b["v"].close()


def test_edges_errors_steps_stats_and_refusals():
    """Sticky error bits and history counts restart for reset envs only; bb_stats' env_steps keeps an unseeded env's step
    counter and drops a seeded one's; refusals leave the handle unchanged; wrong masks and seeds raise ValueError."""
    import torch
    v = gym.VectorEnv(4, 2, 0, 0, 2, 1000, max_orders=64, max_trades=64, max_steps=16)
    v.reset()
    v.step(gym.pack_actions(np.full((4, 2), abi.OP_NEW, np.uint32), bid=1, vol=1, price=50, trader=1))   # ids 0 and 1
    off = gym.pack_actions(np.full((4, 2), abi.OP_NEW, np.uint32), bid=1, vol=1, price=51, trader=1)   # off the tick of 2
    for _ in range(2):
        v.step(off)
    assert (v.env.env_errors() == 0x200).all() and v.env.stats()["env_steps"] == 12
    v.reset(np.array([True, False, False, False]))
    assert list(v.env.env_errors()) == [0, 0x200, 0x200, 0x200]
    assert [v.env.n_steps(e) for e in range(4)] == [0, 3, 3, 3]
    assert v.env.stats()["env_steps"] == 12   # the unseeded env keeps its step counter
    v.reset(np.array([0, 1, 0, 0], np.uint8), np.array([0, 7, 0, 0], np.uint64))
    assert v.env.stats()["env_steps"] == 9 and v.env.n_steps(1) == 0
    # a cancel of an id held from before the reset names no order of the new episode; envs 2 and 3 still hold it
    v.step(gym.pack_actions(np.array([[abi.OP_CANCEL, abi.OP_NOOP]] * 4, np.uint32), order_id=1))
    assert list(v.env.env_errors()) == [0x10, 0x10, 0x200, 0x200]
    for bad in (np.ones(3, bool), np.ones((4, 1), bool), np.ones(4, np.float32), np.ones(4, np.int32), [1, 0, 1, 0],
                torch.ones(4, dtype=torch.int32, device="cuda"), torch.ones(5, dtype=torch.bool, device="cuda")):
        with pytest.raises(ValueError, match="mask"):
            v.reset(bad)
    for bad in (np.ones(3, np.uint64), np.ones(4, np.float64), torch.ones(4, dtype=torch.int32, device="cuda")):
        with pytest.raises(ValueError, match="seeds"):
            v.reset(np.ones(4, bool), bad)
    with pytest.raises(ValueError, match="mask"):
        v.reset(seeds=np.zeros(4, np.uint64))
    with pytest.raises(ValueError, match="null"):
        v.env.reset_device(0)
    v.close()
    e = core.BatchedEnv(1, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8, max_queue=16)
    e.submit([abi.ACT_NEW], [1], [1], [0], [10])
    p = e.device_alloc(8)
    with pytest.raises(ValueError, match="pending"):
        e.reset_device(p)
    e.step()
    assert e.n_orders(0) == 1
    e.device_free(p)
    e.close()


def test_deep_engine_masked_reset():
    """Deep engine: replay, reset books 0 and 2, replay again: the reset books equal a fresh book that replayed the stream
    once, book 1 (an empty slice the second time) is unchanged; the obs rows and cursors of reset books are rewritten."""
    import torch
    from oracle import oracle as orc
    n_books = 3
    streams = [workloads.c5_stream(1500, 2, 300, seed=70 + i, mid_ticks=3000, depth_ticks=256) for i in range(n_books)]
    n = len(streams[0])
    env = core.BatchedEnv(n_books, 5, 0, 1, 1000, max_orders=n + 64, max_trades=4 * n, max_steps=64, max_queue=32,
                          price_window=(2688, 3328), deep_chunks=n // 8 + 1400)
    d_instrs = torch.from_numpy(np.concatenate(streams).view(np.uint8)).cuda()
    d_offs = torch.from_numpy((np.arange(n_books + 1, dtype=np.uint64) * n).view(np.int64)).cuda()
    torch.cuda.synchronize()
    env.replay_device(d_instrs.data_ptr(), d_offs.data_ptr())
    env.synchronize()
    before = (env.get_orders(1), env.get_trades(1), env.history(1))
    mask = torch.tensor([1, 0, 1], dtype=torch.uint8, device="cuda")
    obs = torch.full((n_books, 45), 7, dtype=torch.int32, device="cuda")
    cursor = torch.full((n_books,), 9, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    env.reset_device(mask.data_ptr(), 0, obs.data_ptr(), cursor.data_ptr())
    env.synchronize()
    assert list(cursor.cpu().numpy()) == [0, 9, 0]
    o = obs.cpu().numpy().view(np.uint32)
    assert np.array_equal(o[0], _fresh_record()) and np.array_equal(o[2], _fresh_record()) and (o[1] == 7).all()
    assert env.n_orders(0) == 0 and env.n_steps(0) == 0 and env.n_trades(2) == 0
    again = np.concatenate([streams[0], streams[2]])
    d2 = torch.from_numpy(again.view(np.uint8)).cuda()
    o2 = torch.from_numpy(np.array([0, n, n, 2 * n], np.uint64).view(np.int64)).cuda()
    torch.cuda.synchronize()
    env.replay_device(d2.data_ptr(), o2.data_ptr())
    env.synchronize()
    for b in (0, 2):
        ob = orc.OrderBook(0, 1)
        ob.replay(streams[b])
        assert env.get_orders(b) == ob.get_orders() and env.get_trades(b) == ob.get_trades(), b
    assert (env.get_orders(1), env.get_trades(1)) == before[:2] and np.array_equal(env.history(1), before[2])
    assert not env.env_errors().any()
    env.close()


def test_episodes_example():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "vector_env_episodes_torch.py")], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    assert "episodes completed" in out.stdout and "error_envs: 0" in out.stdout
