"""GPU suite for the device-resident book snapshots of the vector loops (bb_save_device / bb_restore_device,
VectorEnv / MarketVectorEnv.save / restore): units saved into slots of a device store and restored from any slot, with the
slot's random streams or re-seeded ones.  Everything is checked bit for bit against the oracle's envs copied the same way
(tests/episode_snapshot_oracle.py): a slot is an oracle env kept aside."""
import os
import subprocess
import sys

import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import episode_snapshot_oracle as ess
from . import market_split_oracle as mks
from .test_gpu_deep import compare_book
from .test_gpu_gym import _oracle_step, _random_actions
from .test_gpu_market_agents_rows import TICKS as AGENT_TICKS
from .test_gpu_market_agents_rows import learner_block, mixed_agents, oracle_market, random_agents
from .test_gpu_market_agents_rows import oracle_rows as agent_rows
from .test_gpu_market_device import TICKS, assert_books_equal, oracle_rows, random_block
from .test_gpu_reset import ENGINES, _trade_rows

pytestmark = pytest.mark.gpu
ERR_SLOT = 0x1000   # BB_ERR_SLOT


def _as(kind, a):
    """`a` as a numpy array, a torch CUDA tensor of the same width, or a DLPack-only view of one."""
    import torch
    if kind == "np":
        return a
    t = torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a.view(np.int64)).cuda()
    torch.cuda.synchronize()
    if kind == "dlpack":
        from .test_gpu_reset import DLPackOnly
        return DLPackOnly(t)
    return t


def _random_save(rng, units, n_slots):
    """A save map: each slot takes a random unit, or keeps its state (NO_SLOT)."""
    sel = rng.integers(0, units, n_slots).astype(np.uint32)
    sel[rng.random(n_slots) < 0.3] = gym.NO_SLOT
    return sel


def _random_restore(rng, units, n_slots, seeded):
    """A restore map: about a third of the units from random slots, the others untouched; seeds or None."""
    slots = np.full(units, gym.NO_SLOT, np.uint32)
    pick = rng.random(units) < 0.35
    slots[pick] = rng.integers(0, n_slots, int(pick.sum()))
    seeds = rng.integers(0, 2**63, units).astype(np.uint64) if seeded else None
    return slots, seeds


@pytest.mark.parametrize("engine,tick", [("paged", 1), ("paged", 2), ("fast", 1), ("dense", 1)], ids=["paged_t1", "paged_t2", "fast", "dense"])
def test_vector_env_snapshots_match_the_oracle(oracle, engine, tick):
    """Random rows; at random steps random units saved into random slots and random units restored from random slots, some
    with seeds: ids, observations (the rows restore returns included), order and trade reads bit-exact at every step;
    orders, trades, history and error bits of every env at the end."""
    n_envs, rows, n_steps, seed, cap, n_slots = 32, 6, 36, 13, 64, 5
    rng = np.random.default_rng(5 + tick + len(engine))
    v = gym.VectorEnv(n_envs, rows, seed, 0, tick, 1000, max_orders=1024, max_trades=4096, max_steps=64, **ENGINES[engine])
    store = v.snapshots(n_slots)
    assert store.nbytes > n_slots * 1024 * 64
    orcs = [oracle.StepEnv(seed + e, 0, tick, 1000) for e in range(n_envs)]
    slots = [oracle.StepEnv(0, 0, tick, 1000) for _ in range(n_slots)]
    flagged, slot_flagged = np.zeros(n_envs, bool), np.zeros(n_slots, bool)
    issued = np.zeros(n_envs, np.int64)
    seen = [[] for _ in range(n_envs)]   # every trade trades() reported, or the restored log
    prev = v.reset().numpy()
    v.save(store)   # slot k <- env k
    for k in range(n_slots):
        ess.sim_copy(slots[k], orcs[k])
    n_saved = n_restored = n_seeded = 0
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
        if rng.random() < 0.4:
            sel = _random_save(rng, n_envs, n_slots)
            v.save(store, _as(["np", "torch", "dlpack"][s % 3], sel))
            for k in np.flatnonzero(sel != gym.NO_SLOT):
                ess.sim_copy(slots[k], orcs[sel[k]])
                slot_flagged[k] = flagged[sel[k]]
            n_saved += int((sel != gym.NO_SLOT).sum())
        if s % 3 == 2 or rng.random() < 0.25:
            sl, seeds = _random_restore(rng, n_envs, n_slots, rng.random() < 0.4)
            out = v.restore(store, _as(["np", "torch"][s % 2], sl), None if seeds is None else _as("torch", seeds)).numpy()
            for e in range(n_envs):
                if sl[e] != gym.NO_SLOT:
                    ess.sim_copy(orcs[e], slots[sl[e]], seed=None if seeds is None else int(seeds[e]))
                    flagged[e], issued[e] = slot_flagged[sl[e]], len(orcs[e].get_orders())
                    seen[e] = list(orcs[e].get_trades())
                    assert np.array_equal(out[e], orcs[e].level_2_data_array()), (s, e)
                else:
                    assert np.array_equal(out[e], prev[e]), (s, e)
            n_restored += int((sl != gym.NO_SLOT).sum())
            n_seeded += int((sl != gym.NO_SLOT).sum()) if seeds is not None else 0
            prev = out
    assert n_saved > 10 and n_restored > 30 and 0 < n_seeded < n_restored
    for e in range(n_envs):
        assert v.env.get_trades(e) == orcs[e].get_trades() and v.env.get_orders(e) == orcs[e].get_orders(), e
        assert np.array_equal(v.env.history(e), orcs[e]._history()), e
    err = v.env.env_errors()
    assert np.array_equal((err & 0x200) != 0, flagged) and not (err & ~np.uint32(0x200)).any()
    v.close()
    assert store.ptr == 0   # (the env's close freed its store)


@pytest.mark.parametrize("kw", [dict(price_window=(20, 180), live_cap=254), dict()], ids=["dense_c3", "fast_c3"])
def test_vector_env_snapshots_with_background_agents(oracle, kw):
    """With built-in agents: saved and restored units, unseeded and seeded, equal the oracle's agents_update + rows +
    step_keyed on copied envs at every step; a unit restored from another unit's slot draws with its own env id."""
    groups = workloads.c3_groups()
    n_envs, rows, n_steps, seed, n_slots = 16, 4, 28, 77, 4
    rng = np.random.default_rng(9)
    v = gym.VectorEnv(n_envs, rows, 0, 0, 1, 1_000_000, agents=groups, agent_seed=seed, max_orders=8192, max_trades=8192,
                      max_steps=64, max_queue=160, **kw)
    store = v.snapshots(n_slots)
    orcs = [oracle.StepEnv(0, 0, 1, 1_000_000) for _ in range(n_envs)]
    slots = [oracle.StepEnv(0, 0, 1, 1_000_000) for _ in range(n_slots)]
    for o in orcs + slots:
        o.set_groups(groups)
    v.reset()
    mine = [[] for _ in range(n_envs)]
    slot_mine = [[] for _ in range(n_slots)]
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
        if s % 4 == 1:
            sel = rng.permutation(n_envs)[:n_slots].astype(np.uint32)
            v.save(store, sel)
            for k in range(n_slots):
                ess.sim_copy(slots[k], orcs[sel[k]])
                slot_mine[k] = list(mine[sel[k]])
        if s % 4 == 3:
            seeded = s % 8 == 7
            sl, seeds = _random_restore(rng, n_envs, n_slots, seeded)
            out = v.restore(store, sl, seeds).numpy()
            for e in np.flatnonzero(sl != gym.NO_SLOT):
                ess.sim_copy(orcs[e], slots[sl[e]], seed=int(seeds[e]) if seeded else None)
                mine[e] = list(slot_mine[sl[e]])
                assert np.array_equal(out[e], orcs[e].level_2_data_array())
            kinds.add(seeded)
    assert kinds == {False, True}
    v.check_errors()
    for e in range(n_envs):
        assert v.env.get_trades(e) == orcs[e].get_trades() and v.env.get_orders(e) == orcs[e].get_orders(), e
        assert np.array_equal(v.env.history(e), orcs[e]._history()), e
    v.close()


MARKET_CASES = [("fast", 2, None), ("paged", 3, None), ("dense", 4, "random"), ("fast", 2, "mixed")]


@pytest.mark.parametrize("engine,A,pop", MARKET_CASES, ids=[f"{e}-{A}-{p or 'rows_only'}" for e, A, p in MARKET_CASES])
def test_market_vector_env_snapshots_match_the_oracle(oracle, engine, A, pop):
    """Markets saved and restored as units, rows only and against market agents: every book of a restored market takes its
    slot's state; ids, observations and trades reads bit-exact against oracle.MarketEnv copied the same way."""
    ticks, n_markets, seed, aseed, n_steps, cap, n_slots = (TICKS if pop is None else AGENT_TICKS)[A], 8, 31, 0xB0A5, 26, 128, 3
    agents = None if pop is None else random_agents(A) if pop == "random" else mixed_agents(A)
    rows = 4 * A if agents is None else 6
    kw = dict(max_orders=8192, max_trades=16384, max_steps=64, **ENGINES[engine])
    if agents:
        kw["max_queue"] = 128
    v = gym.MarketVectorEnv(n_markets, rows, seed, 0, ticks, 1000, agents=agents, agent_seed=aseed, **kw)
    store = v.snapshots(n_slots)
    v.reset()

    def make(m):
        return oracle_market(oracle, agents, ticks, 1000) if agents else oracle.MarketEnv(seed + m, 0, ticks, 1000)

    orcs = [make(m) for m in range(n_markets)]
    slots = [make(0) for _ in range(n_slots)]
    slot_mine = [None] * n_slots
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    seen = [[[] for _ in range(A)] for _ in range(n_markets)]
    rng = np.random.default_rng(A * 17 + len(engine))
    n_restored = 0
    for s in range(n_steps):
        issued = [[len(o.get_orders(a)) for a in range(A)] for o in orcs]
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
        if s % 5 == 1:
            sel = _random_save(rng, n_markets, n_slots)
            if s == 1:
                sel[:] = np.arange(n_slots)
            v.save(store, _as("torch", sel))
            for k in np.flatnonzero(sel != gym.NO_SLOT):
                ess.market_copy(slots[k], orcs[sel[k]])
                slot_mine[k] = [list(x) for x in mine[sel[k]]]
        if s % 3 == 2:
            sl, seeds = _random_restore(rng, n_markets, n_slots, s % 2 == 1)
            out = v.restore(store, sl, seeds).numpy()
            for mk in range(n_markets):
                if sl[mk] != gym.NO_SLOT:
                    ess.market_copy(orcs[mk], slots[sl[mk]], seed=None if seeds is None else int(seeds[mk]))
                    mine[mk] = [list(x) for x in slot_mine[sl[mk]]]
                    seen[mk] = [list(orcs[mk].get_trades(a)) for a in range(A)]
                    assert all(np.array_equal(out[mk, a], _market_record(orcs[mk], a)) for a in range(A)), (s, mk)
                else:
                    assert np.array_equal(out[mk], obs[mk]), (s, mk)
            n_restored += int((sl != gym.NO_SLOT).sum())
    assert n_restored > 5
    v.check_errors()
    for mk, o in enumerate(orcs):
        assert_books_equal(v.env, mk, A, o)
    v.close()


def _market_record(o, a):
    """Asset a's level-2 record of an oracle market as its book is now (what its last step recorded)."""
    from oracle import oracle as orc
    out = np.zeros(45, np.uint32)
    orc.lib().orc_book_l2(o.asset(a)._book(), orc._ptr(out))
    return out


def test_broadcast_and_untouched_units_match_a_twin():
    """One slot restored into half the units, then into every unit, in one call each: units that were not restored stay
    bit-identical to a twin handle that never restored; units restored from one slot continue identically (rows only)."""
    n_envs, rows, seed = 24, 5, 3
    rng = np.random.default_rng(8)
    make = lambda: gym.VectorEnv(n_envs, rows, seed, 0, 1, 1000, max_orders=2048, max_trades=4096, max_steps=128, **ENGINES["fast"])
    a, twin = make(), make()
    store = a.snapshots(2)
    a.reset(), twin.reset()

    def block():
        return gym.pack_actions(np.full((n_envs, rows), abi.OP_NEW, np.uint32), bid=rng.random((n_envs, rows)) < 0.5,
                                vol=rng.integers(1, 20, (n_envs, rows)), price=rng.integers(45, 56, (n_envs, rows)), trader=3)

    for _ in range(10):
        b = block()
        a.step(b), twin.step(b)
    a.save(store, np.array([5, n_envs + 3], np.uint32))   # slot 1 <- no unit: marked empty
    half = np.where(np.arange(n_envs) % 2 == 0, 0, gym.NO_SLOT).astype(np.uint32)
    a.restore(store, half)
    for _ in range(8):
        b = block()
        ra, rt = a.step(b)[0].numpy(), twin.step(b)[0].numpy()
        assert np.array_equal(ra[1::2], rt[1::2])
    for e in range(1, n_envs, 2):
        assert a.env.get_orders(e) == twin.env.get_orders(e) and a.env.get_trades(e) == twin.env.get_trades(e)
        assert np.array_equal(a.env.history(e), twin.env.history(e))
    out = a.restore(store, np.zeros(n_envs, np.uint32)).numpy()
    assert (out == out[0]).all()
    same = gym.pack_actions(np.full((n_envs, rows), abi.OP_NEW, np.uint32), bid=np.tile(rng.random(rows) < 0.5, (n_envs, 1)),
                            vol=np.tile(rng.integers(1, 20, rows), (n_envs, 1)), price=np.tile(rng.integers(45, 56, rows), (n_envs, 1)), trader=3)
    for _ in range(6):
        obs, ids = (x.numpy() for x in a.step(same))
        assert (obs == obs[0]).all() and (ids == ids[0]).all()
    assert all(a.env.get_trades(e) == a.env.get_trades(0) for e in range(n_envs)) and len(a.env.get_trades(0)) > 0
    a.restore(store, np.full(n_envs, 1, np.uint32))   # the emptied slot: every env flagged, nothing restored
    assert (a.env.env_errors() == ERR_SLOT).all() and a.env.get_orders(0) == a.env.get_orders(1)
    a.close(), twin.close()


def test_error_bits_and_tick_check():
    """Per-env ticks: a slot saved from an env of tick 2 restores into envs of tick 2 and flags those of tick 1; an empty slot,
    a slot out of range and a slot emptied by a save from an out-of-range unit flag BB_ERR_SLOT and change nothing."""
    ticks = [1, 2, 1, 2]
    v = gym.VectorEnv(4, 2, 0, 0, ticks, 1000, max_orders=64, max_trades=64, max_steps=16)
    st = v.snapshots(3)
    v.reset()
    v.step(gym.pack_actions(np.full((4, 2), abi.OP_NEW, np.uint32), bid=[[1, 0]] * 4, vol=3, price=[[50, 60]] * 4, trader=1))
    before = [v.env.get_orders(e) for e in range(4)]
    v.save(st, np.array([1, 99, gym.NO_SLOT], np.uint32))   # slot 0 <- env 1 (tick 2); slot 1 emptied; slot 2 never saved
    v.step(gym.pack_actions(np.full((4, 2), abi.OP_NOOP, np.uint32)))
    assert not v.env.env_errors().any()
    v.restore(st, np.array([0, gym.NO_SLOT, gym.NO_SLOT, 0], np.uint32))
    assert list(v.env.env_errors()) == [ERR_SLOT, 0, 0, 0] and v.env.n_steps(3) == 0 and v.env.n_steps(0) == 2
    assert v.env.get_orders(3) == before[1] and v.env.get_orders(0) == before[0]
    v.restore(st, np.array([1, 2, 3, gym.NO_SLOT], np.uint32))
    assert list(v.env.env_errors()) == [ERR_SLOT, ERR_SLOT, ERR_SLOT, 0]
    assert [v.env.get_orders(e) for e in range(3)] == before[:3]
    with pytest.raises(RuntimeError, match="0x1000"):
        v.check_errors()
    v.close()


def test_refusals():
    """NULL arguments, a store of another handle, a store that predates bb_reserve / bb_set_agents / bb_set_tick_sizes and
    pending host instructions are refused with the handle unchanged; malformed unit and slot arrays raise ValueError."""
    import torch
    v = gym.VectorEnv(4, 2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=16)
    w = gym.VectorEnv(4, 2, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=16)
    v.reset(), w.reset()
    st, other = v.snapshots(2), w.snapshots(2)
    _, nbytes = v.env.store_create(2, allocate=False)
    assert nbytes == st.nbytes
    v.save(st)
    with pytest.raises(ValueError, match="another handle"):
        v.save(other)
    with pytest.raises(ValueError, match="another handle"):
        v.restore(other, np.zeros(4, np.uint32))
    with pytest.raises(ValueError, match="null"):
        v.env.save_device(st.ptr, 0)
    with pytest.raises(ValueError, match="null"):
        v.env.restore_device(0, v.obs.ptr)
    for bad in (np.zeros(3, np.uint32), np.zeros(4, np.float32), np.full(4, -1), torch.zeros(4, dtype=torch.int64, device="cuda")):
        with pytest.raises(ValueError, match="slots"):
            v.restore(st, bad)
    with pytest.raises(ValueError, match="units"):
        v.save(st, np.zeros(3, np.uint32))
    for change in (lambda e: e.reserve(max_orders=128), lambda e: e.set_agents([core.random_group(4, (40, 60), (1, 5), 1, 0.5)]),
                   lambda e: e.set_tick_sizes([1, 1, 1, 1])):
        s2 = v.snapshots(1)
        change(v.env)
        with pytest.raises(ValueError, match="predates"):
            v.save(s2)
        with pytest.raises(ValueError, match="predates"):
            v.restore(s2, np.zeros(4, np.uint32))
        s2.close()
    e = core.BatchedEnv(1, 0, 0, 1, 1000, max_orders=64, max_trades=64, max_steps=8, max_queue=16)
    s3, _ = e.store_create(1)
    e.submit([abi.ACT_NEW], [1], [1], [0], [10])
    p = e.device_alloc(8)
    with pytest.raises(ValueError, match="pending"):
        e.save_device(s3, p)
    e.step()
    assert e.n_orders(0) == 1
    e.device_free(p)
    e.store_destroy(s3)
    e.close()
    v.close(), w.close()


def test_deep_engine_snapshot():
    """Deep engine: replay a preload, save, replay more, restore: the books equal the oracle's books at the save point, and
    a replay of the same continuation from them equals the one from the original state."""
    import torch
    from oracle import oracle as orc
    n_books = 2
    streams = [workloads.c5_stream(3000, 2, 400, seed=80 + i, mid_ticks=3000, depth_ticks=256) for i in range(n_books)]
    h, n = min(len(s) for s in streams) // 2, max(len(s) for s in streams)
    env = core.BatchedEnv(n_books, 5, 0, 1, 1000, max_orders=n + 64, max_trades=4 * n, max_steps=64, max_queue=32,
                          price_window=(2688, 3328), deep_chunks=n // 8 + 1400)
    store, _ = env.store_create(n_books)

    def replay(part):
        parts = [s[part] for s in streams]
        env.replay(np.concatenate(parts), np.cumsum([0] + [len(p) for p in parts]).astype(np.uint64))

    replay(slice(0, h))
    units = torch.arange(n_books, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    env.save_device(store, units.data_ptr())
    replay(slice(h, n))
    after = [(env.get_orders(b), env.get_trades(b)) for b in range(n_books)]
    obs = torch.full((n_books, 45), 7, dtype=torch.int32, device="cuda")
    cursor = torch.zeros(n_books, dtype=torch.int32, device="cuda")
    env.restore_device(store, units.data_ptr(), 0, obs.data_ptr(), cursor.data_ptr())
    env.synchronize()
    for b in range(n_books):
        ob = orc.OrderBook(0, 1)
        ob.replay(streams[b][:h])
        compare_book(env, b, ob)
        assert np.array_equal(obs.cpu().numpy().view(np.uint32)[b], ob.level_2_data())
        assert int(cursor[b]) == len(ob.get_trades()) and env.n_steps(b) == 0
    replay(slice(h, n))
    assert [(env.get_orders(b), env.get_trades(b)) for b in range(n_books)] == after
    assert not env.env_errors().any()
    env.store_destroy(store)
    env.close()


def _policy(torch, obs_i32, rows):
    n = obs_i32.shape[0]
    flat = obs_i32.reshape(n, -1).to(torch.int64)
    r = torch.arange(rows, device="cuda").unsqueeze(0)
    e = torch.arange(n, device="cuda").unsqueeze(1)
    a = torch.zeros((n, rows, 8), dtype=torch.int64, device="cuda")
    a[:, :, 2] = abi.OP_NEW + ((e + r + flat[:, :1]) % 2) * abi.F_BID
    a[:, :, 4] = 45 + (flat[:, 4:5] + 5 * r + e) % 11
    a[:, :, 5] = 1 + (flat[:, :1] + r) % 20
    a[:, :, 6] = 3
    return a.to(torch.int32)


def test_step_save_restore_inside_a_cuda_graph():
    """{policy; step; save every env into its slot when a counter says so; restore the envs a mask selects from slots
    chosen on the device, with device seeds} captured once and replayed against the same loop run eagerly on a twin."""
    import torch
    n, rows, n_slots, seed = 48, 3, 6, 5
    twins = []
    for _ in range(2):
        v = gym.VectorEnv(n, rows, seed, 0, 1, 1000, max_orders=4096, max_trades=8192, max_steps=8)
        s = torch.cuda.Stream()
        v.env.set_stream(s.cuda_stream)
        v.reset()
        st = v.snapshots(n_slots)
        v.save(st)
        twins.append(dict(v=v, s=s, st=st, obs=torch.as_tensor(v.obs, device="cuda").view(torch.int32),
                          it=torch.zeros((), dtype=torch.int64, device="cuda")))
    torch.cuda.synchronize()
    env_ids = torch.arange(n, device="cuda")

    def body(t):
        t["v"].step(_policy(torch, t["obs"], rows))
        t["it"] += 1
        units = torch.where((t["it"] % 3 == 0), (t["it"] * 7 + torch.arange(n_slots, device="cuda")) % n, gym.NO_SLOT)
        t["v"].save(t["st"], units.to(torch.int32))
        done = (env_ids + t["it"]) % 4 == 0
        slots = torch.where(done, (env_ids + t["it"]) % n_slots, gym.NO_SLOT).to(torch.int32)
        t["v"].restore(t["st"], slots, (env_ids * 31 + t["it"]).to(torch.int64))
        t["v"].env.clear_history()

    a, b = twins
    for t in (a, b):   # warm-up outside the capture
        with torch.cuda.stream(t["s"]):
            body(t)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=a["s"]):
        body(a)
    for it in range(12):
        g.replay()
        with torch.cuda.stream(b["s"]):
            body(b)
        torch.cuda.synchronize()
        assert np.array_equal(a["v"].obs.numpy(), b["v"].obs.numpy()) and np.array_equal(a["v"].ids.numpy(), b["v"].ids.numpy()), it
    for e in range(0, n, 5):
        assert a["v"].env.get_trades(e) == b["v"].env.get_trades(e) and a["v"].env.get_orders(e) == b["v"].env.get_orders(e)
    assert not a["v"].env.env_errors().any()
    assert sum(len(a["v"].env.get_trades(e)) for e in range(n)) > 0
    a["v"].close(), b["v"].close()


def test_market_save_after_host_steps_refuses_capture():
    """On a multi-asset handle right after a host bb_step, save and restore first push the host's shuffle streams to the
    books; inside a stream capture that is refused."""
    import torch
    from bourse_b200 import market
    m = market.MarketEnv(0, 0, [1, 2], 1000, n_markets=2, max_orders=64, max_trades=64, max_steps=8, max_queue=16)
    env = m._env
    store, _ = env.store_create(2)
    units = torch.arange(2, dtype=torch.int32, device="cuda")
    m.submit([abi.ACT_NEW, abi.ACT_NEW], [0, 0], side=[True, False], vol=[1, 2], trader=[1, 1], price=[50, 50], market=[0, 0])
    m.step()
    s2 = torch.cuda.Stream()
    env.set_stream(s2.cuda_stream)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with pytest.raises(ValueError, match="bb_step"):
        with torch.cuda.graph(g, stream=s2):
            env.save_device(store, units.data_ptr())
    env.save_device(store, units.data_ptr())   # outside a capture it goes through
    env.restore_device(store, units.data_ptr())
    env.synchronize()
    assert not env.env_errors().any()
    env.store_destroy(store)
    env.close()


def test_warm_start_example():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "vector_env_warm_start_torch.py")], capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    assert "warm start" in out.stdout and "error_envs: 0" in out.stdout
