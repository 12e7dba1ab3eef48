"""GPU suite: Env steps on the deep-book engine (bb_step_device on a deep handle: k_env_deep_stage + k_deepw<.., ENV>, and
gym.VectorEnv(price_window=..., deep_chunks=...)).  Every env is compared bit for bit with an oracle StepEnv(seed + e, start,
tick, step_size) fed the same rows through place_order / cancel_order / modify_order and step: ids and observations at
every step, orders, trades, history and error bits at the end.  Deep books are preloaded by replaying a C5 stream into the
device book and, through the oracle's book replay, into the oracle env's book."""
import ctypes as C

import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import episode_reset_oracle as ers

pytestmark = pytest.mark.gpu

WINDOW = (2688, 3328)   # 640 levels around the C5 mid of 3000
MID = 3000
STEP = 1000
ERR_CAP_PAGES, ERR_CAP_QUEUE, ERR_BAD_ID, ERR_TIME_ORDER, ERR_PRICE = 0x4, 0x8, 0x10, 0x100, 0x200


def deep_vector(n_envs, rows, seed, tick=1, n_orders=4096, chunks=None, max_queue=None, step_size=STEP, trading=True, **kw):
    return gym.VectorEnv(n_envs, rows, seed, 0, tick, step_size, trading, max_orders=n_orders, max_trades=4 * n_orders, max_steps=256,
                         max_queue=max_queue or max(rows, 16), price_window=WINDOW,
                         deep_chunks=chunks or (n_orders // 8 + 2 * (WINDOW[1] - WINDOW[0]) + 64), **kw)


def oracle_replay(o, instrs):
    """Replay a packed stream into an oracle StepEnv's book (the device side: BatchedEnv.replay)."""
    from oracle import oracle as orc
    instrs = np.ascontiguousarray(instrs, dtype=abi.INSTR_DTYPE)
    obs = np.zeros((1, 45), np.uint32)
    err = C.c_uint64()
    n = orc.lib().orc_book_replay(C.c_void_p(o._book()), instrs.ctypes.data, len(instrs), obs.ctypes.data, 0, C.byref(err))
    assert n >= 0, (n, err.value)


def closed(s):
    """A replay stream without market-data records (the env's history holds step records only), closed by a no-op one
    nanosecond after its last event: the next Env step's first event runs at the book's time, which must come after every
    resting order's key time (the deep engine's precondition; equal keys would be the reference's N1 collision)."""
    s = s.copy()
    s["op_flags"] &= ~np.uint32(abi.F_EMIT)
    end = np.zeros(1, dtype=abi.INSTR_DTYPE)
    end["t"], end["op_flags"] = s["t"][-1] + np.uint64(1), abi.OP_NOOP
    return np.concatenate([s, end])


def c5_preload(n_resting, per_step, seed):
    """A C5 book as a replay stream (closed)."""
    return closed(workloads.c5_stream(n_resting, 1, per_step, seed=seed, mid_ticks=MID, depth_ticks=256))


def preload(v, orcs, streams):
    """Replay stream e into env e of the vector env and of its oracle."""
    v.env.replay(np.concatenate(streams), np.cumsum([0] + [len(s) for s in streams]).astype(np.uint64))
    for o, s in zip(orcs, streams):
        oracle_replay(o, s)


def random_rows(rng, n_envs, rows, issued, ticks, zero=None, mid=MID, spread=24, p_empty=0.05):
    """Random mixes: limit and market NEWs (some off the env's tick, some of volume 0 or over 192), CANCELs and MODIFYs
    (price only, volume only, both, neither) of ids among every id issued so far and those the slice itself creates, and
    no-ops; a few envs get an empty step.  `zero[e]`: the env's resting zero-volume orders.  A zero-volume order is never
    re-priced without volume: placed exactly on a level of the other side it would break the engine's "one side per
    level" precondition (flagged BB_ERR_LOCKED), which these mixes keep."""
    a = np.zeros((n_envs, rows), dtype=gym.ACTION_DTYPE)
    for e in range(n_envs):
        if rng.random() < p_empty:
            continue
        tick, nxt = int(ticks[e]), int(issued[e])
        for r in range(rows):
            u = rng.random()
            if u < 0.08:
                continue
            x = a[e, r]
            if u < 0.6 or nxt == 0:
                bid = rng.random() < 0.5
                of = abi.OP_NEW | (abi.F_BID if bid else 0)
                v = rng.random()
                x["vol"] = 0 if v < 0.03 else int(rng.integers(193, 400)) if v < 0.08 else int(rng.integers(1, 50))
                x["trader"] = int(rng.integers(0, 1000))
                # (a zero-volume limit order rests on its own side, beyond the crossing range: placed exactly on a level of the
                # other side it would be the engine's flagged "locked level" precondition)
                far = (spread + int(rng.integers(1, 8))) * (-1 if bid else 1) if v < 0.03 else None
                if far is None and rng.random() < 0.08:
                    of |= abi.F_MARKET
                    nxt += 1
                else:
                    off_tick = tick > 1 and rng.random() < 0.05
                    x["price"] = tick * (mid // tick + (far if far is not None else int(rng.integers(-spread, spread + 1)))) + (1 if off_tick else 0)
                    nxt += 0 if off_tick else 1
                x["op_flags"] = of
            else:
                x["op_flags"] = abi.OP_CANCEL if u < 0.8 else abi.OP_MODIFY
                if u >= 0.8:
                    k = int(rng.integers(0, 4))   # price only, volume only, both, neither
                    x["op_flags"] |= (abi.F_HAS_PRICE if k in (0, 2) else 0) | (abi.F_HAS_VOL if k in (1, 2) else 0)
                    x["price"] = tick * (mid // tick + int(rng.integers(-spread, spread + 1)))
                    x["vol"] = int(rng.integers(0 if k == 1 else 1, 60))   # (volume 0 only in place: a reduce)
        # targets: any id issued before, or (a third of them) an id this slice creates, before or after the row
        for r in range(rows):
            x = a[e, r]
            if int(x["op_flags"]) & 0xFF in (abi.OP_CANCEL, abi.OP_MODIFY):
                if nxt == 0:
                    x["op_flags"] = abi.OP_NOOP
                elif nxt > issued[e] and rng.random() < 0.35:
                    x["order_id"] = int(rng.integers(issued[e], nxt))
                else:
                    x["order_id"] = int(rng.integers(0, nxt))
        # orders that are, or may become, zero-volume in this step: price changes of them carry a volume
        z = set(zero[e]) if zero is not None else set()
        ids = issued[e] + np.cumsum([(int(x["op_flags"]) & 0xFF) == abi.OP_NEW and not (int(x["op_flags"]) & abi.F_MARKET)
                                      and (int(x["price"]) % int(ticks[e]) == 0) for x in a[e]]) - 1
        for r in range(rows):
            x = a[e, r]
            of = int(x["op_flags"])
            if of & 0xFF == abi.OP_NEW and not of & abi.F_MARKET and int(x["vol"]) == 0:
                z.add(int(ids[r]))
            if of & 0xFF == abi.OP_MODIFY and of & abi.F_HAS_VOL and not of & abi.F_HAS_PRICE and int(x["vol"]) == 0:
                z.add(int(x["order_id"]))
        for r in range(rows):
            x = a[e, r]
            of = int(x["op_flags"])
            if of & 0xFF == abi.OP_MODIFY and of & abi.F_HAS_PRICE and (not of & abi.F_HAS_VOL or int(x["vol"]) == 0) and int(x["order_id"]) in z:
                x["op_flags"] = of | abi.F_HAS_VOL
                x["vol"] = int(rng.integers(1, 60))
    return a


def oracle_step(o, rows):
    """One env's rows through the oracle env, then step: the ids and whether a row was off the tick."""
    ids = np.full(len(rows), abi.NO_ID, np.uint64)
    bad = False
    for r, x in enumerate(rows):
        of, k = int(x["op_flags"]), int(x["op_flags"]) & 0xFF
        if k == abi.OP_NEW:
            try:
                ids[r] = o.place_order(bool(of & abi.F_BID), int(x["vol"]), int(x["trader"]), None if of & abi.F_MARKET else int(x["price"]))
            except ValueError:
                bad = True
        elif k == abi.OP_CANCEL:
            o.cancel_order(int(x["order_id"]))
        elif k == abi.OP_MODIFY:
            o.modify_order(int(x["order_id"]), int(x["price"]) if of & abi.F_HAS_PRICE else None, int(x["vol"]) if of & abi.F_HAS_VOL else None)
    o.step()
    return ids, bad


def run_steps(v, orcs, rng, n_steps, ticks, check=None, reads=False):
    """Random steps on every env, each compared with its oracle; returns the envs flagged for off-tick rows."""
    n_envs, rows = v.n_envs, v.rows
    issued = np.array([len(o.get_orders()) for o in orcs], np.int64)
    flagged = np.zeros(n_envs, bool)
    seen = [list(o.get_trades()) for o in orcs]
    check = range(n_envs) if check is None else check
    for s in range(n_steps):
        zero = [[i for i, o in enumerate(orcs[e].get_orders()) if o[1] == 1 and o[4] == 0] for e in range(n_envs)]
        a = random_rows(rng, n_envs, rows, issued, ticks, zero)
        obs, ids = v.step(a)
        if reads:
            got = v.orders(ids)
            tcols, count = v.trades(512)
            st, vol, pr = (got[k].numpy() for k in ("status", "vol", "price"))
            tc = {k: c.numpy() for k, c in tcols.items()}
            cnt = count.numpy()
        obs, ids = obs.numpy(), ids.numpy()
        for e in range(n_envs):
            want, bad = oracle_step(orcs[e], a[e])
            flagged[e] |= bad
            issued[e] = len(orcs[e].get_orders())
            if e not in check:
                continue
            assert np.array_equal(ids[e], want), (s, e)
            assert np.array_equal(obs[e], orcs[e].level_2_data_array()), (s, e)
            if reads:
                table = orcs[e].get_orders()
                for r in range(rows):
                    if want[r] != abi.NO_ID:
                        o = table[int(want[r])]
                        assert (st[e, r], vol[e, r], pr[e, r]) == (o[1], o[4], o[6]), (s, e, r)
                n = min(int(cnt[e]), 512)
                seen[e] += [(int(tc["t"][e, i]), bool(tc["side_is_bid"][e, i]), int(tc["price"][e, i]), int(tc["vol"][e, i]),
                             int(tc["active_id"][e, i]), int(tc["passive_id"][e, i])) for i in range(n)]
                assert int(cnt[e]) <= 512 and seen[e] == orcs[e].get_trades(), (s, e)
    return flagged


def assert_envs_equal(v, orcs, envs):
    for e in envs:
        assert v.env.get_orders(e) == orcs[e].get_orders(), e
        assert v.env.get_trades(e) == orcs[e].get_trades(), e
        assert np.array_equal(v.env.history(e), orcs[e]._history()), e


@pytest.mark.parametrize("n_envs,n_steps,rows", [(4, 40, 24), (300, 5, 8)], ids=["roomy", "compact"])
def test_random_mixes_match_the_oracle(oracle, n_envs, n_steps, rows):
    """Fresh deep books, per-env ticks 1, 2, 3, random mixes over many steps (the roomy instantiation with 1-2 books per SM,
    the compact one with 300 books); order and trade reads on the device after every step of the roomy case."""
    seed = 31
    ticks = [1 + e % 3 for e in range(n_envs)]
    rng = np.random.default_rng(n_envs)
    v = deep_vector(n_envs, rows, seed, tick=ticks)
    orcs = [oracle.StepEnv(seed + e, 0, ticks[e], STEP) for e in range(n_envs)]
    obs0 = v.reset().numpy()
    assert np.array_equal(obs0[0], orcs[0].level_2_data_array())
    flagged = run_steps(v, orcs, rng, n_steps, ticks, reads=n_envs < 10)
    assert_envs_equal(v, orcs, range(n_envs) if n_envs < 10 else range(0, n_envs, 7))
    err = v.env.env_errors()
    assert np.array_equal(err, np.where(flagged, ERR_PRICE, 0).astype(np.uint32))
    assert flagged.any() and sum(len(o.get_trades()) for o in orcs) > 5 * n_envs
    v.close()


@pytest.mark.parametrize("n_envs", [2, 300], ids=["roomy", "compact"])
def test_deep_books_replay_steps_replay(oracle, n_envs):
    """Books preloaded with a C5 stream (thousands of resting orders), Env steps on them, a replayed stream continuing at
    the envs' time, and Env steps again: every env equals its oracle env driven the same way."""
    seed, rows = 4, 16
    n_rest = 4000 if n_envs < 10 else 600
    n_orders = n_rest + 4000
    ticks = [1] * n_envs
    v = deep_vector(n_envs, rows, seed, n_orders=n_orders)
    v.reset()
    orcs = [oracle.StepEnv(seed + e, 0, 1, STEP) for e in range(n_envs)]
    preload(v, orcs, [c5_preload(n_rest, 200, 50 + e) for e in range(n_envs)])
    t_pre = orcs[0].time
    rng = np.random.default_rng(7)
    check = range(n_envs) if n_envs < 10 else range(0, n_envs, 13)
    run_steps(v, orcs, rng, 12 if n_envs < 10 else 3, ticks, check=check)
    t = orcs[0].time
    assert t == t_pre + (12 if n_envs < 10 else 3) * STEP
    more = []
    for e in range(n_envs):   # a continuation: new orders, cancels and modifies of ids the steps issued too
        s = workloads.c5_stream(0, 1, 300, seed=90 + e, mid_ticks=MID)
        s["t"] += np.uint64(orcs[e].time + 1)
        new = (s["op_flags"] & 0xFF) == abi.OP_NEW
        s["order_id"] = np.where(new, 0, s["order_id"] % np.uint32(len(orcs[e].get_orders())))
        more.append(closed(s))
    preload(v, orcs, more)
    run_steps(v, orcs, rng, 6 if n_envs < 10 else 2, ticks, check=check)
    assert_envs_equal(v, orcs, check)
    assert not v.env.env_errors().any(), v.env.env_errors()
    assert min(len(orcs[e].get_trades()) for e in check) > 20
    v.close()


def test_same_step_edges(oracle):
    """Per env, across many steps (so the shuffle puts them both ways round): a CANCEL and a MODIFY of orders the same
    slice creates, rows naming ids the slice creates later, zero-volume orders, volumes over 192 (serial path) and empty
    steps; plus envs whose rows break a rule: a bad id, an off-tick price at ticks 2 and 3, a limit price outside the
    window.  Each rule-breaking env is flagged as the engine flags replayed streams; every other env stays exact."""
    seed, n_envs, rows, n_steps = 3, 6, 8, 30
    ticks = [1, 1, 1, 2, 3, 1]
    v = deep_vector(n_envs, rows, seed, tick=ticks)
    v.reset()
    orcs = [oracle.StepEnv(seed + e, 0, ticks[e], STEP) for e in range(n_envs)]
    rng = np.random.default_rng(3)
    flagged = np.zeros(n_envs, bool)
    for s in range(n_steps):
        a = np.zeros((n_envs, rows), dtype=gym.ACTION_DTYPE)
        for e in range(n_envs):
            n0 = len(orcs[e].get_orders())
            if s % 7 == 6:
                continue   # an empty step
            t = ticks[e]
            # rows 0-1: two NEWs; row 2 cancels the first, row 3 modifies the second; row 4 cancels the NEW of row 5
            bid = bool(s % 2)
            for r, (vol, off) in enumerate([(int(rng.integers(1, 30)), 2), (int(rng.integers(0, 3)), 3)]):
                a[e, r] = (0, abi.OP_NEW | (abi.F_BID if bid else 0), 0, t * (MID // t + (-off if bid else off)), vol, 9, 0)
            a[e, 2] = (0, abi.OP_CANCEL, n0, 0, 0, 0, 0)
            a[e, 3] = (0, abi.OP_MODIFY | abi.F_HAS_VOL | (abi.F_HAS_PRICE if s % 3 == 0 else 0), n0 + 1, t * (MID // t + 1), int(rng.integers(1, 9)), 0, 0)
            a[e, 4] = (0, abi.OP_CANCEL, n0 + 2, 0, 0, 0, 0)
            a[e, 5] = (0, abi.OP_NEW | (0 if bid else abi.F_BID), 0, t * (MID // t), int(rng.integers(150, 260)), 4, 0)
            # rows 6-7: an aggressive order over 192 that sweeps the other side, and a no-op
            a[e, 6] = (0, abi.OP_NEW | abi.F_MARKET | (0 if bid else abi.F_BID), 0, 0, int(rng.integers(193, 300)), 5, 0)
            if e == 2 and s == 10:
                a[e, 7] = (0, abi.OP_CANCEL, n0 + 50, 0, 0, 0, 0)         # an id beyond the post-submission count
            if e in (3, 4) and s == 12:
                a[e, 7] = (0, abi.OP_NEW, 0, t * (MID // t) + 1, 5, 0, 0)  # off the env's tick
            if e == 5 and s == 14:
                a[e, 7] = (0, abi.OP_NEW, 0, WINDOW[1] + 40, 5, 0, 0)      # rests outside the window
        obs, ids = v.step(a)
        obs, ids = obs.numpy(), ids.numpy()
        for e in range(n_envs):
            if (e == 2 and s >= 10) or (e == 5 and s >= 14):
                continue   # the reference panics on a bad id; an order outside the window cannot rest on this book
            want, bad = oracle_step(orcs[e], a[e])
            flagged[e] |= bad
            assert np.array_equal(ids[e], want), (s, e)
            assert np.array_equal(obs[e], orcs[e].level_2_data_array()), (s, e)
    assert_envs_equal(v, orcs, [0, 1, 3, 4])
    err = v.env.env_errors()
    assert list(err) == [0, 0, ERR_BAD_ID, ERR_PRICE, ERR_PRICE, ERR_CAP_PAGES], [hex(x) for x in err]
    assert list(flagged) == [False, False, False, True, True, False]
    assert min(len(orcs[e].get_trades()) for e in (0, 1, 3, 4)) > 20
    v.close()


def test_queue_capacity_trading_off_and_time_order(oracle):
    """Ragged slices through core.BatchedEnv.step_device: a slice over max_queue runs its first max_queue rows and flags
    BB_ERR_CAP_QUEUE; trading switched off (limit orders rest, market orders are rejected); and step_size < max_queue,
    where resting orders of one step can share key times with the next one's: the engine flags BB_ERR_TIME_ORDER there."""
    import torch
    seed, mq = 8, 16
    for trading, step_size in ((True, STEP), (False, STEP), (True, 4)):
        n_envs = 3
        env = core.BatchedEnv(n_envs, seed, 0, 1, step_size, trading, max_orders=2048, max_trades=4096, max_steps=64, max_queue=mq,
                              price_window=WINDOW, deep_chunks=2048)
        orcs = [oracle.StepEnv(seed + e, 0, 1, step_size, trading) for e in range(n_envs)]
        rng = np.random.default_rng(int(trading) + step_size)
        lens = [mq + 5, mq, 3]
        d_ids = torch.zeros(sum(lens), dtype=torch.int64, device="cuda")
        d_obs = torch.zeros((n_envs, 45), dtype=torch.int32, device="cuda")
        offs = torch.from_numpy(np.cumsum([0] + lens).astype(np.int64)).cuda()
        for s in range(12):
            blocks = []
            for e in range(n_envs):
                blk = np.zeros(lens[e], dtype=abi.INSTR_DTYPE)
                for r in range(lens[e]):
                    bid = rng.random() < 0.5
                    mkt = trading and rng.random() < 0.1 or (not trading and r == 0)
                    price = MID + (-1 if bid else 1) * int(rng.integers(1, 4 if step_size < mq else 20)) * (1 if trading else 2)
                    blk[r] = (0, abi.OP_NEW | (abi.F_BID if bid else 0) | (abi.F_MARKET if mkt else 0), 0, 0 if mkt else price,
                              int(rng.integers(1, 30)), 1, 0)
                blocks.append(blk)
            d_rows = torch.from_numpy(np.concatenate(blocks).view(np.uint8)).cuda()
            torch.cuda.synchronize()
            env.step_device(d_rows.data_ptr(), offs.data_ptr(), sum(lens), d_ids.data_ptr(), d_obs.data_ptr())
            env.synchronize()
            ids = d_ids.cpu().numpy().view(np.uint64)
            obs = d_obs.cpu().numpy().view(np.uint32)
            for e in range(n_envs):
                want, _ = oracle_step(orcs[e], blocks[e][:mq])
                got = ids[sum(lens[:e]):sum(lens[:e + 1])]
                assert np.array_equal(got[:mq], want[:mq]) and (got[mq:] == abi.NO_ID).all(), (trading, step_size, s, e)
                if step_size >= mq:
                    assert np.array_equal(obs[e], orcs[e].level_2_data_array()), (trading, s, e)
        err = env.env_errors()
        if step_size >= mq:
            assert list(err) == [ERR_CAP_QUEUE, 0, 0], [hex(x) for x in err]
            for e in range(n_envs):
                assert env.get_orders(e) == orcs[e].get_orders() and env.get_trades(e) == orcs[e].get_trades(), e
                assert np.array_equal(env.history(e), orcs[e]._history()), e
            if not trading:
                assert not any(orcs[e].get_trades() for e in range(n_envs))
        else:
            # 16 events a step, 4 ns apart: the full envs rest orders at keys an earlier step already used
            assert err[0] & ERR_TIME_ORDER and err[1] & ERR_TIME_ORDER and not err[2] & ERR_TIME_ORDER, [hex(x) for x in err]
        env.close()


def test_reset_save_restore_and_reads(oracle):
    """One preloaded deep book saved into a slot and restored into every env, without and with seeds, then stepped; a
    masked reset with seeds mid-run equals a fresh oracle env with that seed; orders() / trades() equal the host reads."""
    seed, n_envs, rows = 12, 8, 12
    v = deep_vector(n_envs, rows, seed, n_orders=8000)
    v.reset()
    src = [oracle.StepEnv(seed, 0, 1, STEP)]
    stream = c5_preload(3000, 300, 61)
    v.env.replay(stream, np.array([0] + [len(stream)] * n_envs, np.uint64))   # env 0 only
    oracle_replay(src[0], stream)
    store = v.snapshots(1)
    v.save(store, np.array([0], np.uint32))
    for seeds in (None, np.arange(100, 100 + n_envs, dtype=np.uint64)):
        out = v.restore(store, np.zeros(n_envs, np.uint32), seeds).numpy()
        orcs = []
        for e in range(n_envs):
            o = oracle.StepEnv(seed if seeds is None else int(seeds[e]), 0, 1, STEP)
            oracle_replay(o, stream)
            orcs.append(o)
            assert v.env.get_orders(e) == o.get_orders(), e
        assert (out[:, 1:] == out[0, 1:]).all()
        rng = np.random.default_rng(5 if seeds is None else 6)
        run_steps(v, orcs, rng, 8, [1] * n_envs, reads=True)
        mask = np.arange(n_envs) % 3 == 1
        rs = np.arange(7, 7 + n_envs, dtype=np.uint64)
        v.reset(mask, rs)
        for e in np.flatnonzero(mask):
            ers.sim_reset(orcs[e], 0, seed=int(rs[e]))
        run_steps(v, orcs, rng, 6, [1] * n_envs, reads=True)
        assert_envs_equal(v, orcs, range(n_envs))
    assert not v.env.env_errors().any()
    v.close()


def test_step_inside_a_cuda_graph(oracle):
    """{policy; step} on deep books captured once and replayed K times equals the same loop run eagerly on a twin, and both
    equal the oracle."""
    import torch
    n_envs, rows, k, seed = 24, 4, 12, 2
    twins = []
    for _ in range(2):
        v = deep_vector(n_envs, rows, seed, n_orders=6000)
        v.reset()
        st = torch.cuda.Stream()
        v.env.set_stream(st.cuda_stream)
        twins.append((v, st))
    orcs = [oracle.StepEnv(seed + e, 0, 1, STEP) for e in range(n_envs)]
    streams = [c5_preload(1500, 200, 70 + e) for e in range(n_envs)]
    for v, _ in twins:
        v.env.replay(np.concatenate(streams), np.cumsum([0] + [len(s) for s in streams]).astype(np.uint64))
    for o, s in zip(orcs, streams):
        oracle_replay(o, s)
    acts = [torch.zeros((n_envs, rows, 8), dtype=torch.int32, device="cuda") for _ in twins]
    obs_t = [torch.as_tensor(v.obs, device="cuda") for v, _ in twins]
    for v, _ in twins:
        v._observe()
    torch.cuda.synchronize()

    def policy(i):   # rows from the last observation: limit orders around the touch, a cancel of an early id
        ob = obs_t[i].to(torch.int64)
        e = torch.arange(n_envs, device="cuda").unsqueeze(1)
        r = torch.arange(rows, device="cuda").unsqueeze(0)
        a = acts[i]
        bid = (e + r + ob[:, :1]) % 2
        a[:, :, 2] = (torch.where(r == rows - 1, abi.OP_CANCEL, abi.OP_NEW + bid * abi.F_BID)).to(torch.int32)
        a[:, :, 3] = ((ob[:, 3:4] + 7 * e + r) % 1000).to(torch.int32)
        a[:, :, 4] = (MID - 20 + (ob[:, 4:5] + 5 * r + e) % 41).to(torch.int32)
        a[:, :, 5] = (1 + (ob[:, :1] + r) % 60).to(torch.int32)
        a[:, :, 6] = 3

    v, st = twins[0]
    with torch.cuda.stream(st):
        policy(0)
        v.step(acts[0])   # warm-up outside the capture
    st.synchronize()
    blocks = [acts[0].cpu().numpy().copy()]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        policy(0)
        v.step(acts[0])
    for _ in range(k):
        g.replay()
        torch.cuda.synchronize()
        blocks.append(acts[0].cpu().numpy().copy())
    w, sw = twins[1]
    for _ in range(k + 1):
        with torch.cuda.stream(sw):
            policy(1)
            w.step(acts[1])
        sw.synchronize()
    assert np.array_equal(v.obs.numpy(), w.obs.numpy()) and np.array_equal(v.ids.numpy(), w.ids.numpy())
    for blk in blocks:
        rows_np = blk.reshape(n_envs, rows * 8).view(np.uint32).copy().view(gym.ACTION_DTYPE).reshape(n_envs, rows)
        for e in range(n_envs):
            oracle_step(orcs[e], rows_np[e])
    for e in range(n_envs):
        assert np.array_equal(v.obs.numpy()[e], orcs[e].level_2_data_array()), e
        for x in (v, w):
            assert x.env.get_orders(e) == orcs[e].get_orders() and x.env.get_trades(e) == orcs[e].get_trades(), e
            assert np.array_equal(x.env.history(e), orcs[e]._history()), e
    assert not v.env.env_errors().any() and not w.env.env_errors().any()
    assert sum(len(o.get_trades()) for o in orcs) > 1000
    v.close(), w.close()


def test_refusals():
    with pytest.raises(ValueError, match="deep-book engine"):
        gym.VectorEnv(4, 2, 0, 0, 1, STEP, agents=workloads.c3_groups(), price_window=WINDOW, deep_chunks=1024)
    env = core.BatchedEnv(2, 0, 0, 1, STEP, max_orders=64, max_trades=64, max_steps=8, max_queue=16, price_window=WINDOW, deep_chunks=256)
    with pytest.raises(ValueError, match="no host-queued Env steps"):
        env.step()   # the host-queued Env path stays refused
    env.reserve_queue(40)   # regrows the staging stream: a slice of 40 rows then runs whole
    rows = np.zeros(80, dtype=abi.INSTR_DTYPE)
    rows["op_flags"], rows["price"], rows["vol"] = abi.OP_NEW | abi.F_BID, MID - 5, 1
    import torch
    d_rows = torch.from_numpy(rows.view(np.uint8)).cuda()
    offs = torch.tensor([0, 40, 80], dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    env.step_device(d_rows.data_ptr(), offs.data_ptr(), 80)
    env.synchronize()
    assert [env.n_orders(e) for e in range(2)] == [40, 40] and not env.env_errors().any()
    env.close()
