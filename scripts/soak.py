"""Randomised soak of the CUDA paths against the oracle: every round draws an engine (deep books included for the
single-asset and external-row rounds), a population (single-asset, market twins, or background agents + external rows), sizes and a launch split, runs it on the GPU and compares a sample of books
bit for bit (level-2 history, trade log, order table).  python scripts/soak.py <seconds> [first_seed]"""
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from bourse_b200 import abi, core, gym, market  # noqa: E402
from oracle import oracle as orc  # noqa: E402

sys.path.insert(0, "tests")
from bourse_b200 import workloads  # noqa: E402
from tests.test_oracle_hypothesis import random_adversarial_stream  # noqa: E402

MODES = ["single", "market", "ext", "replay", "replay"]
budget, seed0 = float(sys.argv[1]), int(sys.argv[2]) if len(sys.argv) > 2 else 0
only = [int(x) for x in sys.argv[3:]]   # optional: just these seeds
t_end = time.time() + budget


def rand_groups(rng, dense):
    gs = []
    for _ in range(int(rng.integers(1, 4))):
        lo = int(rng.integers(20, 60)); hi = lo + int(rng.integers(2, 40))
        gs.append(("r", (int(rng.integers(5, 60)), (lo, hi), (int(rng.integers(1, 30)), int(rng.integers(30, 80))), 2, float(rng.uniform(0.1, 1.0)))))
    if not dense and rng.random() < 0.6:
        gs.append(("m", (1000, int(rng.integers(2, 24)), 1, float(rng.uniform(0.0, 0.5)), int(rng.integers(1, 20)), float(rng.uniform(0.2, 1.0)),
                         float(rng.uniform(1, 8)), float(rng.uniform(0.1, 1.0)), float(rng.uniform(0.0, 2.0)), 0.0, float(rng.uniform(0.3, 1.5)))))
    if not dense and rng.random() < 0.4:
        gs.append(("n", (2000, int(rng.integers(2, 16)), 1, float(rng.uniform(0, 0.5)), float(rng.uniform(0, 0.3)), float(rng.uniform(0, 0.5)),
                         int(rng.integers(1, 20)), float(rng.uniform(-0.5, 1.0)), float(rng.uniform(0.3, 1.2)))))
    order = rng.permutation(len(gs))
    return [gs[i] for i in order]


def build(mod, gs):
    f = {"r": mod.random_group, "m": mod.momentum_group, "n": mod.noise_group}
    return [f[k](*a) for k, a in gs]


rounds = fails = capacity = 0
seed = seed0
while time.time() < t_end and (not only or rounds < len(only)):
    if only:
        seed = only[rounds]
    rng = np.random.default_rng(seed)
    last_env = None
    mode = MODES[int(rng.integers(len(MODES)))]
    if mode == "replay":
        # immediate-mode streams (k_apply<REPLAY>) on every book geometry: C2-style streams with strict / flat / jittered
        # time (equal-key collisions N1, backwards time) or the adversarial tiny-domain streams of the hypothesis tests
        rounds += 1
        seed += 1
        geo = int(rng.integers(5))
        tick = int(rng.integers(1, 3))
        adversarial = rng.random() < 0.5
        n_books = int(rng.integers(1, 40))
        if adversarial:
            streams = [random_adversarial_stream(rng, int(rng.integers(1, 150)), tick) for _ in range(n_books)]
            kwr = [dict(pages_smem=8, pages_total=32), dict(pages_smem=32, pages_total=32), dict(pages_smem=64, pages_total=64),
                   dict(pages_smem=3, pages_total=96), dict(pages_smem=40, pages_total=40)][geo]
            kwr["price_granule"] = 1
        else:
            tm = ["strict", "flat", "jitter"][int(rng.integers(3))]
            hw = int(rng.integers(8, 400))
            dense_ok = tm == "strict" and hw <= 100
            streams = [workloads.replay_stream(int(rng.integers(200, 3000)), int(rng.integers(1 << 30)), tick_size=tick, half_width=hw,
                                               time_mode=tm, min_vol=int(rng.integers(0, 2))) for _ in range(n_books)]
            kwr = [dict(pages_smem=4, pages_total=128), dict(pages_smem=64, pages_total=64), dict(pages_smem=100, pages_total=100),
                   dict(pages_smem=16, pages_total=256),
                   dict(price_window=((1000 - hw) * tick - 8, (1000 + hw) * tick + 8), live_cap=254) if dense_ok else dict(pages_smem=200, pages_total=200)][geo]
        desc = f"seed {seed - 1} replay {'adversarial' if adversarial else 'c2-style'} tick {tick} {kwr} books {n_books}"
        try:
            off = np.zeros(n_books + 1, np.uint64); off[1:] = np.cumsum([len(x) for x in streams])
            n_max = int(max(len(x) for x in streams))
            e = core.BatchedEnv(n_books, 0, 0, tick, 1000, obs_words=abi.OBS_L2, max_orders=n_max + 8, max_trades=4 * n_max + 64,
                                max_steps=n_max + 8, max_queue=16, **kwr)
            last_env = e
            try:
                e.replay(np.concatenate(streams), off)
            except MemoryError:
                pass          # a flagged capacity (dense window slots, pages): checked per book below
            err = e.env_errors()
            for b in range(n_books):
                if err[b]:
                    assert not (int(err[b]) & ~0x1CF), hex(int(err[b]))
                    continue
                ob = orc.OrderBook(0, tick); obs = ob.replay(streams[b], obs_cap=len(streams[b]))
                assert np.array_equal(e.history(b), obs) and e.get_orders(b) == ob.get_orders() and e.get_trades(b) == ob.get_trades(), b
            if err.any():
                capacity += 1
        except Exception as ex:  # noqa: BLE001
            fails += 1
            print("FAIL", desc, "->", repr(ex)[:200], flush=True)
        continue
    dense = rng.random() < 0.4
    kw = dict(price_window=(0, 256), live_cap=254) if dense else (dict() if rng.random() < 0.6 else dict(pages_smem=int(rng.integers(2, 12)), pages_total=64))
    gs = rand_groups(rng, dense)
    if mode != "market" and rng.random() < 0.25:
        # the deep-book engine: C3 centred inside its window (every RandomAgents price must rest there), the rows' prices too
        dense, kw = False, dict(price_window=(0, 256), deep_chunks=16384 // 8 + 2 * 256 + 64)
        gs = [("r", (int(g["n_agents"]), (int(g["tick_lo"]), int(g["tick_hi"])), (int(g["vol_lo"]), int(g["vol_hi"])), int(g["tick_size"]),
                     float(g["rate"]))) for g in workloads.c3_groups_around(100)]
    n_steps = int(rng.integers(5, 60)); split = int(rng.integers(1, n_steps + 1)); rs = int(rng.integers(1 << 30))
    desc = f"seed {seed} {mode} {'dense' if dense else kw} groups {[k for k, _ in gs]} steps {n_steps}/{split}"
    try:
        if mode == "single":
            n_envs = int(rng.integers(1, 200))
            e = core.BatchedEnv(n_envs, 0, 0, 1, 1_000_000, obs_words=abi.OBS_L2, max_orders=16384, max_trades=32768, max_steps=64, max_queue=512, **kw)
            last_env = e
            e.set_agents(build(core, gs)); e.run_agents(split, rs); e.run_agents(n_steps - split, rs) if n_steps > split else None
            assert not e.env_errors().any(), "env errors"
            for env_id in sorted(set(int(x) for x in rng.integers(0, n_envs, 4))):
                o = orc.StepEnvNumpy(0, 0, 1, 1_000_000); o.set_groups(build(orc, gs)); o.run_agents(n_steps, rs, env_id=env_id, keyed=True)
                assert np.array_equal(e.history(env_id), o._history()) and e.get_trades(env_id) == o.get_trades() and e.get_orders(env_id) == o.get_orders(), env_id
        elif mode == "market":
            A = int(rng.integers(2, 5)); n_m = int(rng.integers(1, 60)); assets = [int(rng.integers(A)) for _ in gs]
            e = core.BatchedEnv(n_m * A, 0, 0, 1, 1_000_000, obs_words=abi.OBS_L2, max_orders=16384, max_trades=32768, max_steps=64, max_queue=512, assets=A, **kw)
            last_env = e
            e.set_agents(build(core, gs), assets=assets); e.run_agents(split, rs); e.run_agents(n_steps - split, rs) if n_steps > split else None
            assert not e.env_errors().any(), "env errors"
            for m in sorted(set(int(x) for x in rng.integers(0, n_m, 3))):
                o = orc.MarketEnv(0, 0, [1] * A, 1_000_000); o.set_groups(build(orc, gs), assets); o.run_agents(n_steps, rs, market_id=m, keyed=True)
                for a in range(A):
                    assert np.array_equal(e.history(m * A + a), o.history(a)) and e.get_trades(m * A + a) == o.get_trades(a) and e.get_orders(m * A + a) == o.get_orders(a), (m, a)
        else:
            n_envs = int(rng.integers(1, 64)); rows = int(rng.integers(1, 71))  # up to 70: rounds cross the 32-row passes of submit_rows
            v = gym.VectorEnv(n_envs, rows, 0, 0, 1, 1_000_000, agents=build(core, gs), agent_seed=rs, max_orders=16384, max_trades=32768, max_steps=64, max_queue=512, **kw)
            last_env = v.env
            os_ = [orc.StepEnv(0, 0, 1, 1_000_000) for _ in range(n_envs)]
            [o.set_groups(build(orc, gs)) for o in os_]
            v.reset(); mine = [[] for _ in range(n_envs)]
            for s in range(min(n_steps, 25)):
                u = rng.random((n_envs, rows))
                op = np.where(u < 0.6, abi.OP_NEW, np.where(u < 0.85, abi.OP_CANCEL, abi.OP_NOOP)).astype(np.uint32)
                oid = np.zeros((n_envs, rows), np.uint64)
                for en in range(n_envs):
                    for r in range(rows):
                        if op[en, r] == abi.OP_CANCEL:
                            if mine[en]: oid[en, r] = mine[en][int(rng.integers(len(mine[en])))]
                            else: op[en, r] = abi.OP_NOOP
                bid = rng.random((n_envs, rows)) < 0.5; vol = rng.integers(1, 40, (n_envs, rows)); mk = rng.random((n_envs, rows)) < 0.1
                price = 2 * rng.integers(20, 90, (n_envs, rows))
                obs, ids = v.step(gym.pack_actions(op, bid=bid, vol=vol, trader=77, price=price, order_id=oid, market=mk))
                obs, ids = obs.numpy(), ids.numpy()
                for en, o in enumerate(os_):
                    o.agents_update(rs, en)
                    for r in range(rows):
                        if op[en, r] == abi.OP_NEW:
                            i = o.place_order(bool(bid[en, r]), int(vol[en, r]), 77, None if mk[en, r] else int(price[en, r])); mine[en].append(i)
                            assert ids[en, r] == i
                        elif op[en, r] == abi.OP_CANCEL: o.cancel_order(int(oid[en, r]))
                    o.step_keyed(rs, en)
                    assert np.array_equal(obs[en], o.level_2_data_array()), (s, en)
            v.check_errors()
            for en in range(0, n_envs, 7):
                assert v.env.get_trades(en) == os_[en].get_trades() and v.env.get_orders(en) == os_[en].get_orders()
            v.close()
    except Exception as ex:  # noqa: BLE001
        bits = 0
        try:
            bits = int(np.bitwise_or.reduce(last_env.env_errors())) if last_env is not None else 0
        except Exception:  # noqa: BLE001
            pass
        # a flagged capacity limit (price pages / window 0x4, resting-order slots 0x80, queue 0x8, ...) is the documented
        # behaviour for a population that outgrows the configured book, not a parity failure
        if bits and not (bits & ~0x1CF):
            capacity += 1
        else:
            fails += 1
            print("FAIL", desc, "error bits 0x%x" % bits, "->", repr(ex)[:200], flush=True)
    rounds += 1
    seed += 1
print(f"soak: {rounds} rounds, {fails} parity failures, {capacity} rounds stopped by a flagged capacity limit, seeds {seed0}..{seed - 1}")
