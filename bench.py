#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: lockstep order-book matching + Env step + in-kernel
agents + observation emission.

Workload (config C3 of BASELINE.json / SURVEY.md 8d, per GPU): 4096 envs x (50+50) RandomAgents
(crates/step_sim/examples/random_agents/main.rs:10-19) x 1000 env-steps, level-1 observation per
env-step, Env(0, tick 1, step 1_000_000).  One bench "step" = one full pass of that workload
(reset + 1000 env-steps for every env).  Weak scaling: every rank runs its own 4096 envs, keyed by
global env id; no per-step collective, one NCCL all-gather of the statistics at the end.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # + the last timed pass's outputs, DIR/*.npy
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference        # the reference's CPU algorithm (oracle) on the host cores
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "orders_per_sec"
UNIT = "orders/s"
N_ENVS_PER_GPU = 4096
N_SIM_STEPS = 1000
SEED = 101


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx, self.proc, self.lines = device_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, m in zip(sm, mx) if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(n_envs: int, n_steps: int, threads: int) -> dict:
    """The reference's algorithm on the host cores: C++ oracle, one env per core at a time, reference-style
    shared Xoroshiro stream per env (crates/step_sim/src/runner.rs:46-69).  kind "port": the Rust
    reference cannot be built in this image (no cargo/rustc)."""
    from bourse_b200 import workloads
    from oracle import oracle as orc

    orc.build()
    r = orc.bench_agents(n_envs, threads, n_steps, SEED, workloads.c3_groups(), keyed=False, start_time=0, tick_size=1,
                         step_size=1_000_000)
    return {"value": r["instructions"] / r["seconds"], "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_envs} envs x {n_steps} env-steps of the C3 workload ({r['instructions']} instructions, "
                      f"{r['seconds']:.2f} s wall), oracle/ C++ restatement, reference-style Xoroshiro stream per env",
            "env_steps_per_sec": r["env_steps"] / r["seconds"], "seconds": r["seconds"], "instructions": r["instructions"]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = host_cores()
    vals, secs = [], []
    for i in range(args.warmup + args.steps):
        r = cpu_baseline(N_ENVS_PER_GPU, N_SIM_STEPS, cores)   # the arm's whole config: all 4096 envs x 1000 env-steps per step
        if i >= args.warmup:
            vals.append(r)
            secs.append(r["seconds"])
    tot_i = sum(r["instructions"] for r in vals)
    tot_s = sum(secs)
    v = tot_i / tot_s
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        # the SAME config object as the b200 arm prints (the driver compares them); what a reference step is goes below
        "config": workload_config(args.gpus),
        "note": f"each step = all {N_ENVS_PER_GPU} envs x {N_SIM_STEPS} env-steps of one GPU's shard, on the host cores; the CPU arm is the "
                "oracle's C++ restatement (std::map where the reference uses BTreeMap), not the Rust build",
        "env_steps_per_sec": sum(r["env_steps_per_sec"] * r["seconds"] for r in vals) / tot_s,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": vals[-1]["sample"]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


DUMP_HISTORY_BYTES = 8 << 20   # per workload; with the row caps below, c3 + c4 + c5 stay under 64 MB in all
DUMP_LOG_ENVS, DUMP_LOG_ROWS = 2, 32768
TRADE_COLS = ("t", "side", "price", "vol", "active", "passive")
ORDER_COLS = ("side", "status", "arr_time", "end_time", "vol", "start_vol", "price", "trader")


def dump_outputs(env, out_dir: str, prefix: str):
    """Writes what a caller of the timed path holds after its last pass, for a fixed (seed 0) sample of the envs, as
    float64 .npy files (every field is an integer below 2**53, so float64 holds it exactly):
      <prefix>_envs      sampled env indices (local to this rank)
      <prefix>_history   [env, step, word] observation history of the sampled envs
      <prefix>_trades    [row] env, trade index, then t, side, price, vol, active id, passive id  (first DUMP_LOG_ENVS envs)
      <prefix>_orders    [row] env, order id, then side, status, arr_time, end_time, vol, start_vol, price, trader  (same envs)
    Trade and order tables longer than DUMP_LOG_ROWS are sampled (seed 0) to that many rows."""
    rng = np.random.default_rng(0)
    row_bytes = max(1, env.n_steps(0)) * env.obs_words * 8
    envs = np.sort(rng.choice(env.n_envs, min(env.n_envs, 256, max(1, DUMP_HISTORY_BYTES // row_bytes)), replace=False))
    out = {"envs": envs, "history": np.stack([env.history(int(e)) for e in envs])}
    for name, cols, read in (("trades", TRADE_COLS, env.trades_arrays), ("orders", ORDER_COLS, env.orders_arrays)):
        rows = []
        for e in envs[:DUMP_LOG_ENVS]:
            c = read(int(e))
            n = len(c[cols[0]])
            idx = np.arange(n) if n <= DUMP_LOG_ROWS else np.sort(rng.choice(n, DUMP_LOG_ROWS, replace=False))
            rows.append(np.stack([np.full(len(idx), e), idx] + [c[k][idx] for k in cols], axis=1).astype(np.float64))
        out[name] = np.concatenate(rows)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{prefix}_{name}.npy"), np.asarray(a, dtype=np.float64))


def workload_config(n_gpus: int, sample: str | None = None) -> dict:
    c = {"workload": "C3: 4096 envs/GPU x (50+50) RandomAgents x 1000 env-steps, level-1 obs per env-step, "
                     "Env(start 0, tick 1, step 1_000_000), agents tick_size 2 (crates/step_sim/examples/random_agents/main.rs)",
         "n_envs_per_gpu": N_ENVS_PER_GPU, "n_envs_total": N_ENVS_PER_GPU * n_gpus, "env_steps_per_bench_step": N_SIM_STEPS,
         "agents_per_env": 100, "obs": "level-1 (9 x u32) per env-step", "seed": SEED,
         "parallelism": f"envs sharded over {n_gpus} GPU(s), no per-step collective",
         "l2_policy": "working set (order + history slabs, ~7 GB touched per pass) far exceeds the 126 MB L2; "
                      "a 512 MB buffer is also written between timed passes"}
    if sample:
        c["sample"] = sample
    return c


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from bourse_b200 import abi, core, workloads

    # A dedicated (non-default) torch stream: the library launches on exactly this stream, so the CUDA events below
    # are recorded on the stream the kernels run on.  (Passing the default stream's handle, 0, would make the library
    # fall back to its own non-blocking stream, which events on the legacy default stream do not order against.)
    ctx = Ctx()
    rank, world, local, stream, flush, barrier = ctx.rank, ctx.world, ctx.local, ctx.stream, ctx.flush, ctx.barrier
    n_envs = args.envs
    groups = workloads.c3_groups()
    from bourse_b200.sharding import shard_range
    env_base, n_envs = shard_range(args.envs * world, world, rank)   # weak scaling: args.envs per GPU
    # engine: "dense" = dense tick-indexed ladder + shared-memory order slots (csrc/dense.cuh): C3's resting prices lie
    # in [20, 180) (ticks 10..89 x tick_size 2) and at most 100 orders rest per book (one per RandomAgent), inside the engine's window / slot limits;
    # "paged" = the general engine (any u32 price, any depth).  Both are bit-identical on this workload (tests).
    # (the window and the slot count follow from the population: core.dense_kwargs_for -> price_window (20, 179), live_cap 100)
    eng_kw = core.dense_kwargs_for(groups) if args.engine == "dense" else {}
    env = core.BatchedEnv(n_envs, 0, 0, 1, 1_000_000, device=local, env_id_base=env_base, obs_words=abi.OBS_L1,
                          max_orders=args.max_orders, max_trades=args.max_trades, max_steps=args.sim_steps, max_queue=128, **eng_kw)
    env.set_agents(groups)
    env.set_stream(stream.cuda_stream)
    n_steps = args.sim_steps

    def one_pass():
        env.reset()
        env.run_agents(n_steps, SEED, sync=False)

    # ---- device-resident timing: reset + persistent kernel, CUDA events on the launching stream
    for _ in range(args.warmup):
        one_pass()
        flush.fill_(1)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for a, m, b in ev:
        a.record(stream)
        env.reset()
        m.record(stream)
        env.run_agents(n_steps, SEED, sync=False)
        b.record(stream)
        flush.fill_(1)  # untimed L2 flush between passes (same stream, after the `b` event)
    barrier()
    wall_ms = (time.perf_counter() - wall0) * 1e3   # host clock over the same region: events + flushes + launch gaps
    step_ms = [a.elapsed_time(b) for a, _, b in ev]
    kern_ms = [m.elapsed_time(b) for _, m, b in ev]
    clocks = sampler.stop() if rank == 0 else None
    stats = env.stats()
    if stats["error_envs"]:
        raise SystemExit(f"device flagged errors in {stats['error_envs']} envs: {np.unique(env.env_errors())}")
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs, "c3")
    total_ms = sum(step_ms)

    # ---- end-to-end through the public API with HOST buffers: agent table up, full obs history + stats down
    hist_host = torch.empty((n_envs, n_steps, abi.OBS_L1), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
    h2d = len(groups) * abi.GROUP_DTYPE.itemsize
    d2h = hist_host.nbytes + 64 + n_envs * 36
    for _ in range(1):
        env.reset(); env.set_agents(groups); env.run_agents_to_host(n_steps, SEED, hist_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        env.reset()
        env.set_agents(groups)            # host -> device: the agent population
        # synchronous; device -> host: every env-step's observation, streamed out chunk by chunk while the run goes on
        env.run_agents_to_host(n_steps, SEED, hist_host)
        st = env.stats()                  # device -> host: aggregate statistics (+ final level-1 of every env)
    barrier()
    e2e_s = time.perf_counter() - t0
    checksum = int(hist_host[:, -1, :].astype(np.uint64).sum())

    # ---- the same, plus everything else the reference's sim_runner leaves in HOST memory: every env's trade log and order
    # table (orderbook.rs:113-115) copied out after the run (bb_trades_all / bb_orders_all, one strided copy each, pinned)
    e2e_logs = None
    if not args.no_logs:
        _, n_tr = env.trades_all(0, out=np.empty((n_envs, 0), dtype=abi.TRADE_REC_DTYPE))
        _, n_or = env.orders_all(0, out=np.empty((n_envs, 0), dtype=abi.ORDER_REC_DTYPE))
        cap_t, cap_o = int(n_tr.max()) + 1024, int(n_or.max()) + 1024
        tr_host = torch.empty((n_envs, cap_t, 32), dtype=torch.uint8, pin_memory=True).numpy().view(abi.TRADE_REC_DTYPE).reshape(n_envs, cap_t)
        or_host = torch.empty((n_envs, cap_o, 64), dtype=torch.uint8, pin_memory=True).numpy().view(abi.ORDER_REC_DTYPE).reshape(n_envs, cap_o)
        n_log = args.steps
        for i in range(n_log + 1):
            if i == 1:
                barrier()
                t0 = time.perf_counter()
            env.reset(); env.set_agents(groups); env.run_agents_to_host(n_steps, SEED, hist_host)
            st = env.stats()
            _, n_tr = env.trades_all(cap_t, out=tr_host)
            _, n_or = env.orders_all(cap_o, out=or_host)
        barrier()
        logs_s = (time.perf_counter() - t0) / n_log
        assert int(n_tr.sum()) == stats["trades"] and int(n_or.sum()) == stats["orders_created"]
        traded = int(sum(int(tr_host[e, :n_tr[e]]["vol"].sum(dtype=np.uint64)) for e in range(0, n_envs, 256)))
        e2e_logs = {"seconds_per_pass": logs_s, "d2h_bytes_per_step": int(hist_host.nbytes + tr_host.nbytes + or_host.nbytes + 64 + n_envs * 44),
                    "trade_records": int(n_tr.sum()), "order_records": int(n_or.sum()), "sampled_traded_volume": traded}
        del tr_host, or_host

    # ---- aggregate over ranks: max time, summed work; the ONLY collective of the run is this all-gather (NCCL)
    from bourse_b200.sharding import gather_env_stats
    agg = gather_env_stats(env, total_ms, ctx.comm)
    agg_e2e = gather_env_stats(env, e2e_s * 1e3, ctx.comm)
    if rank == 0:
        max_ms, max_e2e = agg["elapsed_ms_max"], agg_e2e["elapsed_ms_max"] * 1e-3
        instr_per_pass = agg["instructions"]     # stats are per pass (reset each pass)
        env_steps_per_pass = agg["env_steps"]
        value = instr_per_pass * args.steps / (max_ms * 1e-3)
        peak, peak_src = measured_peak_gbs()
        alg_bytes = workloads.algorithmic_bytes(stats, abi.OBS_L1)          # this rank's k_sim launch
        k_ms = sum(kern_ms) / len(kern_ms)
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        traffic = profile_traffic("c3")
        cores = host_cores()
        cpu = cpu_baseline(N_ENVS_PER_GPU, N_SIM_STEPS, cores) if world == 1 and not args.no_cpu else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic", "config": workload_config(world), "engine": args.engine,
            "env_steps_per_sec": env_steps_per_pass * args.steps / (max_ms * 1e-3),
            "orders_per_pass": instr_per_pass, "trades_per_pass": agg["trades"], "l1_checksums": agg["l1_checksums"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": "k_sim", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes,
                         "peak_source": peak_src},
            "e2e": {"value": instr_per_pass * args.steps / max_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * max_e2e / args.steps,
                    "api": "BatchedEnv.reset/set_agents/run_agents_to_host/stats (C ABI bb_reset, bb_set_agents, bb_run_agents_to_host, bb_stats)", "obs_checksum": checksum},
            # everything sim_runner leaves on the host, i.e. the history AND every trade log and order table (PCIe-bound)
            **({"e2e_with_logs": {"value": instr_per_pass / world / e2e_logs["seconds_per_pass"] * world, "unit": UNIT,
                                  "ms_per_step": 1e3 * e2e_logs["seconds_per_pass"], "d2h_bytes_per_step": e2e_logs["d2h_bytes_per_step"],
                                  "trade_records": e2e_logs["trade_records"], "order_records": e2e_logs["order_records"],
                                  "api": "... + BatchedEnv.trades_all / orders_all (bb_trades_all, bb_orders_all)"}} if e2e_logs else {}),
            "gpu_launches": 2 * args.steps, "clocks": clocks,   # timed region: k_init + k_sim per pass
            # sanity: host wall clock over the timed loop (includes the untimed L2 flushes); must be >= the event total
            "wall_ms_timed_loop": wall_ms, "event_ms_timed_loop": total_ms,
        }
        if cpu:
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    # ---- BASELINE configs 4 and 5 beside the headline (same launch, same ranks): C4 at 8192 envs per GPU (65,536 on 8 GPUs),
    # C5 with the 1024 books of the config split over the ranks (capped at 512 per GPU: 1024 deep books do not fit 180 GB)
    secondary = {}
    if not args.no_secondary:
        env.close()
        del hist_host
        torch.cuda.empty_cache()
        c4 = measure_c4(ctx, 8192, N_SIM_STEPS, args.steps, args.warmup, args.max_orders, args.max_trades, False, args.dump_outputs)
        c5_books = min(512, max(1, 1024 // world))
        c5 = measure_c5(ctx, c5_books, args.steps, args.warmup, "deep", 10, world == 1 and not args.no_cpu, args.dump_outputs)
        c5["scaling"] = "strong (1024 books over the ranks)" if c5_books * world == 1024 else f"{c5_books * world} of the 1024 books (one GPU holds at most 512)"
        secondary = {"c4": c4, "c5": c5}
    if rank == 0:
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line))
    ctx.finish()
    return 0


def run_c1(args):
    """C1: examples/random_trades.py semantics (seed 101, 200 steps, 100 Python RandomAgent(i, 0.5, (10,100), (20,50), 2),
    StepEnv(101, 0, tick, 100_000)) through the Python surface; wall time next to the same loop on the oracle's StepEnv.
    A functional config: the time is the CPython agent loop plus one small kernel launch per env.step()."""
    from bourse_b200 import core
    from bourse_b200.step_sim import run
    from bourse_b200.step_sim.agents import RandomAgent
    from oracle import oracle as orc

    orc.build()
    out = {}
    for tick in (2, 1):
        res = {}
        for name, mod in (("b200", core), ("oracle", orc)):
            best = None
            for _ in range(max(args.steps, 1)):
                env = mod.StepEnv(101, 0, tick, 100_000)
                agents = [RandomAgent(i, 0.5, (10, 100), (20, 50), tick) for i in range(100)]
                t0 = time.perf_counter()
                if name == "b200":
                    data = run(env, agents, 200, 101)
                else:   # same loop, oracle classes (runner asserts the product's StepEnv type)
                    rng = np.random.default_rng(101)
                    for _s in range(200):
                        for a in agents:
                            a.update(rng, env)
                        env.step()
                    data = env.get_market_data()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            res[name] = (best, data)
        same = all(np.array_equal(res["b200"][1][k], res["oracle"][1][k]) for k in res["oracle"][1])
        n_orders = len(res["b200"][1]["bid_price"])
        out[f"tick_{tick}"] = {"b200_wall_s": res["b200"][0], "oracle_wall_s": res["oracle"][0], "market_data_identical": bool(same),
                               "n_arrays": len(res["b200"][1]), "n_steps": n_orders}
    print(json.dumps({"metric": "wall_s", "unit": "s", "config": {"workload": "C1: examples/random_trades.py semantics, tick sizes 2 (the file) and 1 "
                      "(BASELINE.json), 100 Python RandomAgents x 200 steps through StepEnv"}, **out}))
    return 0


def gym_action_blocks(n_blocks: int, block_envs: int, rows: int, seed: int) -> np.ndarray:
    """Synthetic policy output for the vectorised loop: per env and step `rows` rows — ~60 % limit orders around 1000
    (+-8 ticks, so books trade), 5 % market orders, 25 % cancels and 10 % no-ops; cancel targets are drawn from ids the env
    is certain to have issued by that step (the first two rows of every step are orders)."""
    from bourse_b200 import abi, gym
    rng = np.random.default_rng(seed)
    shape = (n_blocks, block_envs, rows)
    u = rng.random(shape)
    op = np.where(u < 0.65, abi.OP_NEW, np.where(u < 0.90, abi.OP_CANCEL, abi.OP_NOOP)).astype(np.uint32)
    op[:, :, :2] = abi.OP_NEW                  # two orders per step for sure, so that ids below 2 * step always exist
    op[0, :, 2:][op[0, :, 2:] == abi.OP_CANCEL] = abi.OP_NOOP
    issued = np.maximum(1, 2 * np.arange(n_blocks)[:, None, None])
    return gym.pack_actions(op, bid=rng.random(shape) < 0.5, vol=rng.integers(1, 50, shape), trader=rng.integers(0, 1000, shape),
                            price=rng.integers(992, 1009, shape), order_id=(rng.random(shape) * issued).astype(np.uint64),
                            market=rng.random(shape) < 0.08)


def run_gym(args):
    """SURVEY 8f rank 4: the device-resident vectorised loop (bourse_b200.gym.VectorEnv): per step one action block
    [n_envs, rows] already in device memory -> ONE launch (bb_step_device: ids assigned on the device, Env::step, level-2
    records written to the observation buffer).
    One bench step = reset + `--sim-steps` env-steps (default 256); nothing crosses PCIe inside the timed region."""
    import torch

    from bourse_b200 import abi, gym, workloads

    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    n_envs, rows = args.envs, 8
    n_steps = args.sim_steps if args.sim_steps != N_SIM_STEPS else 256
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    blocks = gym_action_blocks(n_steps, 256, rows, SEED)                       # [step][env % 256][row]
    eng_kw = dict(price_window=(960, 1056), live_cap=254) if args.engine == "dense" else dict(pages_smem=10)
    bg = None
    if args.bg_agents:
        # a learner's rows against the C3 background population (50 + 50 RandomAgents, prices 20..178): every step is
        # { agents.update; rows; Env::step } in ONE launch (bb_run_agents_with_rows); the rows quote inside the agents' range
        bg = workloads.c3_groups()
        blocks["price"] = np.where((blocks["op_flags"] & abi.F_MARKET) != 0, blocks["price"], 2 * (40 + blocks["price"] % 21))
        eng_kw = dict(price_window=(20, 180), live_cap=254) if args.engine == "dense" else dict(pages_smem=10)
        eng_kw.update(agents=bg, agent_seed=SEED, max_queue=128)
    v = gym.VectorEnv(n_envs, rows, SEED, 0, 1, 1_000_000 if bg else 1000, device=local, max_orders=32768 if bg else 4096,
                      max_trades=32768 if bg else 8192, max_steps=n_steps + 8, **eng_kw)
    dev = torch.from_numpy(blocks.view(np.uint8).reshape(n_steps, 256, rows * 32)).cuda()
    dev = dev.repeat(1, (n_envs + 255) // 256, 1)[:, :n_envs].contiguous()       # [step][env][row bytes]
    v.env.set_stream(stream.cuda_stream)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for i in range(args.warmup + args.steps):
        v.reset()
        if i >= args.warmup:
            ev[i - args.warmup][0].record(stream)
        for s in range(n_steps):
            v.step(dev[s])
        if i >= args.warmup:
            ev[i - args.warmup][1].record(stream)
        flush.fill_(1)
    torch.cuda.synchronize()
    v.check_errors()
    ms = [a.elapsed_time(b) for a, b in ev]
    k_ms = sum(ms) / len(ms)
    stats = v.env.stats()
    cpu = None
    if not args.no_cpu and not bg:
        from oracle import oracle as orc
        orc.build()
        cores = host_cores()
        r = orc.bench_env_rows(4096 * cores, cores, n_steps, blocks, SEED)
        cpu = {"value": r["instructions"] / r["seconds"], "unit": UNIT, "cores": cores, "kind": "port",
               "env_steps_per_sec": r["env_steps"] / r["seconds"],
               "sample": f"{4096 * cores} envs x {n_steps} steps of the same action blocks, one env per core at a time ({r['seconds']:.2f} s)"}
    peak, peak_src = measured_peak_gbs()
    alg = workloads.algorithmic_bytes(stats, abi.OBS_L2, n_envs * n_steps * rows)
    print(json.dumps({
        "metric": METRIC, "value": stats["instructions"] / (k_ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": k_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"vectorised device-resident loop: {n_envs} envs x {rows} action rows x {n_steps} steps (65% orders, 25% cancels, "
                               f"10% no-ops){' + 100 background RandomAgents per env in the same shuffled queue' if bg else ''}, level-2 observation of every "
                               f"env after every step, {args.engine} engine"},
        "env_steps_per_sec": n_envs * n_steps / (k_ms * 1e-3), "us_per_vector_step": 1e3 * k_ms / n_steps, "orders_per_pass": stats["instructions"],
        "trades_per_pass": stats["trades"], "gpu_launches": args.steps * (2 + n_steps),
        "roofline": {"bound": "hbm", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak,
                     "traffic": None, "kernel": "k_sim<.., EXT> (one launch per vector step)" if bg else "k_apply<ENV> (one launch per vector step)", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg / n_steps,
                     "peak_source": peak_src},
        **({"cpu_baseline": cpu} if cpu else {})}))
    v.close()
    return 0


class Ctx:
    """Per-rank CUDA context shared by the workload runners: one torch stream the library launches on (so that CUDA events
    recorded on it bracket the kernels), the L2-flush buffer, rank / world, and the max-over-ranks barrier."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: bourse_b200 has no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1 and not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        self.flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
        # the job's statistics all-gather goes through the library's own NCCL communicator (bb_comm_*), not torch
        from bourse_b200.sharding import Comm
        self.comm = Comm.from_env(self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def events(self, n):
        return [(self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)) for _ in range(n)]

    def finish(self):
        self.comm.close()
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def roofline_block(alg_bytes: float, k_ms: float, kernel: str, traffic=None) -> dict:
    peak, peak_src = measured_peak_gbs()
    ach = alg_bytes / (k_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "kernel": kernel,
            "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src}


def measure_c4(ctx: Ctx, per_gpu: int, n_steps: int, steps: int, warmup: int, max_orders: int, max_trades: int, with_cpu: bool,
               dump_dir: str | None = None) -> dict:
    """BASELINE config C4, one GPU's shard per rank: `per_gpu` envs x (40+40 RandomAgents + 20-trader MomentumAgent) x
    n_steps env-steps, level-2 (45-word) record per env-step.  The general (paged) engine: whenever a book's ask side is
    swept empty the MomentumAgent's mid price is ~2^31 (orderbook.rs:272-276 with the empty-side sentinel) and its limit
    bids rest THERE, as the best bid — measured: every one of the 8192 envs leaves any dense window within 1000 steps."""
    from bourse_b200 import abi, core, workloads
    from bourse_b200.sharding import gather_env_stats, shard_range

    base, n_envs = shard_range(per_gpu * ctx.world, ctx.world, ctx.rank)
    groups, obs = workloads.c4_groups(), abi.OBS_L2
    env = core.BatchedEnv(n_envs, 0, 0, 1, 1_000_000, device=ctx.local, env_id_base=base, obs_words=obs, max_orders=max_orders,
                          max_trades=max_trades, max_steps=n_steps, max_queue=128)
    env.set_agents(groups)
    env.set_stream(ctx.stream.cuda_stream)
    ev = ctx.events(steps)
    for i in range(warmup + steps):
        if i == warmup:
            ctx.barrier()
        env.reset()
        if i >= warmup:
            ev[i - warmup][0].record(ctx.stream)
        env.run_agents(n_steps, 7, sync=False)
        if i >= warmup:
            ev[i - warmup][1].record(ctx.stream)
        ctx.flush.fill_(1)
    ctx.barrier()
    ms = [a.elapsed_time(b) for a, b in ev]
    stats = env.stats()
    if stats["error_envs"]:
        raise SystemExit(f"C4: device flagged errors in {stats['error_envs']} envs")
    if dump_dir and ctx.rank == 0:
        dump_outputs(env, dump_dir, "c4")
    agg = gather_env_stats(env, sum(ms), ctx.comm)
    k_ms = sum(ms) / len(ms)
    out = {"workload": f"C4 shard: {per_gpu} envs/GPU x (40+40 RandomAgents + 20-trader MomentumAgent) x {n_steps} env-steps, "
                       "level-2 (45 x u32) record per env-step, paged engine",
           "value": agg["instructions"] * steps / (agg["elapsed_ms_max"] * 1e-3), "unit": UNIT, "ms_per_step": agg["elapsed_ms_max"] / steps,
           "env_steps_per_sec": agg["env_steps"] * steps / (agg["elapsed_ms_max"] * 1e-3), "orders_per_pass": agg["instructions"],
           "trades_per_pass": agg["trades"], "n_envs_total": per_gpu * ctx.world, "l1_checksums": agg["l1_checksums"],
           "roofline": roofline_block(workloads.algorithmic_bytes(stats, obs), k_ms, "k_sim<FAST,MOM>", profile_traffic("c4"))}
    if with_cpu and ctx.rank == 0:
        from oracle import oracle as orc
        orc.build()
        cores = host_cores()
        r = orc.bench_agents(64 * cores, cores, n_steps, 7, groups, keyed=False, start_time=0, tick_size=1, step_size=1_000_000)
        out["cpu_baseline"] = {"value": r["instructions"] / r["seconds"], "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": f"{64 * cores} envs x {n_steps} env-steps of the C4 population, one env per core at a time ({r['seconds']:.2f} s)"}
    env.close()
    return out


C5_WINDOW, C5_CHUNKS = (7936, 12160), 98304


def measure_c5(ctx: Ctx, per_gpu: int, steps: int, warmup: int, engine: str, pages_smem: int, with_cpu: bool,
               dump_dir: str | None = None) -> dict:
    """BASELINE config C5, one GPU's shard per rank: `per_gpu` books x 1,000,000 resting orders (pre-loaded, untimed), then
    100 steps x 10,000 events per book with a 30% cancel/modify rate, replayed from device memory (timed)."""
    import torch
    from bourse_b200 import abi, core, workloads
    from bourse_b200.sharding import gather_env_stats, shard_range

    base, n_envs = shard_range(per_gpu * ctx.world, ctx.world, ctx.rank)
    n_rest, n_steps, per_step, n_distinct = 1_000_000, 100, 10_000, 8
    obs = abi.OBS_L2
    streams = [workloads.c5_stream(n_rest, n_steps, per_step, seed=100 + i) for i in range(n_distinct)]
    dev = torch.device("cuda", ctx.local)
    reps = (n_envs + n_distinct - 1) // n_distinct
    d1 = torch.from_numpy(np.concatenate([x[:n_rest] for x in streams]).view(np.uint8)).to(dev).view(n_distinct, -1).repeat(reps, 1)[:n_envs].contiguous()
    d2 = torch.from_numpy(np.concatenate([x[n_rest:] for x in streams]).view(np.uint8)).to(dev).view(n_distinct, -1).repeat(reps, 1)[:n_envs].contiguous()
    o1 = torch.arange(0, n_envs + 1, dtype=torch.int64, device=dev) * n_rest
    o2 = torch.arange(0, n_envs + 1, dtype=torch.int64, device=dev) * (n_steps * per_step)
    if engine == "deep":
        # deep-book engine (csrc/deepw.cuh): one CTA per book; window = every price the stream can rest at (10000 +- 2048,
        # rounded out to 32-level words), 98304 queue chunks of 31 entries per book
        eng_kw = dict(price_window=C5_WINDOW, deep_chunks=C5_CHUNKS)
        eng_name = ("deep-book engine (one CTA per book: fetch / chain / replay / retire warps — the ladder chain in event order, the queues "
                    "replayed one lane per price level, trades placed by a warp prefix sum; chunked array queues in HBM)")
    else:
        # Price pages resident in shared memory: as many as let the whole shard stay resident in ONE wave (a book's image is
        # ~0.5 KB per page; 148 SMs x 227 KB).  128-296 books per GPU: all 192 pages (2 books per CTA); 512: ~100 pages.
        books_per_sm = -(-n_envs // 148)
        books_per_sm = 1 if books_per_sm <= 1 else 2 if books_per_sm <= 2 else 4 * (-(-books_per_sm // 4))
        c5_pages = pages_smem if pages_smem != 10 else max(10, min(192, (227 * 1024 // books_per_sm - 8192) // 512))
        eng_kw = dict(pages_smem=c5_pages, pages_total=192)
        eng_name = f"paged engine, {c5_pages} of 192 price pages per book resident in shared memory"
    env = core.BatchedEnv(n_envs, 0, 0, 1, 1_000_000, device=ctx.local, env_id_base=base, obs_words=obs, max_orders=1_750_000,
                          max_trades=1 << 20, max_steps=n_steps, max_queue=32, **eng_kw)
    env.set_stream(ctx.stream.cuda_stream)
    torch.cuda.synchronize()
    ev = ctx.events(steps)
    pre_stats = None
    for i in range(warmup + steps):
        if i == warmup:
            ctx.barrier()
        env.reset()
        env.replay_device(d1.data_ptr(), o1.data_ptr())      # untimed: build the 1M-order book
        if pre_stats is None:
            env.synchronize(); pre_stats = env.stats()
            pre_agg = gather_env_stats(env, 0.0, ctx.comm)
        if i >= warmup:
            ev[i - warmup][0].record(ctx.stream)
        env.replay_device(d2.data_ptr(), o2.data_ptr())
        if i >= warmup:
            ev[i - warmup][1].record(ctx.stream)
        ctx.flush.fill_(1)
    ctx.barrier()
    ms = [a.elapsed_time(b) for a, b in ev]
    stats = env.stats()
    if stats["error_envs"]:
        raise SystemExit(f"C5: device flagged errors in {stats['error_envs']} envs")
    if dump_dir and ctx.rank == 0:
        dump_outputs(env, dump_dir, "c5")
    # only the timed phase counts
    stats = {k: (stats[k] - pre_stats[k] if k in ("instructions", "orders_created", "trades", "traded_volume", "transitions", "env_steps") else stats[k]) for k in stats}
    stats["env_steps"] = n_envs * n_steps
    agg = gather_env_stats(env, sum(ms), ctx.comm)
    for k in ("instructions", "orders_created", "trades", "traded_volume", "transitions"):   # the pre-load is the same on every rank
        agg[k] -= pre_agg[k]
    agg["env_steps"] = per_gpu * ctx.world * n_steps
    k_ms = sum(ms) / len(ms)
    out = {"workload": f"C5 shard: {per_gpu} books/GPU x 1,000,000 resting orders (pre-loaded, untimed), then 100 steps x 10,000 events per "
                       "book (15% cancel, 15% modify, 60% limit within +-32 ticks, 10% market), level-2 record per step, replayed from "
                       "device memory; " + eng_name,
           "value": agg["instructions"] * steps / (agg["elapsed_ms_max"] * 1e-3), "unit": UNIT, "ms_per_step": agg["elapsed_ms_max"] / steps,
           # (one CTA per book, up to four resident per SM: with at most one book per SM the pass time IS a book's time)
           **({"us_per_event_per_book": 1e3 * k_ms / (n_steps * per_step)} if n_envs <= 148 and engine == "deep" else {}),
           "env_steps_per_sec": agg["env_steps"] * steps / (agg["elapsed_ms_max"] * 1e-3), "orders_per_pass": agg["instructions"],
           "trades_per_pass": agg["trades"], "n_books_total": per_gpu * ctx.world, "l1_checksums": agg["l1_checksums"][:1],
           "roofline": roofline_block(workloads.algorithmic_bytes(stats, obs, n_envs * n_steps * per_step), k_ms,
                                      "k_deepw" if engine == "deep" else "k_apply<REPLAY,PAGED_RES>", profile_traffic("c5_" + engine, per_book=n_envs))}
    if with_cpu and ctx.rank == 0:
        from oracle import oracle as orc
        orc.build()
        cores = host_cores()
        r = orc.bench_replay_suffix(cores, 1, streams[0], n_rest)
        out["cpu_baseline"] = {"value": r["instructions"] / r["seconds"], "unit": UNIT, "cores": cores, "kind": "port",
                               "us_per_event_per_book": 1e6 * r["seconds"] / (n_steps * per_step),
                               "sample": f"{cores} books (one per core), each pre-loaded with {n_rest} resting orders (untimed) and then fed the "
                                         f"{n_steps * per_step} events of one C5 stream, all threads together ({r['seconds']:.2f} s)"}
    env.close()
    del d1, d2
    torch.cuda.empty_cache()
    return out


def profile_traffic(key: str, per_book: int = 0):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, one ncu capture per kernel, committed under
    profiles/): ncu cannot run inside a timed bench, so the figure comes from profiles/kernel_traffic.json.  per_book: the
    launch's book count when it may differ from the profiled one (books are independent: the traffic scales with them)."""
    tp = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    try:
        e = json.load(open(tp))[key]
        return e["dram_bytes_per_book"] * per_book if per_book else e["dram_bytes_per_launch"]
    except Exception:
        return None


def secondary_line(args, ctx, res: dict) -> dict:
    """A full JSON line for a secondary workload (--workload c4 | c5) from a measure_* result."""
    line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic", "config": {"workload": res["workload"]}}
    line.update({k: v for k, v in res.items() if k not in ("workload", "value", "unit", "ms_per_step")})
    return line


def run_gpu_other(args):
    """Secondary workloads of BASELINE.json (not the headline line): --workload c1 | c2 | c4 | c5 | market, one GPU's shard
    per rank."""
    import torch
    import torch.distributed as dist

    from bourse_b200 import abi, core, workloads
    from bourse_b200.sharding import gather_stats, shard_range

    if args.workload == "c1":
        return run_c1(args)
    ctx = Ctx()
    rank, world, local, stream, flush, barrier = ctx.rank, ctx.world, ctx.local, ctx.stream, ctx.flush, ctx.barrier
    ev = ctx.events(args.steps)
    if args.workload == "c4":
        res = measure_c4(ctx, args.envs if args.envs != N_ENVS_PER_GPU else 8192, args.sim_steps, args.steps, args.warmup, args.max_orders,
                         args.max_trades, world == 1 and not args.no_cpu, args.dump_outputs)
        if rank == 0:
            print(json.dumps(secondary_line(args, ctx, res)))
        ctx.finish()
        return 0
    if args.workload == "c5":
        res = measure_c5(ctx, args.envs if args.envs != N_ENVS_PER_GPU else 128, args.steps, args.warmup, args.engine, args.pages_smem,
                         world == 1 and not args.no_cpu, args.dump_outputs)
        if rank == 0:
            print(json.dumps(secondary_line(args, ctx, res)))
        ctx.finish()
        return 0
    if args.workload == "c2":
        # C2: replayed place/cancel/modify stream (55/5/25/15 % limit/market/cancel/modify) of 10^6 events into ONE book
        # (--envs 1, the config as stated: a single sequential dependency chain) or into --envs books at once
        n_books = args.envs if args.envs != N_ENVS_PER_GPU else 1
        n_ev, n_distinct = 1_000_000, min(8, n_books)
        deep = args.engine == "deep"   # (the deep engine's one-side-per-level precondition excludes the trading-off windows)
        streams = [workloads.replay_stream(n_ev, s, tick_size=1, trading_windows=not deep) for s in range(n_distinct)]
        dev = torch.device("cuda", local)
        reps = (n_books + n_distinct - 1) // n_distinct
        d = torch.from_numpy(np.concatenate(streams).view(np.uint8)).to(dev).view(n_distinct, -1).repeat(reps, 1)[:n_books].contiguous()
        off = torch.arange(0, n_books + 1, dtype=torch.int64, device=dev) * n_ev
        n_emit = int(((streams[0]["op_flags"] & abi.F_EMIT) != 0).sum())
        eng_kw = dict(price_window=(896, 1152), deep_chunks=65536) if deep else dict(pages_smem=args.pages_smem if args.pages_smem != 10 else 64, pages_total=64)
        env = core.BatchedEnv(n_books, 0, 0, 1, 100_000, device=local, obs_words=abi.OBS_L2, max_orders=1 << 20, max_trades=1 << 20,
                              max_steps=n_emit + 8, max_queue=32, **eng_kw)
        env.set_stream(stream.cuda_stream)
        torch.cuda.synchronize()
        for i in range(args.warmup + args.steps):
            if i == args.warmup:
                barrier()
            env.reset()
            if i >= args.warmup:
                ev[i - args.warmup][0].record(stream)
            env.replay_device(d.data_ptr(), off.data_ptr())
            if i >= args.warmup:
                ev[i - args.warmup][1].record(stream)
            flush.fill_(1)
        barrier()
        ms = [a.elapsed_time(b) for a, b in ev]
        stats = env.stats()
        if stats["error_envs"]:
            raise SystemExit(f"device flagged errors in {stats['error_envs']} envs")
        stats["env_steps"] = n_books * n_emit
        peak, peak_src = measured_peak_gbs()
        k_ms = sum(ms) / len(ms)
        alg = workloads.algorithmic_bytes(stats, abi.OBS_L2, n_books * n_ev)
        from oracle import oracle as orc
        orc.build()
        cores = host_cores()
        r = orc.bench_replay(min(n_books, cores), min(n_books, cores), 1, streams[0])
        print(json.dumps({
            "metric": METRIC, "value": stats["instructions"] / (k_ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": k_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"C2: replayed stream of {n_ev} instructions (55% limit, 5% market, 25% cancel, 15% modify; cancel/modify "
                                   f"targets uniform over all issued ids{'' if not deep else '; no trading-off windows'}) into each of {n_books} book(s), level-2 record every 64 events, "
                                   f"{'deep-book engine (one CTA per book)' if deep else 'paged engine'}"},
            "orders_per_pass": stats["instructions"], "trades_per_pass": stats["trades"],
            "roofline": {"bound": "hbm", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak,
                         "traffic": None, "kernel": "k_deepw" if deep else "k_apply", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg, "peak_source": peak_src},
            "cpu_baseline": {"value": r["instructions"] / r["seconds"], "unit": UNIT, "cores": min(n_books, cores), "kind": "port",
                             "sample": f"the same stream into {min(n_books, cores)} book(s), one per core ({r['seconds']:.2f} s; counts every row incl. no-ops)"}}))
        return 0
    if args.workload == "market":
        # SURVEY 8f rank 3: the reference's multi-asset example (crates/step_sim/examples/multi_asset/main.rs:12-22) —
        # MarketEnv::<2> with 4 RandomMarketAgents groups (100 agents per asset), market_sim_runner — batched over
        # `--envs / 2` lockstep markets per GPU; one level-2 record per asset and step (MarketEnv keeps Level2DataRecords)
        n_assets = 2
        per_gpu = args.envs
        base, n_envs = shard_range(per_gpu * world, world, rank, multiple=n_assets)   # markets stay whole
        groups, g_assets = workloads.market_example_groups()
        obs, n_steps = abi.OBS_L2, args.sim_steps
        eng_kw = dict(price_window=(20, 180), live_cap=128) if args.engine == "dense" else {}
        env = core.BatchedEnv(n_envs, 0, 0, 1, 1_000_000, device=local, env_id_base=base, obs_words=obs, max_orders=args.max_orders,
                              max_trades=args.max_trades, max_steps=n_steps, max_queue=args.max_queue or 80, assets=n_assets, **eng_kw)
        env.set_agents(groups, assets=g_assets)
        env.set_stream(stream.cuda_stream)
        for i in range(args.warmup + args.steps):
            if i == args.warmup:
                barrier()
            env.reset()
            if i >= args.warmup:
                ev[i - args.warmup][0].record(stream)
            env.run_agents(n_steps, SEED, sync=False)
            if i >= args.warmup:
                ev[i - args.warmup][1].record(stream)
            flush.fill_(1)
        ext = 0
        name = (f"multi-asset example: {per_gpu // n_assets} markets/GPU x 2 assets x (50+50) RandomMarketAgents per asset x {n_steps} "
                f"steps (market_sim_runner), level-2 record per asset and step, {args.engine} engine")
    barrier()
    ms = [a.elapsed_time(b) for a, b in ev]
    stats = env.stats()
    if stats["error_envs"]:
        raise SystemExit(f"device flagged errors in {stats['error_envs']} envs")
    from bourse_b200.sharding import gather_env_stats
    agg = gather_env_stats(env, sum(ms), ctx.comm)
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        k_ms = sum(ms) / len(ms)
        alg = workloads.algorithmic_bytes(stats, obs, ext)
        cpu = None
        if world == 1 and not args.no_cpu:   # the reference's algorithm (oracle port) on the host cores, bounded sample
            from oracle import oracle as orc
            orc.build()
            cores = host_cores()
            r = orc.bench_market_agents(32 * cores, cores, n_steps, SEED, groups, g_assets, n_assets, keyed=False)
            cpu = {"value": r["instructions"] / r["seconds"], "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{32 * cores} two-asset markets x {n_steps} steps, one market per core at a time, reference-style "
                             f"shared Xoroshiro stream ({r['seconds']:.2f} s)"}
        print(json.dumps({
            "metric": METRIC, "value": agg["instructions"] * args.steps / (agg["elapsed_ms_max"] * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": agg["elapsed_ms_max"] / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": {"workload": name},
            "env_steps_per_sec": agg["env_steps"] * args.steps / (agg["elapsed_ms_max"] * 1e-3), "orders_per_pass": agg["instructions"],
            "trades_per_pass": agg["trades"],
            "roofline": {"bound": "hbm", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "k_sim<DENSE,0,MKT>",
                         "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg, "peak_source": peak_src},
            **({"cpu_baseline": cpu} if cpu else {})}))
    ctx.finish()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=N_ENVS_PER_GPU)
    ap.add_argument("--sim-steps", type=int, default=N_SIM_STEPS)
    ap.add_argument("--max-orders", type=int, default=65536)
    ap.add_argument("--max-trades", type=int, default=65536)
    ap.add_argument("--max-queue", type=int, default=0, help="per-env instructions per step (0 = the workload's default)")
    ap.add_argument("--pages-smem", type=int, default=10,
                    help="c5 / c2: 32-level price pages per book resident in shared memory (of 192 / 64); the default 10 means 'all of them'")
    ap.add_argument("--bg-agents", action="store_true", help="gym: the C3 background population trades in every env (bb_run_agents_with_rows)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-logs", action="store_true", help="skip the e2e_with_logs leg (full trade log + order table to the host)")
    ap.add_argument("--no-secondary", action="store_true", help="headline run only: skip the C4 / C5 block")
    ap.add_argument("--engine", default=None, choices=["dense", "paged", "deep"],
                    help="default: dense for c3 / market (shallow books inside a known price window), paged for gym")
    ap.add_argument("--workload", default="c3", choices=["c1", "c2", "c3", "c4", "c5", "market", "gym"],
                    help="c3 = the headline line; the others are the secondary configs (market = the multi-asset example)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed pass computed (a seeded sample: observation history, "
                         "trade log, order table) as DIR/<workload>_<name>.npy, float64, under 64 MB; c3 (with the c4 / c5 "
                         "block), c4 and c5 only; rank 0's shard when --gpus > 1")
    args = ap.parse_args()
    if args.dump_outputs:
        if args.impl != "b200" or args.workload not in ("c3", "c4", "c5"):
            ap.error("--dump-outputs covers the b200 c3, c4 and c5 workloads")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.engine is None:
        # c2: one CTA per book (k_deepw) while at most two books share an SM, the paged engine (one warp per book) beyond
        c2_deep = args.workload == "c2" and (args.envs == N_ENVS_PER_GPU or args.envs <= 296)
        args.engine = ("paged" if args.workload == "gym" and not args.bg_agents else "deep" if args.workload == "c5" or c2_deep else "dense")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "gym":
        return run_gym(args)
    if args.workload != "c3":
        return run_gpu_other(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
