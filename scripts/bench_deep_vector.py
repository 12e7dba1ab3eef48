"""Per-step time of the device-resident Env loop on deep books (gym.VectorEnv with price_window + deep_chunks:
bb_step_device on the deep-book engine, k_env_deep_stage + k_deepw<.., ENV>).

Books are preloaded to C5 depth: four distinct C5 books (workloads.c5_stream: 1,000,000 resting orders, then one step of
10,000 events; market-data records stripped) are replayed into books 0-3, saved into a store and restored into every book
(book u from slot u % 4).  Then, for 148, 296 and 512 books and 1, 8 and 32 rows per env, the per-step time of a VectorEnv
step with a fixed device-resident action block (60 % limit NEWs within 32 ticks of the mid, 10 % market orders, 15 %
cancels and 15 % modifies of preloaded ids; the same block every step): issued eagerly from Python (CUDA events around --steps steps after --warmup
steps) and replayed from a CUDA graph of --graph-steps steps (CUDA events around the replays).  Every (books, rows) case
starts from freshly restored books.

The fixed cost of a step is measured, not estimated: the same loop with rows that are all no-ops (the step then runs the
staging launch and a k_deepw launch whose only event is the closing record), and a k_deepw replay launch over empty slices
(bb_replay_device with every slice empty: the launch's set-up, the book image in and out, nothing else).

Bytes moved between HBM and shared memory per book and launch come from deep_layout (bourse_b200.cu): k_deepw bulk-copies
the book image up to the level counts in at its start and out at its end (`smem_image` bytes each way); k_env_deep_stage
keeps only the step's permutation (2 bytes per queued row) in shared memory and copies nothing in or out.

--bg-agents times the same books with background agents instead: workloads.c3_groups_around(MID) (C3's two RandomAgents
groups re-centred on the C5 mid) through VectorEnv(agents=...), whose steps (bb_run_agents_with_rows: k_env_agents_stage +
k_deepw<.., ENV>) refuse CUDA-graph capture, so every loop here is issued eagerly: per (books, rows) the deep step with the
agents, the deep step with the rows only, and the FAST engine running the same population and rows on shallow books that
start empty (their cancels name the agents' first ids).  The action block has no MODIFY rows (agent steps drop them);
--rows defaults to 1,8 there.

Prints the card and its power limit, then one JSON line; --out writes the JSON there too.

    python scripts/bench_deep_vector.py --steps 200 --warmup 20 --graph-steps 50 --out deep_vector.json
    python scripts/bench_deep_vector.py --bg-agents --steps 200 --warmup 20 --out deep_agents.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bourse_b200 import abi, gym, workloads  # noqa: E402

C5_WINDOW, C5_CHUNKS, MID = (7936, 12160), 98304, 10_000   # as bench.py's C5 (every price the stream can rest at)
N_REST, PER_STEP, N_DISTINCT = 1_000_000, 10_000, 4
STEP = 1_000_000


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def smem_image_bytes(window) -> int:
    """deep_layout(W).smem_image (bourse_b200.cu, deep.cuh): header, chunk allocator and free stack, both bitmaps, both
    summaries, level volumes; the level counts and queue heads / tails stay in HBM."""
    W = (window[1] - window[0] + 31) // 32 * 32
    bm = 192 + 4 * 256                 # DP_OFF_BM = DP_OFF_FS + 4 * DP_FS_CAP
    sm = bm + 8 * (W // 32)
    lvol = (sm + 8 * 8 + 15) // 16 * 16
    return lvol + 4 * W                # = lcnt


def action_block(rng, n_books, rows, modify=True):
    a = np.zeros((n_books, rows), dtype=gym.ACTION_DTYPE)
    u = rng.random((n_books, rows))
    new = u < 0.7
    market = (u >= 0.6) & new
    bid = rng.random((n_books, rows)) < 0.5
    a["op_flags"] = np.where(new, abi.OP_NEW, np.where(u < 0.85, abi.OP_CANCEL, abi.OP_MODIFY | abi.F_HAS_VOL | abi.F_HAS_PRICE))
    a["op_flags"] |= np.where(new & bid, abi.F_BID, 0).astype(np.uint32) | np.where(market, abi.F_MARKET, 0).astype(np.uint32)
    a["price"] = np.where(market, 0, MID + rng.integers(-32, 33, (n_books, rows)))
    a["vol"] = rng.integers(1, 51, (n_books, rows))
    a["trader"] = rng.integers(0, 1000, (n_books, rows))
    a["order_id"] = np.where(new, 0, rng.integers(0, N_REST, (n_books, rows)))
    if not modify:
        a["op_flags"] = np.where(u < 0.85, a["op_flags"], abi.OP_NOOP)
    return a


def timed_eager(v, acts, st, steps, warmup):
    """us per step of `steps` VectorEnv steps issued from Python after `warmup` steps (CUDA events on the env's stream)."""
    import torch
    with torch.cuda.stream(st):
        for _ in range(warmup):
            v.step(acts)
    st.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    with torch.cuda.stream(st):
        for _ in range(steps):
            v.step(acts)
    e1.record(st)
    e1.synchronize()
    return round(e0.elapsed_time(e1) * 1e3 / steps, 2)


def bg_agents_cases(args, res, streams, books_list, rows_list):
    import torch
    groups = workloads.c3_groups_around(MID)
    n_pre = len(streams[0])
    n_steps_max = args.warmup + args.steps + 8
    per_step = sum(int(g["n_agents"]) for g in groups) + max(rows_list)   # a bound on the ids a step can take
    res["engine"] = "deep with background agents (k_env_agents_stage + k_deepw<.., ENV>), against deep rows-only and FAST with agents"
    res["agents"] = "workloads.c3_groups_around(10000): 50 + 50 RandomAgents, tick size 2, ticks (4990, 5010) and (4960, 5040)"
    rng = np.random.default_rng(0)
    for n_books in books_list:
        for rows in rows_list:
            blk = action_block(rng, n_books, rows, modify=False)
            acts = torch.from_numpy(blk.view(np.uint8).reshape(n_books, rows, 32)).cuda()
            # the shallow books start empty: their cancels name the agents' first ids instead of preloaded ones
            shallow = blk.copy()
            shallow["order_id"] %= 16
            acts_shallow = torch.from_numpy(shallow.view(np.uint8).reshape(n_books, rows, 32)).cuda()
            case = {"books": n_books, "rows_per_env": rows}
            for key, kw in (("deep_agents_us_per_step", dict(agents=groups, price_window=C5_WINDOW, deep_chunks=C5_CHUNKS)),
                            ("deep_rows_only_us_per_step", dict(price_window=C5_WINDOW, deep_chunks=C5_CHUNKS)),
                            ("fast_agents_us_per_step", dict(agents=groups))):
                deep = "deep_chunks" in kw
                v = gym.VectorEnv(n_books, rows, 0, 0, 1, STEP, agent_seed=7, max_orders=(n_pre if deep else 0) + per_step * n_steps_max + 64,
                                  max_trades=1 << 18, max_steps=n_steps_max, **kw)
                st = torch.cuda.Stream()
                v.env.set_stream(st.cuda_stream)
                v.reset()
                if deep:   # C5 books: the distinct preloads saved and restored into every book
                    v.env.replay(np.concatenate(streams), np.array([n_pre * min(i, N_DISTINCT) for i in range(n_books + 1)], np.uint64))
                    store = v.snapshots(N_DISTINCT)
                    v.save(store, np.arange(N_DISTINCT, dtype=np.uint32))
                    v.restore(store, torch.from_numpy((np.arange(n_books) % N_DISTINCT).astype(np.int32)).cuda())
                v.env.synchronize()
                torch.cuda.synchronize()
                case[key] = timed_eager(v, acts if deep else acts_shallow, st, args.steps, args.warmup)
                err = v.env.env_errors()
                if err.any():
                    raise SystemExit(f"deep vector bench: env errors {[hex(x) for x in np.unique(err)]} at {n_books} books, {rows} rows, {key}")
                v.close()
            res["cases"].append(case)
            print(json.dumps(case), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--books", default="148,296,512")
    ap.add_argument("--rows", default="1,8,32")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--graph-steps", type=int, default=50)
    ap.add_argument("--graph-reps", type=int, default=4)
    ap.add_argument("--out", default=None)
    ap.add_argument("--bg-agents", action="store_true", help="background agents: deep with agents, deep rows-only, FAST with agents (eager)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_deep_vector: no CUDA device (this benchmark measures the GPU; there is no CPU fallback)")
    name, power = card()
    print(f"card: {name}, power limit: {power}", flush=True)
    books_list = [int(x) for x in args.books.split(",")]
    rows_list = [int(x) for x in ("1,8" if args.bg_agents and args.rows == "1,8,32" else args.rows).split(",")]
    streams = []
    for i in range(N_DISTINCT):
        s = workloads.c5_stream(N_REST, 1, PER_STEP, seed=100 + i)
        s["op_flags"] &= ~np.uint32(abi.F_EMIT)
        end = np.zeros(1, dtype=abi.INSTR_DTYPE)   # a no-op 1 ns later: the first step's events come after every key time
        end["t"], end["op_flags"] = s["t"][-1] + np.uint64(1), abi.OP_NOOP
        streams.append(np.concatenate([s, end]))
    n_pre = len(streams[0])
    n_steps_max = args.warmup + args.steps + args.graph_steps * (args.graph_reps + 2) + 8
    img = smem_image_bytes(C5_WINDOW)
    res = {"card": name, "power_limit": power, "engine": "deep (k_env_deep_stage + k_deepw<.., ENV>)", "window": C5_WINDOW,
           "deep_chunks": C5_CHUNKS, "preload": f"C5: {N_REST} resting orders + {PER_STEP} events per book, {N_DISTINCT} distinct books "
           "saved and restored into every book", "step_size": STEP, "steps": args.steps, "warmup": args.warmup,
           "graph_steps": args.graph_steps, "graph_reps": args.graph_reps,
           "smem_bytes_per_book_per_launch": {"k_deepw_in": img, "k_deepw_out": img,
                                              "k_env_deep_stage": "2 bytes per queued row (permutation, not copied in or out)"},
           "cases": []}
    rng = np.random.default_rng(0)
    for n_books in [] if args.bg_agents else books_list:
        for rows in [0] + rows_list:   # rows 0: one no-op row per env (the fixed cost of a step)
            r_eff = max(rows, 1)
            v = gym.VectorEnv(n_books, r_eff, 0, 0, 1, STEP, max_orders=n_pre + r_eff * n_steps_max + 64, max_trades=1 << 18,
                              max_steps=n_steps_max, max_queue=max(r_eff, 16), price_window=C5_WINDOW, deep_chunks=C5_CHUNKS)
            st = torch.cuda.Stream()
            v.env.set_stream(st.cuda_stream)
            v.reset()
            v.env.replay(np.concatenate(streams), np.array([n_pre * min(i, N_DISTINCT) for i in range(n_books + 1)], np.uint64))
            store = v.snapshots(N_DISTINCT)
            v.save(store, np.arange(N_DISTINCT, dtype=np.uint32))
            slots = torch.from_numpy((np.arange(n_books) % N_DISTINCT).astype(np.int32)).cuda()
            blk = action_block(rng, n_books, r_eff) if rows else np.zeros((n_books, 1), dtype=gym.ACTION_DTYPE)
            acts = torch.from_numpy(blk.view(np.uint8).reshape(n_books, r_eff, 32)).cuda()
            v.env.synchronize()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            case = {"books": n_books, "rows_per_env": rows}
            if rows == 0:   # the fixed cost of a k_deepw launch alone: a replay over empty slices
                empty_instr = torch.zeros(32, dtype=torch.uint8, device="cuda")
                empty_offs = torch.zeros(n_books + 1, dtype=torch.int64, device="cuda")
                torch.cuda.synchronize()
                for _ in range(10):
                    v.env.replay_device(empty_instr.data_ptr(), empty_offs.data_ptr())
                e0.record(st)
                for _ in range(100):
                    v.env.replay_device(empty_instr.data_ptr(), empty_offs.data_ptr())
                e1.record(st)
                e1.synchronize()
                case["k_deepw_empty_replay_us"] = round(e0.elapsed_time(e1) * 1e3 / 100, 2)
                case["note"] = "fixed cost of a step: one no-op row per env (staging launch + k_deepw with the closing record only)"
            # eager: steps issued from Python on freshly restored books
            v.restore(store, slots)
            with torch.cuda.stream(st):
                for _ in range(args.warmup):
                    v.step(acts)
            st.synchronize()
            e0.record(st)
            with torch.cuda.stream(st):
                for _ in range(args.steps):
                    v.step(acts)
            e1.record(st)
            e1.synchronize()
            case["eager_us_per_step"] = round(e0.elapsed_time(e1) * 1e3 / args.steps, 2)
            # CUDA graph of graph_steps steps, replayed graph_reps times, on freshly restored books
            v.restore(store, slots)
            v.env.clear_history()
            with torch.cuda.stream(st):
                v.step(acts)
            st.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                for _ in range(args.graph_steps):
                    v.step(acts)
            with torch.cuda.stream(st):   # (a graph replays on the current stream: the events must be on it too)
                g.replay()
                st.synchronize()
                e0.record(st)
                for _ in range(args.graph_reps):
                    g.replay()
                e1.record(st)
            e1.synchronize()
            graph_us = e0.elapsed_time(e1) * 1e3 / (args.graph_reps * args.graph_steps)
            case["graph_us_per_step"] = round(graph_us, 2)
            case["env_steps_per_s_graph"] = round(n_books / graph_us * 1e6)
            err = v.env.env_errors()
            if err.any():
                raise SystemExit(f"deep vector bench: env errors {[hex(x) for x in np.unique(err)]} at {n_books} books, {rows} rows")
            del g
            v.close()
            res["cases"].append(case)
            print(json.dumps(case), flush=True)
    if args.bg_agents:
        bg_agents_cases(args, res, streams, books_list, rows_list)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
