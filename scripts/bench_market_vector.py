"""Per-step time of the device-resident market loop (gym.MarketVectorEnv, bb_step_device_market) against the single-asset
device loop on the same books and rows (gym.VectorEnv, bb_step_device) and the host path for markets
(market.MarketEnv.submit + step).

The rows are bench.gym_action_blocks for 8192 envs x 2 rows; the market runs see them as 2048 markets x 4 assets x 8 rows,
book m * 4 + a receiving exactly the rows env m * 4 + a gets in the VectorEnv run.  Device loops are timed with CUDA events
over --steps warmed steps, in windows of 100 steps that each start from reset books (nothing crosses PCIe inside a window); the host path with a host clock around steps that end in
a synchronisation.  Prints the card and its power limit, then one JSON line.

--bg-agents times the same two device loops with background agents instead: the C3 population (50 + 50 RandomAgents) on
every book — as RandomMarketAgents on every asset of every market (bb_run_agents_with_rows_market), and as
VectorEnv(agents=c3_groups()) on the 8192 single-asset books (bb_run_agents_with_rows) — with the rows repriced into the
agents' range as `bench.py --workload gym --bg-agents` does.

--reads measures the device-resident order and trade reads (bb_orders_device / bb_trades_device) in the C3 loops of
--bg-agents on the FAST engine, for 4096 single-asset envs (VectorEnv) and 2048 markets x 4 assets (MarketVectorEnv): the
time per vector step without reads and with `trades(cap=64)` + `orders(k=8)` after every step (the difference is what the
reads add to a step; plain and with-reads runs alternate, twice each), and the time per call of each read alone: CUDA
events around 200 back-to-back calls on the books a window left behind, issued from Python and replayed from a CUDA graph
(`time_calls`).  Those trades() calls find no new trades: they read the headers and write the padded windows.  The k = 8
queried ids per env / market are fixed ids below 500 (every book has issued them after the warm-up steps).

--resets measures the per-unit reset (bb_reset_device, `reset(mask)`) in the rows-only loops on the FAST engine, for 4096
single-asset envs (VectorEnv) and 2048 markets x 4 assets (MarketVectorEnv): the time per step of the step alone and of
the step followed by `reset(mask)` with 0 %, 1 % and 100 % of the units selected (fixed device masks).  Each variant is
captured once as a CUDA graph of 100 steps and replayed from reset books, timed with CUDA events; the plain and with-reset
passes alternate, --passes times each, and the best pass of each counts.

--snapshots measures bb_save_device / bb_restore_device (`save` / `restore`) on warmed C3 books on the FAST engine, for
4096 single-asset envs (VectorEnv) and 2048 markets x 4 assets (MarketVectorEnv): after --warmup-steps steps of the C3
population, a store with one slot per unit; each call saves 1 % or 100 % of the units into their own slots, or restores
them from those slots (with the observation rows and trade cursors), replayed 50 times from a CUDA graph and timed with CUDA
events, --passes times, best pass.  The bytes a call copies come from the prefix lengths of the selected books (blob,
orders and trades logged, agent state); bytes/s is that over the time per call (a save reads and writes each byte once, as
does a restore, so the DRAM traffic is twice it).

    python scripts/bench_market_vector.py --steps 1000 --warmup 20
    python scripts/bench_market_vector.py --bg-agents --steps 1000 --warmup 20
    python scripts/bench_market_vector.py --reads --steps 1000 --warmup 20
    python scripts/bench_market_vector.py --resets --passes 3
    python scripts/bench_market_vector.py --snapshots --passes 3
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import gym_action_blocks  # noqa: E402
from bourse_b200 import abi, gym, market, workloads  # noqa: E402

N_MARKETS, ASSETS, ROWS_PER_BOOK = 2048, 4, 2
N_BOOKS, ROWS = N_MARKETS * ASSETS, ASSETS * ROWS_PER_BOOK
ENGINES = {"fast": dict(), "dense": dict(price_window=(960, 1056), live_cap=254)}
KW = dict(max_orders=8192, max_trades=16384, max_steps=256)
WINDOW = 100
# background agents: the C3 population's prices are 20..178 (bench.py --workload gym --bg-agents)
BG_ENGINES = {"fast": dict(), "dense": dict(price_window=(20, 180), live_cap=254)}
BG_KW = dict(max_orders=8192, max_trades=16384, max_steps=256, max_queue=128)
# --snapshots: room for the orders and trades of 300 warm-up steps of C3 (about 13,500 and 6,500 per book)
SNAP_KW = dict(max_orders=16384, max_trades=16384, max_steps=256, max_queue=128)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def market_blocks(blocks):
    """[n, 8192, 2] env rows -> [n, 2048, 8] market rows: book m * 4 + a's two rows, asset a, in asset order."""
    out = blocks.reshape(len(blocks), N_MARKETS, ROWS).copy()
    out["aux"] = np.repeat(np.arange(ASSETS, dtype=np.uint32), ROWS_PER_BOOK)
    return out


def windows(steps, warmup):
    """(untimed steps, timed steps) after each reset: every book restarts from empty every WINDOW steps, so resting orders
    stay within the dense engine's slots, as bench.py --workload gym resets between passes."""
    out, left = [], steps
    while left:
        out.append((warmup, min(WINDOW, left)))
        left -= out[-1][1]
    return out


def time_device(loop, d_blocks, steps, warmup, after_step=None):
    """us per `loop.step` (followed by `after_step()` when given) on a stream of its own: CUDA events around the timed steps
    of each window, summed."""
    import torch
    stream = torch.cuda.Stream()
    loop.env.set_stream(stream.cuda_stream)
    n, total, errors = len(d_blocks), 0.0, 0
    for pre, timed in windows(steps, warmup):
        loop.reset()
        for s in range(pre):
            loop.step(d_blocks[s % n])
        stream.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for s in range(pre, pre + timed):
            loop.step(d_blocks[s % n])
            if after_step:
                after_step()
        t1.record(stream)
        stream.synchronize()
        total += t0.elapsed_time(t1) * 1e3
        errors |= int(np.bitwise_or.reduce(loop.env.env_errors()))
    loop.env.set_stream(0)
    return total / steps, errors


def c3_market_agents():
    """The C3 population as RandomMarketAgents on every asset of a market."""
    agents = []
    for a in range(ASSETS):
        for g in workloads.c3_groups():
            agents.append(market.RandomMarketAgents(a, int(g["n_agents"]), (int(g["tick_lo"]), int(g["tick_hi"])),
                                                    (int(g["vol_lo"]), int(g["vol_hi"])), int(g["tick_size"]), float(g["rate"])))
    return agents


def time_calls(loop, call, reps=200):
    """us per `call()` on the loop's stream, two ways: CUDA events around `reps` back-to-back calls from Python (bounded by
    the host's enqueue rate when the kernels are short), and around one replay of a CUDA graph holding `reps` calls (the
    device's time per call, launch gaps included).  One untimed call first allocates the outputs."""
    import torch
    stream = torch.cuda.Stream()
    loop.env.set_stream(stream.cuda_stream)
    call()
    stream.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(reps):
        call()
    t1.record(stream)
    stream.synchronize()
    eager = t0.elapsed_time(t1) * 1e3 / reps
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        for _ in range(reps):
            call()
    g.replay()   # (untimed)
    torch.cuda.synchronize()
    t0.record(stream)
    with torch.cuda.stream(stream):
        g.replay()
    t1.record(stream)
    stream.synchronize()
    loop.env.set_stream(0)
    return eager, t0.elapsed_time(t1) * 1e3 / reps


def bench_reads(args, name, power):
    """--reads: see the module docstring."""
    import torch
    k, cap, n_envs = 8, 64, N_BOOKS // 2
    res = {"card": name, "power_limit": power, "engine": "fast", "agents": "C3 (50 + 50 RandomAgents) on every book",
           "orders_k": k, "trades_cap": cap, "steps": args.steps, "warmup": args.warmup, "rows_per_book": ROWS_PER_BOOK,
           "us_per_step": {}, "us_per_call": {}, "errors": {}}
    rng = np.random.default_rng(9)
    c3 = workloads.c3_groups()
    for label, units in (("vector_env_4096", n_envs), ("market_vector_2048x4", N_MARKETS)):
        books = units if label.startswith("vector") else N_BOOKS
        blocks = gym_action_blocks(args.blocks, books, ROWS_PER_BOOK, seed=5)
        blocks["price"] = np.where((blocks["op_flags"] & abi.F_MARKET) != 0, blocks["price"], 2 * (40 + blocks["price"] % 21))
        if label.startswith("vector"):
            loop = gym.VectorEnv(n_envs, ROWS_PER_BOOK, 0, 0, 1, 1_000_000, agents=c3, agent_seed=5, **BG_KW)
            d_blocks = [torch.from_numpy(x.view(np.uint8).reshape(n_envs, -1)).cuda() for x in blocks]
            q_assets = None
        else:
            loop = gym.MarketVectorEnv(N_MARKETS, ROWS, 0, 0, [1] * ASSETS, 1_000_000, agents=c3_market_agents(), agent_seed=5, **BG_KW)
            d_blocks = [torch.from_numpy(x.view(np.uint8).reshape(N_MARKETS, -1)).cuda() for x in market_blocks(blocks)]
            q_assets = torch.from_numpy(np.tile(np.arange(k, dtype=np.int32) % ASSETS, (units, 1))).cuda()
        q_ids = torch.from_numpy(rng.integers(0, 500, (units, k))).cuda()
        torch.cuda.synchronize()

        def orders():
            return loop.orders(q_ids) if q_assets is None else loop.orders(q_ids, q_assets)

        def reads():
            loop.trades(cap)
            orders()

        for _ in range(2):   # plain and with reads, twice each, alternated
            for tag, fn in (("plain", None), ("with_reads", reads)):
                us, err = time_device(loop, d_blocks, args.steps, args.warmup, fn)
                res["us_per_step"].setdefault(f"{label}_{tag}", []).append(us)
                res["errors"][f"{label}_{tag}"] = res["errors"].get(f"{label}_{tag}", 0) | err
        for tag, fn in (("orders", orders), ("trades", lambda: loop.trades(cap))):
            eager, graph = time_calls(loop, fn)
            res["us_per_call"][f"{label}_{tag}_eager"], res["us_per_call"][f"{label}_{tag}_graph"] = eager, graph
        plain, with_reads = (min(res["us_per_step"][f"{label}_{t}"]) for t in ("plain", "with_reads"))
        res["us_per_step"][f"{label}_added_by_reads"] = with_reads - plain
        res["errors"][f"{label}_after_reads"] = int(np.bitwise_or.reduce(loop.env.env_errors()))
        loop.close()
    return res


def bench_resets(args, name, power):
    """--resets: see the module docstring."""
    import torch
    K, n_envs = 100, N_BOOKS // 2
    res = {"card": name, "power_limit": power, "engine": "fast", "agents": None, "steps_per_graph": K, "passes": args.passes,
           "rows_per_book": ROWS_PER_BOOK, "us_per_step": {}, "errors": {}}
    fractions = (("reset_0pct", 0.0), ("reset_1pct", 0.01), ("reset_100pct", 1.0))
    for label, units in (("vector_env_4096", n_envs), ("market_vector_2048x4", N_MARKETS)):
        books = units if label.startswith("vector") else N_BOOKS
        blocks = gym_action_blocks(min(args.blocks, K), books, ROWS_PER_BOOK, seed=5)
        if label.startswith("vector"):
            loop = gym.VectorEnv(n_envs, ROWS_PER_BOOK, 0, 0, 1, 1000, **KW)
        else:
            loop = gym.MarketVectorEnv(N_MARKETS, ROWS, 0, 0, [1] * ASSETS, 1000, **KW)
            blocks = market_blocks(blocks)
        d_blocks = [torch.from_numpy(x.view(np.uint8).reshape(units, -1)).cuda() for x in blocks]
        rng = np.random.default_rng(3)
        masks = {tag: torch.from_numpy(rng.permutation(units) < round(f * units)).cuda() for tag, f in fractions}
        stream = torch.cuda.Stream()
        loop.env.set_stream(stream.cuda_stream)
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):   # the first launches query kernel attributes: outside any capture
            loop.step(d_blocks[0])
            loop.reset(masks["reset_1pct"])
        graphs = {}
        for tag in ("plain",) + tuple(t for t, _ in fractions):
            loop.reset()   # (also restarts the history ring of VectorEnv.step, so no clear is captured)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for s in range(K):
                    loop.step(d_blocks[s % len(d_blocks)])
                    if tag != "plain":
                        loop.reset(masks[tag])
            graphs[tag] = g
        for _ in range(args.passes):   # plain and with-reset graphs alternate
            for tag, g in graphs.items():
                loop.reset()
                stream.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record(stream)
                with torch.cuda.stream(stream):
                    g.replay()
                t1.record(stream)
                stream.synchronize()
                res["us_per_step"].setdefault(f"{label}_{tag}", []).append(t0.elapsed_time(t1) * 1e3 / K)
                res["errors"][f"{label}_{tag}"] = res["errors"].get(f"{label}_{tag}", 0) | int(np.bitwise_or.reduce(loop.env.env_errors()))
        plain = min(res["us_per_step"][f"{label}_plain"])
        for tag, _ in fractions:
            res["us_per_step"][f"{label}_added_by_{tag}"] = min(res["us_per_step"][f"{label}_{tag}"]) - plain
        del graphs
        loop.env.set_stream(0)
        loop.close()
    return res


def bench_snapshots(args, name, power):
    """--snapshots: see the module docstring."""
    import torch
    R, n_envs = 50, N_BOOKS // 2
    c3 = workloads.c3_groups()
    agents_per_book = sum(int(g["n_agents"]) for g in c3)
    blob = 128 + (12 + 512) * 32   # the FAST engine's book blob: header, 32-entry page directory, 32 pages
    res = {"card": name, "power_limit": power, "engine": "fast", "agents": "C3 (50 + 50 RandomAgents) on every book",
           "warmup_steps": args.warmup_steps, "calls_per_graph": R, "passes": args.passes, "us_per_call": {}, "bytes_per_call": {},
           "GB_per_s": {}, "errors": {}}
    for label, units in (("vector_env_4096", n_envs), ("market_vector_2048x4", N_MARKETS)):
        books = units if label.startswith("vector") else N_BOOKS
        A = books // units
        blocks = gym_action_blocks(args.blocks, books, ROWS_PER_BOOK, seed=5)
        blocks["price"] = np.where((blocks["op_flags"] & abi.F_MARKET) != 0, blocks["price"], 2 * (40 + blocks["price"] % 21))
        if label.startswith("vector"):
            loop = gym.VectorEnv(n_envs, ROWS_PER_BOOK, 0, 0, 1, 1_000_000, agents=c3, agent_seed=5, **SNAP_KW)
        else:
            loop = gym.MarketVectorEnv(N_MARKETS, ROWS, 0, 0, [1] * ASSETS, 1_000_000, agents=c3_market_agents(), agent_seed=5, **SNAP_KW)
            blocks = market_blocks(blocks)
        d_blocks = [torch.from_numpy(x.view(np.uint8).reshape(units, -1)).cuda() for x in blocks]
        loop.reset()
        for s in range(args.warmup_steps):
            loop.step(d_blocks[s % len(d_blocks)])
        store = loop.snapshots(units)
        res[f"{label}_store_bytes"] = store.nbytes
        n_ord = np.array([loop.env.n_orders(b) for b in range(books)], np.int64)
        n_tr = np.array([loop.env.n_trades(b) for b in range(books)], np.int64)
        per_book = blob + 64 * np.minimum(n_ord, SNAP_KW["max_orders"]) + 32 * np.minimum(n_tr, SNAP_KW["max_trades"]) + 4 * agents_per_book
        per_unit = per_book.reshape(units, A).sum(axis=1)
        res[f"{label}_mean_orders_logged"], res[f"{label}_mean_trades_logged"] = float(n_ord.mean()), float(n_tr.mean())
        rng = np.random.default_rng(3)
        stream = torch.cuda.Stream()
        loop.env.set_stream(stream.cuda_stream)
        calls = {}
        for tag, f in (("1pct", 0.01), ("100pct", 1.0)):
            sel = rng.permutation(units) < round(f * units)
            own = np.where(sel, np.arange(units), gym.NO_SLOT).astype(np.uint32)   # unit u <-> slot u
            d_sel = torch.from_numpy(own.view(np.int32)).cuda()
            calls[f"save_{tag}"] = (lambda d=d_sel: loop.save(store, d), int(per_unit[sel].sum()))
            calls[f"restore_{tag}"] = (lambda d=d_sel: loop.restore(store, d), int(per_unit[sel].sum()))
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):   # every slot filled, and the first launches (attribute queries) outside any capture
            loop.save(store)
            for fn, _ in calls.values():
                fn()
        stream.synchronize()
        graphs = {}
        for tag, (fn, nbytes) in calls.items():
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for _ in range(R):
                    fn()
            graphs[tag] = g
            res["bytes_per_call"][f"{label}_{tag}"] = nbytes
        for _ in range(args.passes):
            for tag, g in graphs.items():
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record(stream)
                with torch.cuda.stream(stream):
                    g.replay()
                t1.record(stream)
                stream.synchronize()
                res["us_per_call"].setdefault(f"{label}_{tag}", []).append(t0.elapsed_time(t1) * 1e3 / R)
        for tag in graphs:
            best = min(res["us_per_call"][f"{label}_{tag}"])
            res["GB_per_s"][f"{label}_{tag}"] = res["bytes_per_call"][f"{label}_{tag}"] / best / 1e3
        res["errors"][label] = int(np.bitwise_or.reduce(loop.env.env_errors()))
        del graphs
        loop.env.set_stream(0)
        loop.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20, help="untimed steps after each reset")
    ap.add_argument("--blocks", type=int, default=64, help="distinct action blocks, cycled")
    ap.add_argument("--bg-agents", action="store_true", help="the C3 population trades in every book (see the module docstring)")
    ap.add_argument("--reads", action="store_true", help="time orders() / trades() in the C3 loops (see the module docstring)")
    ap.add_argument("--resets", action="store_true", help="time reset(mask) in the rows-only loops (see the module docstring)")
    ap.add_argument("--snapshots", action="store_true", help="time save / restore on warmed C3 books (see the module docstring)")
    ap.add_argument("--warmup-steps", type=int, default=300, help="--snapshots: C3 steps before the store is filled")
    ap.add_argument("--passes", type=int, default=3, help="--resets / --snapshots: timed passes of each variant")
    args = ap.parse_args()
    import torch

    name, power = card()
    print(f"card: {name}, power limit: {power}", flush=True)
    if args.reads:
        print(json.dumps(bench_reads(args, name, power)), flush=True)
        return
    if args.resets:
        print(json.dumps(bench_resets(args, name, power)), flush=True)
        return
    if args.snapshots:
        print(json.dumps(bench_snapshots(args, name, power)), flush=True)
        return
    blocks = gym_action_blocks(args.blocks, N_BOOKS, ROWS_PER_BOOK, seed=5)
    if args.bg_agents:   # limit prices into the agents' range, as bench.py run_gym does
        blocks["price"] = np.where((blocks["op_flags"] & abi.F_MARKET) != 0, blocks["price"], 2 * (40 + blocks["price"] % 21))
    mblocks = market_blocks(blocks)
    res = {"card": name, "power_limit": power, "markets": N_MARKETS, "assets": ASSETS, "rows_per_market": ROWS,
           "steps": args.steps, "warmup": args.warmup, "us_per_step": {}, "errors": {}}

    def as_device(b):
        return [torch.from_numpy(x.view(np.uint8).reshape(x.shape[0], -1)).cuda() for x in b]

    d_env, d_mkt = as_device(blocks), as_device(mblocks)
    torch.cuda.synchronize()
    if args.bg_agents:
        c3 = workloads.c3_groups()
        res["agents"] = "C3 (50 + 50 RandomAgents) on every book"
        agents = c3_market_agents()
        for eng, ekw in BG_ENGINES.items():
            v = gym.MarketVectorEnv(N_MARKETS, ROWS, 0, 0, [1] * ASSETS, 1_000_000, agents=agents, agent_seed=5, **BG_KW, **ekw)
            res["us_per_step"][f"market_vector_bg_{eng}"], res["errors"][f"market_vector_bg_{eng}"] = time_device(v, d_mkt, args.steps, args.warmup)
            v.close()
            ve = gym.VectorEnv(N_BOOKS, ROWS_PER_BOOK, 0, 0, 1, 1_000_000, agents=c3, agent_seed=5, **BG_KW, **ekw)
            res["us_per_step"][f"vector_env_bg_{eng}"], res["errors"][f"vector_env_bg_{eng}"] = time_device(ve, d_env, args.steps, args.warmup)
            ve.close()
        print(json.dumps(res), flush=True)
        return
    for eng, ekw in ENGINES.items():
        v = gym.MarketVectorEnv(N_MARKETS, ROWS, 0, 0, [1] * ASSETS, 1000, **KW, **ekw)
        res["us_per_step"][f"market_vector_{eng}"], res["errors"][f"market_vector_{eng}"] = time_device(v, d_mkt, args.steps, args.warmup)
        v.close()
        ve = gym.VectorEnv(N_BOOKS, ROWS_PER_BOOK, 0, 0, 1, 1000, **KW, **ekw)
        res["us_per_step"][f"vector_env_{eng}"], res["errors"][f"vector_env_{eng}"] = time_device(ve, d_env, args.steps, args.warmup)
        ve.close()
    # host path: the same market rows through MarketEnv.submit + step (no-op rows are not submitted)
    host = []
    for b in mblocks:
        f = b["op_flags"].ravel()
        keep = (f & 0xFF) != abi.OP_NOOP
        op = (f & 0xFF)[keep]
        mk = np.repeat(np.arange(N_MARKETS, dtype=np.uint32), ROWS)[keep]
        flags = np.where(f[keep] & abi.F_MARKET, abi.F_MARKET, abi.F_HAS_PRICE).astype(np.uint32)
        host.append(dict(action=op, asset=b["aux"].ravel()[keep], side=(f[keep] & abi.F_BID) != 0, vol=b["vol"].ravel()[keep],
                         trader=b["trader"].ravel()[keep], price=b["price"].ravel()[keep],
                         order_id=b["order_id"].ravel()[keep].astype(np.uint64), market=mk, flags=flags))
    m = market.MarketEnv(0, 0, [1] * ASSETS, 1000, n_markets=N_MARKETS, **KW)
    total, errors = 0.0, 0
    for pre, timed in windows(args.steps, args.warmup):
        m._env.reset()
        for s in range(pre):
            m.submit(**host[s % len(host)]); m.step()
        t0 = time.perf_counter()
        for s in range(pre, pre + timed):
            m.submit(**host[s % len(host)])
            m.step()   # (synchronous: bb_step checks the device's error flag)
        total += time.perf_counter() - t0
        errors |= int(np.bitwise_or.reduce(m.env_errors()))
    res["us_per_step"]["market_env_host"] = total * 1e6 / args.steps
    res["errors"]["market_env_host"] = errors
    m._env.close()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
