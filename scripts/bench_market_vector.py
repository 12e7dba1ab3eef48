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

    python scripts/bench_market_vector.py --steps 1000 --warmup 20
    python scripts/bench_market_vector.py --bg-agents --steps 1000 --warmup 20
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


def time_device(loop, d_blocks, steps, warmup):
    """us per `loop.step` on a stream of its own: CUDA events around the timed steps of each window, summed."""
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
        t1.record(stream)
        stream.synchronize()
        total += t0.elapsed_time(t1) * 1e3
        errors |= int(np.bitwise_or.reduce(loop.env.env_errors()))
    loop.env.set_stream(0)
    return total / steps, errors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20, help="untimed steps after each reset")
    ap.add_argument("--blocks", type=int, default=64, help="distinct action blocks, cycled")
    ap.add_argument("--bg-agents", action="store_true", help="the C3 population trades in every book (see the module docstring)")
    args = ap.parse_args()
    import torch

    name, power = card()
    print(f"card: {name}, power limit: {power}", flush=True)
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
        agents = []
        for a in range(ASSETS):
            for g in c3:
                agents.append(market.RandomMarketAgents(a, int(g["n_agents"]), (int(g["tick_lo"]), int(g["tick_hi"])),
                                                        (int(g["vol_lo"]), int(g["vol_hi"])), int(g["tick_size"]), float(g["rate"])))
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
