"""Synthetic workloads of BASELINE.json (made concrete in SURVEY.md 8d).

`replay_stream` builds config C2: a place/cancel/modify mix for ONE book as a packed ``bb_instr``
array (immediate-mode semantics, explicit time per instruction).  `c3_groups` / `c4_groups` are the
agent populations of configs C3 / C4.  Host-side generation only; nothing here touches book state.
"""
from __future__ import annotations

import numpy as np

from . import abi
from .core import momentum_group, random_group


def replay_stream(n: int, seed: int, tick_size: int = 1, mid_ticks: int = 1000, half_width: int = 64,
                  step_size: int = 100_000, emit_every: int = 64, max_vol: int = 100, trading_windows: bool = True,
                  time_mode: str = "strict", min_vol: int = 1) -> np.ndarray:
    """C2 stream: 55% limit, 5% market, 25% cancel, 15% modify (1/3 vol-only, 1/3 price-only, 1/3 both).

    time_mode: "strict" (t strictly increasing: +1 per event, +step_size every `emit_every`),
               "flat" (time never advances: exercises the reference's equal-key collisions, N1),
               "jitter" (time may move backwards: exercises sorted queue insertion).
    """
    rng = np.random.Generator(np.random.PCG64(seed))
    u = rng.random(n)
    op = np.full(n, abi.OP_MODIFY, dtype=np.uint32)
    op[u < 0.85] = abi.OP_CANCEL
    op[u < 0.60] = abi.OP_NEW
    market = (u >= 0.55) & (u < 0.60)
    flags = np.zeros(n, dtype=np.uint32)
    vol = rng.integers(min_vol, max_vol + 1, size=n, dtype=np.uint32)
    if trading_windows and n >= 2000:  # trading switched off for ~1% of the stream
        n_win = max(1, n // 5000)
        starts = rng.integers(0, n - 60, size=n_win)
        for s in starts:
            op[s], vol[s], market[s] = abi.OP_SET_TRADING, 0, False
            op[s + 50], vol[s + 50], market[s + 50] = abi.OP_SET_TRADING, 1, False
    is_new = op == abi.OP_NEW
    issued_before = np.cumsum(is_new) - is_new
    target = np.floor(rng.random(n) * np.maximum(issued_before, 1)).astype(np.uint32)
    needs_target = (op == abi.OP_CANCEL) | (op == abi.OP_MODIFY)
    op[needs_target & (issued_before == 0)] = abi.OP_NOOP
    side = rng.random(n) < 0.5
    price = (rng.integers(mid_ticks - half_width, mid_ticks + half_width + 1, size=n).astype(np.uint32) * tick_size).astype(np.uint32)
    kind = rng.integers(0, 3, size=n)
    is_mod = op == abi.OP_MODIFY
    flags[is_new & side] |= abi.F_BID
    flags[is_new & market] |= abi.F_MARKET
    flags[is_mod & (kind != 1)] |= abi.F_HAS_VOL
    flags[is_mod & (kind != 0)] |= abi.F_HAS_PRICE
    idx = np.arange(n, dtype=np.uint64)
    if emit_every:
        flags[(idx % emit_every) == emit_every - 1] |= abi.F_EMIT
    if time_mode == "strict":
        t = idx + 1 + (idx // max(emit_every, 1)) * step_size
    elif time_mode == "flat":
        t = np.zeros(n, dtype=np.uint64) + 5
    elif time_mode == "jitter":
        t = (rng.integers(0, 50, size=n) + (idx // 8)).astype(np.uint64)
    else:
        raise ValueError(time_mode)
    out = np.zeros(n, dtype=abi.INSTR_DTYPE)
    out["t"] = t
    out["op_flags"] = op | flags
    out["order_id"] = np.where(needs_target, target, 0)
    out["price"] = np.where(is_new & market, 0, price)
    out["vol"] = vol
    out["trader"] = rng.integers(0, 1000, size=n, dtype=np.uint32)
    return out


def c3_groups():
    """crates/step_sim/examples/random_agents/main.rs:10-19 — 50 + 50 RandomAgents."""
    return [random_group(50, (40, 60), (10, 20), 2, 0.8), random_group(50, (10, 90), (50, 70), 2, 0.2)]


def c3_groups_around(mid: int):
    """C3's two RandomAgents groups (same widths, volumes, rates and tick size 2) re-centred on the price `mid`: for a deep
    book's window, e.g. ticks (4990, 5010) and (4960, 5040) around the C5 mid of 10,000."""
    c = mid // 2
    return [random_group(50, (c - 10, c + 10), (10, 20), 2, 0.8), random_group(50, (c - 40, c + 40), (50, 70), 2, 0.2)]


def c4_groups():
    """SURVEY.md 8d config C4: 40 + 40 RandomAgents and a 20-trader MomentumAgent."""
    return [random_group(40, (40, 60), (10, 20), 2, 0.8), random_group(40, (10, 90), (50, 70), 2, 0.2),
            momentum_group(80, 20, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0)]


def market_example_groups():
    """crates/step_sim/examples/multi_asset/main.rs:15-20 — MarketEnv::<2>, (50 + 50) RandomMarketAgents on each asset.
    Returns (groups, asset of each group) for BatchedEnv.set_agents(groups, assets=...)."""
    return c3_groups() + c3_groups(), [0, 0, 1, 1]


def algorithmic_bytes(stats: dict, obs_words: int, ext_instructions: int = 0) -> int:
    """SURVEY.md 8d: 25*I_ext + 42*N_created + 26*N_transitions + 33*N_trades + OBS*E."""
    return (25 * ext_instructions + 42 * stats["orders_created"] + 26 * stats["transitions"] + 33 * stats["trades"]
            + 4 * obs_words * stats["env_steps"])


def c5_stream(n_resting: int, n_steps: int, events_per_step: int, seed: int, mid_ticks: int = 10_000, depth_ticks: int = 2048,
              step_size: int = 1_000_000) -> np.ndarray:
    """Config C5 (deep-book stress, SURVEY.md 8d) for ONE book as a replay stream.

    Phase 1 pre-loads `n_resting` non-crossing limit orders, half per side, uniformly over `depth_ticks` ticks per side
    (bids below `mid_ticks`, asks above), vol U{1..50}.  Phase 2 is `n_steps` x `events_per_step` events: 15% cancel and
    15% modify (1/3 vol-only, 1/3 price-only, 1/3 both) with targets uniform over every id issued so far, 60% new limit
    orders within +-32 ticks of `mid_ticks` (either side, so about half of them cross), 10% market orders; a level-2 record
    is emitted at the end of every step.  Time is strictly increasing (+1 per event, +step_size per step)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n2 = n_steps * events_per_step
    n = n_resting + n2
    out = np.zeros(n, dtype=abi.INSTR_DTYPE)
    idx = np.arange(n, dtype=np.uint64)
    # phase 1
    side1 = rng.random(n_resting) < 0.5
    off = rng.integers(1, depth_ticks + 1, size=n_resting)
    price1 = np.where(side1, mid_ticks - off, mid_ticks + off).astype(np.uint32)
    out["op_flags"][:n_resting] = abi.OP_NEW | np.where(side1, abi.F_BID, 0).astype(np.uint32)
    out["price"][:n_resting] = price1
    out["vol"][:n_resting] = rng.integers(1, 51, size=n_resting, dtype=np.uint32)
    # phase 2
    u = rng.random(n2)
    op = np.full(n2, abi.OP_NEW, dtype=np.uint32)
    op[u < 0.30] = abi.OP_MODIFY
    op[u < 0.15] = abi.OP_CANCEL
    market = u >= 0.90
    is_new = op == abi.OP_NEW
    side2 = rng.random(n2) < 0.5
    flags = np.zeros(n2, dtype=np.uint32)
    flags[is_new & side2] |= abi.F_BID
    flags[is_new & market] |= abi.F_MARKET
    kind = rng.integers(0, 3, size=n2)
    is_mod = op == abi.OP_MODIFY
    flags[is_mod & (kind != 1)] |= abi.F_HAS_VOL
    flags[is_mod & (kind != 0)] |= abi.F_HAS_PRICE
    issued_before = n_resting + np.cumsum(is_new) - is_new
    target = np.floor(rng.random(n2) * issued_before).astype(np.uint32)
    price2 = rng.integers(mid_ticks - 32, mid_ticks + 33, size=n2).astype(np.uint32)
    k = np.arange(n2)
    flags[(k % events_per_step) == events_per_step - 1] |= abi.F_EMIT
    out["op_flags"][n_resting:] = op | flags
    out["order_id"][n_resting:] = np.where(is_new, 0, target)
    out["price"][n_resting:] = np.where(is_new & market, 0, price2)
    out["vol"][n_resting:] = rng.integers(1, 51, size=n2, dtype=np.uint32)
    out["trader"] = (idx % 1000).astype(np.uint32)
    t = idx + 1
    t[n_resting:] += (k // events_per_step).astype(np.uint64) * np.uint64(step_size)
    out["t"] = t
    return out


def shallow_replay_stream(n: int, seed: int, tick_size: int = 1, mid_ticks: int = 1000, half_width: int = 24,
                          max_live: int = 120, step_size: int = 100_000, emit_every: int = 64, max_vol: int = 100) -> np.ndarray:
    """C2-style replay stream for SHALLOW books (the dense-window engine's domain): 45% limit, 5% market, 35% cancel,
    15% modify.  The generator tracks the ids that may still rest (issued as limit orders, not yet cancelled): cancels
    take the oldest of them, modifies a random one, and a limit order issued while `max_live` ids are outstanding is
    turned into a cancel, so at most `max_live` orders ever rest.  Time is strictly increasing; trading is switched
    off for ~1% windows (limit orders then rest unmatched, N6)."""
    from collections import deque

    rng = np.random.Generator(np.random.PCG64(seed))
    u = rng.random(n)
    vol = rng.integers(1, max_vol + 1, size=n, dtype=np.uint32)
    side = rng.random(n) < 0.5
    price = (rng.integers(mid_ticks - half_width, mid_ticks + half_width + 1, size=n).astype(np.uint32) * tick_size).astype(np.uint32)
    kind = rng.integers(0, 3, size=n)
    pick = rng.random(n)
    toggles = {}
    if n >= 2000:
        for s in rng.integers(0, n - 60, size=max(1, n // 5000)):
            toggles[int(s)] = 0
            toggles[int(s) + 50] = 1
    out = np.zeros(n, dtype=abi.INSTR_DTYPE)
    fifo, issued = deque(), 0
    for i in range(n):
        of, oid, p, v = abi.OP_NOOP, 0, 0, int(vol[i])
        if i in toggles:
            of, v = abi.OP_SET_TRADING, toggles[i]
        elif u[i] < 0.45 and len(fifo) < max_live:      # limit order
            of, p = abi.OP_NEW | (abi.F_BID if side[i] else 0), int(price[i])
            fifo.append(issued)
            issued += 1
        elif 0.45 <= u[i] < 0.50:                        # market order
            of = abi.OP_NEW | abi.F_MARKET | (abi.F_BID if side[i] else 0)
            issued += 1
        elif u[i] < 0.85:                                # cancel the oldest outstanding id (also when the book is "full")
            if fifo:
                of, oid = abi.OP_CANCEL, fifo.popleft()
        elif fifo:                                       # modify a random outstanding id
            oid = fifo[int(pick[i] * len(fifo))]
            of = abi.OP_MODIFY | (abi.F_HAS_VOL if kind[i] != 1 else 0) | (abi.F_HAS_PRICE if kind[i] != 0 else 0)
            p = int(price[i])
        if (i % emit_every) == emit_every - 1:
            of |= abi.F_EMIT
        out[i] = (i + 1 + (i // emit_every) * step_size, of, oid, p, v, i % 1000, 0)
    return out
