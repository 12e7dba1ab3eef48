"""Drop-in mirror of the reference's Python extension module ``bourse.core``.

Same class names, constructor/method signatures, return layouts and error behaviour as the PyO3
classes (reference: ``rust/src/order_book.rs:35-398``, ``rust/src/step_sim.rs:55-608``,
``rust/src/step_sim_numpy.rs:66-517``, tuples ``rust/src/types.rs:4-40``), backed by the CUDA library
through the C ABI (``include/bourse_b200.h``) — every book lives on the GPU and every mutation is a
kernel launch.  There is no CPU implementation behind these classes.

``BatchedEnv`` is the native shape of the new framework: thousands of independent envs advanced in
lockstep, with the same per-env semantics.
"""
from __future__ import annotations

import ctypes as C
import math
import typing

import numpy as np

from . import abi

MAX_PRICE = 2**32 - 1


class PanicException(Exception):
    """Raised where the reference would panic (e.g. an unknown order id, orderbook.rs:642)."""


def _check(lib, h, rc):
    if rc == abi.BB_OK:
        return
    msg = lib.bb_last_error(h)
    msg = msg.decode() if msg else f"bourse_b200 error {rc}"
    if rc == abi.BB_EPRICE:
        raise ValueError(msg)
    if rc == abi.BB_EBADID:
        raise PanicException(msg)
    if rc == abi.BB_ECAP:
        raise MemoryError(msg)
    if rc == abi.BB_EINVAL:
        raise ValueError(msg)
    raise RuntimeError(msg)


class BatchedEnv:
    """`n_envs` independent Env instances (crates/step_sim/src/env.rs:58-71) on one GPU.

    Price ladder capacity: each book holds `pages_total` 32-level price pages (per side and 32-price
    block), `pages_smem` of them resident in shared memory.  With `pages_total == pages_smem` (the
    default, 10) and `price_granule == 1` the specialised kernels run; a book that needs more pages
    flags BB_ERR_CAP_PAGES.  Give `pages_total > pages_smem` for wide or deep books (HBM pages).

    `price_window=(lo, hi)` selects the dense-window engine instead (include/bourse_b200.h, bb_config.win_levels):
    fastest for shallow books whose resting prices stay in [lo, hi) with at most `live_cap` (default 128, max 254)
    resting orders per book; leaving those limits flags an env error rather than producing different results.

    `deep_chunks=N` (with `price_window`, up to 8192 levels) selects the deep-book engine: one CTA per book (fetch / chain /
    replay / retire warps, csrc/deepw.cuh) and chunked array queues in HBM (N 256-byte chunks of 31 queue entries per book)
    — for books with ~10^6 resting orders, driven by replayed streams (`replay`, `replay_device`) or by device-resident Env
    steps (`step_device`, `gym.VectorEnv`; rows as on the other engines, `step_size >= max_queue`), with or without in-kernel
    agents (`set_agents`: RandomAgents price ranges inside the window; `run_agents`, `run_agents_with_rows`).  The
    host-queued Env calls (`submit`, `step`) raise.

    `assets=A` (> 1) groups consecutive books into multi-asset markets with MarketEnv semantics
    (crates/step_sim/src/market_env.rs:108-121); see `bourse_b200.market`.

    `tick_size` is one tick for every env, or a sequence of `n_envs` ticks, one per env (bb_set_tick_sizes): each book then
    checks limit prices against its own tick and lays out its level-2 record at its own tick offsets.  Without an explicit
    `price_granule` or `price_window` the ladder granule of a sequence is the gcd of its ticks.  On the paged engine a book
    whose tick is k times the granule spreads its levels k times more thinly over the 32-price pages and may need a larger
    `pages_total`; the dense and deep engines are unaffected."""

    def __init__(self, n_envs: int, seed: int, start_time: int, tick_size: typing.Union[int, typing.Sequence[int]], step_size: int,
                 trading: bool = True, *,
                 device: int = 0, env_id_base: int = 0, obs_words: int = abi.OBS_L2, max_orders: int = 1 << 16,
                 max_trades: int = 1 << 16, max_steps: int = 1 << 12, max_queue: int = 256, pages_smem: int = 0,
                 pages_total: int = 0, price_granule: int = 0, price_window: typing.Optional[typing.Tuple[int, int]] = None,
                 live_cap: int = 0, assets: int = 0, deep_chunks: int = 0):
        self._lib = abi.load()
        ticks = None
        if not isinstance(tick_size, (int, np.integer)):
            ticks = [int(t) for t in tick_size]
            if len(ticks) != n_envs:
                raise ValueError(f"tick_size: one tick per env expected ({n_envs}), got {len(ticks)}")
            if min(ticks) <= 0:
                raise ValueError("tick sizes must be > 0")
            tick_size = math.gcd(*ticks)   # the paged engine's ladder granule: every book's prices are multiples of it
        cfg = abi.Config()
        cfg.struct_size = C.sizeof(abi.Config)
        cfg.device, cfg.n_envs, cfg.env_id_base = device, n_envs, env_id_base
        cfg.start_time, cfg.step_size, cfg.seed = start_time, step_size, seed
        cfg.tick_size, cfg.price_granule, cfg.trading = tick_size, price_granule, int(trading)
        cfg.obs_words, cfg.max_orders, cfg.max_trades = obs_words, max_orders, max_trades
        cfg.max_steps, cfg.max_queue = max_steps, max_queue
        cfg.pages_smem, cfg.pages_total = pages_smem, pages_total
        cfg.assets = assets   # > 1: books [m * assets, (m + 1) * assets) form one market (shared shuffled queue per step)
        if price_window is not None:   # dense-window engine for shallow books: prices in [lo, hi), <= live_cap resting orders
            lo, hi = price_window
            if hi <= lo:
                raise ValueError("price_window must be (lo, hi) with hi > lo")
            cfg.win_lo, cfg.win_levels, cfg.live_cap = lo, hi - lo, live_cap
            cfg.price_granule = 1
        # deep-book engine (csrc/deep.cuh): one CTA per book, replayed streams only; needs price_window as well
        if deep_chunks and price_window is None:
            raise ValueError("deep_chunks needs price_window=(lo, hi) (at most 8192 levels)")
        cfg.deep_chunks = deep_chunks
        self._h = C.c_void_p()
        self.n_envs, self.obs_words, self.device = n_envs, obs_words, device
        self.tick_size = int(tick_size)   # a sequence of ticks: their gcd (`tick_sizes` holds each env's)
        self.tick_sizes = np.full(n_envs, tick_size, dtype=np.uint32)
        self.max_orders, self.max_trades, self.max_steps, self.max_queue = max_orders, max_trades, max_steps, max_queue
        rc = self._lib.bb_create(C.byref(cfg), C.byref(self._h))
        if rc != abi.BB_OK:
            msg = self._lib.bb_last_error(None)
            self._h = C.c_void_p()
            raise RuntimeError(f"bb_create failed ({rc}): {msg.decode() if msg else ''}")
        if ticks is not None and any(t != tick_size for t in ticks):
            try:
                self.set_tick_sizes(ticks)
            except Exception:
                self.close()
                raise

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.bb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        _check(self._lib, self._h, rc)

    # ------------------------------------------------------------------ control
    def reserve(self, max_orders: int = 0, max_trades: int = 0, max_steps: int = 0):
        """Grow the per-env order table / trade log / history to at least these capacities (bb_reserve); contents are kept."""
        self._ck(self._lib.bb_reserve(self._h, max_orders, max_trades, max_steps))
        self.max_orders, self.max_steps = max(self.max_orders, max_orders), max(self.max_steps, max_steps)
        if self.max_trades:
            self.max_trades = max(self.max_trades, max_trades)

    def reserve_queue(self, max_queue: int):
        """Grow the number of transactions one env may queue for one step (bb_reserve_queue); MemoryError when the step's
        shuffle would no longer fit in shared memory."""
        self._ck(self._lib.bb_reserve_queue(self._h, max_queue))
        self.max_queue = max(self.max_queue, max_queue)

    def grow_if_needed(self, env: int = 0, headroom_orders: int = 0, headroom_steps: int = 0, headroom_trades: int = 0):
        """Single-env convenience used by OrderBook / StepEnv: double a table once it is more than half full (plus the
        given headroom), so that the classes grow without bound like the reference's Vecs."""
        o, t, s = self.n_orders(env) + headroom_orders, self.n_trades(env) + headroom_trades, self.n_steps(env) + headroom_steps
        want_o = 2 * self.max_orders if 2 * o > self.max_orders else 0
        want_t = 2 * self.max_trades if self.max_trades and 2 * t > self.max_trades else 0
        want_s = 2 * self.max_steps if 2 * s > self.max_steps else 0
        if want_o or want_t or want_s:
            self.reserve(max(want_o, 2 * o if want_o else 0), max(want_t, 4 * t if want_t else 0), max(want_s, 2 * s if want_s else 0))

    def clear_history(self):
        """Restart every env's per-step record history at 0 (bb_clear_history); books and logs are untouched."""
        self._ck(self._lib.bb_clear_history(self._h))

    def clear_errors(self):
        """Zero every env's sticky error word (bb_clear_errors)."""
        self._ck(self._lib.bb_clear_errors(self._h))

    def set_tick_sizes(self, ticks):
        """Give each book its own tick (bb_set_tick_sizes; MarketEnv::new, market_env.rs:73-90): `n_envs` ticks, or on a
        multi-asset handle `assets` ticks (asset a's tick for book a of every market).  ValueError, nothing changed, for a
        tick of 0 or one that is not a multiple of the price granule, or while any env holds orders or queued transactions
        (`reset()` first).  The ticks survive `reset()`."""
        t = np.ascontiguousarray(ticks, dtype=np.uint32)
        self._ck(self._lib.bb_set_tick_sizes(self._h, abi.ptr(t), len(t)))
        self.tick_sizes = np.resize(t, self.n_envs) if len(t) != self.n_envs else t.copy()

    def reset(self): self._ck(self._lib.bb_reset(self._h))
    def synchronize(self): self._ck(self._lib.bb_synchronize(self._h))
    def set_stream(self, cuda_stream: int): self._ck(self._lib.bb_set_stream(self._h, C.c_void_p(cuda_stream)))
    def set_trading(self, on: bool, env: int = abi.ALL_ENVS): self._ck(self._lib.bb_set_trading(self._h, env, int(on)))
    def set_time(self, env: int, t: int): self._ck(self._lib.bb_set_time(self._h, env, t))

    def time(self, env: int = 0) -> int:
        t = C.c_uint64()
        self._ck(self._lib.bb_time(self._h, env, C.byref(t)))
        return t.value

    # ------------------------------------------------------------------ Env mode
    def submit(self, action, side=None, vol=None, trader=None, price=None, order_id=None, env=None, flags=None):
        """Batched Env::place_order / cancel_order / modify_order; returns u64 ids (NO_ID where none)."""
        action = np.ascontiguousarray(action, dtype=np.uint32)
        n = len(action)

        def arr(x, dt):
            if x is None:
                return None
            x = np.ascontiguousarray(x, dtype=dt)
            if len(x) != n:
                raise ValueError("instruction arrays must have equal length")
            return x

        if side is not None:
            side = arr(np.asarray(side).astype(np.uint8), np.uint8)
        vol, trader, price = arr(vol, np.uint32), arr(trader, np.uint32), arr(price, np.uint32)
        order_id, env, flags = arr(order_id, np.uint64), arr(env, np.uint32), arr(flags, np.uint32)
        out = np.empty(n, dtype=np.uint64)
        done = C.c_uint64()
        rc = self._lib.bb_submit(self._h, n, abi.ptr(env), abi.ptr(action), abi.ptr(side), abi.ptr(vol), abi.ptr(trader),
                                 abi.ptr(price), abi.ptr(order_id), abi.ptr(flags), abi.ptr(out), C.byref(done))
        self._ck(rc)
        return out

    def step(self, n_steps: int = 1): self._ck(self._lib.bb_step(self._h, n_steps))

    # ------------------------------------------------------------------ device-resident loop (bourse_b200.gym)
    def step_device(self, d_instrs_ptr: int, d_offsets_ptr: int, n_rows: int, d_out_ids_ptr: int = 0, d_obs_ptr: int = 0):
        """One Env::step whose instruction rows are already in device memory (bb_step_device); asynchronous.  `d_obs_ptr`:
        device buffer [n_envs, obs_words] that receives the end-of-step observation records from the same launch."""
        self._ck(self._lib.bb_step_device(self._h, C.c_void_p(d_instrs_ptr), C.c_void_p(d_offsets_ptr), n_rows,
                                          C.c_void_p(d_out_ids_ptr) if d_out_ids_ptr else None,
                                          C.c_void_p(d_obs_ptr) if d_obs_ptr else None))

    def step_device_market(self, d_instrs_ptr: int, d_offsets_ptr: int, n_rows: int, d_out_ids_ptr: int = 0, d_obs_ptr: int = 0):
        """One MarketEnv::step for every market of a multi-asset handle whose rows are already in device memory
        (bb_step_device_market); asynchronous.  `d_offsets_ptr`: u64 [n_markets + 1] delimiting each market's rows; each
        row's `aux` is its asset.  `d_out_ids_ptr` receives the per-book ids, `d_obs_ptr` [n_envs, obs_words] the records."""
        self._ck(self._lib.bb_step_device_market(self._h, C.c_void_p(d_instrs_ptr), C.c_void_p(d_offsets_ptr), n_rows,
                                                 C.c_void_p(d_out_ids_ptr) if d_out_ids_ptr else None,
                                                 C.c_void_p(d_obs_ptr) if d_obs_ptr else None))

    def run_agents_with_rows(self, seed: int, d_instrs_ptr: int, d_offsets_ptr: int, n_rows: int, d_out_ids_ptr: int = 0,
                             d_obs_ptr: int = 0):
        """One env-step of { built-in agents update; the caller's device-resident rows; Env::step } (bb_run_agents_with_rows)."""
        self._ck(self._lib.bb_run_agents_with_rows(self._h, seed, C.c_void_p(d_instrs_ptr), C.c_void_p(d_offsets_ptr), n_rows,
                                                   C.c_void_p(d_out_ids_ptr) if d_out_ids_ptr else None,
                                                   C.c_void_p(d_obs_ptr) if d_obs_ptr else None))

    def run_agents_with_rows_market(self, seed: int, d_instrs_ptr: int, d_offsets_ptr: int, n_rows: int, d_out_ids_ptr: int = 0,
                                    d_obs_ptr: int = 0):
        """One market step of { market agents update; the caller's device-resident rows; MarketEnv::step } for every market
        of a multi-asset handle with market agents (bb_run_agents_with_rows_market); asynchronous.  Rows, offsets and ids
        are laid out as for `step_device_market`."""
        self._ck(self._lib.bb_run_agents_with_rows_market(self._h, seed, C.c_void_p(d_instrs_ptr), C.c_void_p(d_offsets_ptr), n_rows,
                                                          C.c_void_p(d_out_ids_ptr) if d_out_ids_ptr else None,
                                                          C.c_void_p(d_obs_ptr) if d_obs_ptr else None))

    def orders_device(self, d_ids_ptr: int, d_assets_ptr: int, n_per_unit: int, side_is_bid: int = 0, status: int = 0,
                      arr_time: int = 0, end_time: int = 0, vol: int = 0, start_vol: int = 0, price: int = 0, trader: int = 0):
        """Order records of a [units, n_per_unit] block of device-resident ids (bb_orders_device); asynchronous.  A unit is an
        env, or a market on a multi-asset handle, where `d_assets_ptr` ([units, n_per_unit] u32) names each query's asset
        (0 on a single-asset handle).  The keyword arguments are device pointers of the [units, n_per_unit] output columns;
        0 skips a column."""
        p = C.c_void_p
        self._ck(self._lib.bb_orders_device(self._h, p(d_ids_ptr), p(d_assets_ptr), n_per_unit, p(side_is_bid), p(status), p(arr_time),
                                            p(end_time), p(vol), p(start_vol), p(price), p(trader)))

    def trades_device(self, d_cursor_ptr: int, cap: int, count: int = 0, t: int = 0, side_is_bid: int = 0, price: int = 0,
                      vol: int = 0, active_id: int = 0, passive_id: int = 0):
        """Each book's trades since `d_cursor_ptr[book]` (u32 [n_envs], advanced) into [n_envs, cap] device columns
        (bb_trades_device); asynchronous.  `count` (u32 [n_envs]) receives the number of trades each book had to report."""
        p = C.c_void_p
        self._ck(self._lib.bb_trades_device(self._h, p(d_cursor_ptr), cap, p(count), p(t), p(side_is_bid), p(price), p(vol),
                                            p(active_id), p(passive_id)))

    def reset_device(self, mask_ptr: int, seeds_ptr: int = 0, obs_ptr: int = 0, cursor_ptr: int = 0):
        """Reset the units (envs, or markets on a multi-asset handle) whose u8 entry of the device mask `mask_ptr` is
        non-zero (bb_reset_device); asynchronous.  `seeds_ptr`: u64 [units] re-seeding them, or 0 to continue their random
        streams.  `obs_ptr` [n_envs, obs_words] receives the fresh records of reset books, `cursor_ptr` (u32 [n_envs], a
        trades_device cursor) has their entries zeroed."""
        p = C.c_void_p
        self._ck(self._lib.bb_reset_device(self._h, p(mask_ptr), p(seeds_ptr or None), p(obs_ptr or None), p(cursor_ptr or None)))

    def set_agent_params_device(self, params_ptr: int, keys_ptr: int = 0, mask_ptr: int = 0):
        """Per-unit agent parameters and Philox keys (bb_set_agent_params_device): the units (envs, or markets) whose u8
        entry of the device mask `mask_ptr` is non-zero (0: every unit) take their row of the device records `params_ptr`
        ([units][n_groups] bb_agent_group, 0 keeps the records) and their u64 key of `keys_ptr` (0 keeps the keys).  A unit
        with a record outside the declared population is flagged BB_ERR_PARAMS and keeps what it had; asynchronous."""
        p = C.c_void_p
        self._ck(self._lib.bb_set_agent_params_device(self._h, p(params_ptr or None), p(keys_ptr or None), p(mask_ptr or None)))

    def store_create(self, n_slots: int, allocate: bool = True) -> typing.Tuple[int, int]:
        """(store handle, bytes) of a device store of `n_slots` unit snapshots (bb_store_create), sized from the current
        capacities; with `allocate=False` only the size is computed and the handle is 0.  Free it with `store_destroy`
        (the env's `close` frees every store left)."""
        s, nbytes = C.c_void_p(), C.c_uint64()
        self._ck(self._lib.bb_store_create(self._h, n_slots, C.byref(s) if allocate else None, C.byref(nbytes)))
        return (s.value or 0), nbytes.value

    def store_destroy(self, store: int): self._ck(self._lib.bb_store_destroy(C.c_void_p(store)))

    def save_device(self, store: int, units_ptr: int):
        """Slot k of `store` receives unit u32 [n_slots] `units_ptr`[k] (bb_save_device; NO_SLOT keeps the slot, a unit
        index >= units empties it); asynchronous."""
        self._ck(self._lib.bb_save_device(self._h, C.c_void_p(store), C.c_void_p(units_ptr)))

    def restore_device(self, store: int, slots_ptr: int, seeds_ptr: int = 0, obs_ptr: int = 0, cursor_ptr: int = 0):
        """Unit u takes the state saved in slot u32 [units] `slots_ptr`[u] of `store` (bb_restore_device; NO_SLOT leaves it);
        `seeds_ptr` u64 [units] re-seeds the restored units' shuffle streams, 0 takes the slot's.  `obs_ptr` [n_envs,
        obs_words] receives the restored books' records, `cursor_ptr` (a trades_device cursor) their logged trade counts;
        asynchronous."""
        p = C.c_void_p
        self._ck(self._lib.bb_restore_device(self._h, p(store), p(slots_ptr), p(seeds_ptr or None), p(obs_ptr or None),
                                             p(cursor_ptr or None)))

    def level_2_data_device(self, d_out_ptr: int): self._ck(self._lib.bb_level2_device(self._h, C.c_void_p(d_out_ptr)))
    def level_1_data_device(self, d_out_ptr: int): self._ck(self._lib.bb_level1_device(self._h, C.c_void_p(d_out_ptr)))

    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._ck(self._lib.bb_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr: int): self._ck(self._lib.bb_device_free(self._h, C.c_void_p(ptr)))

    def memcpy(self, dst: int, src: int, nbytes: int, kind: int):
        """kind 1 host->device, 2 device->host, 3 device->device; synchronous on the env's stream."""
        self._ck(self._lib.bb_memcpy(self._h, C.c_void_p(dst), C.c_void_p(src), nbytes, kind))

    # ------------------------------------------------------------------ immediate mode / replay
    def replay(self, instrs: np.ndarray, env_offsets=None):
        instrs = np.ascontiguousarray(instrs, dtype=abi.INSTR_DTYPE)
        if env_offsets is None:
            if self.n_envs != 1:
                raise ValueError("env_offsets required when n_envs > 1")
            env_offsets = np.array([0, len(instrs)], dtype=np.uint64)
        env_offsets = np.ascontiguousarray(env_offsets, dtype=np.uint64)
        if len(env_offsets) != self.n_envs + 1 or env_offsets[-1] != len(instrs):
            raise ValueError("env_offsets must have n_envs + 1 entries ending at len(instrs)")
        self._ck(self._lib.bb_replay(self._h, abi.ptr(instrs), abi.ptr(env_offsets)))

    def replay_device(self, d_instrs_ptr: int, d_offsets_ptr: int):
        self._ck(self._lib.bb_replay_device(self._h, C.c_void_p(d_instrs_ptr), C.c_void_p(d_offsets_ptr)))

    # ------------------------------------------------------------------ in-kernel agents
    def set_agents(self, groups, assets=None):
        """Define the in-kernel agent set.  `assets` (multi-asset handles only): the asset each group trades, i.e. the
        *Market twin of the group's agent type (bb_set_agents_market)."""
        arr = np.zeros(len(groups), dtype=abi.GROUP_DTYPE)
        for i, g in enumerate(groups):
            arr[i] = g
        if assets is None:
            self._ck(self._lib.bb_set_agents(self._h, abi.ptr(arr), len(arr)))
        else:
            a = np.ascontiguousarray(assets, dtype=np.uint32)
            if len(a) != len(arr):
                raise ValueError("one asset index per agent group")
            self._ck(self._lib.bb_set_agents_market(self._h, abi.ptr(arr), abi.ptr(a), len(arr)))

    def run_agents(self, n_steps: int, seed: int, sync: bool = True):
        self._ck(self._lib.bb_run_agents(self._h, seed, n_steps))
        if sync:
            self.synchronize()

    def run_agents_to_host(self, n_steps: int, seed: int, out: typing.Optional[np.ndarray] = None,
                           chunk_steps: int = 0) -> np.ndarray:
        """`run_agents` with the observation history streamed into `out[n_envs, n_steps, obs_words]` (host memory,
        ideally pinned) while the simulation runs; returns `out`."""
        if out is None:
            out = np.empty((self.n_envs, n_steps, self.obs_words), dtype=np.uint32)
        assert out.shape == (self.n_envs, n_steps, self.obs_words) and out.dtype == np.uint32 and out.flags.c_contiguous
        self._ck(self._lib.bb_run_agents_to_host(self._h, seed, n_steps, chunk_steps, abi.ptr(out)))
        return out

    # ------------------------------------------------------------------ reads
    def level_1_data(self) -> np.ndarray:
        out = np.empty((self.n_envs, 9), dtype=np.uint32)
        self._ck(self._lib.bb_level1(self._h, abi.ptr(out)))
        return out

    def level_2_data(self) -> np.ndarray:
        out = np.empty((self.n_envs, 45), dtype=np.uint32)
        self._ck(self._lib.bb_level2(self._h, abi.ptr(out)))
        return out

    def book_level_1(self, env: int = 0) -> np.ndarray:
        out = np.empty(8, dtype=np.uint32)
        self._ck(self._lib.bb_book_level1(self._h, env, abi.ptr(out)))
        return out

    def book_level_2(self, env: int = 0) -> np.ndarray:
        out = np.empty(45, dtype=np.uint32)
        self._ck(self._lib.bb_book_level2(self._h, env, abi.ptr(out)))
        return out

    def n_steps(self, env: int = 0) -> int:
        n = C.c_uint32()
        self._ck(self._lib.bb_n_steps(self._h, env, C.byref(n)))
        return n.value

    def history(self, env: int = 0, first: int = 0, n: typing.Optional[int] = None) -> np.ndarray:
        if n is None:
            n = self.n_steps(env) - first
        out = np.empty((n, self.obs_words), dtype=np.uint32)
        self._ck(self._lib.bb_history(self._h, env, first, n, abi.ptr(out)))
        return out

    def history_all(self, n_steps: int, out: typing.Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty((self.n_envs, n_steps, self.obs_words), dtype=np.uint32)
        self._ck(self._lib.bb_history_all(self._h, n_steps, abi.ptr(out)))
        return out

    def n_orders(self, env: int = 0) -> int:
        n = C.c_uint64()
        self._ck(self._lib.bb_n_orders(self._h, env, C.byref(n)))
        return n.value

    def n_trades(self, env: int = 0) -> int:
        n = C.c_uint64()
        self._ck(self._lib.bb_n_trades(self._h, env, C.byref(n)))
        return n.value

    def orders_arrays(self, env: int = 0):
        n = self.n_orders(env)
        cols = dict(side=np.empty(n, np.uint8), status=np.empty(n, np.uint8), arr_time=np.empty(n, np.uint64),
                    end_time=np.empty(n, np.uint64), vol=np.empty(n, np.uint32), start_vol=np.empty(n, np.uint32),
                    price=np.empty(n, np.uint32), trader=np.empty(n, np.uint32))
        self._ck(self._lib.bb_orders(self._h, env, 0, n, *[abi.ptr(c) for c in cols.values()]))
        return cols

    def trades_arrays(self, env: int = 0):
        n = self.n_trades(env)
        cols = dict(t=np.empty(n, np.uint64), side=np.empty(n, np.uint8), price=np.empty(n, np.uint32),
                    vol=np.empty(n, np.uint32), active=np.empty(n, np.uint64), passive=np.empty(n, np.uint64))
        self._ck(self._lib.bb_trades(self._h, env, 0, n, *[abi.ptr(c) for c in cols.values()]))
        return cols

    def orders_all(self, cap_per_env: int, out: typing.Optional[np.ndarray] = None):
        """Every env's order table in one strided copy (bb_orders_all): (records [n_envs, cap_per_env] of abi.ORDER_REC_DTYPE,
        counts [n_envs]).  `out`: a preallocated (ideally pinned) array to fill."""
        if out is None:
            out = np.empty((self.n_envs, cap_per_env), dtype=abi.ORDER_REC_DTYPE)
        assert out.shape == (self.n_envs, cap_per_env) and out.dtype == abi.ORDER_REC_DTYPE and out.flags.c_contiguous
        counts = np.empty(self.n_envs, dtype=np.uint32)
        self._ck(self._lib.bb_orders_all(self._h, cap_per_env, abi.ptr(out), abi.ptr(counts)))
        return out, counts

    def trades_all(self, cap_per_env: int, out: typing.Optional[np.ndarray] = None):
        """Every env's trade log in one strided copy (bb_trades_all): (records [n_envs, cap_per_env] of abi.TRADE_REC_DTYPE,
        counts [n_envs])."""
        if out is None:
            out = np.empty((self.n_envs, cap_per_env), dtype=abi.TRADE_REC_DTYPE)
        assert out.shape == (self.n_envs, cap_per_env) and out.dtype == abi.TRADE_REC_DTYPE and out.flags.c_contiguous
        counts = np.empty(self.n_envs, dtype=np.uint32)
        self._ck(self._lib.bb_trades_all(self._h, cap_per_env, abi.ptr(out), abi.ptr(counts)))
        return out, counts

    def get_orders(self, env: int = 0):
        """list[PyOrder] = (side, status, arr, end, vol, start_vol, price, trader, id) — rust/src/types.rs:19-31"""
        c = self.orders_arrays(env)
        return [(bool(c["side"][i]), int(c["status"][i]), int(c["arr_time"][i]), int(c["end_time"][i]), int(c["vol"][i]),
                 int(c["start_vol"][i]), int(c["price"][i]), int(c["trader"][i]), i) for i in range(len(c["side"]))]

    def get_trades(self, env: int = 0):
        """list[PyTrade] = (t, side, price, vol, active_id, passive_id) — rust/src/types.rs:4-17"""
        c = self.trades_arrays(env)
        return [(int(c["t"][i]), bool(c["side"][i]), int(c["price"][i]), int(c["vol"][i]), int(c["active"][i]),
                 int(c["passive"][i])) for i in range(len(c["t"]))]

    def order_keys(self, env: int = 0) -> np.ndarray:
        """Time component of every order's queue key (OrderEntry.key.2, orderbook.rs:36-44)."""
        n = self.n_orders(env)
        out = np.zeros(n, dtype=np.uint64)
        self._ck(self._lib.bb_order_keys(self._h, env, 0, n, abi.ptr(out)))
        return out

    def load_book(self, env: int, t: int, trade_vol: int, trading: bool, c: dict):
        """Overwrite one env's book from snapshot columns (bourse_b200.snapshot.dict_to_columns)."""
        self._ck(self._lib.bb_load_book(
            self._h, env, t, trade_vol, int(trading), len(c["side"]), abi.ptr(c["side"]), abi.ptr(c["status"]),
            abi.ptr(c["arr_time"]), abi.ptr(c["end_time"]), abi.ptr(c["vol"]), abi.ptr(c["start_vol"]), abi.ptr(c["price"]),
            abi.ptr(c["trader"]), abi.ptr(c["key_time"]), len(c["tr_t"]), abi.ptr(c["tr_t"]), abi.ptr(c["tr_side"]),
            abi.ptr(c["tr_price"]), abi.ptr(c["tr_vol"]), abi.ptr(c["tr_active"]), abi.ptr(c["tr_passive"])))

    def order_status(self, order_id: int, env: int = 0) -> int:
        s = C.c_uint8()
        self._ck(self._lib.bb_order_status(self._h, env, order_id, C.byref(s)))
        return s.value

    def env_errors(self) -> np.ndarray:
        out = np.empty(self.n_envs, dtype=np.uint32)
        self._ck(self._lib.bb_env_errors(self._h, abi.ptr(out)))
        return out

    def stats(self) -> dict:
        s = abi.Stats()
        self._ck(self._lib.bb_stats(self._h, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in abi.Stats._fields_}


def random_group(n_agents, tick_range, vol_range, tick_size, activity_rate):
    """RandomAgents::new argument order (crates/step_sim/src/agents/random_agent.rs:66-81)."""
    g = np.zeros(1, dtype=abi.GROUP_DTYPE)[0]
    g["kind"], g["n_agents"] = abi.GROUP_RANDOM, n_agents
    g["tick_lo"], g["tick_hi"] = tick_range
    g["vol_lo"], g["vol_hi"] = vol_range
    g["tick_size"], g["rate"] = tick_size, activity_rate
    return g


def dense_kwargs_for(groups) -> dict:
    """Engine keywords for `BatchedEnv` derived from an in-kernel agent population: when every group is a RandomAgents
    group the resting prices are bounded by the groups' tick ranges (`tick * tick_size`, random_agent.rs:96-106) and every
    agent holds at most one order, so the dense-window engine's window and slot count follow from the parameters:
    `price_window = [min price, max price + 1)`, `live_cap = number of agents` (<= 254).  MomentumAgent / NoiseAgent quote
    around the mid price, which is ~2^31 whenever one side of the book is empty (orderbook.rs:272-276): no window holds
    them, so any such group (or more than 254 agents, or a window beyond 1024 levels) returns {} — the general engine."""
    lo, hi, n = None, 0, 0
    for g in groups:
        if int(g["kind"]) != abi.GROUP_RANDOM:
            return {}
        ts = int(g["tick_size"])
        glo, ghi = int(g["tick_lo"]) * ts, (int(g["tick_hi"]) - 1) * ts + 1
        lo, hi, n = (glo if lo is None else min(lo, glo)), max(hi, ghi), n + int(g["n_agents"])
    if lo is None or n > 254 or hi - lo > 1024:
        return {}
    return dict(price_window=(lo, hi), live_cap=max(n, 1))


def momentum_group(agent_id_start, n_agents, tick_size, p_cancel, trade_vol, decay, demand, scale, order_ratio,
                   price_dist_mu, price_dist_sigma, live_cap: int = 0):
    """MomentumAgent::new + MomentumParams (crates/step_sim/src/agents/momentum_agent.rs:16-35, 118-134).
    `live_cap`: room for the agent's list of resting limit orders (the reference's Vec, momentum_agent.rs:99-102); 0 = 254."""
    g = np.zeros(1, dtype=abi.GROUP_DTYPE)[0]
    g["kind"], g["n_agents"] = abi.GROUP_MOMENTUM, n_agents
    g["tick_lo"], g["vol_lo"], g["vol_hi"] = agent_id_start, trade_vol, live_cap
    g["tick_size"], g["rate"] = tick_size, p_cancel
    g["decay"], g["demand"], g["scale"], g["order_ratio"] = decay, demand, scale, order_ratio
    g["mu"], g["sigma"] = price_dist_mu, price_dist_sigma
    return g


def noise_group(agent_id_start, n_agents, tick_size, p_limit, p_market, p_cancel, trade_vol, price_dist_mu,
                price_dist_sigma, live_cap: int = 0):
    """NoiseAgent::new + NoiseAgentParams (crates/step_sim/src/agents/noise_agent.rs:14-44, 98-114); `live_cap` as above."""
    g = np.zeros(1, dtype=abi.GROUP_DTYPE)[0]
    g["kind"], g["n_agents"] = abi.GROUP_NOISE, n_agents
    g["tick_lo"], g["vol_lo"], g["vol_hi"] = agent_id_start, trade_vol, live_cap
    g["tick_size"], g["rate"] = tick_size, p_cancel
    g["decay"], g["demand"] = p_limit, p_market
    g["mu"], g["sigma"] = price_dist_mu, price_dist_sigma
    return g


class OrderBook:
    """``bourse.core.OrderBook`` (rust/src/order_book.rs:35-375): immediate-mode book on the GPU."""

    def __init__(self, start_time: int, tick_size: int, trading: bool = True, *, max_orders: int = 1 << 18,
                 max_trades: int = 1 << 18, **kw):
        kw.setdefault("pages_smem", 16)   # a single book can afford a large resident ladder ...
        kw.setdefault("pages_total", 256)  # ... and HBM overflow pages for arbitrarily wide price ranges
        self._env = BatchedEnv(1, 0, start_time, tick_size, 1, trading, max_orders=max_orders, max_trades=max_trades,
                               max_steps=kw.pop("max_steps", 1 << 10), **kw)
        self._t = start_time
        self._trading = bool(trading)
        self._one = np.zeros(1, dtype=abi.INSTR_DTYPE)
        self._calls = 0

    def _apply(self, op_flags, order_id=0, price=0, vol=0, trader=0):
        x = self._one
        x["t"], x["op_flags"], x["order_id"] = self._t, op_flags, order_id
        x["price"], x["vol"], x["trader"] = price, vol, trader
        self._calls += 1
        if self._calls & 63 == 0:      # the reference's order table and trade log grow without bound: so do these
            self._env.grow_if_needed(0, headroom_orders=64, headroom_trades=self._env.n_orders(0) + 128)
        self._env.replay(x)

    def set_time(self, t: int): self._t = t; self._env.set_time(0, t)
    def enable_trading(self): self._trading = True; self._env.set_trading(True, 0)
    def disable_trading(self): self._trading = False; self._env.set_trading(False, 0)

    def _l1(self): return [int(x) for x in self._env.book_level_1(0)]
    def bid_ask(self): l = self._l1(); return (l[0], l[1])
    def bid_vol(self): return self._l1()[2]
    def ask_vol(self): return self._l1()[3]
    def best_bid_vol(self): return self._l1()[4]
    def best_ask_vol(self): return self._l1()[5]
    def best_bid_vol_and_orders(self): l = self._l1(); return (l[4], l[6])
    def best_ask_vol_and_orders(self): l = self._l1(); return (l[5], l[7])
    def level_2_data(self) -> np.ndarray: return self._env.book_level_2(0)
    def trade_vol(self) -> int: return int(self._env.book_level_2(0)[0])

    def order_status(self, order_id: int) -> int: return self._env.order_status(order_id, 0)

    def place_order(self, bid: bool, vol: int, trader_id: int, price: typing.Optional[int] = None) -> int:
        if price is not None and price % self._env.tick_size != 0:  # orderbook.rs:367-383
            raise ValueError(f"Price {price} was not a multiple of tick-size {self._env.tick_size}")
        oid = self._env.n_orders(0)
        f = abi.OP_NEW | (abi.F_BID if bid else 0) | (abi.F_MARKET if price is None else 0)
        self._apply(f, 0, price or 0, vol, trader_id)
        return oid

    def cancel_order(self, order_id: int): self._apply(abi.OP_CANCEL, order_id)

    def modify_order(self, order_id: int, new_price: typing.Optional[int] = None, new_vol: typing.Optional[int] = None):
        f = abi.OP_MODIFY | (abi.F_HAS_PRICE if new_price is not None else 0) | (abi.F_HAS_VOL if new_vol is not None else 0)
        self._apply(f, order_id, new_price or 0, new_vol or 0)

    def replay(self, instrs: np.ndarray) -> np.ndarray:
        """Apply a packed instruction stream (config C2); returns the [n_emit, 45] records of F_EMIT rows."""
        first = self._env.n_steps(0)
        n_new = int(((np.asarray(instrs["op_flags"]) & 0xFF) == abi.OP_NEW).sum()) if len(instrs) else 0
        n_emit = int(((np.asarray(instrs["op_flags"]) & abi.F_EMIT) != 0).sum()) if len(instrs) else 0
        # every trade either fills a passive order completely or is the last fill of its aggressor: <= 2 per instruction
        self._env.grow_if_needed(0, headroom_orders=n_new, headroom_steps=n_emit, headroom_trades=2 * len(instrs))
        self._env.replay(instrs)
        if len(instrs):
            self._t = int(instrs["t"][-1])
        return self._env.history(0, first)

    def get_trades(self): return self._env.get_trades(0)
    def get_orders(self): return self._env.get_orders(0)

    def save_json_snapshot(self, path: str, pretty: bool = False):
        from .snapshot import save_json
        save_json(self, path, pretty)


class _StepEnvBase:
    def __init__(self, seed: int, start_time: int, tick_size: int, step_size: int, trading: bool = True, *,
                 max_orders: int = 1 << 18, max_trades: int = 1 << 18, max_steps: int = 1 << 14, max_queue: int = 4096, **kw):
        kw.setdefault("pages_smem", 16)
        kw.setdefault("pages_total", 256)
        self._env = BatchedEnv(1, seed, start_time, tick_size, step_size, trading, obs_words=abi.OBS_L2,
                               max_orders=max_orders, max_trades=max_trades, max_steps=max_steps, max_queue=max_queue, **kw)
        # Single-row submissions (the per-agent calls of the reference's Python agents: Env::place_order / cancel_order /
        # modify_order, env.rs:173-219) only QUEUE a transaction until the next step, and the id a new order gets is the next
        # one in sequence (orderbook.rs:356-396).  They are therefore collected here — ids handed out from a host counter, the
        # tick check of create_order done at the call so that its ValueError is raised where the reference raises it — and
        # reach the library as ONE bb_submit per step (or before anything that reads the book's tables): a ctypes call per
        # order cost more than everything else in examples/random_trades.py.
        self._pend: typing.List[tuple] = []
        self._pend_new = 0   # new orders among them
        # host copy of the order table's status column: [0, _status_n) known, everything below _first_live final
        self._status, self._status_n, self._first_live, self._status_stale = np.zeros(1024, np.uint8), 0, 0, False
        self._tick = tick_size
        self._next_id = 0    # the id the next new order gets (None: unknown, ask the library)
        self._n_issued = 0   # upper bound of the order ids handed out (exact unless a submission raised)
        self._queued = 0     # rows handed to the library since the last step

    def _submit_rows(self, action, *a, **kw):
        out = self._env.submit(action, *a, **kw)
        self._queued += len(action)   # transactions waiting for the next step (the reference's Env::transactions, env.rs:93-96)
        return out

    def _sync_ids(self):
        if self._next_id is None:
            self._next_id = self._env.n_orders(0)

    def _submit1(self, action, side=0, vol=0, trader=0, price=0, order_id=0, flags=abi.F_HAS_PRICE | abi.F_HAS_VOL) -> int:
        oid = abi.NO_ID
        if action == abi.ACT_NEW:
            if not (flags & abi.F_MARKET) and price % self._tick:   # create_order's tick check, orderbook.rs:367-383
                raise ValueError(f"Price {price} was not a multiple of tick-size {self._tick}")
            self._sync_ids()
            self._ensure_orders(1)
            oid = self._next_id
            self._next_id += 1
            self._pend_new += 1
        self._pend.append((action, side, vol, trader, price, order_id, flags))
        return oid

    def _flush(self):
        """Hand the collected transactions to the library (in submission order)."""
        if not self._pend:
            return
        a = np.array(self._pend, dtype=np.uint64)
        self._pend, self._pend_new = [], 0
        try:
            out = self._submit_rows(a[:, 0].astype(np.uint32), a[:, 1].astype(np.uint8), a[:, 2].astype(np.uint32), a[:, 3].astype(np.uint32),
                                   a[:, 4].astype(np.uint32), a[:, 5], flags=a[:, 6].astype(np.uint32))
        except Exception:
            self._next_id = None   # (whatever was accepted before the failing row keeps its id)
            raise
        new = out[a[:, 0] == abi.ACT_NEW]
        if len(new) and int(new[-1]) + 1 != self._next_id:   # ids are handed out in sequence: cannot happen
            raise RuntimeError("order ids out of step with the library")

    def enable_trading(self): self._flush(); self._env.set_trading(True, 0)
    def disable_trading(self): self._flush(); self._env.set_trading(False, 0)
    # The reference's order table, trade log and per-step records are Vecs that grow without bound (orderbook.rs:113-115,
    # data.rs:9-57); the tables here are preallocated, so the single-env classes reserve ahead (bb_reserve):
    # orders at submission (ids are handed out on the host), history and trade log before every step.
    def _ensure_orders(self, n_more: int):
        e = self._env
        self._sync_ids()                      # ids handed out so far, the transactions still collected here included
        need = self._next_id + n_more
        if need > e.max_orders:
            e.reserve(max_orders=max(2 * e.max_orders, 2 * need))
        self._n_issued = need

    def step(self):
        e = self._env
        self._flush()
        self._sync_ids()
        self._n_steps = getattr(self, "_n_steps", 0) + 1
        if self._n_steps > e.max_steps:
            e.reserve(max_steps=2 * e.max_steps)
        if e.max_trades:
            # a trade either fills a passive order completely or is the last fill of its aggressor, so one step adds at most
            # (orders in existence) trades; the exact count is only asked for when that bound runs into the capacity
            self._trades_ub = getattr(self, "_trades_ub", 0) + self._next_id + 64
            if self._trades_ub > e.max_trades:
                self._trades_ub = e.n_trades(0) + self._next_id + 64
                if self._trades_ub > e.max_trades:
                    e.reserve(max_trades=max(2 * e.max_trades, 2 * self._trades_ub))
        self._status_stale = True
        # the reference's transaction queue is an unbounded Vec; the step's shuffle here happens in shared memory, so the queue
        # capacity is reserved ahead of need (and once more if a submission that raised half-way left the count short)
        if self._queued > e.max_queue:
            try:
                e.reserve_queue(min(65535, max(2 * e.max_queue, self._queued)))
            except MemoryError:
                pass   # (the count includes rows that queue nothing; bb_step knows the exact one and refuses cleanly)
        try:
            e.step(1)
        except MemoryError as err:
            if "max_queue" not in str(err) or e.max_queue >= 65535:
                raise
            e.reserve_queue(min(65535, 4 * max(e.max_queue, self._queued)))
            e.step(1)
        self._queued = 0

    def get_orders(self): self._flush(); return self._env.get_orders(0)
    def get_trades(self): return self._env.get_trades(0)

    def order_status(self, order_id: int) -> int:
        # an order submitted since the last step is New (0) until the step places it; transactions still collected here do not
        # change any status before the step either
        if self._next_id is None:
            self._flush()
            self._sync_ids()
        if order_id >= self._next_id:
            self._flush()
            return self._env.order_status(order_id, 0)   # (raises like the reference: unknown id)
        n_done = self._next_id - self._pend_new           # orders the library knows
        if order_id >= n_done:
            return 0
        # Statuses only change in a step, and Filled / Cancelled / Rejected are final: the first query after a step brings the
        # statuses from the oldest order that could still change (New / Active at the last look) to the newest one over in ONE
        # copy, and the queries of the step are served from the host column — not one library call per query.
        if self._status_n < n_done or self._status_stale:
            st, lo = self._status, self._first_live
            if len(st) < n_done:
                st = np.concatenate([st, np.zeros(max(n_done, 2 * len(st)) - len(st), np.uint8)])
            e = self._env
            e._ck(e._lib.bb_orders(e._h, 0, lo, n_done - lo, None, abi.ptr(st[lo:]), None, None, None, None, None, None))
            open_ = np.flatnonzero(st[lo:n_done] <= 1)
            self._first_live = lo + int(open_[0]) if len(open_) else n_done
            self._status, self._status_n, self._status_stale = st, n_done, False
        st = self._status
        return int(st[order_id])

    def _l2(self) -> np.ndarray:
        return self._env.level_2_data()[0]

    def get_market_data(self) -> typing.Dict[str, np.ndarray]:
        """45 u32 arrays keyed as rust/src/step_sim.rs:562-607."""
        h = self._env.history(0)
        d = {"trade_vol": h[:, 0].copy(), "bid_price": h[:, 1].copy(), "ask_price": h[:, 2].copy(),
             "ask_vol": h[:, 3].copy(), "bid_vol": h[:, 4].copy()}
        for i in range(10):
            d[f"bid_vol_{i}"] = h[:, 5 + 4 * i].copy()
            d[f"n_bid_{i}"] = h[:, 6 + 4 * i].copy()
            d[f"ask_vol_{i}"] = h[:, 7 + 4 * i].copy()
            d[f"n_ask_{i}"] = h[:, 8 + 4 * i].copy()
        return d


class StepEnv(_StepEnvBase):
    """``bourse.core.StepEnv`` (rust/src/step_sim.rs:55-608)."""

    @property
    def time(self): return self._env.time(0)
    @property
    def bid_ask(self): l = self._l2(); return (int(l[1]), int(l[2]))
    @property
    def ask_vol(self): return int(self._l2()[3])
    @property
    def bid_vol(self): return int(self._l2()[4])
    @property
    def best_bid_vol(self): return int(self._l2()[5])
    @property
    def best_bid_vol_and_orders(self): l = self._l2(); return (int(l[5]), int(l[6]))
    @property
    def best_ask_vol(self): return int(self._l2()[7])
    @property
    def best_ask_vol_and_orders(self): l = self._l2(); return (int(l[7]), int(l[8]))
    @property
    def trade_vol(self): return int(self._l2()[0])

    def place_order(self, bid: bool, vol: int, trader_id: int, price: typing.Optional[int] = None) -> int:
        if price is None:
            return self._submit1(abi.ACT_NEW, 1 if bid else 0, vol, trader_id, 0, 0, abi.F_MARKET)
        return self._submit1(abi.ACT_NEW, 1 if bid else 0, vol, trader_id, price)

    def cancel_order(self, order_id: int):
        self._submit1(abi.ACT_CANCEL, order_id=order_id)

    def modify_order(self, order_id: int, new_price: typing.Optional[int] = None, new_vol: typing.Optional[int] = None):
        f = (abi.F_HAS_PRICE if new_price is not None else 0) | (abi.F_HAS_VOL if new_vol is not None else 0)
        self._submit1(abi.ACT_MODIFY, vol=new_vol or 0, price=new_price or 0, order_id=order_id, flags=f)

    def get_prices(self): h = self._env.history(0); return h[:, 1].copy(), h[:, 2].copy()
    def get_volumes(self): h = self._env.history(0); return h[:, 4].copy(), h[:, 3].copy()
    def get_touch_volumes(self): h = self._env.history(0); return h[:, 5].copy(), h[:, 7].copy()
    def get_touch_order_counts(self): h = self._env.history(0); return h[:, 6].copy(), h[:, 8].copy()
    def get_trade_volumes(self): return self._env.history(0)[:, 0].copy()
    def level_1_data_array(self): return self._l2()[1:9].copy()   # 8 values, no trade_vol (step_sim.rs:381-395)
    def level_2_data_array(self): return self._l2().copy()


class StepEnvNumpy(_StepEnvBase):
    """``bourse.core.StepEnvNumpy`` (rust/src/step_sim_numpy.rs:66-517)."""

    def submit_limit_orders(self, orders):
        sides, vols, traders, prices = orders
        n = len(sides)
        self._flush()
        self._ensure_orders(n)
        self._next_id = None
        return self._submit_rows(np.full(n, abi.ACT_NEW, np.uint32), np.asarray(sides), vols, traders, prices)

    def submit_cancellations(self, order_ids):
        order_ids = np.asarray(order_ids, dtype=np.uint64)
        self._flush()
        self._submit_rows(np.full(len(order_ids), abi.ACT_CANCEL, np.uint32), order_id=order_ids)

    def submit_instructions(self, instructions):
        action, sides, vols, traders, prices, order_ids = instructions
        action = np.asarray(action, dtype=np.uint32)
        # the reference treats every code other than 1 / 2 as a no-op (step_sim_numpy.rs:254-268)
        action = np.where((action == 1) | (action == 2), action, 0).astype(np.uint32)
        self._flush()
        self._ensure_orders(int((action == 1).sum()))
        self._next_id = None
        return self._submit_rows(action, np.asarray(sides), vols, traders, prices, order_ids)

    def level_1_data(self): return self._l2()[:9].copy()
    def level_2_data(self): return self._l2().copy()


def order_book_from_json(path: str, **kw) -> OrderBook:
    from .snapshot import load_json
    return load_json(path, **kw)
