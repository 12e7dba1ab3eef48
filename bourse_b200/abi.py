"""ctypes binding of the C ABI in include/bourse_b200.h (no torch, numpy buffers at the edge).

This is the Python-side FFI stub a maintainer of the reference would add in place of the PyO3
module `bourse.core` (/root/reference/rust/src/lib.rs:7-15); see INTEGRATION.md.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# BOURSE_B200_LIB: developer override used to A/B kernel variants built side by side (scripts/ab.sh)
LIB_PATH = os.environ.get("BOURSE_B200_LIB") or os.path.join(HERE, "libbourse_b200.so")

BB_OK, BB_EPRICE, BB_EBADID, BB_ECAP, BB_ECUDA, BB_EINVAL, BB_EDEVICE = 0, -1, -2, -3, -4, -5, -6
OBS_L1, OBS_L2 = 9, 45
NO_ID = 2**64 - 1
STATUS_NONE = 0xFF   # bb_orders_device: status of a query that names no order
ALL_ENVS = 0xFFFFFFFF
NO_SLOT = 0xFFFFFFFF   # bb_save_device / bb_restore_device: leave this slot / unit as it is
OP_NOOP, OP_NEW, OP_CANCEL, OP_MODIFY, OP_SET_TRADING, OP_RESTORE = 0, 1, 2, 3, 4, 5
F_BID, F_MARKET, F_HAS_PRICE, F_HAS_VOL, F_EMIT = 1 << 8, 1 << 9, 1 << 10, 1 << 11, 1 << 12
ACT_NOOP, ACT_NEW, ACT_CANCEL, ACT_MODIFY = 0, 1, 2, 3
GROUP_RANDOM, GROUP_MOMENTUM, GROUP_NOISE = 0, 1, 2

INSTR_DTYPE = np.dtype(
    [("t", "<u8"), ("op_flags", "<u4"), ("order_id", "<u4"), ("price", "<u4"), ("vol", "<u4"),
     ("trader", "<u4"), ("aux", "<u4")], align=True)
GROUP_DTYPE = np.dtype(
    [("kind", "<u4"), ("n_agents", "<u4"), ("tick_lo", "<u4"), ("tick_hi", "<u4"), ("vol_lo", "<u4"),
     ("vol_hi", "<u4"), ("tick_size", "<u4"), ("rate", "<f4"), ("decay", "<f8"), ("demand", "<f8"),
     ("scale", "<f8"), ("order_ratio", "<f8"), ("mu", "<f8"), ("sigma", "<f8")], align=True)
ORDER_REC_DTYPE = np.dtype(
    [("price", "<u4"), ("vol", "<u4"), ("link0", "<u4"), ("link1", "<u4"), ("key_time", "<u8"), ("meta", "<u4"), ("start_vol", "<u4"),
     ("arr_time", "<u8"), ("end_time", "<u8"), ("trader", "<u4"), ("pad", "<u4", (3,))], align=True)
TRADE_REC_DTYPE = np.dtype(
    [("t", "<u8"), ("price", "<u4"), ("vol", "<u4"), ("active_id", "<u4"), ("passive_id", "<u4"), ("side_is_bid", "<u4"), ("pad", "<u4")],
    align=True)
assert INSTR_DTYPE.itemsize == 32 and GROUP_DTYPE.itemsize == 80 and ORDER_REC_DTYPE.itemsize == 64 and TRADE_REC_DTYPE.itemsize == 32


class Config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("n_envs", C.c_uint32),
                ("env_id_base", C.c_uint32), ("start_time", C.c_uint64), ("step_size", C.c_uint64),
                ("seed", C.c_uint64), ("tick_size", C.c_uint32), ("price_granule", C.c_uint32),
                ("trading", C.c_uint32), ("obs_words", C.c_uint32), ("max_orders", C.c_uint32),
                ("max_trades", C.c_uint32), ("max_steps", C.c_uint32), ("max_queue", C.c_uint32),
                ("pages_smem", C.c_uint32), ("pages_total", C.c_uint32), ("win_lo", C.c_uint32),
                ("win_levels", C.c_uint32), ("live_cap", C.c_uint32), ("assets", C.c_uint32), ("deep_chunks", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("instructions", "orders_created", "trades", "traded_volume",
                                          "env_steps", "transitions", "error_envs", "l1_checksum")]


EXPORTS = [
    "bb_abi_version", "bb_create", "bb_destroy", "bb_reset", "bb_last_error", "bb_set_stream", "bb_synchronize",
    "bb_submit", "bb_step", "bb_replay", "bb_replay_device", "bb_set_agents", "bb_run_agents", "bb_run_agents_to_host", "bb_level1",
    "bb_level2", "bb_book_level1", "bb_book_level2", "bb_n_steps", "bb_history", "bb_history_all",
    "bb_n_orders", "bb_n_trades", "bb_orders", "bb_trades", "bb_order_status", "bb_time", "bb_set_time",
    "bb_set_trading", "bb_env_errors", "bb_stats", "bb_history_device", "bb_order_keys", "bb_load_book",
    "bb_set_agents_market", "bb_step_device", "bb_level2_device", "bb_level1_device", "bb_device_alloc", "bb_device_free", "bb_memcpy", "bb_run_agents_with_rows", "bb_reserve", "bb_reserve_queue", "bb_clear_history", "bb_clear_errors",
    "bb_orders_all", "bb_trades_all", "bb_set_tick_sizes", "bb_step_device_market", "bb_run_agents_with_rows_market", "bb_orders_device", "bb_trades_device", "bb_reset_device", "bb_store_create", "bb_store_destroy", "bb_save_device", "bb_restore_device", "bb_comm_unique_id", "bb_comm_init_rank", "bb_comm_init_all", "bb_comm_n_ranks", "bb_comm_destroy", "bb_comm_last_error", "bb_gather_stats",
]

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raises if it has not been built (there is no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m bourse_b200.build` (nvcc, sm_100a). "
            "bourse_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    P = C.POINTER

    def sig(name, res, *args):
        try:
            f = getattr(L, name)
        except AttributeError:
            if os.environ.get("BOURSE_B200_LIB"):  # older variant under A/B test: symbol simply unavailable
                return
            raise
        f.restype = res
        f.argtypes = list(args)

    sig("bb_abi_version", i32)
    sig("bb_create", i32, P(Config), P(vp))
    sig("bb_destroy", i32, vp)
    sig("bb_reset", i32, vp)
    sig("bb_reserve", i32, vp, u32, u32, u32)
    sig("bb_reserve_queue", i32, vp, u32)
    sig("bb_set_tick_sizes", i32, vp, vp, u32)
    sig("bb_clear_history", i32, vp)
    sig("bb_clear_errors", i32, vp)
    sig("bb_last_error", C.c_char_p, vp)
    sig("bb_set_stream", i32, vp, vp)
    sig("bb_synchronize", i32, vp)
    sig("bb_submit", i32, vp, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp, P(u64))
    sig("bb_step", i32, vp, u32)
    sig("bb_replay", i32, vp, vp, vp)
    sig("bb_replay_device", i32, vp, vp, vp)
    sig("bb_set_agents", i32, vp, vp, u32)
    sig("bb_set_agents_market", i32, vp, vp, vp, u32)
    sig("bb_step_device", i32, vp, vp, vp, u64, vp, vp)
    sig("bb_step_device_market", i32, vp, vp, vp, u64, vp, vp)
    sig("bb_orders_device", i32, vp, vp, vp, u64, vp, vp, vp, vp, vp, vp, vp, vp)
    sig("bb_trades_device", i32, vp, vp, u32, vp, vp, vp, vp, vp, vp, vp)
    sig("bb_reset_device", i32, vp, vp, vp, vp, vp)
    sig("bb_store_create", i32, vp, u32, P(vp), P(u64))
    sig("bb_store_destroy", i32, vp)
    sig("bb_save_device", i32, vp, vp, vp)
    sig("bb_restore_device", i32, vp, vp, vp, vp, vp, vp)
    sig("bb_level2_device", i32, vp, vp)
    sig("bb_level1_device", i32, vp, vp)
    sig("bb_device_alloc", i32, vp, u64, P(vp))
    sig("bb_device_free", i32, vp, vp)
    sig("bb_memcpy", i32, vp, vp, vp, u64, i32)
    sig("bb_run_agents", i32, vp, u64, u32)
    sig("bb_run_agents_with_rows", i32, vp, u64, vp, vp, u64, vp, vp)
    sig("bb_run_agents_with_rows_market", i32, vp, u64, vp, vp, u64, vp, vp)
    sig("bb_run_agents_to_host", i32, vp, u64, u32, u32, vp)
    sig("bb_level1", i32, vp, vp)
    sig("bb_level2", i32, vp, vp)
    sig("bb_book_level1", i32, vp, u32, vp)
    sig("bb_book_level2", i32, vp, u32, vp)
    sig("bb_n_steps", i32, vp, u32, P(u32))
    sig("bb_history", i32, vp, u32, u32, u32, vp)
    sig("bb_history_all", i32, vp, u32, vp)
    sig("bb_n_orders", i32, vp, u32, P(u64))
    sig("bb_n_trades", i32, vp, u32, P(u64))
    sig("bb_orders", i32, vp, u32, u64, u64, vp, vp, vp, vp, vp, vp, vp, vp)
    sig("bb_trades", i32, vp, u32, u64, u64, vp, vp, vp, vp, vp, vp)
    sig("bb_order_status", i32, vp, u32, u64, P(C.c_uint8))
    sig("bb_time", i32, vp, u32, P(u64))
    sig("bb_set_time", i32, vp, u32, u64)
    sig("bb_set_trading", i32, vp, u32, i32)
    sig("bb_env_errors", i32, vp, vp)
    sig("bb_stats", i32, vp, P(Stats))
    sig("bb_history_device", i32, vp, P(vp), P(u64), P(u32))
    sig("bb_order_keys", i32, vp, u32, u64, u64, vp)
    sig("bb_load_book", i32, vp, u32, u64, u32, i32, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp, u64, vp, vp, vp, vp, vp, vp)
    sig("bb_orders_all", i32, vp, u32, vp, vp)
    sig("bb_trades_all", i32, vp, u32, vp, vp)
    sig("bb_comm_unique_id", i32, vp)
    sig("bb_comm_init_rank", i32, vp, i32, i32, i32, P(vp))
    sig("bb_comm_init_all", i32, i32, vp, P(vp))
    sig("bb_comm_n_ranks", i32, vp)
    sig("bb_comm_destroy", i32, vp)
    sig("bb_comm_last_error", C.c_char_p)
    sig("bb_gather_stats", i32, vp, vp, u32, vp, vp, vp)
    _lib = L
    return L


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
