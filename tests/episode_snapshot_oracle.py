"""Test infrastructure: the snapshot restore of `bb_restore_device` on the oracle's envs
(tests/episode_snapshot/episode_snapshot.cpp).  `sim_copy(dst, src)` makes an `oracle.StepEnv` / `StepEnvNumpy` a copy of
another, and `market_copy` an `oracle.MarketEnv`: env, agent groups with their state, step counter and shuffle stream, with
the per-step records cleared; `seed` re-seeds the copy's shuffle stream as the constructor does and keeps the step counter.
A saved slot is an oracle env kept aside (`sim_copy(slot, env)`), a restore copies it back (`sim_copy(env, slot)`).

The library is compiled on first use into a temporary directory (the repository tree may be read-only), with the oracle
Makefile's compiler and flags, as tests/episode_reset_oracle.py does."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

from .market_split_oracle import _flags

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "episode_snapshot", "episode_snapshot.cpp")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        from oracle import oracle as orc
        orc.lib()   # (builds liboracle.so if needed: the handles come from it)
        cxx, flags = _flags()
        tmp = tempfile.mkdtemp(prefix="episode_snapshot_")
        out = os.path.join(tmp, "libepisode_snapshot.so")
        try:
            res = subprocess.run([cxx, *flags, "-fvisibility=hidden", "-shared", "-o", out, SRC], capture_output=True, text=True)
            if res.returncode != 0:
                raise RuntimeError("compiling episode_snapshot.cpp failed:\n" + res.stderr)
            L = C.CDLL(out)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)   # (a loaded library stays mapped)
        for name in ("ess_sim_copy", "ess_market_copy"):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64]
        _lib = L
    return _lib


def sim_copy(dst, src, seed=None):
    """`dst` (an oracle StepEnv / StepEnvNumpy) becomes a copy of `src` with no history; `seed` re-seeds its shuffle stream."""
    lib().ess_sim_copy(dst._h, src._h, int(seed is not None), 0 if seed is None else int(seed))


def market_copy(dst, src, seed=None):
    """`dst` (an oracle MarketEnv) becomes a copy of `src` with no history; `seed` re-seeds its shuffle stream."""
    lib().ess_market_copy(dst._h, src._h, int(seed is not None), 0 if seed is None else int(seed))
