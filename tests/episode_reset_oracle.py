"""Test infrastructure: the per-env reset of `bb_reset_device` on the oracle's envs (tests/episode_reset/episode_reset.cpp).
`sim_reset` rebuilds an `oracle.StepEnv` / `StepEnvNumpy` and `market_reset` an `oracle.MarketEnv` from their construction
parameters, agent groups kept with their state cleared; `seed=None` keeps the env's shuffle stream and step counter, a seed
re-seeds the stream as the constructor does and restarts the step counter.

The library is compiled on first use into a temporary directory (the repository tree may be read-only), with the oracle
Makefile's compiler and flags, as tests/market_split_oracle.py does."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

from .market_split_oracle import _flags

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "episode_reset", "episode_reset.cpp")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        from oracle import oracle as orc
        orc.lib()   # (builds liboracle.so if needed: the handles come from it)
        cxx, flags = _flags()
        tmp = tempfile.mkdtemp(prefix="episode_reset_")
        out = os.path.join(tmp, "libepisode_reset.so")
        try:
            res = subprocess.run([cxx, *flags, "-fvisibility=hidden", "-shared", "-o", out, SRC], capture_output=True, text=True)
            if res.returncode != 0:
                raise RuntimeError("compiling episode_reset.cpp failed:\n" + res.stderr)
            L = C.CDLL(out)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)   # (a loaded library stays mapped)
        for name in ("ers_sim_reset", "ers_market_reset"):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_uint64]
        _lib = L
    return _lib


def sim_reset(env, start_time: int, trading: bool = True, seed=None):
    """`env` (an oracle StepEnv / StepEnvNumpy) back to a fresh Env at `start_time`, its tick and step size kept."""
    lib().ers_sim_reset(env._h, start_time, int(trading), int(seed is not None), 0 if seed is None else int(seed))


def market_reset(m, start_time: int, trading: bool = True, seed=None):
    """`m` (an oracle MarketEnv) back to a fresh MarketEnv at `start_time`, its ticks and step size kept."""
    lib().ers_market_reset(m._h, start_time, int(trading), int(seed is not None), 0 if seed is None else int(seed))
