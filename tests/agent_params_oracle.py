"""Test infrastructure: `bb_set_agent_params_device` on the oracle's envs (tests/agent_params/agent_params.cpp).
`sim_set_group` overwrites the parameters of agent group `gi` of an `oracle.StepEnv` / `StepEnvNumpy`, and
`market_set_group` those of an `oracle.MarketEnv`, in place: held orders, momentum state and live-order lists are kept.
The oracle's own `set_groups` can only append groups.

The library is compiled on first use into a temporary directory (the repository tree may be read-only), with the oracle
Makefile's compiler and flags, as tests/market_split_oracle.py does."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from bourse_b200 import abi

from .market_split_oracle import _flags

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "agent_params", "agent_params.cpp")
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        from oracle import oracle as orc
        orc.lib()   # (builds liboracle.so if needed: the handles come from it)
        cxx, flags = _flags()
        tmp = tempfile.mkdtemp(prefix="agent_params_")
        out = os.path.join(tmp, "libagent_params.so")
        try:
            res = subprocess.run([cxx, *flags, "-fvisibility=hidden", "-shared", "-o", out, SRC], capture_output=True, text=True)
            if res.returncode != 0:
                raise RuntimeError("compiling agent_params.cpp failed:\n" + res.stderr)
            L = C.CDLL(out)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)   # (a loaded library stays mapped)
        for name in ("aps_sim_set_group", "aps_market_set_group"):
            getattr(L, name).restype = C.c_int
            getattr(L, name).argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        _lib = L
    return _lib


def _record(group) -> np.ndarray:
    r = np.zeros(1, dtype=abi.GROUP_DTYPE)
    r[0] = group
    return r


def sim_set_group(env, gi: int, group):
    """Group `gi` of `env` (an oracle StepEnv / StepEnvNumpy) runs with the parameters of `group` (a GROUP_DTYPE record
    of the same kind) from its next update on."""
    r = _record(group)
    if lib().aps_sim_set_group(env._h, gi, r.ctypes.data):
        raise ValueError(f"group {gi}: no such group, or another kind")


def market_set_group(m, gi: int, group):
    """The same for group `gi` of an oracle MarketEnv."""
    r = _record(group)
    if lib().aps_market_set_group(m._h, gi, r.ctypes.data):
        raise ValueError(f"group {gi}: no such group, or another kind")
