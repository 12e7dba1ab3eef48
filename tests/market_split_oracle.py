"""Test infrastructure: one keyed market step of the oracle's MarketSim in two halves, `agents_update` and `step_keyed`, so
that a test can place and cancel orders between them on an `oracle.MarketEnv` (tests/market_split/market_split.cpp).

The library is compiled on first use into a temporary directory (the repository tree may be read-only), with the
oracle Makefile's compiler and flags, so that the agents' floating-point code is compiled exactly as liboracle's."""
import ctypes as C
import os
import re
import shutil
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "market_split", "market_split.cpp")
_lib = None


def _flags():
    with open(os.path.join(ROOT, "oracle", "Makefile")) as f:
        text = f.read()
    cxx = re.search(r"^CXX \?= (.+)$", text, re.M).group(1).strip()
    return os.environ.get("CXX", cxx), re.search(r"^CXXFLAGS \?= (.+)$", text, re.M).group(1).split()


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        from oracle import oracle as orc
        orc.lib()   # (builds liboracle.so if needed: the handles come from it)
        cxx, flags = _flags()
        tmp = tempfile.mkdtemp(prefix="market_split_")
        out = os.path.join(tmp, "libmarket_split.so")
        try:
            res = subprocess.run([cxx, *flags, "-fvisibility=hidden", "-shared", "-o", out, SRC], capture_output=True, text=True)
            if res.returncode != 0:
                raise RuntimeError("compiling market_split.cpp failed:\n" + res.stderr)
            L = C.CDLL(out)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)   # (a loaded library stays mapped)
        for name in ("mks_agents_update", "mks_step_keyed"):
            getattr(L, name).restype = C.c_int
            getattr(L, name).argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        L.mks_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def agents_update(m, seed: int, market_id: int = 0):
    """First half of one keyed market step on `m` (an oracle.MarketEnv): every group queues its instructions on its asset
    (Philox contract).  ValueError where an agent's limit price is off its book's tick, as MarketEnv.run_agents."""
    if lib().mks_agents_update(m._h, seed, market_id):
        raise ValueError(lib().mks_last_error().decode())


def step_keyed(m, seed: int, market_id: int = 0):
    """Second half: MarketEnv::step with the keyed shuffle over the whole queue, the caller's own instructions included."""
    if lib().mks_step_keyed(m._h, seed, market_id):
        raise IndexError("order id out of range")
