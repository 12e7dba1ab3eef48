"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes front-end over ``oracle/liboracle.so`` (the C++ CPU restatement of the reference's order
book / Env / agents, see ``oracle/book.hpp`` and ``oracle/env.hpp`` for the reference file:line
each function follows).  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this module; the product package
``bourse_b200`` never does.

The class names and method signatures follow the reference's Python surface
(``rust/src/order_book.rs:35-398``, ``rust/src/step_sim.rs:55-608``,
``rust/src/step_sim_numpy.rs:66-517``) so the same test body can drive the oracle and the CUDA path.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")

# 32-byte instruction record; identical layout to ``bb_instr`` (include/bourse_b200.h)
INSTR_DTYPE = np.dtype(
    [("t", "<u8"), ("op_flags", "<u4"), ("order_id", "<u4"), ("price", "<u4"), ("vol", "<u4"),
     ("trader", "<u4"), ("aux", "<u4")], align=True)
# 80-byte agent group record; identical layout to ``bb_agent_group``
GROUP_DTYPE = np.dtype(
    [("kind", "<u4"), ("n_agents", "<u4"), ("tick_lo", "<u4"), ("tick_hi", "<u4"), ("vol_lo", "<u4"),
     ("vol_hi", "<u4"), ("tick_size", "<u4"), ("rate", "<f4"), ("decay", "<f8"), ("demand", "<f8"),
     ("scale", "<f8"), ("order_ratio", "<f8"), ("mu", "<f8"), ("sigma", "<f8")], align=True)
assert INSTR_DTYPE.itemsize == 32 and GROUP_DTYPE.itemsize == 80

OP_NOOP, OP_NEW, OP_CANCEL, OP_MODIFY, OP_SET_TRADING = 0, 1, 2, 3, 4
F_BID, F_MARKET, F_HAS_PRICE, F_HAS_VOL, F_EMIT = 1 << 8, 1 << 9, 1 << 10, 1 << 11, 1 << 12

MAX_PRICE = 2**32 - 1


def build(force: bool = False) -> str:
    """Compile liboracle.so with the Makefile next to this file (gcc only)."""
    srcs = [os.path.join(_HERE, f) for f in ("oracle_capi.cpp", "book.hpp", "env.hpp", "rng.hpp")]
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-s", "-B", "liboracle.so"], check=True)
    return _LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        build()
    L = C.CDLL(_LIB_PATH)
    vp, u64, u32, i32, dbl = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_double
    P = C.POINTER

    def sig(name, res, *args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = list(args)

    sig("orc_book_new", vp, u64, u32, i32)
    sig("orc_book_free", None, vp)
    sig("orc_book_set_time", None, vp, u64)
    sig("orc_book_time", u64, vp)
    sig("orc_book_set_trading", None, vp, i32)
    sig("orc_book_create", i32, vp, i32, u32, u32, i32, u32, P(u64))
    sig("orc_book_place_id", i32, vp, u64)
    sig("orc_book_place", i32, vp, i32, u32, u32, i32, u32, P(u64))
    sig("orc_book_cancel", i32, vp, u64)
    sig("orc_book_modify", i32, vp, u64, i32, u32, i32, u32)
    sig("orc_book_order_status", i32, vp, u64)
    sig("orc_book_trade_vol", u32, vp)
    sig("orc_book_mid_price", dbl, vp)
    sig("orc_book_l1", None, vp, vp)
    sig("orc_book_l2", None, vp, vp)
    sig("orc_book_n_orders", u64, vp)
    sig("orc_book_n_trades", u64, vp)
    sig("orc_book_orders", None, vp, vp, vp, vp, vp, vp, vp, vp, vp)
    sig("orc_book_trades", None, vp, vp, vp, vp, vp, vp, vp)
    sig("orc_book_replay", C.c_int64, vp, vp, u64, vp, u64, P(u64))
    sig("orc_sim_new", vp, u64, u64, u32, u64, i32)
    sig("orc_sim_free", None, vp)
    sig("orc_sim_book", vp, vp)
    sig("orc_sim_keep_records", None, vp, i32)
    sig("orc_sim_place", i32, vp, i32, u32, u32, i32, u32, P(u64))
    sig("orc_sim_cancel", None, vp, u64)
    sig("orc_sim_modify", None, vp, u64, i32, u32, i32, u32)
    sig("orc_sim_step", i32, vp)
    sig("orc_sim_n_queued", u64, vp)
    sig("orc_sim_set_trading", None, vp, i32)
    sig("orc_sim_l2", None, vp, vp)
    sig("orc_sim_n_steps", u64, vp)
    sig("orc_sim_history", None, vp, vp)
    sig("orc_sim_set_groups", None, vp, vp, u32)
    sig("orc_sim_run", i32, vp, i32, u64, u32, u64)
    sig("orc_sim_n_instructions", u64, vp)
    sig("orc_sim_agents_update", i32, vp, u64, u32)
    sig("orc_sim_step_keyed", i32, vp, u64, u32)
    sig("orc_bench_agents", dbl, u32, u32, u64, u64, i32, u64, u32, u64, vp, u32, vp)
    sig("orc_bench_replay", dbl, u32, u32, u32, vp, u64, vp)
    sig("orc_market_new", vp, u64, u64, vp, u32, u64, i32)
    sig("orc_market_free", None, vp)
    sig("orc_market_book", vp, vp, u32)
    sig("orc_market_place", i32, vp, u32, i32, u32, u32, i32, u32, vp)
    sig("orc_market_cancel", None, vp, u32, u64)
    sig("orc_market_modify", None, vp, u32, u64, i32, u32, i32, u32)
    sig("orc_market_step", i32, vp)
    sig("orc_market_n_steps", u64, vp, u32)
    sig("orc_market_history", None, vp, u32, vp)
    sig("orc_market_set_groups", None, vp, vp, vp, u32)
    sig("orc_market_run", i32, vp, i32, u64, u32, u64)
    sig("orc_market_n_instructions", u64, vp)
    sig("orc_bench_market_agents", dbl, u32, u32, u64, u64, i32, u64, vp, u32, u64, vp, vp, u32, vp)
    sig("orc_bench_replay_suffix", dbl, u32, u32, vp, u64, u64, vp)
    sig("orc_bench_env_rows", dbl, u32, u32, u64, u32, vp, u32, u32, u64, u32, u64, vp)
    sig("orc_last_error", C.c_char_p)
    sig("orc_philox", None, u32, u32, u32, u32, u32, u32, vp)
    sig("orc_xoroshiro", None, u64, u32, vp)
    sig("orc_xoroshiro_state", None, u64, u64, u32, vp, vp, vp, u32, vp)
    sig("orc_shuffle_perm", None, u64, u32, vp)
    sig("orc_round_price", u32, dbl, dbl, i32)
    _lib = L
    return L


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _check_agents(rc):
    """An agent run returns -1 where a reference agent's create_order would raise PriceError and the agent's unwrap
    panic: raised here as ValueError with the reference's message.  The steps completed before it keep their records."""
    if rc:
        raise ValueError(lib().orc_last_error().decode())


def random_group(n_agents, tick_range, vol_range, tick_size, activity_rate):
    """RandomAgents::new argument order (crates/step_sim/src/agents/random_agent.rs:66-81)."""
    g = np.zeros(1, dtype=GROUP_DTYPE)[0]
    g["kind"], g["n_agents"] = 0, n_agents
    g["tick_lo"], g["tick_hi"] = tick_range
    g["vol_lo"], g["vol_hi"] = vol_range
    g["tick_size"], g["rate"] = tick_size, activity_rate
    return g


def momentum_group(agent_id_start, n_agents, tick_size, p_cancel, trade_vol, decay, demand, scale,
                   order_ratio, price_dist_mu, price_dist_sigma):
    """MomentumAgent::new + MomentumParams (crates/step_sim/src/agents/momentum_agent.rs:16-35,118-134)."""
    g = np.zeros(1, dtype=GROUP_DTYPE)[0]
    g["kind"], g["n_agents"] = 1, n_agents
    g["tick_lo"], g["vol_lo"] = agent_id_start, trade_vol
    g["tick_size"], g["rate"] = tick_size, p_cancel
    g["decay"], g["demand"], g["scale"], g["order_ratio"] = decay, demand, scale, order_ratio
    g["mu"], g["sigma"] = price_dist_mu, price_dist_sigma
    return g


def noise_group(agent_id_start, n_agents, tick_size, p_limit, p_market, p_cancel, trade_vol, price_dist_mu, price_dist_sigma):
    """NoiseAgent::new + NoiseAgentParams (crates/step_sim/src/agents/noise_agent.rs:14-44, 98-114)."""
    g = np.zeros(1, dtype=GROUP_DTYPE)[0]
    g["kind"], g["n_agents"] = 2, n_agents
    g["tick_lo"], g["vol_lo"] = agent_id_start, trade_vol
    g["tick_size"], g["rate"] = tick_size, p_cancel
    g["decay"], g["demand"] = p_limit, p_market
    g["mu"], g["sigma"] = price_dist_mu, price_dist_sigma
    return g


def groups_array(groups) -> np.ndarray:
    out = np.zeros(len(groups), dtype=GROUP_DTYPE)
    for i, g in enumerate(groups):
        out[i] = g
    return out


class _BookView:
    """Read-only accessors shared by OrderBook and the Env-backed classes."""

    def _book(self):
        raise NotImplementedError

    def orders_arrays(self):
        """Column arrays of the order table (same keys as bourse_b200.core.BatchedEnv.orders_arrays)."""
        L, b = lib(), self._book()
        n = L.orc_book_n_orders(b)
        side = np.zeros(n, np.uint8); status = np.zeros(n, np.uint8)
        arr = np.zeros(n, np.uint64); end = np.zeros(n, np.uint64)
        vol = np.zeros(n, np.uint32); sv = np.zeros(n, np.uint32)
        price = np.zeros(n, np.uint32); trader = np.zeros(n, np.uint32)
        L.orc_book_orders(b, _ptr(side), _ptr(status), _ptr(arr), _ptr(end), _ptr(vol), _ptr(sv), _ptr(price), _ptr(trader))
        return dict(side=side, status=status, arr_time=arr, end_time=end, vol=vol, start_vol=sv, price=price, trader=trader)

    def trades_arrays(self):
        L, b = lib(), self._book()
        n = L.orc_book_n_trades(b)
        t = np.zeros(n, np.uint64); side = np.zeros(n, np.uint8)
        price = np.zeros(n, np.uint32); vol = np.zeros(n, np.uint32)
        act = np.zeros(n, np.uint64); pas = np.zeros(n, np.uint64)
        L.orc_book_trades(b, _ptr(t), _ptr(side), _ptr(price), _ptr(vol), _ptr(act), _ptr(pas))
        return dict(t=t, side=side, price=price, vol=vol, active=act, passive=pas)

    def get_orders(self):
        c = self.orders_arrays()
        return [(bool(c["side"][i]), int(c["status"][i]), int(c["arr_time"][i]), int(c["end_time"][i]), int(c["vol"][i]),
                 int(c["start_vol"][i]), int(c["price"][i]), int(c["trader"][i]), i) for i in range(len(c["side"]))]

    def get_trades(self):
        c = self.trades_arrays()
        return [(int(c["t"][i]), bool(c["side"][i]), int(c["price"][i]), int(c["vol"][i]), int(c["active"][i]),
                 int(c["passive"][i])) for i in range(len(c["t"]))]

    def order_status(self, order_id: int) -> int:
        s = lib().orc_book_order_status(self._book(), order_id)
        if s < 0:
            raise IndexError(f"No order with id {order_id} exists")
        return s


class OrderBook(_BookView):
    """Oracle twin of ``bourse.core.OrderBook`` (rust/src/order_book.rs:35-375)."""

    def __init__(self, start_time: int, tick_size: int, trading: bool = True):
        self._h = lib().orc_book_new(start_time, tick_size, int(trading))
        self.tick_size = tick_size

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_book_free(self._h)
            self._h = None

    def _book(self):
        return self._h

    def set_time(self, t): lib().orc_book_set_time(self._h, t)
    def enable_trading(self): lib().orc_book_set_trading(self._h, 1)
    def disable_trading(self): lib().orc_book_set_trading(self._h, 0)

    def _l1(self):
        out = np.zeros(8, np.uint32)
        lib().orc_book_l1(self._h, _ptr(out))
        return [int(x) for x in out]

    def bid_ask(self): l = self._l1(); return (l[0], l[1])
    def bid_vol(self): return self._l1()[2]
    def ask_vol(self): return self._l1()[3]
    def best_bid_vol(self): return self._l1()[4]
    def best_ask_vol(self): return self._l1()[5]
    def best_bid_vol_and_orders(self): l = self._l1(); return (l[4], l[6])
    def best_ask_vol_and_orders(self): l = self._l1(); return (l[5], l[7])
    def trade_vol(self): return lib().orc_book_trade_vol(self._h)
    def mid_price(self): return lib().orc_book_mid_price(self._h)

    def level_2_data(self) -> np.ndarray:
        out = np.zeros(45, np.uint32)
        lib().orc_book_l2(self._h, _ptr(out))
        return out

    def create_order(self, bid, vol, trader_id, price=None) -> int:
        oid = C.c_uint64()
        rc = lib().orc_book_create(self._h, int(bid), vol, trader_id, int(price is not None), price or 0, C.byref(oid))
        if rc:
            raise ValueError(f"Price {price} was not a multiple of tick-size {self.tick_size}")
        return oid.value

    def place_created(self, order_id):
        if lib().orc_book_place_id(self._h, order_id):
            raise IndexError(order_id)

    def place_order(self, bid, vol, trader_id, price=None) -> int:
        oid = C.c_uint64()
        rc = lib().orc_book_place(self._h, int(bid), vol, trader_id, int(price is not None), price or 0, C.byref(oid))
        if rc:
            raise ValueError(f"Price {price} was not a multiple of tick-size {self.tick_size}")
        return oid.value

    def cancel_order(self, order_id):
        if lib().orc_book_cancel(self._h, order_id):
            raise IndexError(f"No order with id {order_id} exists")

    def modify_order(self, order_id, new_price=None, new_vol=None):
        rc = lib().orc_book_modify(self._h, order_id, int(new_price is not None), new_price or 0,
                                   int(new_vol is not None), new_vol or 0)
        if rc:
            raise IndexError(f"No order with id {order_id} exists")

    def replay(self, instrs: np.ndarray, obs_cap: int = 0):
        """Apply a packed INSTR_DTYPE stream; returns the [n_emit, 45] L2 records of F_EMIT rows."""
        instrs = np.ascontiguousarray(instrs, dtype=INSTR_DTYPE)
        obs = np.zeros((max(obs_cap, 1), 45), np.uint32)
        err_at = C.c_uint64()
        n = lib().orc_book_replay(self._h, _ptr(instrs), len(instrs), _ptr(obs), obs_cap, C.byref(err_at))
        if n < 0:
            raise ValueError(f"replay error {n} at instruction {err_at.value}")
        return obs[:n]


class _EnvBase(_BookView):
    def __init__(self, seed, start_time, tick_size, step_size, trading=True):
        self._h = lib().orc_sim_new(seed, start_time, tick_size, step_size, int(trading))
        self.tick_size = tick_size

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_sim_free(self._h)
            self._h = None

    def _book(self):
        return lib().orc_sim_book(self._h)

    def enable_trading(self): lib().orc_sim_set_trading(self._h, 1)
    def disable_trading(self): lib().orc_sim_set_trading(self._h, 0)

    def step(self):
        if lib().orc_sim_step(self._h):
            raise IndexError("an instruction referenced an order id that does not exist")

    def _l2(self) -> np.ndarray:
        out = np.zeros(45, np.uint32)
        lib().orc_sim_l2(self._h, _ptr(out))
        return out

    def _history(self) -> np.ndarray:
        n = lib().orc_sim_n_steps(self._h)
        out = np.zeros((max(n, 1), 45), np.uint32)
        lib().orc_sim_history(self._h, _ptr(out))
        return out[:n]

    def get_market_data(self):
        h = self._history()
        d = {"trade_vol": h[:, 0].copy(), "bid_price": h[:, 1].copy(), "ask_price": h[:, 2].copy(),
             "ask_vol": h[:, 3].copy(), "bid_vol": h[:, 4].copy()}
        for i in range(10):
            d[f"bid_vol_{i}"] = h[:, 5 + 4 * i].copy()
            d[f"n_bid_{i}"] = h[:, 6 + 4 * i].copy()
            d[f"ask_vol_{i}"] = h[:, 7 + 4 * i].copy()
            d[f"n_ask_{i}"] = h[:, 8 + 4 * i].copy()
        return d

    # agent-driven runs (crates/step_sim/src/runner.rs:46-69)
    def set_groups(self, groups):
        arr = groups_array(groups)
        lib().orc_sim_set_groups(self._h, _ptr(arr), len(arr))

    def run_agents(self, n_steps, seed, env_id=0, keyed=True):
        _check_agents(lib().orc_sim_run(self._h, int(keyed), seed, env_id, n_steps))

    def agents_update(self, seed, env_id=0):
        """First half of one keyed step: the built-in agents queue their instructions (Philox contract)."""
        _check_agents(lib().orc_sim_agents_update(self._h, seed, env_id))

    def step_keyed(self, seed, env_id=0):
        """Second half: Env::step with the keyed shuffle over everything queued, the caller's own instructions included."""
        if lib().orc_sim_step_keyed(self._h, seed, env_id):
            raise IndexError("order id out of range")

    def n_instructions(self):
        return lib().orc_sim_n_instructions(self._h)


class StepEnv(_EnvBase):
    """Oracle twin of ``bourse.core.StepEnv`` (rust/src/step_sim.rs:55-608)."""

    @property
    def time(self): return lib().orc_book_time(self._book())
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

    def place_order(self, bid, vol, trader_id, price=None) -> int:
        oid = C.c_uint64()
        rc = lib().orc_sim_place(self._h, int(bid), vol, trader_id, int(price is not None), price or 0, C.byref(oid))
        if rc:
            raise ValueError(f"Price {price} was not a multiple of tick-size {self.tick_size}")
        return oid.value

    def cancel_order(self, order_id): lib().orc_sim_cancel(self._h, order_id)

    def modify_order(self, order_id, new_price=None, new_vol=None):
        lib().orc_sim_modify(self._h, order_id, int(new_price is not None), new_price or 0,
                             int(new_vol is not None), new_vol or 0)

    def get_prices(self): h = self._history(); return h[:, 1].copy(), h[:, 2].copy()
    def get_volumes(self): h = self._history(); return h[:, 4].copy(), h[:, 3].copy()
    def get_touch_volumes(self): h = self._history(); return h[:, 5].copy(), h[:, 7].copy()
    def get_touch_order_counts(self): h = self._history(); return h[:, 6].copy(), h[:, 8].copy()
    def get_trade_volumes(self): return self._history()[:, 0].copy()
    def level_1_data_array(self): return self._l2()[1:9].copy()   # 8 values, no trade_vol (step_sim.rs:381-395)
    def level_2_data_array(self): return self._l2()


class StepEnvNumpy(_EnvBase):
    """Oracle twin of ``bourse.core.StepEnvNumpy`` (rust/src/step_sim_numpy.rs:66-517)."""

    def submit_limit_orders(self, orders):
        sides, vols, traders, prices = orders
        ids = np.zeros(len(sides), np.uint64)
        oid = C.c_uint64()
        for i in range(len(sides)):
            rc = lib().orc_sim_place(self._h, int(bool(sides[i])), int(vols[i]), int(traders[i]), 1, int(prices[i]), C.byref(oid))
            if rc:  # rows before i stay queued (lazy map + collect, step_sim_numpy.rs:166-179)
                raise ValueError(f"Price {int(prices[i])} was not a multiple of tick-size {self.tick_size}")
            ids[i] = oid.value
        return ids

    def submit_cancellations(self, order_ids):
        for i in order_ids:
            lib().orc_sim_cancel(self._h, int(i))

    def submit_instructions(self, instructions):
        action, sides, vols, traders, prices, order_ids = instructions
        ids = np.full(len(action), 2**64 - 1, np.uint64)
        oid = C.c_uint64()
        for i in range(len(action)):
            if action[i] == 1:
                rc = lib().orc_sim_place(self._h, int(bool(sides[i])), int(vols[i]), int(traders[i]), 1, int(prices[i]), C.byref(oid))
                if rc:
                    raise ValueError(f"Price {int(prices[i])} was not a multiple of tick-size {self.tick_size}")
                ids[i] = oid.value
            elif action[i] == 2:
                lib().orc_sim_cancel(self._h, int(order_ids[i]))
        return ids

    def level_1_data(self): return self._l2()[:9].copy()
    def level_2_data(self): return self._l2()


def bench_agents(n_envs, n_threads, n_steps, seed, groups, keyed=False, start_time=0, tick_size=1,
                 step_size=1_000_000):
    arr = groups_array(groups)
    out = np.zeros(3, np.uint64)
    secs = lib().orc_bench_agents(n_envs, n_threads, n_steps, seed, int(keyed), start_time, tick_size, step_size,
                                  _ptr(arr), len(arr), _ptr(out))
    return {"seconds": secs, "instructions": int(out[0]), "trades": int(out[1]), "env_steps": int(out[2])}


def bench_market_agents(n_markets, n_threads, n_steps, seed, groups, assets, n_assets, keyed=False, start_time=0, tick_size=1,
                        step_size=1_000_000):
    arr = groups_array(groups)
    a = np.ascontiguousarray(assets, dtype=np.uint32)
    ticks = np.full(n_assets, tick_size, np.uint32)
    out = np.zeros(3, np.uint64)
    secs = lib().orc_bench_market_agents(n_markets, n_threads, n_steps, seed, int(keyed), start_time, _ptr(ticks), n_assets,
                                         step_size, _ptr(arr), _ptr(a), len(arr), _ptr(out))
    return {"seconds": secs, "instructions": int(out[0]), "trades": int(out[1]), "env_steps": int(out[2])}


def bench_env_rows(n_envs, n_threads, n_steps, blocks, seed, tick_size=1, step_size=1000):
    """`blocks`: INSTR_DTYPE array [n_blocks, block_envs, rows], cycled over the steps (see orc_bench_env_rows)."""
    blocks = np.ascontiguousarray(blocks, dtype=INSTR_DTYPE)
    nb, be, rows = blocks.shape
    out = np.zeros(3, np.uint64)
    secs = lib().orc_bench_env_rows(n_envs, n_threads, n_steps, rows, _ptr(blocks), nb, be, seed, tick_size, step_size, _ptr(out))
    return {"seconds": secs, "instructions": int(out[0]), "trades": int(out[1]), "env_steps": int(out[2])}


def bench_replay(n_books, n_threads, tick_size, instrs):
    instrs = np.ascontiguousarray(instrs, dtype=INSTR_DTYPE)
    out = np.zeros(2, np.uint64)
    secs = lib().orc_bench_replay(n_books, n_threads, tick_size, _ptr(instrs), len(instrs), _ptr(out))
    return {"seconds": secs, "instructions": int(out[0]), "trades": int(out[1])}


def bench_replay_suffix(n_threads, tick_size, instrs, n_pre):
    """One book per thread: untimed replay of instrs[:n_pre], then the timed replay of the rest (all threads together)."""
    instrs = np.ascontiguousarray(instrs, dtype=INSTR_DTYPE)
    out = np.zeros(2, np.uint64)
    secs = lib().orc_bench_replay_suffix(n_threads, tick_size, _ptr(instrs), n_pre, len(instrs), _ptr(out))
    return {"seconds": secs, "instructions": int(out[0]), "trades": int(out[1])}


class _AssetView(_BookView):
    """Read-only view of one asset's book inside a MarketEnv (orders / trades / status getters)."""

    def __init__(self, market, asset):
        self._m, self._a = market, asset

    def _book(self):
        return lib().orc_market_book(self._m._h, self._a)


class MarketEnv:
    """bourse_de::MarketEnv (crates/step_sim/src/market_env.rs:47-300): `len(tick_sizes)` assets, one shuffled
    transaction queue per step.  Order ids are (asset, id) pairs (MarketOrderId)."""

    def __init__(self, seed, start_time, tick_sizes, step_size, trading=True):
        ts = np.ascontiguousarray(tick_sizes, dtype=np.uint32)
        self.n_assets = len(ts)
        self._h = lib().orc_market_new(seed, start_time, _ptr(ts), len(ts), step_size, int(trading))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_market_free(self._h)
            self._h = None

    def asset(self, a):
        return _AssetView(self, a)

    def place_order(self, asset, bid, vol, trader_id, price=None):
        out = C.c_uint64()
        rc = lib().orc_market_place(self._h, asset, int(bid), vol, trader_id, int(price is not None), price or 0, C.byref(out))
        if rc:
            raise ValueError(f"Price {price} was not a multiple of tick-size")
        return (asset, out.value)

    def cancel_order(self, order_id): lib().orc_market_cancel(self._h, order_id[0], order_id[1])

    def modify_order(self, order_id, new_price=None, new_vol=None):
        lib().orc_market_modify(self._h, order_id[0], order_id[1], int(new_price is not None), new_price or 0,
                                int(new_vol is not None), new_vol or 0)

    def step(self):
        if lib().orc_market_step(self._h):
            raise IndexError("order id out of range")

    def history(self, asset):
        n = lib().orc_market_n_steps(self._h, asset)
        out = np.zeros((n, 45), np.uint32)
        if n:
            lib().orc_market_history(self._h, asset, _ptr(out))
        return out

    def set_groups(self, groups, assets):
        """Market agent twins: group i (random_group / momentum_group / noise_group) trades asset assets[i]
        (RandomMarketAgents random_agent.rs:165-247, MomentumMarketAgent momentum_agent.rs:282-409, NoiseMarketAgent
        noise_agent.rs:226-345); groups update in list order each step."""
        arr = groups_array(groups)
        a = np.ascontiguousarray(assets, dtype=np.uint32)
        assert len(a) == len(arr) and (a < self.n_assets).all()
        lib().orc_market_set_groups(self._h, _ptr(arr), _ptr(a), len(arr))

    def run_agents(self, n_steps, seed, market_id=0, keyed=True):
        """market_sim_runner (runner.rs:107-131); keyed=True uses the Philox contract keyed by market id."""
        _check_agents(lib().orc_market_run(self._h, int(keyed), seed, market_id, n_steps))

    def n_instructions(self): return lib().orc_market_n_instructions(self._h)

    def time(self): return lib().orc_book_time(lib().orc_market_book(self._h, 0))
    def get_orders(self, asset): return self.asset(asset).get_orders()
    def get_trades(self, asset): return self.asset(asset).get_trades()
    def order_status(self, order_id): return self.asset(order_id[0]).order_status(order_id[1])

    def bid_asks(self):
        out = []
        for a in range(self.n_assets):
            l1 = np.zeros(8, np.uint32)
            lib().orc_book_l1(lib().orc_market_book(self._h, a), _ptr(l1))
            out.append((int(l1[0]), int(l1[1])))
        return out


class Market:
    """bourse_book::Market (crates/order_book/src/market.rs:59-365), immediate mode: an array of oracle OrderBooks."""

    def __init__(self, start_time, tick_size, trading=True):
        self._books = [OrderBook(start_time, int(t), trading) for t in tick_size]
        self._t = start_time

    def get_order_book(self, asset): return self._books[asset]
    def get_time(self): return self._t

    def set_time(self, t):
        self._t = t
        for b in self._books:
            b.set_time(t)

    def enable_trading(self): [b.enable_trading() for b in self._books]
    def disable_trading(self): [b.disable_trading() for b in self._books]
    def bid_vols(self): return [b.bid_vol() for b in self._books]
    def bid_best_vols(self): return [b.best_bid_vol() for b in self._books]
    def bid_best_vol_and_orders(self): return [b.best_bid_vol_and_orders() for b in self._books]
    def ask_vols(self): return [b.ask_vol() for b in self._books]
    def ask_best_vols(self): return [b.best_ask_vol() for b in self._books]
    def ask_best_vol_and_orders(self): return [b.best_ask_vol_and_orders() for b in self._books]
    def bid_asks(self): return [b.bid_ask() for b in self._books]
    def level_2_data(self): return np.stack([b.level_2_data() for b in self._books])
    def order(self, order_id): return self._books[order_id[0]].get_orders()[order_id[1]]

    def create_and_place_order(self, asset, bid, vol, trader_id, price=None):
        return (asset, self._books[asset].place_order(bid, vol, trader_id, price=price))

    def cancel_order(self, order_id): self._books[order_id[0]].cancel_order(order_id[1])

    def modify_order(self, order_id, new_price=None, new_vol=None):
        self._books[order_id[0]].modify_order(order_id[1], new_price=new_price, new_vol=new_vol)

    def get_orders(self, asset): return self._books[asset].get_orders()
    def get_trades(self, asset): return self._books[asset].get_trades()
