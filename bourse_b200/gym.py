"""Vectorised, device-resident environment loop (SURVEY.md 8f rank 4).

The reference's array API — `StepEnvNumpy.submit_instructions(...)` then `step()` then `level_2_data()`
(rust/src/step_sim_numpy.rs:233-275, :139-145, :351-368) — is the shape an RL loop uses, one env at a time with numpy
arrays on the host.  `VectorEnv` is that loop batched over `n_envs` envs with every array resident in DEVICE memory:
actions go in as a `[n_envs, rows_per_env]` block of packed instruction rows, the new order ids and the level-1 / level-2
observations come back as device arrays, and nothing crosses PCIe per step unless the caller asks for a host copy.

Buffers are exchanged through DLPack (`__dlpack__` / `__dlpack_device__`: `torch.from_dlpack(env.obs)`, `cupy.from_dlpack`,
`jax.dlpack`) and the CUDA array interface (`__cuda_array_interface__`, version 3), which torch, cupy and numba all
speak, so this module needs none of them: both give zero-copy views, and a torch / cupy array (anything with `__dlpack__`
or the CUDA array interface) can be passed to `step` directly.  numpy arrays are accepted too (copied host to device).

What happened to the learner's orders is read on the device as well: `orders(...)` returns the records of a block of order
ids (the reference's `get_orders()[id]` / `order_status(id)`) and `trades(cap)` the trades every book logged since the last
call (`get_trades()`), as device arrays, one launch each (bb_orders_device / bb_trades_device).

`MarketVectorEnv` is the same loop for multi-asset markets (`MarketEnv` place / cancel / modify then `step`, one block of
rows per market, each row naming its asset).  Use `VectorEnv` for independent single-asset envs, `MarketVectorEnv` when
assets share a market's shuffled queue, and `market.MarketEnv` for host-driven, order-by-order market use.
"""
from __future__ import annotations

import ctypes as C
import math
import typing

import numpy as np

from . import abi
from .core import BatchedEnv

# ---- DLPack (dlpack.h, v0.8 ABI: DLManagedTensor in a PyCapsule named "dltensor"), pure ctypes ---------------------------
KDL_CUDA, KDL_INT, KDL_UINT, KDL_BOOL = 2, 0, 1, 6


class _DLDevice(C.Structure):
    _fields_ = [("device_type", C.c_int32), ("device_id", C.c_int32)]


class _DLDataType(C.Structure):
    _fields_ = [("code", C.c_uint8), ("bits", C.c_uint8), ("lanes", C.c_uint16)]


class _DLTensor(C.Structure):
    _fields_ = [("data", C.c_void_p), ("device", _DLDevice), ("ndim", C.c_int32), ("dtype", _DLDataType),
                ("shape", C.POINTER(C.c_int64)), ("strides", C.POINTER(C.c_int64)), ("byte_offset", C.c_uint64)]


class _DLManagedTensor(C.Structure):
    pass


_DLDeleter = C.CFUNCTYPE(None, C.POINTER(_DLManagedTensor))
_DLManagedTensor._fields_ = [("dl_tensor", _DLTensor), ("manager_ctx", C.c_void_p), ("deleter", _DLDeleter)]
_api = C.pythonapi
_DLTENSOR = b"dltensor"   # (PyCapsule keeps the POINTER to its name: the bytes object must outlive every capsule)
_api.PyCapsule_New.restype, _api.PyCapsule_New.argtypes = C.py_object, [C.c_void_p, C.c_char_p, C.c_void_p]
_api.PyCapsule_IsValid.restype, _api.PyCapsule_IsValid.argtypes = C.c_int, [C.py_object, C.c_char_p]
_api.PyCapsule_GetPointer.restype, _api.PyCapsule_GetPointer.argtypes = C.c_void_p, [C.py_object, C.c_char_p]
_api.PyCapsule_SetName.restype, _api.PyCapsule_SetName.argtypes = C.c_int, [C.py_object, C.c_char_p]
_LIVE_EXPORTS: dict = {}   # address of an exported DLManagedTensor -> everything that must outlive its consumer


@_DLDeleter
def _dl_deleter(mt_ptr):   # called by the consumer when it drops the tensor: release our bookkeeping (the env owns the memory)
    _LIVE_EXPORTS.pop(C.addressof(mt_ptr.contents), None)


def _dlpack_import(x) -> typing.Tuple[int, int, typing.Any, typing.Tuple[int, ...], typing.Tuple[int, int]]:
    """(device pointer, byte size, keep-alive object, shape, (DLPack type code, bits)) of anything that exports DLPack;
    C-contiguous CUDA tensors only."""
    capsule = x.__dlpack__()
    if not _api.PyCapsule_IsValid(capsule, _DLTENSOR):
        raise ValueError("not a DLPack capsule")
    mt = C.cast(_api.PyCapsule_GetPointer(capsule, _DLTENSOR), C.POINTER(_DLManagedTensor)).contents
    t = mt.dl_tensor
    if t.device.device_type != KDL_CUDA:
        raise ValueError("DLPack tensor is not in CUDA device memory")
    shape = [t.shape[i] for i in range(t.ndim)]
    if t.strides:
        expect = 1
        for i in reversed(range(t.ndim)):
            if shape[i] != 1 and t.strides[i] != expect:
                raise ValueError("device arrays must be C-contiguous")
            expect *= shape[i]
    nbytes = int(np.prod(shape)) * (t.dtype.bits * t.dtype.lanes // 8)
    # the capsule is kept (un-renamed) together with its producer: its own destructor releases the tensor when we drop it
    return int(t.data) + int(t.byte_offset), nbytes, (capsule, x), tuple(shape), (int(t.dtype.code), int(t.dtype.bits))

ACTION_DTYPE = abi.INSTR_DTYPE  # one row = one instruction: (t ignored, op_flags, order_id, price, vol, trader, aux)


class DeviceArray:
    """A C-contiguous array in device memory owned by a `BatchedEnv`; speaks `__cuda_array_interface__`."""

    def __init__(self, env: BatchedEnv, shape: typing.Tuple[int, ...], dtype):
        self._env, self.shape, self.dtype = env, tuple(shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = env.device_alloc(self.nbytes)

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": self.dtype.str, "data": (self.ptr, False), "version": 3, "strides": None}

    def __dlpack_device__(self):
        return (KDL_CUDA, self._env.device)

    def __dlpack__(self, stream=None, **_kw):
        """DLPack export (zero copy): `torch.from_dlpack(arr)`.  The memory stays owned by the env — keep the env alive while
        views exist.  `stream`: the consumer's stream; the producer side is the env's stream, which the caller orders
        against as for any other use of the env's outputs (`env.synchronize()` or stream semantics of `set_stream`)."""
        if self.dtype.kind != "u":
            raise TypeError("only unsigned integer arrays are exported")
        mt = _DLManagedTensor()
        shape = (C.c_int64 * len(self.shape))(*self.shape)
        mt.dl_tensor = _DLTensor(C.c_void_p(self.ptr), _DLDevice(KDL_CUDA, self._env.device), len(self.shape),
                                 _DLDataType(KDL_UINT, 8 * self.dtype.itemsize, 1), shape, None, 0)
        mt.manager_ctx, mt.deleter = None, _dl_deleter
        _LIVE_EXPORTS[C.addressof(mt)] = (mt, shape, self)
        # no capsule destructor: a capsule that is never consumed leaves its ~200-byte bookkeeping entry behind (a ctypes
        # callback must not be handed a capsule that is being deallocated); a consumed one is released by `_dl_deleter`
        return _api.PyCapsule_New(C.addressof(mt), _DLTENSOR, None)

    def numpy(self) -> np.ndarray:
        """Host copy (synchronises the env's stream)."""
        out = np.empty(self.shape, self.dtype)
        self._env.memcpy(out.ctypes.data, self.ptr, self.nbytes, 2)
        return out

    def copy_from_host(self, a: np.ndarray):
        a = np.ascontiguousarray(a)
        assert a.nbytes == self.nbytes, "size mismatch"
        self._env.memcpy(self.ptr, a.ctypes.data, self.nbytes, 1)

    def free(self):
        if self.ptr:
            self._env.device_free(self.ptr)
            self.ptr = 0


def _device_array(x) -> typing.Optional[typing.Tuple[int, typing.Tuple[int, ...], np.dtype, typing.Any]]:
    """(device address, shape, dtype, keep-alive object) of a C-contiguous CUDA array (CUDA array interface or DLPack), or
    None for a host array.  The keep-alive object must outlive the launch that reads the array."""
    cai = getattr(x, "__cuda_array_interface__", None)
    if cai is not None:
        if cai.get("strides") is not None:
            raise ValueError("device arrays must be C-contiguous")
        return int(cai["data"][0]), tuple(cai["shape"]), np.dtype(cai["typestr"]), x
    if hasattr(x, "__dlpack__") and not isinstance(x, np.ndarray):   # DLPack-only producers
        ptr, _, keep, shape, (code, bits) = _dlpack_import(x)
        kind = "i" if code == KDL_INT else "u" if code == KDL_UINT else "b" if code == KDL_BOOL and bits == 8 else "V"
        return ptr, shape, np.dtype(f"{kind}{bits // 8}"), keep
    return None


def pack_actions(op, bid=None, vol=None, trader=None, price=None, order_id=None, market=None, has_price=None, has_vol=None,
                 asset=None) -> np.ndarray:
    """Columns -> packed instruction rows (host numpy, any shape).  `op`: abi.OP_NOOP / OP_NEW / OP_CANCEL / OP_MODIFY.
    NEW rows: `market=True` is a market order (`price=None` in the reference).  MODIFY rows: `has_price` / `has_vol` say
    which of `price` / `vol` is `Some` (default: both).  `asset`: the row's asset for `MarketVectorEnv` (the `aux` column;
    left 0 when not given)."""
    op = np.asarray(op, dtype=np.uint32)
    a = np.zeros(op.shape, dtype=ACTION_DTYPE)

    def col(x, default=0):
        return np.broadcast_to(np.asarray(default if x is None else x), op.shape)

    f = op.copy()
    f |= np.where(col(bid).astype(bool) & (op == abi.OP_NEW), abi.F_BID, 0).astype(np.uint32)
    f |= np.where(col(market).astype(bool) & (op == abi.OP_NEW), abi.F_MARKET, 0).astype(np.uint32)
    mod = op == abi.OP_MODIFY
    f |= np.where(mod & col(has_price, 1).astype(bool), abi.F_HAS_PRICE, 0).astype(np.uint32)
    f |= np.where(mod & col(has_vol, 1).astype(bool), abi.F_HAS_VOL, 0).astype(np.uint32)
    a["op_flags"] = f
    oid = col(order_id).astype(np.uint64)
    a["order_id"] = np.where(oid > 0xFFFFFFFE, 0xFFFFFFFF, oid).astype(np.uint32)  # ids beyond u32 cannot exist: bad id
    a["price"], a["vol"], a["trader"] = col(price), col(vol), col(trader)
    if asset is not None:
        a["aux"] = col(asset)
    return a


# bb_orders_device / bb_trades_device output columns (PyOrder / PyTrade fields, rust/src/types.rs:4-31)
ORDER_COLUMNS = (("side_is_bid", np.uint8), ("status", np.uint8), ("arr_time", np.uint64), ("end_time", np.uint64), ("vol", np.uint32),
                 ("start_vol", np.uint32), ("price", np.uint32), ("trader", np.uint32))
TRADE_COLUMNS = (("t", np.uint64), ("side_is_bid", np.uint8), ("price", np.uint32), ("vol", np.uint32), ("active_id", np.uint64),
                 ("passive_id", np.uint64))


NO_SLOT = abi.NO_SLOT


class Store:
    """A device store of `n_slots` unit snapshots made by `VectorEnv` / `MarketVectorEnv.snapshots` (bb_store_create).  A slot
    holds one unit's full state — books, order tables, trade logs, agent state and random streams — but not its history.
    `nbytes` is its size on the device.  It belongs to its env: `close()` frees it, and so does the env's `close()`."""

    def __init__(self, env: BatchedEnv, n_slots: int):
        self.env, self.n_slots = env, int(n_slots)
        self.ptr, self.nbytes = env.store_create(self.n_slots)

    def close(self):
        if self.ptr:
            self.env.store_destroy(self.ptr)
            self.ptr = 0


class _DeviceLoop:
    """What `VectorEnv` and `MarketVectorEnv` share: the handle, the device buffers, host-action staging, the history ring and
    the order / trade reads."""

    env: BatchedEnv
    obs: DeviceArray
    ids: DeviceArray
    _what = "env"
    _groups: typing.Optional[np.ndarray] = None   # the declared background population, abi.GROUP_DTYPE [n_groups]

    def _buffers(self, obs_shape, rows_shape):
        self.obs = DeviceArray(self.env, obs_shape, np.uint32)
        self.ids = DeviceArray(self.env, rows_shape, np.uint64)
        self._actions = DeviceArray(self.env, rows_shape, ACTION_DTYPE)  # staging for host-side actions
        self._offsets = DeviceArray(self.env, (rows_shape[0] + 1,), np.uint64)
        self._offsets.copy_from_host(np.arange(rows_shape[0] + 1, dtype=np.uint64) * np.uint64(rows_shape[1]))
        self._units, self._book_shape = rows_shape[0], tuple(obs_shape[:-1])
        self._cursor = DeviceArray(self.env, (self.env.n_envs,), np.uint32)  # trades(): each book's next unread trade
        self._cursor.copy_from_host(np.zeros(self.env.n_envs, np.uint32))
        self._reads: dict = {}   # orders() / trades() outputs and query staging, by kind and size: allocated once, then reused
        self._stores: typing.List[Store] = []

    def close(self):
        for st in self._stores:
            st.close()
        for a in (self.obs, self.ids, self._actions, self._offsets, self._cursor):
            a.free()
        for bufs in self._reads.values():
            for a in ((bufs,) if isinstance(bufs, DeviceArray) else bufs.values()):
                a.free()
        self.env.close()

    def _observe(self) -> DeviceArray:
        (self.env.level_1_data_device if self.obs_words == abi.OBS_L1 else self.env.level_2_data_device)(self.obs.ptr)
        return self.obs

    def reset(self, mask=None, seeds=None) -> DeviceArray:
        """Without `mask`: every env back to its freshly created state (`bb_reset`), the trade cursor zeroed.

        With `mask`, a `[units]` array (`units` = `n_envs`, or `n_markets` for `MarketVectorEnv`), only the units whose entry
        is non-zero are reset — gymnasium's per-env autoreset (bb_reset_device): their books are emptied, their history,
        order table, trade log and error bits restart at 0, their agents' state is cleared; every other unit is untouched.
        `mask` is a device array (CUDA array interface or DLPack: a torch `bool` / `uint8` tensor) or a numpy `bool` /
        `uint8` array (copied into a staging buffer).  `seeds` (same shape, 8-byte integers, device or numpy) re-seeds
        the reset units' shuffle streams as `StepEnvNumpy(seed, ...)` / `MarketEnv` construction does and restarts their
        step counters, so a unit reset with its creation seed (`seed + e`) replays episode 1 under the same actions; without
        `seeds` the streams continue (the next episode draws what the unit would have drawn without the reset, agent draws
        included).  One launch writes the reset units' rows of `self.obs` (the fresh record) and zeroes their entries of
        the `trades` cursor; returns `self.obs`.

        Order ids the learner holds for a reset env are void: a CANCEL of one flags `BB_ERR_BAD_ID` as any unknown id does.
        `self.obs` is overwritten for reset units: copy the final observation first if it is needed.  With device arrays
        for `mask` and `seeds` the call has no host synchronisation and can be captured into a CUDA graph together with
        `step` (a seeded `MarketVectorEnv` reset right after host-side `bb_step` shuffles refuses capture)."""
        if mask is None:
            if seeds is not None:
                raise ValueError("seeds re-seed the units a mask selects: pass a mask")
            self._n_steps = 0
            self.env.reset()   # (the agent population survives a reset; its state is cleared with the books)
            self._cursor.copy_from_host(np.zeros(self.env.n_envs, np.uint32))
            return self._observe()
        mask_ptr, keep_mask = self._unit_array(mask, np.uint8, "mask")
        seeds_ptr, keep_seeds = self._unit_array(seeds, np.uint64, "seeds") if seeds is not None else (0, None)
        self._keep = (keep_mask, keep_seeds)   # alive until the next call, as in _action_ptr
        self.env.reset_device(mask_ptr, seeds_ptr, self.obs.ptr, self._cursor.ptr)
        return self.obs

    def snapshots(self, n_slots: int) -> Store:
        """A device store of `n_slots` slots for `save` / `restore`, sized from the env's current capacities (every slot
        empty).  Growing a capacity (`env.reserve`), new agents or new tick sizes make it unusable: create another."""
        st = Store(self.env, n_slots)
        self._stores.append(st)
        return st

    def save(self, store: Store, units=None):
        """Save units into the slots of `store` (bb_save_device): slot k receives unit `units[k]`.  `units` is an
        `[n_slots]` array of 4-byte integers, device (CUDA array interface or DLPack) or numpy; `None` saves unit k into
        slot k.  `NO_SLOT` leaves a slot as it is, an index >= units empties it.  The env is not changed.  One launch on
        the env's stream with no host synchronisation (device `units`), so it can be captured into a CUDA graph."""
        if units is None:
            units = np.arange(store.n_slots, dtype=np.uint32)
        ptr, keep = self._unit_array(units, np.uint32, "units", store.n_slots)
        self._keep = keep   # alive until the next call, as in _action_ptr
        self.env.save_device(store.ptr, ptr)

    def restore(self, store: Store, slots, seeds=None) -> DeviceArray:
        """Restore units from the slots of `store` (bb_restore_device): unit u takes the state saved in slot `slots[u]`
        (`NO_SLOT`: untouched), several units may name one slot.  `slots` is a `[units]` array of 4-byte integers, device
        or numpy.  A restored unit is the saved one — books, order tables, trade logs, time, error bits, agent state —
        with its history count at 0.  Without `seeds` it takes the slot's shuffle stream and step counter, so a unit
        restored from its own snapshot continues bit-identically under the same actions (background agents draw by
        env / market id, so another unit restored from that slot draws other agent instructions).  `seeds` (`[units]`,
        8-byte integers) re-seeds the restored units' shuffle streams as `reset(mask, seeds)` does; the step counter stays
        the slot's.  A slot out of range, empty, or saved at another tick flags the unit (`BB_ERR_SLOT`, `check_errors`
        raises) and leaves it untouched.  The rows of restored units in `self.obs` receive their records, their `trades`
        cursors the restored logs' counts; returns `self.obs`.  Launches on the env's stream with no host synchronisation
        (device arrays), so it can be captured into a CUDA graph with `step`."""
        slots_ptr, keep_slots = self._unit_array(slots, np.uint32, "slots")
        seeds_ptr, keep_seeds = self._unit_array(seeds, np.uint64, "seeds") if seeds is not None else (0, None)
        self._keep = (keep_slots, keep_seeds)
        self.env.restore_device(store.ptr, slots_ptr, seeds_ptr, self.obs.ptr, self._cursor.ptr)
        return self.obs

    def agent_params(self) -> np.ndarray:
        """A host `abi.GROUP_DTYPE` array `[units, n_groups]` filled with the declared background groups: the template for
        `set_agent_params` (edit it, e.g. `p["rate"][:, 0] = rates`, and pass it back)."""
        if self._groups is None:
            raise ValueError("the env has no background agents")
        return np.tile(self._groups, (self._units, 1))

    def set_agent_params(self, params=None, *, keys=None, mask=None):
        """Per-unit background-agent parameters and Philox keys (bb_set_agent_params_device); a unit is an env, or a market
        for `MarketVectorEnv`.  Every unit `mask` selects (default: all) takes its row of `params` and / or its entry of
        `keys`; every later `step` runs group gi of unit u with `params[u, gi]` and draws with the agent seed XOR `keys[u]`
        (agent draws and the step's shuffle).  Keys start at 0, the parameters at the declared groups.

        `params`: the `[units, n_groups]` array `agent_params()` returns, edited, or any C-contiguous device array (CUDA
        array interface / DLPack) of exactly `units * n_groups * 80` bytes in that layout; `None` keeps the parameters.
        `keys`: `[units]` 8-byte integers; `mask`: `[units]` bool / 1-byte integers; each a device array or numpy.  Rows
        must stay inside the declared population: same kind, agent count and tick size; RandomAgents tick and volume
        ranges inside the declared ones; Momentum / Noise agent id start and live-list capacity (`tick_lo`, `vol_hi`)
        unchanged.  A unit with any other row keeps its parameters and key and is flagged (`BB_ERR_PARAMS`,
        `check_errors` raises).  `reset` and `restore` keep parameters and keys.  One launch with no host
        synchronisation (device arrays)."""
        if params is None and keys is None:
            raise ValueError("pass params, keys or both")
        if self._groups is None:
            raise ValueError("the env has no background agents")
        units, ng = self._units, len(self._groups)
        nbytes = units * ng * abi.GROUP_DTYPE.itemsize
        params_ptr, keep_params, host_params = 0, None, None
        if params is not None:
            dev = _device_array(params)
            if dev is not None:
                params_ptr, shape, typ, keep_params = dev
                n = int(np.prod(shape)) * typ.itemsize
                if n != nbytes:
                    raise ValueError(f"params: device array holds {n} bytes, expected {nbytes} ([{units}, {ng}] records of 80 bytes)")
            else:
                host_params = np.asarray(params)
                if host_params.dtype != abi.GROUP_DTYPE or host_params.shape != (units, ng):
                    raise ValueError(f"params must be a [{units}, {ng}] abi.GROUP_DTYPE array (agent_params())")
        keys_ptr, keep_keys = self._unit_array(keys, np.uint64, "keys") if keys is not None else (0, None)
        mask_ptr, keep_mask = self._unit_array(mask, np.uint8, "mask") if mask is not None else (0, None)
        if host_params is not None:
            buf = self._buffer(("params", units, ng), (nbytes,), np.uint8)
            buf.copy_from_host(np.ascontiguousarray(host_params).view(np.uint8).reshape(-1))
            params_ptr = buf.ptr
        self._keep = (keep_params, keep_keys, keep_mask)   # alive until the next call, as in _action_ptr
        self.env.set_agent_params_device(params_ptr, keys_ptr, mask_ptr)

    def _unit_array(self, x, dtype, name, n=None) -> typing.Tuple[int, typing.Any]:
        """(device address, keep-alive object) of an [n] (default: [units]) mask (bool / 1-byte integers), unit or slot
        array (4-byte integers) or seed array (8-byte integers): the caller's device array, or a staging copy of a host
        array."""
        dtype, units = np.dtype(dtype), self._units if n is None else n
        kinds = "biu" if dtype.itemsize == 1 else "iu"
        what = f"{name} must be a [{units}] array of " + ("bool or 1-byte integers" if dtype.itemsize == 1 else f"{dtype.itemsize}-byte integers")
        dev = _device_array(x)
        if dev is not None:
            ptr, shape, typ, keep = dev
            if shape != (units,) or typ.kind not in kinds or typ.itemsize != dtype.itemsize:
                raise ValueError(what)
            return ptr, keep
        a = np.asarray(x)
        if a.shape != (units,) or a.dtype.kind not in kinds or (dtype.itemsize == 1 and a.dtype.itemsize != 1):
            raise ValueError(what)
        if dtype.itemsize == 4 and a.size and (int(a.min()) < 0 or int(a.max()) > 0xFFFFFFFF):
            raise ValueError(what + " in [0, 2^32)")
        buf = self._buffer((name, units), (units,), dtype)
        buf.copy_from_host(a.astype(dtype))
        return buf.ptr, None

    def _buffer(self, key, shape, dtype) -> DeviceArray:
        if key not in self._reads:
            self._reads[key] = DeviceArray(self.env, shape, dtype)
        return self._reads[key]

    def _columns(self, key, shape, columns) -> dict:
        if key not in self._reads:
            self._reads[key] = {name: DeviceArray(self.env, shape, dt) for name, dt in columns}
        return self._reads[key]

    def _query_block(self, x, dtype, name) -> typing.Tuple[int, int]:
        """(device address, k) of a [units, k] query block: the caller's device array (CUDA array interface or DLPack, any
        integer type of `dtype`'s size), or a staging copy of a host array."""
        dtype, units = np.dtype(dtype), self._units
        dev = _device_array(x)
        if dev is not None:
            ptr, shape, typ, self._keep = dev   # alive until the next call: the launch that reads it is already enqueued by then
            if len(shape) != 2 or shape[0] != units or typ.kind not in "iu" or typ.itemsize != dtype.itemsize:
                raise ValueError(f"{name} must be a [{units}, k] array of {dtype.itemsize}-byte integers")
            return ptr, int(shape[1])
        a = np.ascontiguousarray(x, dtype=dtype)
        if a.ndim != 2 or a.shape[0] != units:
            raise ValueError(f"{name} must have shape [{units}, k]")
        buf = self._buffer((name, a.shape[1]), a.shape, dtype)
        buf.copy_from_host(a)
        return buf.ptr, a.shape[1]

    def _orders(self, ids, assets) -> typing.Dict[str, DeviceArray]:
        ids_ptr, k = self._query_block(ids, np.uint64, "ids")
        assets_ptr = 0
        if assets is not None:
            assets_ptr, ka = self._query_block(assets, np.uint32, "assets")
            if ka != k:
                raise ValueError("ids and assets must have the same shape")
        out = self._columns(("orders", k), (self._units, k), ORDER_COLUMNS)
        if k:
            self.env.orders_device(ids_ptr, assets_ptr, k, **{name: a.ptr for name, a in out.items()})
        return out

    def trades(self, cap: int) -> typing.Tuple[typing.Dict[str, DeviceArray], DeviceArray]:
        """The trades every book logged since the last call (bb_trades_device): `(columns, count)`.  `columns` are `DeviceArray`s
        keyed `t, side_is_bid, price, vol, active_id, passive_id` (the PyTrade fields, ids as u64), shaped `[n_envs, cap]` (a
        `MarketVectorEnv`: `[n_markets, assets, cap]`); a book's first `min(count, cap)` slots hold its new trades in log
        order, the rest `active_id = passive_id = abi.NO_ID` and zeros.  `count` (`[n_envs]` / `[n_markets, assets]`) is the
        number of trades each book had to report; it may exceed `cap`, and the ones that did not fit come with the next call.
        The env keeps the read position of every book (zeroed by `reset()`).  Trades a full log (`max_trades`) could not
        hold are not reported; `check_errors` raises for them.  One launch on the env's stream, ordered after the steps
        before it, with no host synchronisation; the outputs are allocated on the first call for a given `cap` and
        overwritten by the next call with that `cap`.  Make that first call before capturing one into a CUDA graph."""
        cols = self._columns(("trades", cap), self._book_shape + (cap,), TRADE_COLUMNS)
        count = self._buffer(("count", cap), self._book_shape, np.uint32)
        self.env.trades_device(self._cursor.ptr, cap, count.ptr, **{name: a.ptr for name, a in cols.items()})
        return cols, count

    def _action_ptr(self, actions) -> int:
        """Device address of the step's action block: the caller's device array, or the staging copy of a host array."""
        shape, nbytes = self._actions.shape, self._actions.nbytes
        dev = _device_array(actions)
        if dev is not None:
            ptr, dshape, typ, self._keep = dev   # alive until the next call: the launch that reads it is already enqueued by then
            n = int(np.prod(dshape)) * typ.itemsize
            if n != nbytes:
                raise ValueError(f"device array holds {n} bytes, expected {nbytes}")
        else:  # host array: one H2D copy
            a = np.ascontiguousarray(actions, dtype=ACTION_DTYPE)
            if a.shape != shape:
                raise ValueError(f"actions must have shape {shape}")
            self._actions.copy_from_host(a)
            ptr = self._actions.ptr
        # an open-ended loop consumes each observation as it is produced: the library's per-step history is a scratch ring here
        self._n_steps += 1
        if self._n_steps > self.env.max_steps:
            self.env.clear_history()
            self._n_steps = 1
        return ptr

    def check_errors(self):
        """Raise if any env flagged an error (capacity, bad order id, off-tick price, a refused `set_agent_params` row);
        synchronises."""
        e = self.env.env_errors()
        if e.any():
            bad = np.flatnonzero(e)
            params = " (0x2000: a set_agent_params row outside the declared population)" if (e & abi.ERR_PARAMS).any() else ""
            raise RuntimeError(f"{len(bad)} {self._what}(s) flagged errors, first {self._what} {bad[0]}: 0x{int(e[bad[0]]):x}{params}")


class VectorEnv(_DeviceLoop):
    """`n_envs` lockstep `StepEnvNumpy(seed + env, start_time, tick_size, step_size, trading)` instances with a fixed action
    block of `rows_per_env` instruction rows per env and step (pad with OP_NOOP rows).

        env = VectorEnv(4096, rows_per_env=8, seed=0, start_time=0, tick_size=1, step_size=1000)
        obs = env.reset()                       # DeviceArray [n_envs, 45] u32, StepEnvNumpy.level_2_data layout
        obs, ids = env.step(actions)            # actions: [n_envs, rows_per_env] packed rows, device or host
        t = torch.as_tensor(obs, device="cuda") # zero-copy

    `ids[e, r]` is the order id row r created in env e, or `abi.NO_ID` (2^64 - 1) for cancel / modify / no-op rows
    (step_sim_numpy.rs:256-267).  Semantics per env are exactly `submit_instructions` + `step`: ids in row order, the
    step's queue shuffled with the env's own Xoroshiro stream, event i at `t + i`.  A NEW row with an off-tick limit
    price creates nothing (the reference raises ValueError there); the env is flagged and `check_errors` raises.
    `tick_size` may be a sequence of `n_envs` ticks, one per env (`core.BatchedEnv`): each env then checks its rows
    against, and lays out its level-2 observation at, its own tick.

    Without background agents a step is ONE kernel launch on the env's stream (`env.set_stream(...)`) with no host
    synchronisation, so a loop of policy + `step` can be captured into a CUDA graph and replayed (tests/test_gpu_gym.py);
    steps that include the built-in agents refuse capture (their history staging is validated on the host).  The library's
    per-step history is a scratch ring for this class: `step` clears it (`bb_clear_history`) whenever `max_steps` records
    have accumulated; a caller replaying a captured step must do the same every `max_steps` replays.

    With background agents, `set_agent_params` gives each env its own group parameters (a market regime per env) and its own
    agent key.  Reproducible but distinct episodes: `reset(mask, seeds)` with the envs' creation seeds replays the same agent
    draws, and `set_agent_params(keys=new_keys, mask=mask)` before it makes them new ones; the same key replays them.

    Deep books: `price_window=(lo, hi)` with `deep_chunks=N` (see `core.BatchedEnv`) runs every env on the deep-book engine,
    for books with thousands to millions of resting orders.  Preload them with `self.env.replay(...)` (or a saved book), copy
    them into many envs with `save` / `restore`, then `step` as above: same semantics, two kernel launches per step and still
    no host synchronisation, so the step can be captured into a CUDA graph.  Every limit price that rests must lie inside the
    window, and `step_size` must be at least `max_queue` (the engine needs strictly increasing times between resting orders;
    otherwise the env is flagged `BB_ERR_TIME_ORDER`).  For the same reason a preload stream should end with a no-op one
    nanosecond after its last event: a step's first event runs at the book's time.  Background agents (`agents=`) run on
    deep books too, two launches per step as well: every RandomAgents price range must lie inside the window (the
    library refuses the population otherwise), and Momentum / Noise quotes that leave it flag `BB_ERR_CAP_PAGES`."""

    def __init__(self, n_envs: int, rows_per_env: int, seed: int, start_time: int, tick_size: typing.Union[int, typing.Sequence[int]], step_size: int,
                 trading: bool = True, *, level_1: bool = False, agents=None, agent_seed: int = 0, **kw):
        """`agents`: optional background population (a list of `core.random_group` / `momentum_group` / `noise_group`
        records).  With it every `step` is `{ agents.update(env); the action rows; env.step() }` in one launch
        (bb_run_agents_with_rows): the rows join the agents' instructions in the step's one shuffled queue (Philox key
        `agent_seed`).  Action rows may then be NEW, CANCEL or no-op (MODIFY is refused).  At one step per launch the
        general engine (no `price_window`) is the faster choice here: 92 us against 117 us per 4096-env step on the dense
        engine, whose per-launch agent-table rebuild only pays off inside the persistent multi-step kernel."""
        n_bg = sum(int(g["n_agents"]) for g in agents) if agents else 0
        kw.setdefault("max_queue", max(rows_per_env + 2 * n_bg, 16))
        if rows_per_env > kw["max_queue"]:
            raise ValueError("rows_per_env exceeds max_queue")
        self._agents, self._agent_seed = agents, agent_seed
        self._groups = np.array(list(agents), dtype=abi.GROUP_DTYPE) if agents else None
        self._n_steps = 0
        self.n_envs, self.rows = n_envs, rows_per_env
        self.env = BatchedEnv(n_envs, seed, start_time, tick_size, step_size, trading, obs_words=abi.OBS_L1 if level_1 else abi.OBS_L2, **kw)
        self.obs_words = abi.OBS_L1 if level_1 else abi.OBS_L2
        try:
            self._buffers((n_envs, self.obs_words), (n_envs, rows_per_env))
            if agents:
                self.env.set_agents(agents)
        except Exception:
            self.env.close()
            raise

    def step(self, actions) -> typing.Tuple[DeviceArray, DeviceArray]:
        ptr = self._action_ptr(actions)
        # one launch: (background agents,) ids, Env::step and the observation records written straight into self.obs
        if self._agents:
            self.env.run_agents_with_rows(self._agent_seed, ptr, self._offsets.ptr, self.n_envs * self.rows, self.ids.ptr, self.obs.ptr)
        else:
            self.env.step_device(ptr, self._offsets.ptr, self.n_envs * self.rows, self.ids.ptr, self.obs.ptr)
        return self.obs, self.ids

    def orders(self, ids) -> typing.Dict[str, DeviceArray]:
        """The records of the orders `ids` names (bb_orders_device; `get_orders()[id]` / `order_status(id)` of every env at
        once).  `ids`: a `[n_envs, k]` block of 8-byte ids, row e naming orders of env e — a device array (CUDA array
        interface / DLPack: `env.ids`, a torch tensor, the id columns of `trades`) or a numpy array (copied as `step` copies
        actions).  Returns `DeviceArray` columns `[n_envs, k]` keyed `side_is_bid, status, arr_time, end_time, vol,
        start_vol, price, trader` (the PyOrder fields).  An `abi.NO_ID` entry reads as status `abi.STATUS_NONE` with zeros
        and is no error, so blocks may be padded; an id the env has not issued reads the same and flags the env
        (`check_errors` raises).  One launch on the env's stream with no host synchronisation (device ids); the columns are
        allocated on the first call for a given `k` and overwritten by the next call with that `k`.  Make that first call
        before capturing one into a CUDA graph."""
        return self._orders(ids, None)


class MarketVectorEnv(_DeviceLoop):
    """`n_markets` lockstep `MarketEnv::new(start_time, tick_sizes, step_size, trading)` instances (market_env.rs:73-90),
    market m shuffling with `Xoroshiro128StarStar::seed_from_u64(seed + m)`, driven by a fixed block of `rows_per_market`
    instruction rows per market and step (pad with OP_NOOP rows; `pack_actions(..., asset=...)` sets each row's asset).

        env = MarketVectorEnv(2048, rows_per_market=8, seed=0, start_time=0, tick_sizes=[1, 2, 5, 10], step_size=1000)
        obs = env.reset()                       # DeviceArray [n_markets, assets, 45] u32
        obs, ids = env.step(actions)            # actions: [n_markets, rows_per_market] packed rows, device or host

    Per market, a step is exactly `MarketEnv::place_order / cancel_order / modify_order` for each row in row order, then
    `MarketEnv::step(rng)` (bb_step_device_market): `ids[m, r]` is the id row r created in its asset's book (order ids are
    per asset, `MarketOrderId = (asset, ids[m, r])`) or `abi.NO_ID`; CANCEL / MODIFY rows target `(asset, order_id)`.  An
    off-tick limit price creates nothing and flags its asset's book (`check_errors` raises).  `obs[m, a]` is asset a's
    end-of-step record.  A step is one kernel launch with no host synchronisation, so it can be captured into a CUDA graph;
    the history is a scratch ring as in `VectorEnv`.  `tick_sizes` has one tick per asset, at least two assets (a
    one-asset market is an Env: use `VectorEnv`).

    With `agents` (the `market.RandomMarketAgents` / `MomentumMarketAgent` / `NoiseMarketAgent` objects that
    `market.MarketEnv.set_agents` takes) every market is populated: a step is `agents.update(env)`, the rows, then
    `MarketEnv::step` (bb_run_agents_with_rows_market), in one launch that refuses CUDA-graph capture.

    Which class: this one for an RL-style loop over many markets, alone (no `agents`) or against built-in agents in the
    same shuffled queue (`agents=`); `market.MarketEnv` (`place_order` / `submit` + `step` on the host) for scripted,
    order-by-order use, and its `run_agents` for markets of built-in agents with no learner.

    With `agents`, `set_agent_params` gives each market its own group parameters (group gi applies to its asset's book) and
    its own agent key; `reset(mask, seeds)` plus `set_agent_params(keys=..., mask=...)` gives reproducible but distinct
    episodes, as for `VectorEnv`."""

    _what = "book"

    def __init__(self, n_markets: int, rows_per_market: int, seed: int, start_time: int, tick_sizes: typing.Sequence[int],
                 step_size: int, trading: bool = True, *, level_1: bool = False, agents=None, agent_seed: int = 0, **kw):
        """`agents`: optional background population, a list of `market.RandomMarketAgents` / `MomentumMarketAgent` /
        `NoiseMarketAgent`.  With it every `step` is `{ agents.update(env); the action rows; MarketEnv::step }` for every
        market in one launch: the rows follow all groups' instructions in the market's one shuffled queue (Philox key
        `agent_seed`), and each row's id in its asset's book comes after the ids the agents took.  Action rows may then be
        NEW, CANCEL or no-op (MODIFY is refused).  At most 4 assets: a market's books are the warps of one CTA."""
        ticks = [int(t) for t in tick_sizes]
        if len(ticks) < 2:
            raise ValueError("MarketVectorEnv needs two or more assets; a one-asset market is an Env: use VectorEnv")
        if min(ticks) <= 0:
            raise ValueError("tick sizes must be > 0")
        A = len(ticks)
        if agents:
            if A > 4:
                raise ValueError("in-kernel market agents support at most 4 assets per market")
            per_asset = [0] * A
            for a in agents:
                if not 0 <= a.asset < A:
                    raise ValueError("agent group asset index out of range")
                per_asset[a.asset] += int(a.group["n_agents"])
            # each book's queue holds its agents' instructions and, at worst, every row of the market
            kw.setdefault("max_queue", max(2 * max(per_asset) + rows_per_market, 16))
        else:
            kw.setdefault("max_queue", max(-(-rows_per_market // A), 16))   # a market's queue holds assets * max_queue rows
        if rows_per_market > A * kw["max_queue"]:
            raise ValueError("rows_per_market exceeds assets * max_queue")
        if A * kw["max_queue"] > 65535:
            raise ValueError("assets * max_queue must stay below 65536")
        self._agents, self._agent_seed = agents, agent_seed
        self._groups = np.array([a.group for a in agents], dtype=abi.GROUP_DTYPE) if agents else None
        self._n_steps = 0
        self.n_markets, self.rows, self.n_assets, self.tick_sizes = n_markets, rows_per_market, A, ticks
        self.obs_words = abi.OBS_L1 if level_1 else abi.OBS_L2
        # as market.MarketEnv: the handle's tick is the gcd of the assets' ticks, each book then gets its asset's own
        granule = math.gcd(*ticks)
        self.env = BatchedEnv(A * n_markets, seed, start_time, granule, step_size, trading, assets=A, obs_words=self.obs_words, **kw)
        try:
            if any(t != granule for t in ticks):
                self.env.set_tick_sizes(ticks)
            self._buffers((n_markets, A, self.obs_words), (n_markets, rows_per_market))
            if agents:
                self.env.set_agents([a.group for a in agents], assets=[a.asset for a in agents])
        except Exception:
            self.env.close()
            raise

    def step(self, actions) -> typing.Tuple[DeviceArray, DeviceArray]:
        ptr = self._action_ptr(actions)
        # one launch: (background agents,) ids, the market-wide shuffle, MarketEnv::step and the observation records written
        # straight into self.obs
        if self._agents:
            self.env.run_agents_with_rows_market(self._agent_seed, ptr, self._offsets.ptr, self.n_markets * self.rows, self.ids.ptr,
                                                 self.obs.ptr)
        else:
            self.env.step_device_market(ptr, self._offsets.ptr, self.n_markets * self.rows, self.ids.ptr, self.obs.ptr)
        return self.obs, self.ids

    def orders(self, ids, assets) -> typing.Dict[str, DeviceArray]:
        """The records of the orders `(assets, ids)` name (bb_orders_device; `MarketEnv.get_orders(asset)[id]` of every
        market at once).  `ids` (8-byte integers) and `assets` (4-byte integers) are `[n_markets, k]` blocks: entry
        `[m, j]` names order `ids[m, j]` of asset `assets[m, j]`'s book in market m, as `step`'s ids and action rows do.
        Device arrays or numpy arrays, as in `VectorEnv.orders`; the returned `DeviceArray` columns are `[n_markets, k]`
        with the same keys.  An `abi.NO_ID` entry reads as status `abi.STATUS_NONE` with zeros and is no error; an id the
        book has not issued, or an asset outside the market, reads the same and flags a book (`check_errors` raises).  One
        launch on the env's stream; outputs are allocated on the first call for a given `k`, overwritten by the next call
        with that `k`."""
        return self._orders(ids, assets)
