"""pack_actions' asset column (no GPU): `asset=` fills bb_instr::aux, the column MarketVectorEnv / bb_step_device_market
read as each row's asset, and leaving it out gives exactly the rows pack_actions gave before the column existed."""
import numpy as np

from bourse_b200 import abi, gym


def _columns(rng, shape):
    return dict(op=rng.integers(0, 5, shape).astype(np.uint32), bid=rng.random(shape) < 0.5, vol=rng.integers(0, 100, shape),
                trader=rng.integers(0, 1000, shape), price=rng.integers(0, 500, shape), order_id=rng.integers(0, 2**33, shape),
                market=rng.random(shape) < 0.2, has_price=rng.random(shape) < 0.5, has_vol=rng.random(shape) < 0.5)


def _reference_pack(op, bid, vol, trader, price, order_id, market, has_price, has_vol):
    """The packing rules restated field by field: what the default output must stay byte-identical to."""
    a = np.zeros(op.shape, dtype=abi.INSTR_DTYPE)
    f = op.astype(np.uint32).copy()
    new, mod = op == abi.OP_NEW, op == abi.OP_MODIFY
    f |= np.where(bid & new, abi.F_BID, 0).astype(np.uint32)
    f |= np.where(market & new, abi.F_MARKET, 0).astype(np.uint32)
    f |= np.where(mod & has_price, abi.F_HAS_PRICE, 0).astype(np.uint32)
    f |= np.where(mod & has_vol, abi.F_HAS_VOL, 0).astype(np.uint32)
    a["op_flags"] = f
    a["order_id"] = np.where(order_id > 0xFFFFFFFE, 0xFFFFFFFF, order_id).astype(np.uint32)
    a["price"], a["vol"], a["trader"] = price, vol, trader
    return a


def test_default_output_unchanged():
    rng = np.random.default_rng(0)
    for shape in [(7,), (4, 5), (2, 3, 6)]:
        c = _columns(rng, shape)
        got = gym.pack_actions(**c)
        assert got.tobytes() == _reference_pack(**c).tobytes()
        assert (got["aux"] == 0).all()
        assert gym.pack_actions(**c, asset=None).tobytes() == got.tobytes()


def test_asset_fills_aux_only():
    rng = np.random.default_rng(1)
    c = _columns(rng, (6, 8))
    asset = rng.integers(0, 5, (6, 8))
    got, base = gym.pack_actions(**c, asset=asset), gym.pack_actions(**c)
    assert np.array_equal(got["aux"], asset.astype(np.uint32))
    for k in ("t", "op_flags", "order_id", "price", "vol", "trader"):
        assert np.array_equal(got[k], base[k]), k
    # a scalar asset broadcasts over the rows
    assert (gym.pack_actions(**c, asset=3)["aux"] == 3).all()
