"""CPU suite for host-side logic that needs no GPU: action packing of the vectorised loop (bourse_b200.gym), the agent-group
records built by the Rust-named constructors (bourse_b200.market / core), shard ranges, and the bench's synthetic policy."""
import types

import numpy as np
import pytest

from bourse_b200 import abi, core, gym, market, sharding, workloads


def test_pack_actions_flags_and_fields():
    op = np.array([abi.OP_NEW, abi.OP_NEW, abi.OP_CANCEL, abi.OP_MODIFY, abi.OP_MODIFY, abi.OP_NOOP], np.uint32)
    a = gym.pack_actions(op, bid=[1, 0, 1, 1, 0, 1], vol=[5, 6, 7, 8, 9, 10], trader=3, price=[50, 52, 0, 60, 61, 99],
                         order_id=[0, 0, 4, 2**40, 6, 0], market=[0, 1, 1, 1, 0, 0], has_price=[1, 1, 1, 0, 1, 1], has_vol=[1, 1, 1, 1, 0, 1])
    assert a.dtype == abi.INSTR_DTYPE and a.shape == (6,)
    f = a["op_flags"]
    assert f[0] == abi.OP_NEW | abi.F_BID                      # limit bid: no MARKET / HAS_* bits on NEW rows
    assert f[1] == abi.OP_NEW | abi.F_MARKET                   # market ask
    assert f[2] == abi.OP_CANCEL                               # side / market columns are ignored outside NEW rows
    assert f[3] == abi.OP_MODIFY | abi.F_HAS_VOL               # new_price = None
    assert f[4] == abi.OP_MODIFY | abi.F_HAS_PRICE             # new_vol = None
    assert f[5] == abi.OP_NOOP
    assert a["order_id"][3] == 0xFFFFFFFF                      # ids beyond u32 cannot exist: kept out of range (bad id)
    assert list(a["vol"]) == [5, 6, 7, 8, 9, 10] and (a["trader"] == 3).all() and (a["t"] == 0).all()


def test_pack_actions_broadcasts_to_blocks():
    op = np.full((4, 3, 2), abi.OP_NEW, np.uint32)
    a = gym.pack_actions(op, bid=True, vol=7, price=np.arange(2) + 10)
    assert a.shape == (4, 3, 2) and (a["price"][..., 1] == 11).all() and (a["op_flags"] == (abi.OP_NEW | abi.F_BID)).all()
    assert a.nbytes == 4 * 3 * 2 * 32


def test_device_array_import():
    class Fake:
        def __init__(self, shape, typestr, strides=None):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (0xABC000, False), "version": 3, "strides": strides}
    ptr, shape, dtype, _ = gym._device_array(Fake((4, 2, 32), "|u1"))
    assert (ptr, shape, dtype) == (0xABC000, (4, 2, 32), np.dtype(np.uint8))
    assert gym._device_array(np.zeros(4)) is None             # host arrays take the copy path
    loop = types.SimpleNamespace(_actions=types.SimpleNamespace(shape=(4, 2), nbytes=256))
    with pytest.raises(ValueError, match="bytes"):            # the action block's size is checked against the env's
        gym._DeviceLoop._action_ptr(loop, Fake((4, 2), "<u4"))
    with pytest.raises(ValueError, match="contiguous"):
        gym._device_array(Fake((4, 2, 32), "|u1", strides=(128, 64, 2)))


def test_market_agent_constructors_follow_the_rust_argument_order():
    r = market.RandomMarketAgents(1, 50, (40, 60), (10, 20), 2, 0.8)          # random_agent.rs:173-202
    g = r.group
    assert r.asset == 1 and g["kind"] == abi.GROUP_RANDOM and g["n_agents"] == 50 and (g["tick_lo"], g["tick_hi"]) == (40, 60)
    assert (g["vol_lo"], g["vol_hi"]) == (10, 20) and g["tick_size"] == 2 and abs(float(g["rate"]) - 0.8) < 1e-6
    mp = market.MomentumParams(tick_size=2, p_cancel=0.1, trade_vol=10, decay=1.0, demand=5.0, scale=0.5, order_ratio=1.0,
                               price_dist_mu=0.0, price_dist_sigma=10.0)
    m = market.MomentumMarketAgent(100, 20, 3, mp)                            # momentum_agent.rs:294-325: (id start, n, asset, params)
    assert m.asset == 3 and m.group["kind"] == abi.GROUP_MOMENTUM and m.group["tick_lo"] == 100 and m.group["n_agents"] == 20
    assert m.group["vol_lo"] == 10 and m.group["sigma"] == 10.0 and m.group["order_ratio"] == 1.0
    np_ = market.NoiseAgentParams(tick_size=2, p_limit=0.5, p_market=0.25, p_cancel=0.1, trade_vol=100, price_dist_mu=0.0, price_dist_sigma=1.0)
    n = market.NoiseMarketAgent(2, 10, 4, np_)                                # noise_agent.rs:236-258: (asset, id start, n, params)
    assert n.asset == 2 and n.group["kind"] == abi.GROUP_NOISE and n.group["tick_lo"] == 10 and n.group["n_agents"] == 4
    assert n.group["decay"] == 0.5 and n.group["demand"] == 0.25 and abs(float(n.group["rate"]) - 0.1) < 1e-6
    same = core.noise_group(10, 4, 2, 0.5, 0.25, 0.1, 100, 0.0, 1.0)
    assert n.group.tobytes() == same.tobytes()


def test_live_list_capacity_travels_in_vol_hi():
    """bb_agent_group::vol_hi of a Momentum / Noise group is the capacity of its live-order list (include/bourse_b200.h);
    0, the default of the constructors, keeps the library's 254."""
    assert core.momentum_group(0, 5, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0)["vol_hi"] == 0
    assert core.momentum_group(0, 5, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0, live_cap=4096)["vol_hi"] == 4096
    assert core.noise_group(10, 4, 2, 0.5, 0.25, 0.1, 100, 0.0, 1.0, live_cap=777)["vol_hi"] == 777
    # C4's population asks for nothing beyond the default: the benched configuration is unchanged
    assert all(int(g["vol_hi"]) == 0 for g in workloads.c4_groups() if int(g["kind"]) != abi.GROUP_RANDOM)


def test_market_example_population():
    groups, assets = workloads.market_example_groups()        # crates/step_sim/examples/multi_asset/main.rs:15-20
    assert assets == [0, 0, 1, 1] and len(groups) == 4
    assert [int(g["n_agents"]) for g in groups] == [50, 50, 50, 50]
    assert groups[0].tobytes() == groups[2].tobytes() and groups[1].tobytes() == groups[3].tobytes()


def test_shard_ranges_keep_markets_whole():
    # consecutive blocks, sizes differ by at most one, cover everything exactly once
    for total, world in ((4096, 8), (1000, 3), (7, 8)):
        spans = [sharding.shard_range(total, world, r) for r in range(world)]
        assert spans[0][0] == 0 and sum(n for _, n in spans) == total
        assert all(spans[i][0] + spans[i][1] == spans[i + 1][0] for i in range(world - 1))
        assert max(n for _, n in spans) - min(n for _, n in spans) <= 1
    # multi-asset markets stay whole: blocks are multiples of `assets`, whatever the remainder
    for total, world, a in ((14, 4, 2), (4096 * 3, 5, 3), (8, 8, 4)):
        spans = [sharding.shard_range(total, world, r, multiple=a) for r in range(world)]
        assert all(b % a == 0 and n % a == 0 for b, n in spans) and sum(n for _, n in spans) == total
        assert all(spans[i][0] + spans[i][1] == spans[i + 1][0] for i in range(world - 1))
    with pytest.raises(ValueError):
        sharding.shard_range(7, 2, 0, multiple=2)


def test_bench_gym_policy_never_names_an_unissued_id():
    import bench

    blocks = bench.gym_action_blocks(32, 16, 8, 3)
    assert blocks.shape == (32, 16, 8) and ((blocks["op_flags"][:, :, :2] & 0xFF) == abi.OP_NEW).all()
    issued = np.zeros(16, np.int64)
    for s in range(32):
        op = blocks["op_flags"][s] & 0xFF
        cancels = op == abi.OP_CANCEL
        assert (blocks["order_id"][s][cancels] < np.broadcast_to(issued[:, None], op.shape)[cancels]).all()
        issued += (op == abi.OP_NEW).sum(axis=1)


def test_data_processing_frames_match_the_reference_layout():
    """src/bourse/data_processing.py:10-105: column names (incl. the reference's `arr time`), side / status mappings."""
    from bourse_b200 import data_processing as dp
    t = dp.trades_to_dataframe([(10, False, 60, 20, 4, 1), (20, True, 55, 10, 5, 2)])
    assert list(t.columns) == ["time", "side", "price", "vol", "active_id", "passive_id"]
    assert list(t["side"]) == ["ask", "bid"] and list(t["vol"]) == [20, 10]
    o = dp.orders_to_dataframe([(True, 2, 0, 10, 0, 10, 50, 11, 0), (False, 1, 0, 2**64 - 1, 5, 20, 60, 12, 1)])
    assert list(o.columns) == ["side", "status", "arr time", "end_time", "vol", "start_vol", "price", "trader_id", "order_id"]
    assert list(o["side"]) == ["bid", "ask"] and list(o["status"]) == ["filled", "active"]
