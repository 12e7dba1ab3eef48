"""GPU suite for the submission of device-resident rows (bb_step_device, bb_run_agents_with_rows): rows that create nothing
get BB_NO_ID and take no id, checked against the oracle."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

pytestmark = pytest.mark.gpu


def test_background_agent_rows_drop_a_new_with_a_trader_id_beyond_19_bits(oracle):
    """bb_run_agents_with_rows: a NEW whose trader id does not fit 19 bits is dropped (BB_NO_ID, BB_ERR_ROW_OP) and the next
    NEW row takes the id it would have taken; every env then keeps matching the oracle without that row."""
    groups = workloads.c3_groups()
    n_envs, rows, seed = 4, 2, 5
    rng = np.random.default_rng(3)
    v = gym.VectorEnv(n_envs, rows, 0, 0, 1, 1_000_000, agents=groups, agent_seed=seed, max_orders=4096, max_trades=4096,
                      max_steps=16, max_queue=160)
    orcs = [oracle.StepEnv(0, 0, 1, 1_000_000) for _ in range(n_envs)]
    for o in orcs:
        o.set_groups(groups)
    v.reset()
    for s in range(6):
        op = np.full((n_envs, rows), abi.OP_NEW, np.uint32)
        bid, vol, price = rng.random((n_envs, rows)) < 0.5, rng.integers(1, 30, (n_envs, rows)), 2 * rng.integers(40, 61, (n_envs, rows))
        trader = np.full((n_envs, rows), 7, np.uint64)
        if s == 0:
            trader[0, 0] = 1 << 19
        obs, ids = v.step(gym.pack_actions(op, bid=bid, vol=vol, trader=trader, price=price))
        obs, ids = obs.numpy(), ids.numpy()
        if s == 0:
            assert ids[0, 0] == abi.NO_ID
            err = v.env.env_errors()
            assert err[0] == 0x400 and (err[1:] == 0).all()
            v.env.clear_errors()
        for e, o in enumerate(orcs):
            o.agents_update(seed, e)
            for r in range(rows):
                if trader[e, r] < (1 << 19):
                    assert ids[e, r] == o.place_order(bool(bid[e, r]), int(vol[e, r]), int(trader[e, r]), int(price[e, r])), (s, e, r)
            o.step_keyed(seed, e)
            assert np.array_equal(obs[e], o.level_2_data_array()), (s, e)
    v.check_errors()
    for e in range(n_envs):
        assert v.env.get_orders(e) == orcs[e].get_orders() and v.env.get_trades(e) == orcs[e].get_trades()
    v.close()


def test_step_device_rows_past_max_queue_get_no_id(oracle):
    """bb_step_device runs the first max_queue rows of an env's slice; the rows past it create nothing, so their ids read
    BB_NO_ID whatever the buffer held before, and the env is flagged BB_ERR_CAP_QUEUE."""
    max_queue, rows = 16, 19
    env = core.BatchedEnv(1, 9, 0, 1, 1000, max_orders=256, max_trades=256, max_steps=8, max_queue=max_queue)
    rng = np.random.default_rng(4)
    bid, vol, price = rng.random(rows) < 0.5, rng.integers(1, 20, rows), rng.integers(45, 56, rows)
    acts = gym.DeviceArray(env, (rows,), gym.ACTION_DTYPE)
    acts.copy_from_host(gym.pack_actions(np.full(rows, abi.OP_NEW, np.uint32), bid=bid, vol=vol, trader=3, price=price))
    offsets = gym.DeviceArray(env, (2,), np.uint64)
    offsets.copy_from_host(np.array([0, rows], np.uint64))
    ids = gym.DeviceArray(env, (rows,), np.uint64)
    sentinel = np.uint64(0x5A5A5A5A5A5A5A5A)
    ids.copy_from_host(np.full(rows, sentinel, np.uint64))
    env.step_device(acts.ptr, offsets.ptr, rows, ids.ptr)
    got = ids.numpy()
    assert (got[max_queue:] == abi.NO_ID).all()
    assert env.env_errors()[0] == 0x08   # BB_ERR_CAP_QUEUE
    o = oracle.StepEnv(9, 0, 1, 1000)
    want = [o.place_order(bool(bid[r]), int(vol[r]), 3, int(price[r])) for r in range(max_queue)]
    o.step()
    assert list(got[:max_queue]) == want
    assert env.get_orders(0) == o.get_orders() and env.get_trades(0) == o.get_trades()
    assert np.array_equal(env.history(0), o._history())
    for a in (acts, offsets, ids):
        a.free()
    env.close()
