"""CPU suite for the oracle side of the snapshot restore (tests/episode_snapshot_oracle.py, what bb_save_device /
bb_restore_device are checked against): a copied env steps identically to its source under the same actions, agents and
markets included; its history starts empty; a re-seeded copy matches an env built by hand with that stream."""
import numpy as np

from oracle import oracle as orc

from . import episode_reset_oracle as ers
from . import episode_snapshot_oracle as ess
from .test_oracle_reset import _drive, _rows, _shuffle_of_next_step, _state

GROUPS = [orc.random_group(30, (40, 60), (10, 20), 1, 0.8),
          orc.momentum_group(100, 6, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0),
          orc.noise_group(200, 5, 1, 0.3, 0.1, 0.2, 7, 0.5, 0.8)]


def test_copy_steps_identically_to_its_source():
    rng = np.random.default_rng(0)
    a = orc.StepEnv(3, 0, 1, 1000)
    for _ in range(10):
        _drive(a, _rows(rng, 6))
    b = orc.StepEnv(99, 0, 1, 1000)
    ess.sim_copy(b, a)
    assert len(b._history()) == 0 and len(a._history()) == 10
    assert b.get_orders() == a.get_orders() and b.get_trades() == a.get_trades() and b.time == a.time
    assert np.array_equal(b.level_2_data_array(), a.level_2_data_array())
    for _ in range(12):
        rows = _rows(rng, 7)
        _drive(a, rows)
        _drive(b, rows)
    assert _state(a)[:2] == _state(b)[:2] and np.array_equal(a._history()[10:], b._history())
    assert _shuffle_of_next_step(a, 12, a.time) == _shuffle_of_next_step(b, 12, b.time)


def test_copy_back_from_a_slot_replays_the_continuation():
    """A slot is an env kept aside: restoring it into the env it came from replays the same continuation."""
    rng = np.random.default_rng(1)
    a = orc.StepEnv(5, 0, 2, 1000)
    for _ in range(8):
        _drive(a, [(bid, vol, 2 * p) for bid, vol, p in _rows(rng, 5)])
    slot = orc.StepEnv(0, 0, 2, 1000)
    ess.sim_copy(slot, a)
    tail = [[(bid, vol, 2 * p) for bid, vol, p in _rows(rng, 6)] for _ in range(9)]
    for rows in tail:
        _drive(a, rows)
    first = _state(a)
    ess.sim_copy(a, slot)
    for rows in tail:
        _drive(a, rows)
    assert _state(a)[:2] == first[:2] and np.array_equal(a._history(), first[2][8:])


def test_reseeded_copy_matches_a_hand_built_stream():
    """A re-seeded copy is the source's book with the shuffle stream a constructor given that seed starts with."""
    rng = np.random.default_rng(2)
    a = orc.StepEnv(3, 0, 1, 1000)
    for _ in range(6):
        _drive(a, _rows(rng, 5))
    c = orc.StepEnv(0, 0, 1, 1000)
    ess.sim_copy(c, a, seed=42)
    assert c.get_orders() == a.get_orders()
    perm = _shuffle_of_next_step(c, 12, c.time)
    fresh = orc.StepEnv(42, 0, 1, 1000)   # the stream a seeded constructor has
    assert perm == _shuffle_of_next_step(fresh, 12, 0) and perm != _shuffle_of_next_step(a, 12, a.time)


def test_copy_with_agents_keeps_the_step_counter():
    seed = 0xABCDEF

    def make():
        e = orc.StepEnv(0, 0, 1, 1_000_000)
        e.set_groups(GROUPS)
        return e

    a, b = make(), make()
    a.run_agents(10, seed, 4)
    ess.sim_copy(b, a, seed=7)   # re-seeding touches only the shuffle stream: agent draws continue from step 10
    a.run_agents(8, seed, 4)
    b.run_agents(8, seed, 4)
    assert _state(a)[:2] == _state(b)[:2] and len(a.get_trades()) > 0
    c = make()
    c.run_agents(10, seed, 4)
    ers.sim_reset(c, 0)
    c.run_agents(8, seed, 4)
    assert _state(c)[:2] != _state(a)[:2]


def test_market_copy():
    ticks, groups, assets, seed = [1, 2, 5], [orc.random_group(20, (40, 60), (10, 20), 10, 0.8),
                                              orc.random_group(15, (40, 60), (10, 20), 10, 0.6)], [0, 2], 77
    a = orc.MarketEnv(4, 0, ticks, 1000)
    a.set_groups(groups, assets)
    a.run_agents(6, seed, market_id=2)
    b = orc.MarketEnv(9, 0, ticks, 1000)
    b.set_groups(groups, assets)
    ess.market_copy(b, a)
    assert all(len(b.history(x)) == 0 and b.get_orders(x) == a.get_orders(x) for x in range(3))
    a.run_agents(7, seed, market_id=2)
    b.run_agents(7, seed, market_id=2)
    for x in range(3):
        assert a.get_orders(x) == b.get_orders(x) and a.get_trades(x) == b.get_trades(x)
        assert np.array_equal(a.history(x)[6:], b.history(x))
    assert sum(len(a.get_trades(x)) for x in range(3)) > 0
