"""CPU suite for the oracle side of the per-env reset (tests/episode_reset_oracle.py, what bb_reset_device is checked
against): a reset with a seed is a freshly constructed env with that seed; a reset without one empties the book and
clears the agents but keeps the shuffle stream and the step counter of the agents' Philox draws."""
import numpy as np

from oracle import oracle as orc

from . import episode_reset_oracle as ers


def _rows(rng, n):
    return [(bool(rng.random() < 0.5), int(rng.integers(1, 30)), int(rng.integers(45, 56))) for _ in range(n)]


def _drive(env, rows):
    for bid, vol, price in rows:
        env.place_order(bid, vol, 7, price)
    env.step()


def _state(env):
    return env.get_orders(), env.get_trades(), env._history().tolist()


def _shuffle_of_next_step(env, k, t0):
    """The permutation the env's next shuffle draws: k bids at one price, each rests at arr_time = t0 + its queue position."""
    for j in range(k):
        env.place_order(True, j + 1, 1, 50)
    env.step()
    return [o[2] - t0 for o in env.get_orders()[-k:]]


def test_seeded_reset_is_a_fresh_env():
    rng = np.random.default_rng(0)
    a = orc.StepEnv(3, 0, 1, 1000)
    for _ in range(12):
        _drive(a, _rows(rng, 6))
    ers.sim_reset(a, 0, seed=9)
    assert a.get_orders() == [] and a.get_trades() == [] and len(a._history()) == 0
    assert np.array_equal(a.level_2_data_array(), orc.StepEnv(9, 0, 1, 1000).level_2_data_array())
    b = orc.StepEnv(9, 0, 1, 1000)
    for _ in range(15):
        rows = _rows(rng, 7)
        _drive(a, rows)
        _drive(b, rows)
    assert _state(a) == _state(b) and len(a.get_trades()) > 0
    assert _shuffle_of_next_step(a, 12, 15_000) == _shuffle_of_next_step(b, 12, 15_000)


def test_unseeded_reset_keeps_the_shuffle_stream():
    rng = np.random.default_rng(1)
    a, twin, fresh = orc.StepEnv(3, 0, 1, 1000), orc.StepEnv(3, 0, 1, 1000), orc.StepEnv(3, 0, 1, 1000)
    for _ in range(10):
        rows = _rows(rng, 5)
        _drive(a, rows)
        _drive(twin, rows)
    ers.sim_reset(a, 0)
    assert a.get_orders() == [] and len(a._history()) == 0 and a.time == 0
    perm = _shuffle_of_next_step(a, 12, 0)
    assert perm == _shuffle_of_next_step(twin, 12, 10_000)   # the twin's stream, never reset, is at the same state
    assert sorted(perm) == list(range(12)) and perm != _shuffle_of_next_step(fresh, 12, 0)


def test_reset_with_agents_keeps_or_restarts_the_step_counter():
    groups = [orc.random_group(30, (40, 60), (10, 20), 1, 0.8),
              orc.momentum_group(100, 6, 1, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0),
              orc.noise_group(200, 5, 1, 0.3, 0.1, 0.2, 7, 0.5, 0.8)]
    seed, env_id = 0xABCDEF, 4

    def make():
        e = orc.StepEnv(0, 0, 1, 1_000_000)
        e.set_groups(groups)
        return e

    ran, idle, fresh = make(), make(), make()
    ran.run_agents(10, seed, env_id)
    for _ in range(10):
        idle.step_keyed(seed, env_id)   # ten steps with nothing queued: same step counter, agents untouched
    ers.sim_reset(ran, 0)
    ers.sim_reset(idle, 0)
    for e in (ran, idle, fresh):
        e.run_agents(8, seed, env_id)
    assert _state(ran) == _state(idle) and len(ran.get_trades()) > 0
    assert _state(ran) != _state(fresh)   # draws keyed by steps 10..17, not 0..7
    ers.sim_reset(ran, 0, seed=5)
    ran.run_agents(8, seed, env_id)
    assert _state(ran)[:2] == _state(fresh)[:2] and np.array_equal(ran._history(), fresh._history())


def test_market_reset():
    ticks, groups, assets = [1, 2, 5], [orc.random_group(20, (40, 60), (10, 20), 10, 0.8), orc.random_group(15, (40, 60), (10, 20), 10, 0.6)], [0, 2]
    seed = 77
    a = orc.MarketEnv(4, 0, ticks, 1000)
    a.set_groups(groups, assets)
    a.run_agents(6, seed, market_id=2)
    ers.market_reset(a, 0)
    assert all(a.get_orders(x) == [] and len(a.history(x)) == 0 and len(a.get_trades(x)) == 0 for x in range(3))
    a.run_agents(5, seed, market_id=2)
    ers.market_reset(a, 0, seed=4)
    fresh = orc.MarketEnv(4, 0, ticks, 1000)
    fresh.set_groups(groups, assets)
    a.run_agents(7, seed, market_id=2)
    fresh.run_agents(7, seed, market_id=2)
    for x in range(3):
        assert a.get_orders(x) == fresh.get_orders(x) and a.get_trades(x) == fresh.get_trades(x)
        assert np.array_equal(a.history(x), fresh.history(x))
    assert sum(len(fresh.get_trades(x)) for x in range(3)) > 0
