"""GPU suite: the journaled event loop of the dense engine's RandomAgents kernel (k_sim, dense.cuh d_flush).

Lane 0 runs a step's events with only the book on its chain: each event's outcome stays in its queue entry, each fill
becomes a trade-journal entry in the queue entries past the step's events, and the warp writes the order records, the
trade log and the trade counters out afterwards.  A journal that fills up suspends the running event, flushes, and
resumes it.  These cases drive the flush paths hard and compare with the oracle bit for bit."""
import numpy as np
import pytest

from bourse_b200 import abi
from bourse_b200.core import random_group

pytestmark = pytest.mark.gpu

STEP = 1_000_000
# Every small agent acts every step (so a step has at least 90 events and a 96-entry queue leaves at most 8 journal
# entries); the few large orders sweep many of the small resting ones.
SWEEP_GROUPS = [random_group(90, (30, 90), (1, 4), 2, 1.0), random_group(6, (20, 100), (200, 600), 2, 0.5)]
WINDOWS = {"dense": (0, 256), "dense_l": (0, 512)}


def _oracle(oracle, groups, seed, env_id, n_steps):
    env = oracle.StepEnvNumpy(0, 0, 1, STEP)
    env.set_groups(groups)
    env.run_agents(n_steps, seed, env_id=env_id, keyed=True)
    return env


def _env(core, n_envs, n_steps, window, **kw):
    kw.setdefault("max_orders", 8192)
    kw.setdefault("max_trades", 1 << 16)
    return core.BatchedEnv(n_envs, 0, 0, 1, STEP, obs_words=abi.OBS_L2, env_id_base=500, max_steps=n_steps,
                           price_window=window, live_cap=128, **kw)


@pytest.mark.parametrize("engine", sorted(WINDOWS))
@pytest.mark.parametrize("max_queue", [96, 256])
def test_journal_overflow_mid_step(core, oracle, engine, max_queue):
    """Sweeps produce more fills in a step than the journal holds (with max_queue 96): the event in progress is suspended
    and resumed, possibly several times, and the result is still the reference's."""
    n_envs, n_steps, seed = 12, 40, 3
    env = _env(core, n_envs, n_steps, WINDOWS[engine], max_queue=max_queue)
    env.set_agents(SWEEP_GROUPS)
    env.run_agents(n_steps, seed)
    assert not env.env_errors().any()
    hist = env.history_all(n_steps)
    busiest = 0
    for e in range(n_envs):
        ce = _oracle(oracle, SWEEP_GROUPS, seed, 500 + e, n_steps)
        assert np.array_equal(hist[e], ce._history()[:, :abi.OBS_L2]), e
        assert env.get_trades(e) == ce.get_trades(), e
        assert env.get_orders(e) == ce.get_orders(), e
        t = ce.trades_arrays()["t"]
        busiest = max(busiest, int(np.bincount(np.asarray(t, dtype=np.int64) // STEP).max()))
    assert busiest > 2 + 96 - 90  # some step overflowed the smallest possible journal


@pytest.mark.parametrize("engine", sorted(WINDOWS))
def test_trade_log_cap_hit_mid_step(core, oracle, engine):
    """max_trades is reached in the middle of a step: ERR_CAP_TRADES, the log holds exactly the first max_trades trades,
    the order table and the observations are the reference's."""
    n_envs, n_steps, seed, cap = 6, 12, 5, 137
    env = _env(core, n_envs, n_steps, WINDOWS[engine], max_queue=96, max_trades=cap)
    env.set_agents(SWEEP_GROUPS)
    try:
        env.run_agents(n_steps, seed)
    except MemoryError:  # the launch's error report, where the call synchronises on it
        pass
    errs = env.env_errors()
    hist = env.history_all(n_steps)
    total, inside = 0, 0
    for e in range(n_envs):
        ce = _oracle(oracle, SWEEP_GROUPS, seed, 500 + e, n_steps)
        ct, gt = ce.trades_arrays(), env.trades_arrays(e)
        total += len(ct["t"])
        assert len(ct["t"]) > cap and int(errs[e]) == 0x02, e
        inside += int(ct["t"][cap - 1]) // STEP == int(ct["t"][cap]) // STEP  # the cap falls inside a step
        assert len(gt["t"]) == cap and all(np.array_equal(ct[k][:cap], gt[k]) for k in ct), e
        assert env.get_orders(e) == ce.get_orders(), e
        assert np.array_equal(hist[e], ce._history()[:, :abi.OBS_L2]), e
    assert inside > 0
    assert env.stats()["trades"] == total


@pytest.mark.parametrize("engine", sorted(WINDOWS))
def test_order_table_after_split_launches(core, oracle, engine):
    """Launches of arbitrary lengths: after each one the order table, the trade log and the observations so far equal the
    oracle's after the same number of steps."""
    n_envs, seed = 8, 21
    pieces = (7, 1, 13, 2, 9)
    env = _env(core, n_envs, sum(pieces), WINDOWS[engine], max_queue=96)
    env.set_agents(SWEEP_GROUPS)
    done = 0
    for k in pieces:
        env.run_agents(k, seed)
        done += k
        assert not env.env_errors().any()
        hist = env.history_all(done)
        for e in range(n_envs):
            ce = _oracle(oracle, SWEEP_GROUPS, seed, 500 + e, done)
            assert env.get_orders(e) == ce.get_orders(), (done, e)
            assert env.get_trades(e) == ce.get_trades(), (done, e)
            assert np.array_equal(hist[e], ce._history()[:, :abi.OBS_L2]), (done, e)
