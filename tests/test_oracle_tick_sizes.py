"""CPU suite: the oracle's per-asset tick sizes (MarketEnv::new(start_time, tick_sizes, ...), market_env.rs:73-90)
against hand-worked answers, and the random mixed-tick market driver the GPU suite (test_gpu_tick_sizes.py) runs."""
import types

import numpy as np

from . import scenarios_ticks as st


def test_known_answers_mixed_ticks(oracle):
    for scenario in st.ALL_KNOWN:
        scenario(types.SimpleNamespace(MarketEnv=oracle.MarketEnv))


def test_random_mixed_tick_markets_are_reproducible(oracle):
    """Two oracle runs of the same mixed-tick stream agree, off-grid rows are refused, and the stream trades enough for
    the GPU comparison to mean something."""
    ticks, n_markets, n_steps = [1, 2, 5], 4, 60
    a, b = (st.OracleMarkets(oracle, 31, ticks, n_markets, 10_000) for _ in range(2))
    n_off = st.drive_markets(np.random.default_rng(8), [a, b], ticks, n_steps, n_markets)
    assert n_off > 10
    n_tr = 0
    for x, y in zip(a.m, b.m):
        for k in range(len(ticks)):
            assert x.get_trades(k) == y.get_trades(k) and x.get_orders(k) == y.get_orders(k)
            assert np.array_equal(x.history(k), y.history(k))
            assert all(o[6] % ticks[k] == 0 for o in x.get_orders(k) if o[6] not in (0, 2**32 - 1))
            n_tr += len(x.get_trades(k))
    assert n_tr > 500


def test_step_env_rows_follow_each_envs_tick(oracle):
    """The per-env row generator stays on each env's grid; its level-2 records step by that env's tick."""
    for tick in range(1, 9):
        rng, o, n = np.random.default_rng(tick), oracle.StepEnv(tick, 0, tick, 1000), 0
        for _ in range(20):
            rows, n = st.env_rows(rng, tick, n)
            st.apply_rows_oracle(o, rows)
            o.step()
        h = o._history()
        for r in h:
            bid, ask = int(r[1]), int(r[2])
            assert (bid == 0 or bid % tick == 0) and (ask == 2**32 - 1 or ask % tick == 0)
