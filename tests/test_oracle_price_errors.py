"""CPU suite: an in-kernel agent whose limit price is off its book's tick.  The reference agents unwrap create_order's
PriceError (orderbook.rs:367-383) and panic; the oracle raises ValueError with the reference's message instead of
aborting the process, and keeps the records of the steps completed before it."""
import numpy as np
import pytest

from . import scenarios_ticks as st


@pytest.mark.parametrize("pop", st.OFFGRID_POPS)
def test_single_asset_off_tick_group_raises_and_keeps_history(oracle, pop):
    # tick 1: every population is on its grid; tick 2: the off-grid group draws an odd price sooner or later
    ok = oracle.StepEnvNumpy(0, 0, 1, st.STEP)
    ok.set_groups(st.offgrid_groups(oracle, pop, 1))
    ok.run_agents(st.N_STEPS, st.SEED, env_id=0)
    assert len(ok._history()) == st.N_STEPS and len(ok.get_trades()) > 100
    failed = []
    for env_id in range(6):
        o = oracle.StepEnvNumpy(0, 0, 2, st.STEP)
        o.set_groups(st.offgrid_groups(oracle, pop, 1))
        try:
            o.run_agents(st.N_STEPS, st.SEED, env_id=env_id)
            continue
        except ValueError as err:
            assert str(err).endswith("was not a multiple of tick-size 2"), err
            assert int(str(err).split()[1]) % 2 == 1
        f = len(o._history())
        failed.append(f)
        # the same run stopped one step short of the failure: identical records, orders and trades
        r = oracle.StepEnvNumpy(0, 0, 2, st.STEP)
        r.set_groups(st.offgrid_groups(oracle, pop, 1))
        r.run_agents(f, st.SEED, env_id=env_id)
        assert np.array_equal(o._history(), r._history()) and o.get_trades() == r.get_trades()
        assert o.get_orders()[:len(r.get_orders())] == r.get_orders()
    assert failed and max(failed) > 0, failed


@pytest.mark.parametrize("pop", st.OFFGRID_POPS)
def test_market_off_tick_group_raises_and_keeps_history(oracle, pop):
    ticks = st.market_ticks(1)
    groups, assets = st.offgrid_market_groups(oracle, pop, 1)
    failed = []
    for mk in range(6):
        o = oracle.MarketEnv(0, 0, ticks, st.STEP)
        o.set_groups(groups, assets)
        try:
            o.run_agents(st.N_STEPS, st.SEED, market_id=mk)
            continue
        except ValueError as err:
            assert str(err).endswith("was not a multiple of tick-size 2"), err
        f = len(o.history(0))
        assert len(o.history(1)) == f
        failed.append(f)
        r = oracle.MarketEnv(0, 0, ticks, st.STEP)
        r.set_groups(groups, assets)
        r.run_agents(f, st.SEED, market_id=mk)
        for a in range(len(ticks)):
            assert np.array_equal(o.history(a), r.history(a)) and o.get_trades(a) == r.get_trades(a)
    assert failed and max(failed) > 0, failed


def test_split_agent_update_raises(oracle):
    """agents_update (the first half of a keyed step) raises the same way and leaves the env usable for reading."""
    o = oracle.StepEnvNumpy(0, 0, 2, 1000)
    o.set_groups([oracle.random_group(40, (40, 60), (10, 20), 1, 0.7)])
    with pytest.raises(ValueError, match=r"^Price \d*[13579] was not a multiple of tick-size 2$"):
        o.agents_update(1, 0)
    assert len(o._history()) == 0 and o.get_trades() == []


def test_momentum_off_its_books_tick_raises(oracle):
    """The market from test_gpu_tick_sizes: a Momentum group with tick 3 on a tick-2 asset raises once it quotes."""
    o = oracle.MarketEnv(0, 0, [1, 2], 100_000)
    o.set_groups([oracle.random_group(40, (40, 60), (10, 20), 1, 0.7), oracle.random_group(40, (40, 60), (10, 20), 2, 0.7),
                  oracle.momentum_group(100, 12, 3, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0)], [0, 1, 1])
    with pytest.raises(ValueError, match="tick-size 2$"):
        o.run_agents(30, 5, market_id=0)
    assert 0 < len(o.history(1)) < 30
