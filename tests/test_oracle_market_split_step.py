"""CPU suite for the two halves of the oracle's keyed market step (tests/market_split_oracle.py, what
bb_run_agents_with_rows_market is checked against): with nothing queued between them they are exactly MarketSim's
run_keyed, and instructions queued between them join the market's one shuffled queue after every group's."""
import numpy as np
import pytest

from oracle import oracle as orc

from . import market_split_oracle as mks


def _populations():
    mom = orc.momentum_group(100, 6, 2, 0.1, 10, 1.0, 5.0, 0.5, 1.0, 0.0, 1.0)
    noise = orc.noise_group(200, 5, 2, 0.3, 0.1, 0.2, 7, 0.5, 0.8)
    return {
        "random": ([orc.random_group(30, (40, 60), (10, 20), 2, 0.8), orc.random_group(20, (10, 90), (50, 70), 2, 0.3)], [0, 1], [1, 2]),
        "random_momentum": ([orc.random_group(25, (40, 60), (10, 20), 2, 0.7), mom, orc.random_group(15, (40, 60), (10, 20), 2, 0.5)],
                            [1, 1, 2], [1, 2, 1]),
        "mixed_noise": ([orc.random_group(20, (40, 60), (10, 20), 2, 0.7), noise, mom, orc.random_group(10, (10, 90), (50, 70), 2, 0.3)],
                        [0, 1, 2, 3], [2, 1, 2, 1]),
    }


@pytest.mark.parametrize("name", list(_populations()))
def test_split_step_equals_run_keyed(name):
    groups, assets, ticks = _populations()[name]
    seed, market_id, n_steps = 0x1234_5678_9ABC, 5, 30
    a = orc.MarketEnv(0, 0, ticks, 1000)
    b = orc.MarketEnv(0, 0, ticks, 1000)
    for m in (a, b):
        m.set_groups(groups, assets)
    a.run_agents(n_steps, seed, market_id=market_id, keyed=True)
    for _ in range(n_steps):
        mks.agents_update(b, seed, market_id)
        mks.step_keyed(b, seed, market_id)
    assert a.n_instructions() == b.n_instructions() > 0
    n_tr = 0
    for k in range(len(ticks)):
        assert np.array_equal(a.history(k), b.history(k)), k
        assert a.get_orders(k) == b.get_orders(k), k
        assert a.get_trades(k) == b.get_trades(k), k
        n_tr += len(a.get_trades(k))
    assert n_tr > 0


def test_rows_between_the_halves_take_ids_after_the_agents():
    """An order placed between the halves gets the id after the agents' ones on its asset's book, and it is processed in the
    step that follows (its record shows the order's volume resting on the book)."""
    m = orc.MarketEnv(0, 0, [1, 2], 1000)
    m.set_groups([orc.random_group(4, (40, 41), (5, 6), 1, 1.0)], [1])
    mks.agents_update(m, 9, 0)
    oid = m.place_order(1, True, 3, 777, 10)
    assert oid == (1, 4)
    mks.step_keyed(m, 9, 0)
    assert m.n_instructions() == 5
    o = m.get_orders(1)
    assert len(o) == 5 and o[4][7] == 777 and o[4][1] == 1   # the learner's bid rests (Active), far below the agents' asks
    assert len(m.get_orders(0)) == 0
