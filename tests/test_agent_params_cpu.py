"""Per-unit agent parameters without a GPU: the oracle helper that restates bb_set_agent_params_device on oracle envs
(tests/agent_params_oracle.py) against the oracle itself, and the host-side checks of `set_agent_params`."""
import types

import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads
from oracle import oracle as orc

from .agent_params_oracle import market_set_group, sim_set_group

SEED = 0x5EED_0001_2345
STEP = 1_000_000
CANCELLED = 3   # Status::Cancelled (oracle/book.hpp, types.rs:51-75)


def _varied(groups, rng):
    """Records inside the envelope of `groups`: narrower RandomAgents ranges, other rates and Momentum / Noise draws."""
    out = [g.copy() for g in groups]
    for g in out:
        g["rate"] = rng.uniform(0.05, 0.95)
        if int(g["kind"]) == abi.GROUP_RANDOM:
            lo, hi = int(g["tick_lo"]), int(g["tick_hi"])
            a = int(rng.integers(lo, hi))
            g["tick_lo"], g["tick_hi"] = a, int(rng.integers(a + 1, hi + 1))
            vlo, vhi = int(g["vol_lo"]), int(g["vol_hi"])
            v = int(rng.integers(vlo, vhi))
            g["vol_lo"], g["vol_hi"] = v, int(rng.integers(v + 1, vhi + 1))
        else:
            g["vol_lo"] = int(rng.integers(1, 30))
            g["decay"], g["demand"] = rng.uniform(0.1, 0.9), rng.uniform(0.1, 0.9)
            g["sigma"] = rng.uniform(0.5, 1.5)
    return out


def _noise_groups():
    return [core.random_group(30, (40, 60), (10, 20), 1, 0.5), core.noise_group(30, 10, 1, 0.3, 0.2, 0.1, 5, 0.0, 1.0)]


def _sim(groups):
    e = orc.StepEnvNumpy(0, 0, 1, STEP)
    e.set_groups(groups)
    return e


def _same(a, b):
    return np.array_equal(a._history(), b._history()) and a.get_orders() == b.get_orders() and a.get_trades() == b.get_trades()


@pytest.mark.parametrize("population", ["c3", "c4", "noise"])
def test_changing_every_group_at_step_0_equals_building_with_them(population):
    groups = {"c3": workloads.c3_groups, "c4": workloads.c4_groups, "noise": _noise_groups}[population]()
    mine = _varied(groups, np.random.default_rng(7))
    built, changed = _sim(mine), _sim(groups)
    for gi, g in enumerate(mine):
        sim_set_group(changed, gi, g)
    built.run_agents(40, SEED, env_id=3)
    changed.run_agents(40, SEED, env_id=3)
    assert len(built.get_trades()) > 0 and _same(built, changed)


@pytest.mark.parametrize("population", ["c3", "c4", "noise"])
def test_changing_a_group_mid_run_keeps_its_agents_state(population):
    groups = {"c3": workloads.c3_groups, "c4": workloads.c4_groups, "noise": _noise_groups}[population]()
    k = 20
    # the same parameters written back: nothing changes, so the held orders, momentum and live lists were kept
    plain, same = _sim(groups), _sim(groups)
    plain.run_agents(k, SEED, env_id=1)
    same.run_agents(k, SEED, env_id=1)
    for gi, g in enumerate(groups):
        sim_set_group(same, gi, g)
    plain.run_agents(k, SEED, env_id=1)
    same.run_agents(k, SEED, env_id=1)
    assert _same(plain, same)
    # other parameters for group 0: the orders its agents held before the change are still cancelled by them after it
    changed = _sim(groups)
    changed.run_agents(k, SEED, env_id=1)
    n_before = len(changed.get_orders())
    g = groups[0].copy()
    g["rate"] = 0.99
    sim_set_group(changed, 0, g)
    changed.run_agents(k, SEED, env_id=1)
    cancelled_after = [o for o in changed.get_orders()[:n_before] if o[1] == CANCELLED and o[3] >= k * STEP]
    assert cancelled_after and not np.array_equal(plain._history()[k:], changed._history()[k:])


def test_market_set_group_matches_building_the_market_with_it():
    groups, assets = workloads.market_example_groups()
    mine = _varied(groups, np.random.default_rng(3))
    built = orc.MarketEnv(0, 0, [1, 2], 1_000_000)
    built.set_groups(mine, assets)
    changed = orc.MarketEnv(0, 0, [1, 2], 1_000_000)
    changed.set_groups(groups, assets)
    for gi, g in enumerate(mine):
        market_set_group(changed, gi, g)
    built.run_agents(30, SEED, market_id=2)
    changed.run_agents(30, SEED, market_id=2)
    for a in (0, 1):
        assert np.array_equal(built.history(a), changed.history(a)) and built.get_trades(a) == changed.get_trades(a)
    assert any(built.get_trades(a) for a in (0, 1))


def test_set_group_refuses_another_kind():
    e = _sim(workloads.c4_groups())
    with pytest.raises(ValueError):
        sim_set_group(e, 2, workloads.c4_groups()[0])
    with pytest.raises(ValueError):
        sim_set_group(e, 3, workloads.c4_groups()[0])


def _loop(units=4, groups=None):
    loop = types.SimpleNamespace(_units=units, _groups=np.array(groups or workloads.c4_groups(), dtype=abi.GROUP_DTYPE))
    loop._unit_array = types.MethodType(gym._DeviceLoop._unit_array, loop)
    return loop


def test_agent_params_template():
    loop = _loop(5)
    p = gym._DeviceLoop.agent_params(loop)
    assert p.dtype == abi.GROUP_DTYPE and p.shape == (5, 3)
    assert all(p[u].tobytes() == loop._groups.tobytes() for u in range(5))
    p["rate"][:, 0] = 0.5   # a copy: the declared groups are untouched
    assert float(loop._groups["rate"][0]) == pytest.approx(0.8)
    with pytest.raises(ValueError, match="no background agents"):
        gym._DeviceLoop.agent_params(types.SimpleNamespace(_units=5, _groups=None))


def test_set_agent_params_host_checks():
    loop = _loop(4)
    call = gym._DeviceLoop.set_agent_params
    with pytest.raises(ValueError, match="params, keys or both"):
        call(loop)
    with pytest.raises(ValueError, match="GROUP_DTYPE"):
        call(loop, np.zeros((4, 2), abi.GROUP_DTYPE))                      # wrong group count
    with pytest.raises(ValueError, match="GROUP_DTYPE"):
        call(loop, np.zeros((3, 3), abi.GROUP_DTYPE))                      # wrong unit count
    with pytest.raises(ValueError, match="GROUP_DTYPE"):
        call(loop, np.zeros((4, 3, 80), np.uint8))                         # host bytes are not records
    with pytest.raises(ValueError, match="keys must be"):
        call(loop, keys=np.zeros(3, np.uint64))
    with pytest.raises(ValueError, match="keys must be"):
        call(loop, keys=np.zeros(4, np.float64))

    class Fake:
        def __init__(self, shape, typestr):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (0xABC000, False), "version": 3, "strides": None}
    with pytest.raises(ValueError, match="mask must be"):
        call(loop, keys=Fake((4,), "<u8"), mask=np.ones(4, np.int32))
    with pytest.raises(ValueError, match="holds 948 bytes, expected 960"):
        call(loop, Fake((4, 3, 79), "|u1"))
    with pytest.raises(ValueError, match="keys must be"):
        call(loop, keys=Fake((4,), "<u4"))
    with pytest.raises(ValueError, match="no background agents"):
        call(types.SimpleNamespace(_units=4, _groups=None), keys=np.zeros(4, np.uint64))
