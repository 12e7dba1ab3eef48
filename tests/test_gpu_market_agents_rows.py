"""GPU suite for background agents in the device-resident market loop (bb_run_agents_with_rows_market,
gym.MarketVectorEnv(agents=...), k_sim<.., MKT, EXT>): per market, one step is `agents.update(env)`, the caller's rows
through MarketEnv::place_order / cancel_order in row order, then MarketEnv::step (runner.rs:107-131 with the caller's calls
in between, market_env.rs:108-121, 163-219).  Everything is checked against one oracle MarketSim per market doing
agents_update, the row calls and step_keyed (tests/market_split_oracle.py), and against market.MarketEnv.run_agents on a
twin handle."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, market

from . import market_split_oracle as mks

pytestmark = pytest.mark.gpu

ERR_CAP_QUEUE, ERR_BAD_ID, ERR_PRICE, ERR_ROW_OP = 0x08, 0x10, 0x200, 0x400
ENGINES = {
    "fast": dict(pages_smem=32, pages_total=32),
    "paged": dict(pages_smem=8, pages_total=64),
    "dense": dict(price_window=(0, 256), live_cap=128),
    "dense_l": dict(price_window=(0, 512), live_cap=254),
}
TICKS = {2: [1, 2], 3: [1, 2, 3], 4: [1, 2, 3, 2]}
# agents quote on a tick of 6, a multiple of every asset's tick, at prices 60 .. 234 (inside the dense windows)
MOM = market.MomentumParams(tick_size=6, p_cancel=0.1, trade_vol=10, decay=1.0, demand=5.0, scale=0.5, order_ratio=1.0,
                            price_dist_mu=0.0, price_dist_sigma=1.0)
NOISE = market.NoiseAgentParams(tick_size=6, p_limit=0.3, p_market=0.1, p_cancel=0.2, trade_vol=7, price_dist_mu=0.5,
                                price_dist_sigma=0.8)


def random_agents(A):
    return [market.RandomMarketAgents(a, 30 - 3 * a, (14, 26), (10, 20), 6, 0.7) for a in range(A)] + \
           [market.RandomMarketAgents(A - 1, 12, (10, 40), (20, 40), 6, 0.3)]


def mixed_agents(A):
    return [market.RandomMarketAgents(a, 25, (14, 26), (10, 20), 6, 0.7) for a in range(A)] + \
           [market.MomentumMarketAgent(100, 8, A - 1, MOM), market.NoiseMarketAgent(0, 200, 6, NOISE),
            market.RandomMarketAgents(1, 10, (10, 40), (20, 40), 6, 0.3)]


def oracle_market(oracle, agents, ticks, step_size):
    o = oracle.MarketEnv(0, 0, ticks, step_size)
    o.set_groups([a.group for a in agents], [a.asset for a in agents])
    return o


def learner_block(rng, ticks, mine, rows):
    """One market's rows: limit NEWs on their asset's tick at the agents' prices, market NEWs, cancels of the learner's own
    earlier ids (`mine[a]`), no-ops.  Trader ids 500+ mark the learner's orders."""
    A = len(ticks)
    cols = {k: np.zeros(rows, np.int64) for k in ("op", "asset", "bid", "vol", "trader", "price", "oid", "mkt")}
    for r in range(rows):
        a, u = int(rng.integers(A)), rng.random()
        cols["asset"][r] = a
        if u < 0.15:
            continue   # OP_NOOP
        if u < 0.75 or not mine[a]:
            cols["op"][r], cols["bid"][r], cols["vol"][r], cols["trader"][r] = abi.OP_NEW, rng.random() < 0.5, rng.integers(1, 25), 500 + r
            if rng.random() < 0.1:
                cols["mkt"][r] = 1
            else:
                cols["price"][r] = ticks[a] * int(rng.integers(90 // ticks[a], 210 // ticks[a]))
        else:
            cols["op"][r], cols["oid"][r] = abi.OP_CANCEL, mine[a][int(rng.integers(len(mine[a])))]
    return gym.pack_actions(cols["op"], bid=cols["bid"], vol=cols["vol"], trader=cols["trader"], price=cols["price"],
                            order_id=cols["oid"], market=cols["mkt"], asset=cols["asset"])


def oracle_rows(o, blk, mine=None):
    """The rows through the oracle market (between its agents_update and step_keyed); returns the ids per row."""
    ids = []
    for x in blk:
        op, a, i = int(x["op_flags"]) & 0xFF, int(x["aux"]), abi.NO_ID
        if op == abi.OP_NEW:
            price = None if x["op_flags"] & abi.F_MARKET else int(x["price"])
            i = o.place_order(a, bool(x["op_flags"] & abi.F_BID), int(x["vol"]), int(x["trader"]), price)[1]
            if mine is not None:
                mine[a].append(i)
        elif op == abi.OP_CANCEL:
            o.cancel_order((a, int(x["order_id"])))
        ids.append(i)
    return ids


def assert_books_equal(env, mk, A, o):
    for a in range(A):
        b = mk * A + a
        assert np.array_equal(env.history(b), o.history(a)), (mk, a)
        assert env.get_orders(b) == o.get_orders(a), (mk, a)
        assert env.get_trades(b) == o.get_trades(a), (mk, a)


CASES = [(e, A, "random") for e in ENGINES for A in (2, 3, 4)] + [(e, A, "mixed") for e in ("fast", "paged") for A in (2, 3, 4)]


@pytest.mark.parametrize("engine,A,pop", CASES, ids=[f"{e}-{A}-{p}" for e, A, p in CASES])
def test_rows_with_market_agents_bit_exact(oracle, engine, A, pop):
    """Per step and market: ids and every book's record equal the oracle's agents_update + row calls + step_keyed; at the end
    histories, orders and trades; the learner traded against the agents; plain agent launches then continue bit-exact."""
    ticks, n_markets, rows, n_steps, seed = TICKS[A], 8, 6, 25, 0xB0A5
    agents = random_agents(A) if pop == "random" else mixed_agents(A)
    v = gym.MarketVectorEnv(n_markets, rows, 0, 0, ticks, 1000, agents=agents, agent_seed=seed, max_orders=8192, max_trades=16384,
                            max_steps=64, max_queue=128, **ENGINES[engine])
    v.reset()
    orcs = [oracle_market(oracle, agents, ticks, 1000) for _ in range(n_markets)]
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    rng = np.random.default_rng(A * 31 + len(engine) + len(pop))
    for s in range(n_steps):
        blk = np.stack([learner_block(rng, ticks, mine[mk], rows) for mk in range(n_markets)])
        obs, ids = v.step(blk)
        obs, ids = obs.numpy(), ids.numpy()
        for mk, o in enumerate(orcs):
            mks.agents_update(o, seed, mk)
            want = oracle_rows(o, blk[mk], mine[mk])
            mks.step_keyed(o, seed, mk)
            assert list(ids[mk]) == want, (s, mk)
            for a in range(A):
                assert np.array_equal(obs[mk, a], o.history(a)[-1]), (s, mk, a)
    v.check_errors()
    crossed = 0
    for mk, o in enumerate(orcs):
        assert_books_equal(v.env, mk, A, o)
        for a in range(A):
            own = set(mine[mk][a])
            crossed += sum((t[4] in own) != (t[5] in own) for t in o.get_trades(a))
    assert crossed > 0   # learner orders matched against agent orders
    # plain agent launches continue the same books
    v.env.run_agents(3, seed)
    for mk in (0, n_markets - 1):
        orcs[mk].run_agents(3, seed, market_id=mk, keyed=True)
        assert_books_equal(v.env, mk, A, orcs[mk])
    assert not v.env.env_errors().any()
    v.close()


@pytest.mark.parametrize("engine", ["fast", "dense"])
def test_noop_rows_equal_run_agents_on_a_twin(engine):
    """Rows that queue nothing change nothing: step for step, the same histories as market.MarketEnv.run_agents(1)."""
    ticks, n_markets, rows, seed = [1, 2, 3], 6, 4, 21
    agents = random_agents(3)
    kw = dict(max_orders=8192, max_trades=16384, max_steps=64, max_queue=200, **ENGINES[engine])
    v = gym.MarketVectorEnv(n_markets, rows, 0, 0, ticks, 1000, agents=agents, agent_seed=seed, **kw)
    m = market.MarketEnv(0, 0, ticks, 1000, n_markets=n_markets, **kw)
    m.set_agents(agents)
    v.reset()
    noop = gym.pack_actions(np.full((n_markets, rows), abi.OP_NOOP, np.uint32), asset=np.arange(rows) % 3)
    for s in range(20):
        obs, ids = v.step(noop)
        m.run_agents(1, seed)
        assert (ids.numpy() == abi.NO_ID).all()
        for mk in range(n_markets):
            for a in range(3):
                assert np.array_equal(obs.numpy()[mk, a], m.get_level_2_data_history(a, mk)[-1]), (s, mk, a)
    for b in range(3 * n_markets):
        assert np.array_equal(v.env.history(b), m._env.history(b)), b
        assert v.env.get_orders(b) == m._env.get_orders(b) and v.env.get_trades(b) == m._env.get_trades(b), b
    assert not v.env.env_errors().any() and not m.env_errors().any()
    v.close()
    m._env.close()


def _row(op, asset, price=0, vol=5, trader=600, oid=0, bid=1):
    return dict(op=op, asset=asset, price=price, vol=vol, trader=trader, oid=oid, bid=bid)


def _block(n_markets, rows, placed):
    """A block of no-ops with `placed[(market, row)] = _row(...)` filled in."""
    cols = {k: np.zeros((n_markets, rows), np.int64) for k in ("op", "asset", "bid", "vol", "trader", "price", "oid")}
    for (mk, r), c in placed.items():
        for k, val in c.items():
            cols[k][mk, r] = val
    return gym.pack_actions(cols["op"], bid=cols["bid"], vol=cols["vol"], trader=cols["trader"], price=cols["price"],
                            order_id=cols["oid"], asset=cols["asset"])


@pytest.mark.parametrize("engine", ["fast", "dense"])
def test_row_error_bits(oracle, engine):
    """Each row error sets exactly its bit on exactly the book of the table in the header; the dropped rows take no id and
    the markets stay bit-exact against the oracle (which never sees those rows) until the unknown-id cancel."""
    ticks, A, n_markets, rows, seed = [1, 2, 3], 3, 3, 3, 5
    agents = random_agents(A)
    v = gym.MarketVectorEnv(n_markets, rows, 0, 0, ticks, 1000, agents=agents, agent_seed=seed, max_orders=8192, max_trades=16384,
                            max_steps=64, **ENGINES[engine])
    v.reset()
    orcs = [oracle_market(oracle, agents, ticks, 1000) for _ in range(n_markets)]

    def step(placed, oracle_rows_too, want_err):
        blk = _block(n_markets, rows, placed)
        obs, ids = v.step(blk)
        obs, ids = obs.numpy(), ids.numpy()
        for mk, o in enumerate(orcs):
            mks.agents_update(o, seed, mk)
            want = [abi.NO_ID] * rows
            for (m2, r), c in placed.items():
                if m2 == mk and (m2, r) in oracle_rows_too:
                    want[r] = o.place_order(c["asset"], bool(c["bid"]), c["vol"], c["trader"], c["price"])[1]
            mks.step_keyed(o, seed, mk)
            assert list(ids[mk]) == want, mk
            for a in range(A):
                assert np.array_equal(obs[mk, a], o.history(a)[-1]), (mk, a)
        err = v.env.env_errors()
        expect = np.zeros(A * n_markets, np.uint32)
        for b, bit in want_err.items():
            expect[b] |= bit
        assert np.array_equal(err, expect), (err, expect)
        v.env.clear_errors()

    for _ in range(3):
        step({}, (), {})
    # a limit NEW off asset 2's tick (3) in market 1, next to an on-tick NEW of the same asset: only the latter takes an id
    step({(1, 0): _row(abi.OP_NEW, 2, price=100), (1, 1): _row(abi.OP_NEW, 2, price=99)}, {(1, 1)}, {1 * A + 2: ERR_PRICE})
    # a row naming no asset of market 0: book 0 of market 0
    step({(0, 2): _row(abi.OP_NEW, 7, price=90)}, (), {0: ERR_ROW_OP})
    # a MODIFY row on asset 1 of market 2: that book
    step({(2, 0): _row(abi.OP_MODIFY, 1, price=90, oid=0)}, (), {2 * A + 1: ERR_ROW_OP})
    # a trader id beyond 19 bits on asset 0 of market 1
    step({(1, 2): _row(abi.OP_NEW, 0, price=90, trader=1 << 19)}, (), {1 * A + 0: ERR_ROW_OP})
    for _ in range(2):
        step({}, (), {})
    for mk in range(n_markets):
        assert_books_equal(v.env, mk, A, orcs[mk])
    # a cancel of an id asset 1 of market 0 has not issued (inside the order table's capacity)
    assert v.env.n_orders(1) < 6000
    v.step(_block(n_markets, rows, {(0, 1): _row(abi.OP_CANCEL, 1, oid=6000)}))
    err = v.env.env_errors()
    assert err[1] == ERR_BAD_ID and not np.delete(err, 1).any(), err
    v.close()


def test_over_long_row_block_drops_the_markets_step():
    """A market whose queue (agents' instructions plus queued rows) exceeds assets * max_queue flags BB_ERR_CAP_QUEUE on each
    of its books and nowhere else."""
    ticks, n_markets, rows = [1, 2], 3, 32
    agents = [market.RandomMarketAgents(a, 2, (14, 26), (10, 20), 6, 1.0) for a in range(2)]
    v = gym.MarketVectorEnv(n_markets, rows, 0, 0, ticks, 1000, agents=agents, agent_seed=3, max_orders=4096, max_trades=4096,
                            max_steps=16, max_queue=16)
    v.reset()
    op = np.full((n_markets, rows), abi.OP_NOOP, np.uint32)
    op[1] = abi.OP_NEW
    obs, ids = v.step(gym.pack_actions(op, bid=1, vol=3, trader=9, price=60, asset=0))
    err = v.env.env_errors().reshape(n_markets, 2)
    assert (err[1] == ERR_CAP_QUEUE).all() and not err[0].any() and not err[2].any(), err
    assert v.env.n_steps(2) == v.env.n_steps(0) == 1   # every book still stepped
    v.close()


def test_refusals(monkeypatch):
    from bourse_b200 import workloads
    import torch

    # single-asset handle
    e = core.BatchedEnv(2, 0, 0, 1, 1000, max_orders=256, max_trades=256, max_steps=8, max_queue=64)
    e.set_agents(workloads.c3_groups())
    p = e.device_alloc(64)
    with pytest.raises(ValueError, match="bb_run_agents_with_rows"):
        e.run_agents_with_rows_market(1, p, p, 0)
    e.device_free(p)
    e.close()
    # market handle without market agents; bb_run_agents_with_rows keeps refusing market handles
    m = core.BatchedEnv(4, 0, 0, 1, 1000, assets=2, max_orders=256, max_trades=256, max_steps=8, max_queue=64)
    p = m.device_alloc(64)
    with pytest.raises(ValueError, match="bb_set_agents_market has not been called"):
        m.run_agents_with_rows_market(1, p, p, 0)
    with pytest.raises(ValueError, match="drives single-asset envs"):
        m.run_agents_with_rows(1, p, p, 0)
    # pending host-queued instructions
    m.set_agents([market.RandomMarketAgents(0, 4, (14, 26), (10, 20), 1, 0.5).group], assets=[0])
    m.submit([abi.ACT_NEW], [1], [1], [0], [10], env=[1])
    with pytest.raises(ValueError, match="pending"):
        m.run_agents_with_rows_market(1, p, p, 0)
    m.device_free(p)
    m.close()
    # five assets with agents: refused before any handle exists
    def no_handle(*a, **k):
        raise AssertionError("a handle was created")
    monkeypatch.setattr(gym, "BatchedEnv", no_handle)
    with pytest.raises(ValueError, match="at most 4 assets"):
        gym.MarketVectorEnv(2, 2, 0, 0, [1] * 5, 1000, agents=random_agents(5))
    with pytest.raises(ValueError, match="65536"):
        gym.MarketVectorEnv(2, 2, 0, 0, [1] * 4, 1000, agents=random_agents(4), max_queue=20000)
    monkeypatch.undo()
    # stream capture
    v = gym.MarketVectorEnv(2, 2, 0, 0, [1, 2], 1000, agents=random_agents(2), agent_seed=1, max_orders=1024, max_trades=1024, max_steps=8)
    stream = torch.cuda.Stream()
    v.env.set_stream(stream.cuda_stream)
    v.reset()
    acts = torch.zeros((2, 2, 8), dtype=torch.int32, device="cuda")
    with torch.cuda.stream(stream):
        v.step(acts)
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with pytest.raises(ValueError, match="cannot be captured"):
        with torch.cuda.graph(g, stream=stream):
            v.step(acts)
    v.close()
