"""GPU suite for device-resident rows on slices longer than a warp, on ragged slices and at the queue-capacity edges.

submit_rows (csrc/kernels.cuh), behind bb_step_device, bb_run_agents_with_rows, bb_step_device_market and
bb_run_agents_with_rows_market, walks a unit's slice 32 rows at a time and carries the next order id, the book's and the
market's queue positions from one pass to the next; k_sim's market-rows path marks queued rows in a bitmask of one bit per
row with per-word prefix counts built 32 words per pass; rows a kernel visits but does not submit get BB_NO_ID from a
rolled loop.  Here every entry point runs on slices of 0 to more than 1024 rows, with offsets that differ from unit to
unit and step to step, rows placed at the pass boundaries, and slices at and just past max_queue / assets * max_queue.

Each test first runs the oracle (oracle.StepEnv / MarketEnv, with agents_update / step_keyed for the agent loops) and
records per step the ids of every row and every book's record; then the device call runs on the same slices and must
match step by step, and at the end in histories, orders, trades and the exact error words of include/bourse_b200.h."""
import numpy as np
import pytest

from bourse_b200 import abi, core, gym, workloads

from . import market_split_oracle as mks
from .test_gpu_gym import _random_actions
from .test_gpu_market_agents_rows import mixed_agents, oracle_market, random_agents
from .test_gpu_market_agents_rows import learner_block, oracle_rows as agent_market_rows
from .test_gpu_market_device import oracle_rows as market_rows, random_block

pytestmark = pytest.mark.gpu

ERR_CAP_QUEUE, ERR_CAP_LIVE, ERR_PRICE, ERR_ROW_OP = 0x08, 0x80, 0x200, 0x400
OP_UNKNOWN = 9   # no operation of the ABI: queues nothing, takes no id
SENTINEL = 0x5A5A5A5A5A5A5A5A
ENGINES = {
    "paged": dict(pages_smem=4, pages_total=64),   # most pages in HBM
    "fast": dict(pages_smem=32, pages_total=32),
    "dense": dict(price_window=(0, 256)),          # 128 resting-order slots
    "dense_l": dict(price_window=(0, 512), live_cap=254),
}


# ---------------------------------------------------------------------------------------------------- plumbing
def launch(env, call, blocks, seed=None, with_ids=True):
    """Run entry point `call` of `env` once on the ragged slices `blocks` (one packed row array per unit, uploaded with
    their offsets); returns (the ids of each unit's rows, the [n_envs, obs_words] records).  The id buffer starts out
    holding a sentinel, so a row the kernel forgets reads as neither an id nor BB_NO_ID.  `with_ids=False` passes no id
    buffer (the handle's own is used)."""
    sizes = [len(b) for b in blocks]
    n = sum(sizes)
    rows = np.concatenate(list(blocks) + [np.zeros(1, gym.ACTION_DTYPE)])   # (a spare row: no buffer is empty)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    acts = gym.DeviceArray(env, rows.shape, gym.ACTION_DTYPE)
    acts.copy_from_host(rows)
    off = gym.DeviceArray(env, offs.shape, np.uint64)
    off.copy_from_host(offs)
    ids = gym.DeviceArray(env, (n + 1,), np.uint64)
    ids.copy_from_host(np.full(n + 1, SENTINEL, np.uint64))
    obs = gym.DeviceArray(env, (env.n_envs, env.obs_words), np.uint32)
    args = (acts.ptr, off.ptr, n, ids.ptr if with_ids else 0, obs.ptr)
    getattr(env, call)(*(args if seed is None else (seed,) + args))
    got_ids, got_obs = ids.numpy(), obs.numpy()
    for a in (acts, off, ids, obs):
        a.free()
    return np.split(got_ids[:n], np.cumsum(sizes)[:-1]), got_obs


def run_plan(env, call, plan, seed=None, with_ids=True):
    """The device side of a plan: per step (slices, wanted ids per unit or None, {book: wanted record})."""
    for s, (blocks, want_ids, want_obs) in enumerate(plan):
        ids, obs = launch(env, call, blocks, seed, with_ids)
        if with_ids:
            for u, w in enumerate(want_ids):
                if w is not None:
                    assert list(ids[u]) == w, (s, u, len(blocks[u]))
        for b, w in want_obs.items():
            assert np.array_equal(obs[b], w), (s, b)


def row(op, **kw):
    return gym.pack_actions(np.array([op], np.uint32), **kw)[0]


def takes_id(blk, ticks, simq=False):
    """Which rows create an order: on-tick limit or market NEWs (`ticks`: the row's book tick, per row or one), and with
    `simq` (k_sim's queue) only trader ids below 2^19."""
    f = blk["op_flags"]
    ok = ((f & 0xFF) == abi.OP_NEW) & (((f & abi.F_MARKET) != 0) | (blk["price"] % np.asarray(ticks, np.uint32) == 0))
    return ok & (blk["trader"] < (1 << 19)) if simq else ok


# ---------------------------------------------------------------------------------------------------- single-asset envs
def env_slice(rng, m, issued, tick, simq=False, fixed=None):
    """m rows for one env whose book has issued `issued` ids: the limit / market NEW, CANCEL, MODIFY and no-op mix of
    test_gpu_gym (cancels and modifies of earlier ids), now and then an unknown op code, off-tick limit NEWs at rows 31,
    32 and 63 (tick > 1), and CANCELs naming ids of the same slice across the pass boundary: row 40 the id row 5 creates,
    row 2 the id row 33 creates.  `simq` (bb_run_agents_with_rows queues NEW and CANCEL only): MODIFYs become CANCELs.
    `fixed` {row: packed row} is placed before the ids are counted."""
    ins = [r for r in (31, 32, 63) if tick > 1 and r < m]
    op, cols = _random_actions(rng, 1, m - len(ins), [issued], tick)
    op[0, rng.random(op.shape[1]) < 0.03] = OP_UNKNOWN
    if simq:
        op[op == abi.OP_MODIFY] = abi.OP_CANCEL
    blk = gym.pack_actions(op, **cols)[0]
    if ins:
        off_tick = gym.pack_actions(np.full(len(ins), abi.OP_NEW, np.uint32), bid=np.arange(len(ins)) % 2, vol=3, trader=4,
                                    price=50 * tick + 1)
        blk = np.insert(blk, [r - k for k, r in enumerate(ins)], off_tick)
    fixed = fixed or {}
    for r, x in fixed.items():
        if r < m:
            blk[r] = x
    refs = [(c, t) for c, t in ((40, 5), (2, 33)) if t < m and c < m and c not in fixed and t not in fixed]
    for c, t in refs:
        blk[t] = row(abi.OP_NEW, bid=t % 2, vol=4, trader=5, price=50 * tick)
        blk[c] = row(abi.OP_CANCEL)
    ids = issued + np.cumsum(takes_id(blk, tick, simq)) - 1
    for c, t in refs:
        blk[c]["order_id"] = ids[t]
    return blk


def oracle_env_rows(o, blk, simq=False):
    """The rows through an oracle StepEnv in row order (place_order / cancel_order / modify_order; with `simq` the rows
    bb_run_agents_with_rows drops are left out); returns (ids, whether a place_order raised PriceError, rows dropped)."""
    ids, bad, dropped = [], False, 0
    for x in blk:
        f = int(x["op_flags"])
        op, i = f & 0xFF, abi.NO_ID
        if simq and (op == abi.OP_MODIFY or (op == abi.OP_NEW and x["trader"] >= (1 << 19))):
            dropped += 1
        elif op == abi.OP_NEW:
            try:
                i = o.place_order(bool(f & abi.F_BID), int(x["vol"]), int(x["trader"]), None if f & abi.F_MARKET else int(x["price"]))
            except ValueError:
                bad = True
        elif op == abi.OP_CANCEL:
            o.cancel_order(int(x["order_id"]))
        elif op == abi.OP_MODIFY:
            o.modify_order(int(x["order_id"]), int(x["price"]) if f & abi.F_HAS_PRICE else None,
                           int(x["vol"]) if f & abi.F_HAS_VOL else None)
        ids.append(i)
    return ids, bad, dropped


def assert_envs_equal(env, orcs, skip=()):
    for e, o in enumerate(orcs):
        if e not in skip:
            assert np.array_equal(env.history(e), o._history()), e
            assert env.get_orders(e) == o.get_orders(), e
            assert env.get_trades(e) == o.get_trades(), e


def slice_lengths(max_queue):
    return sorted({0, 1, 31, 32, 33, 63, 64, 65, 97, max_queue - 1, max_queue, max_queue + 1, max_queue + 70})


# case: (engine, max_queue, ticks "12" = per-env ticks 1 and 2 in turn, or one tick)
STEP_CASES = {
    "paged_t12": ("paged", 160, "12"),
    "fast_t1": ("fast", 160, 1),
    "fast_t12": ("fast", 160, "12"),
    "dense_l_t12": ("dense_l", 160, "12"),
    "dense_t2": ("dense", 64, 2),   # 128 slots: at most 64 rows of a slice run
}


def plan_step_device(oracle, max_queue, ticks, n_steps, seed, rng):
    """bb_step_device: per step every env takes a slice length of slice_lengths(max_queue) (each length once per step,
    rotating over the envs); the oracle sees the first max_queue rows of each slice, the rest get BB_NO_ID."""
    lengths = slice_lengths(max_queue)
    orcs = [oracle.StepEnv(seed + e, 0, t, 1000) for e, t in enumerate(ticks)]
    err = np.zeros(len(ticks), np.uint32)
    plan = []
    for s in range(n_steps):
        blocks = [env_slice(rng, lengths[(e + 3 * s) % len(lengths)], len(o.get_orders()), ticks[e]) for e, o in enumerate(orcs)]
        want_ids, want_obs = [], {}
        for e, o in enumerate(orcs):
            ids, bad, _ = oracle_env_rows(o, blocks[e][:max_queue])
            o.step()
            want_ids.append(ids + [abi.NO_ID] * (len(blocks[e]) - len(ids)))
            want_obs[e] = o.level_2_data_array()
            err[e] |= (ERR_PRICE if bad else 0) | (ERR_CAP_QUEUE if len(blocks[e]) > max_queue else 0)
        plan.append((blocks, want_ids, want_obs))
    return plan, orcs, err


@pytest.mark.parametrize("case", list(STEP_CASES))
def test_step_device_ragged_slices(oracle, case):
    """Every env's ids and record equal the oracle's step for step; a slice past max_queue runs its first max_queue rows,
    its other rows read BB_NO_ID and only that env is flagged BB_ERR_CAP_QUEUE (BB_ERR_PRICE only where one of the rows
    that ran was off the tick), and the env goes on matching."""
    engine, max_queue, tick = STEP_CASES[case]
    n_envs, seed = len(slice_lengths(max_queue)), 17
    ticks = [1 + e % 2 for e in range(n_envs)] if tick == "12" else [tick] * n_envs
    plan, orcs, err = plan_step_device(oracle, max_queue, ticks, 4, seed, np.random.default_rng(len(case)))
    env = core.BatchedEnv(n_envs, seed, 0, ticks, 1000, max_orders=4096, max_trades=8192, max_steps=16, max_queue=max_queue,
                          **ENGINES[engine])
    run_plan(env, "step_device", plan)
    assert np.array_equal(env.env_errors(), err), (env.env_errors(), err)
    assert (err & ERR_CAP_QUEUE).any() and (tick == 1 or (err & ERR_PRICE).any())
    assert_envs_equal(env, orcs)
    env.close()


# case: (engine, agent population, per-env ticks 1 and 2 in turn (C3 quotes on a tick of 2) or all 1, slice lengths)
AGENT_CASES = {
    "fast_c3": ("fast", "c3", "12", (0, 1, 31, 32, 33, 63, 64, 65, 97, 159, 160)),
    "dense_l_c3": ("dense_l", "c3", "12", (0, 1, 31, 32, 33, 63, 64, 65)),
    "paged_c4": ("paged", "c4", 1, (0, 1, 31, 32, 33, 63, 64, 65, 97, 159, 160)),
}
AGENT_MAX_QUEUE = 320   # the agents' events (C3: at most one per agent, 100; C4 about 120) plus 160 rows


def plan_agent_rows(oracle, groups, lengths, ticks, n_steps, seed, rng):
    """bb_run_agents_with_rows: per step and env agents_update, the env's slice, step_keyed.  At step 0 env 0 holds a NEW
    with trader id 2^19 at row 31, one with 2^19 - 1 at row 32 and a MODIFY at row 33.  The last env takes slices of
    33 rows, then at the last step max_queue rows on top of its agents' events: it is flagged and not compared."""
    n_envs = len(ticks)
    over = n_envs - 1
    orcs = [oracle.StepEnv(0, 0, t, 1_000_000) for t in ticks]
    for o in orcs:
        o.set_groups(groups)
    err = np.zeros(n_envs, np.uint32)
    special = {31: row(abi.OP_NEW, bid=1, vol=6, trader=1 << 19, price=50 * ticks[0]),
               32: row(abi.OP_NEW, bid=0, vol=6, trader=(1 << 19) - 1, price=50 * ticks[0]),
               33: row(abi.OP_MODIFY, order_id=0, price=50 * ticks[0], vol=2)}
    plan = []
    for s in range(n_steps):
        blocks, want_ids, want_obs = [], [], {}
        for e, o in enumerate(orcs):
            o.agents_update(seed, e)
            if e == over and s == n_steps - 1:
                blocks.append(gym.pack_actions(np.full(AGENT_MAX_QUEUE, abi.OP_NEW, np.uint32), bid=np.arange(AGENT_MAX_QUEUE) % 2,
                                               vol=5, trader=9, price=50 * ticks[e]))
                want_ids.append(None)
                continue
            m = 33 if e == over else lengths[(e + 3 * s) % len(lengths)]
            if e == 0 and s == 0:
                m = max(m, 65)
            blk = env_slice(rng, m, len(o.get_orders()), ticks[e], simq=True, fixed=special if (e, s) == (0, 0) else None)
            ids, bad, dropped = oracle_env_rows(o, blk, simq=True)
            o.step_keyed(seed, e)
            blocks.append(blk)
            want_ids.append(ids)
            want_obs[e] = o.level_2_data_array()
            err[e] |= (ERR_PRICE if bad else 0) | (ERR_ROW_OP if dropped else 0)
        plan.append((blocks, want_ids, want_obs))
    return plan, orcs, err


@pytest.mark.parametrize("case", list(AGENT_CASES))
def test_agent_rows_ragged_slices(oracle, case):
    """Ragged slices next to the background agents: every env's ids and record equal the oracle's agents_update + row
    calls + step_keyed.  The trader id 2^19 - 1 is accepted and recorded, 2^19 and the MODIFY are dropped without taking
    an id (BB_ERR_ROW_OP); an env whose agent events plus rows exceed max_queue is flagged BB_ERR_CAP_QUEUE, and every
    other env stays exact."""
    engine, pop, tick, lengths = AGENT_CASES[case]
    groups = workloads.c3_groups() if pop == "c3" else workloads.c4_groups()
    n_envs, seed = len(lengths) + 1, 0xC0DE
    ticks = [1 + e % 2 for e in range(n_envs)] if tick == "12" else [tick] * n_envs
    plan, orcs, err = plan_agent_rows(oracle, groups, lengths, ticks, 4, seed, np.random.default_rng(len(case) + 100))
    env = core.BatchedEnv(n_envs, 0, 0, ticks, 1_000_000, max_orders=8192, max_trades=16384, max_steps=16,
                          max_queue=AGENT_MAX_QUEUE, **ENGINES[engine])
    env.set_agents(groups)
    run_plan(env, "run_agents_with_rows", plan, seed)
    got = env.env_errors()
    over = n_envs - 1
    # (what that env raised before its last step, its off-tick rows' BB_ERR_PRICE, stays; the dense engine may also drop
    # the over-long step for want of resting-order slots)
    assert got[over] & ~np.uint32(ERR_CAP_LIVE) == err[over] | ERR_CAP_QUEUE, got
    assert np.array_equal(got[:over], err[:over]), (got, err)
    assert err[0] == ERR_ROW_OP
    # row 31 (2^19) took no id, row 32 (2^19 - 1) the next one, and its order record carries the trader id
    ids0 = plan[0][1][0]
    assert ids0[31] == abi.NO_ID and ids0[33] == abi.NO_ID and ids0[32] != abi.NO_ID
    assert env.get_orders(0)[ids0[32]][7] == (1 << 19) - 1 == orcs[0].get_orders()[ids0[32]][7]   # (trader_id)
    assert_envs_equal(env, orcs, skip=(over,))
    env.close()


# ---------------------------------------------------------------------------------------------------- markets
def with_bad_assets(blk, A, n):
    """`blk` (n - k rows) with k NEWs naming assets >= A inserted so that they sit at rows 31, 32, 63 and 64 of the n."""
    rows = [r for r in (31, 32, 63, 64) if r < n]
    bad = gym.pack_actions(np.full(len(rows), abi.OP_NEW, np.uint32), bid=1, vol=2, trader=3, price=60, asset=A + np.arange(len(rows)))
    return np.insert(blk, [r - k for k, r in enumerate(rows)], bad)


def market_block(rng, ticks, issued, kind, n):
    """One market's slice of `n` rows: "mixed" the rows of random_block over all assets with rows naming no asset at the
    pass boundaries; "one" every row on the last asset (limit prices on its tick)."""
    A = len(ticks)
    if kind == "one":
        iss = [issued[A - 1]]
        blk = random_block(rng, [ticks[A - 1]], iss, n)
        blk["aux"] = A - 1
        issued[A - 1] = iss[0]
        return blk
    return with_bad_assets(random_block(rng, ticks, issued, n - sum(r < n for r in (31, 32, 63, 64))), A, n)


MARKET_MAX_QUEUE = {2: 600, 5: 240, 33: 40}   # assets * max_queue >= 1200: a market's slice of 1100 rows fits


def plan_step_device_market(oracle, A, ticks, n_markets, n_steps, seed, rng):
    """bb_step_device_market: per step the markets take slices of 0, 33, 100 and 1100 mixed rows, exactly assets *
    max_queue rows, max_queue + 60 rows on one asset, and assets * max_queue + 1 / + 40 rows (over: nothing submitted,
    the oracle steps with an empty queue), rotating over the markets."""
    cap = A * MARKET_MAX_QUEUE[A]
    kinds = [("mixed", 0), ("mixed", 33), ("mixed", 100), ("mixed", 1100), ("mixed", cap), ("one", MARKET_MAX_QUEUE[A] + 60),
             ("over", cap + 1), ("over", cap + 40)]
    orcs = [oracle.MarketEnv(seed + mk, 0, ticks, 1000) for mk in range(n_markets)]
    issued = [[0] * A for _ in range(n_markets)]
    err = np.zeros((n_markets, A), np.uint32)
    plan = []
    for s in range(n_steps):
        blocks, want_ids, want_obs = [], [], {}
        for mk, o in enumerate(orcs):
            kind, n = kinds[(mk + s) % len(kinds)]
            if kind == "over":
                blk = market_block(rng, ticks, list(issued[mk]), "mixed", n)
                o.step()
                ids = [abi.NO_ID] * n
                err[mk] |= ERR_CAP_QUEUE
            else:
                blk = market_block(rng, ticks, issued[mk], kind, n)
                ids, bad, row_op = market_rows(o, blk)
                for a in bad:
                    err[mk, a] |= ERR_PRICE
                err[mk, 0] |= ERR_ROW_OP if row_op else 0
            assert len(blk) == n
            blocks.append(blk)
            want_ids.append(ids)
            want_obs.update({mk * A + a: o.history(a)[-1] for a in range(A)})
        plan.append((blocks, want_ids, want_obs))
    return plan, orcs, err


def assert_markets_equal(env, orcs, A, skip=()):
    for mk, o in enumerate(orcs):
        if mk in skip:
            continue
        for a in range(A):
            b = mk * A + a
            assert np.array_equal(env.history(b), o.history(a)), (mk, a)
            assert env.get_orders(b) == o.get_orders(a), (mk, a)
            assert env.get_trades(b) == o.get_trades(a), (mk, a)


@pytest.mark.parametrize("engine", ["fast", "paged"])
@pytest.mark.parametrize("A", [2, 5, 33])
def test_step_device_market_ragged_slices(oracle, engine, A):
    """Per step and market the ids and every book's record equal the oracle's; rows naming no asset at the pass
    boundaries flag book 0 BB_ERR_ROW_OP and shift no id; a market's slice of exactly assets * max_queue rows, or more
    than max_queue rows on one asset, is exact; one row more flags every book of that market BB_ERR_CAP_QUEUE, every row
    reads BB_NO_ID and the books step as with an empty queue.  33 assets: a market spans several CTAs and has more books
    than a warp has lanes."""
    ticks = [(1, 2, 3)[a % 3] for a in range(A)]
    n_markets, seed = 8, 23
    plan, orcs, err = plan_step_device_market(oracle, A, ticks, n_markets, 3, seed, np.random.default_rng(A + len(engine)))
    env = core.BatchedEnv(n_markets * A, seed, 0, 1, 1000, assets=A, max_orders=4096, max_trades=16384, max_steps=16,
                          max_queue=MARKET_MAX_QUEUE[A], **ENGINES[engine])
    env.set_tick_sizes(ticks)
    run_plan(env, "step_device_market", plan)
    got = env.env_errors().reshape(n_markets, A)
    assert np.array_equal(got, err), (got, err)
    assert (err[:, 0] & ERR_ROW_OP).any() and (err & ERR_PRICE).any()
    assert_markets_equal(env, orcs, A)
    env.close()


def queued_block(rng, ticks, mine, n_queued, n_noop, asset=None):
    """A market's slice in which exactly n_queued rows queue: on-tick limit and market NEWs and CANCELs of the learner's
    own earlier ids (`mine[a]`), on the assets in turn (or all on `asset`), with n_noop no-ops among them."""
    A = len(ticks)
    cols = {k: np.zeros(n_queued, np.int64) for k in ("op", "asset", "bid", "vol", "trader", "price", "oid", "mkt")}
    a0 = int(rng.integers(A))
    for r in range(n_queued):
        a = (a0 + r) % A if asset is None else asset
        cols["asset"][r] = a
        if rng.random() < 0.7 or not mine[a]:
            cols["op"][r], cols["bid"][r], cols["vol"][r], cols["trader"][r] = abi.OP_NEW, rng.random() < 0.5, rng.integers(1, 25), 500 + r % 1000
            if rng.random() < 0.1:
                cols["mkt"][r] = 1
            else:
                cols["price"][r] = ticks[a] * int(rng.integers(90 // ticks[a], 210 // ticks[a]))
        else:
            cols["op"][r], cols["oid"][r] = abi.OP_CANCEL, mine[a][int(rng.integers(len(mine[a])))]
    blk = gym.pack_actions(cols["op"], bid=cols["bid"], vol=cols["vol"], trader=cols["trader"], price=cols["price"],
                           order_id=cols["oid"], market=cols["mkt"], asset=cols["asset"])
    noop = gym.pack_actions(np.full(n_noop, abi.OP_NOOP, np.uint32), asset=rng.integers(A, size=n_noop))
    return np.insert(blk, np.sort(rng.integers(0, n_queued + 1, n_noop)), noop)


MKT_AGENT_QUEUED = (0, 31, 32, 33, 1023, 1024, 1025, 1100)
MKT_AGENT_MAX_QUEUE = 320   # 4 * 320 = 1280 >= 1100 rows plus the agents' events; no book's own events exceed 320


def plan_agent_rows_market(oracle, agents, ticks, n_steps, seed, rng):
    """bb_run_agents_with_rows_market on 4 assets: per step the first 8 markets queue 0 .. 1100 rows (rotating), with
    a few no-ops between them.  Market 8 puts max_queue + 20 rows on asset 0 at the last step (that book's own events
    exceed max_queue, the market's fit), market 9 assets * max_queue + 5 rows spread over the assets (the market's queue
    exceeds assets * max_queue); both take empty slices before that and are not compared."""
    A, n_markets = len(ticks), len(MKT_AGENT_QUEUED) + 2
    orcs = [oracle_market(oracle, agents, ticks, 1000) for _ in range(n_markets)]
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    plan = []
    for s in range(n_steps):
        blocks, want_ids, want_obs = [], [], {}
        for mk, o in enumerate(orcs):
            if mk >= len(MKT_AGENT_QUEUED):
                last = s == n_steps - 1
                n_q = (MKT_AGENT_MAX_QUEUE + 20 if mk == 8 else A * MKT_AGENT_MAX_QUEUE + 5) if last else 0
                blocks.append(queued_block(rng, ticks, mine[mk], n_q, 3, asset=0 if mk == 8 else None))
                want_ids.append(None)
                if not last:
                    mks.agents_update(o, seed, mk)
                    mks.step_keyed(o, seed, mk)
                    want_obs.update({mk * A + a: o.history(a)[-1] for a in range(A)})
                continue
            mks.agents_update(o, seed, mk)
            blk = queued_block(rng, ticks, mine[mk], MKT_AGENT_QUEUED[(mk + 3 * s) % len(MKT_AGENT_QUEUED)], int(rng.integers(0, 9)))
            want_ids.append(agent_market_rows(o, blk, mine[mk]))
            mks.step_keyed(o, seed, mk)
            blocks.append(blk)
            want_obs.update({mk * A + a: o.history(a)[-1] for a in range(A)})
        plan.append((blocks, want_ids, want_obs))
    return plan, orcs


@pytest.mark.parametrize("engine", ["fast", "paged"])
def test_market_agent_rows_past_a_thousand_queued_rows(oracle, engine):
    """Markets of 4 assets with max_queue = 320 (assets * max_queue > 1024: the row mask has more than 32 words, its
    prefix counts take two passes) queue 0, 31, 32, 33, 1023, 1024, 1025 and 1100 rows next to the market agents: ids
    and records equal the oracle step for step.  A book whose own events exceed max_queue is flagged on that book alone;
    a market over assets * max_queue on every book; every other market stays exact."""
    ticks, seed = [1, 2, 3, 2], 0xFEED
    agents = random_agents(4)
    plan, orcs = plan_agent_rows_market(oracle, agents, ticks, 3, seed, np.random.default_rng(len(engine) + 7))
    # (layout arithmetic: 2 * 1280 bytes of permutation, as many of draws and 2 * 40 mask words per warp fit in shared
    # memory on FAST and paged; bb_create refuses what does not)
    env = core.BatchedEnv(len(orcs) * 4, 0, 0, 1, 1000, assets=4, max_orders=8192, max_trades=32768, max_steps=16,
                          max_queue=MKT_AGENT_MAX_QUEUE, **ENGINES[engine])
    env.set_tick_sizes(ticks)
    env.set_agents([a.group for a in agents], assets=[a.asset for a in agents])
    run_plan(env, "run_agents_with_rows_market", plan, seed)
    got = env.env_errors().reshape(len(orcs), 4)
    n = len(MKT_AGENT_QUEUED)
    assert not got[:n].any(), got
    assert list(got[n]) == [ERR_CAP_QUEUE, 0, 0, 0], got
    assert (got[n + 1] == ERR_CAP_QUEUE).all(), got
    assert all(env.n_steps(b) == 3 for b in range(n * 4, (n + 2) * 4))   # the flagged markets' books still stepped
    assert_markets_equal(env, orcs, 4, skip=(n, n + 1))
    env.close()


MKT_AGENT_CASES = [(2, "mixed", "fast"), (3, "random", "dense_l"), (3, "mixed", "paged")]


@pytest.mark.parametrize("A,pop,engine", MKT_AGENT_CASES, ids=[f"{e}-{A}-{p}" for A, p, e in MKT_AGENT_CASES])
def test_market_agent_rows_ragged_slices(oracle, A, pop, engine):
    """The market agents of test_gpu_market_agents_rows next to slices of 33 to 65 rows that differ from market to market
    and step to step: ids and records equal the oracle's."""
    ticks, n_markets, seed = [1, 2, 3][:A], 6, 0xB0A5
    agents = random_agents(A) if pop == "random" else mixed_agents(A)
    rng = np.random.default_rng(A * 13 + len(engine))
    orcs = [oracle_market(oracle, agents, ticks, 1000) for _ in range(n_markets)]
    mine = [[[] for _ in range(A)] for _ in range(n_markets)]
    plan = []
    for s in range(6):
        blocks = [learner_block(rng, ticks, mine[mk], int(rng.integers(33, 66))) for mk in range(n_markets)]
        want_ids, want_obs = [], {}
        for mk, o in enumerate(orcs):
            mks.agents_update(o, seed, mk)
            want_ids.append(agent_market_rows(o, blocks[mk], mine[mk]))
            mks.step_keyed(o, seed, mk)
            want_obs.update({mk * A + a: o.history(a)[-1] for a in range(A)})
        plan.append((blocks, want_ids, want_obs))
    env = core.BatchedEnv(n_markets * A, 0, 0, 1, 1000, assets=A, max_orders=8192, max_trades=16384, max_steps=16,
                          max_queue=128, **ENGINES[engine])
    env.set_tick_sizes(ticks)
    env.set_agents([a.group for a in agents], assets=[a.asset for a in agents])
    run_plan(env, "run_agents_with_rows_market", plan, seed)
    assert not env.env_errors().any(), env.env_errors()
    assert_markets_equal(env, orcs, A)
    env.close()


# ---------------------------------------------------------------------------------------------------- no id buffer
def test_internal_id_buffer_regrows(oracle):
    """d_out_ids = NULL with n_rows growing from call to call: the handle's id buffer (which k_apply also reads the new
    ids back from) regrows, and records and books still equal the oracle's, on single-asset envs and on markets."""
    rng, seed = np.random.default_rng(99), 5
    n_envs, max_queue, tick = 16, 640, 2
    orcs = [oracle.StepEnv(seed + e, 0, tick, 1000) for e in range(n_envs)]
    err = np.zeros(n_envs, np.uint32)
    plan = []
    for hi in (2, 70, 200, 640):
        blocks = [env_slice(rng, int(rng.integers(hi // 2, hi + 1)), len(o.get_orders()), tick) for o in orcs]
        want_obs = {}
        for e, o in enumerate(orcs):
            err[e] |= ERR_PRICE if oracle_env_rows(o, blocks[e])[1] else 0
            o.step()
            want_obs[e] = o.level_2_data_array()
        plan.append((blocks, None, want_obs))
    env = core.BatchedEnv(n_envs, seed, 0, tick, 1000, max_orders=8192, max_trades=16384, max_steps=16, max_queue=max_queue,
                          **ENGINES["fast"])
    run_plan(env, "step_device", plan, with_ids=False)
    assert np.array_equal(env.env_errors(), err), (env.env_errors(), err)
    assert_envs_equal(env, orcs)
    env.close()

    A, n_markets, ticks = 3, 4, [1, 2, 3]
    morcs = [oracle.MarketEnv(seed + mk, 0, ticks, 1000) for mk in range(n_markets)]
    issued = [[0] * A for _ in range(n_markets)]
    plan = []
    for hi in (3, 90, 400, 1100):
        blocks = [random_block(rng, ticks, issued[mk], int(rng.integers(hi // 2, hi + 1)), off_tick=False) for mk in range(n_markets)]
        want_obs = {}
        for mk, o in enumerate(morcs):
            market_rows(o, blocks[mk])
            want_obs.update({mk * A + a: o.history(a)[-1] for a in range(A)})
        plan.append((blocks, None, want_obs))
    env = core.BatchedEnv(n_markets * A, seed, 0, 1, 1000, assets=A, max_orders=8192, max_trades=16384, max_steps=16,
                          max_queue=400, **ENGINES["fast"])
    env.set_tick_sizes(ticks)
    run_plan(env, "step_device_market", plan, with_ids=False)
    assert not env.env_errors().any(), env.env_errors()
    assert_markets_equal(env, morcs, A)
    env.close()
