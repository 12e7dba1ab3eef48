"""Multi-asset markets on the batched GPU simulator.

Mirrors the reference's Rust-level `bourse_de::MarketEnv` (crates/step_sim/src/market_env.rs:47-300) over
`bourse_book::Market` (crates/order_book/src/market.rs:59-365): `ASSETS` independent order books that share one
transaction queue per step.  The queue is shuffled as a whole and event i of the shuffled queue executes at
`start_time + i` on its asset's book (market_env.rs:108-121).  The reference does not expose these types through
`bourse.core`; the method names and argument order below are the Rust ones, with `MarketOrderId` as an
`(asset, id)` tuple.

Books of one market are consecutive envs of a `BatchedEnv(assets=A)` handle, so `n_markets` independent markets
advance in lockstep on one GPU exactly like plain envs do.  Each asset has its own tick size, as in the reference
(market_env.rs:73-90): prices are checked against the asset's tick and its level-2 records step by that tick.  On the
paged engine the ladder granule is the gcd of the ticks (unless `price_granule` is given), and an asset whose tick is
k times the granule spreads its levels k times more thinly over the 32-price pages, so it may need a larger `pages_total`.
"""
from __future__ import annotations

import math
import typing

import numpy as np

from . import abi
from .core import BatchedEnv, OrderBook

MarketOrderId = typing.Tuple[int, int]


class Market:
    """`bourse_book::Market::<ASSETS>::new(start_time, tick_size, trading)` (market.rs:74-86): an array of independent
    order books addressed by asset index, immediate mode.  Each asset is a `bourse_b200.core.OrderBook`, so tick sizes
    may differ per asset as in the reference."""

    def __init__(self, start_time: int, tick_size: typing.Sequence[int], trading: bool = True, *, book_cls=OrderBook, **kw):
        self._books = [book_cls(start_time, int(t), trading, **kw) for t in tick_size]
        self._t = start_time

    def get_order_book(self, asset: int): return self._books[asset]
    def get_time(self) -> int: return self._t

    def set_time(self, t: int):  # market.rs:113-117
        self._t = t
        for b in self._books:
            b.set_time(t)

    def enable_trading(self):
        for b in self._books:
            b.enable_trading()

    def disable_trading(self):
        for b in self._books:
            b.disable_trading()

    def bid_vols(self): return [b.bid_vol() for b in self._books]
    def bid_best_vols(self): return [b.best_bid_vol() for b in self._books]
    def bid_best_vol_and_orders(self): return [b.best_bid_vol_and_orders() for b in self._books]
    def ask_vols(self): return [b.ask_vol() for b in self._books]
    def ask_best_vols(self): return [b.best_ask_vol() for b in self._books]
    def ask_best_vol_and_orders(self): return [b.best_ask_vol_and_orders() for b in self._books]
    def bid_asks(self): return [b.bid_ask() for b in self._books]
    def level_2_data(self) -> np.ndarray: return np.stack([b.level_2_data() for b in self._books])

    def order(self, order_id: MarketOrderId):
        """The order tuple `(side, status, arr_time, end_time, vol, start_vol, price, trader_id, order_id)`."""
        return self._books[order_id[0]].get_orders()[order_id[1]]

    def create_and_place_order(self, asset: int, bid: bool, vol: int, trader_id: int, price: typing.Optional[int] = None) -> MarketOrderId:
        return (asset, self._books[asset].place_order(bid, vol, trader_id, price=price))  # market.rs:270-280

    def cancel_order(self, order_id: MarketOrderId): self._books[order_id[0]].cancel_order(order_id[1])

    def modify_order(self, order_id: MarketOrderId, new_price: typing.Optional[int] = None, new_vol: typing.Optional[int] = None):
        self._books[order_id[0]].modify_order(order_id[1], new_price=new_price, new_vol=new_vol)

    def get_orders(self, asset: int): return self._books[asset].get_orders()
    def get_trades(self, asset: int): return self._books[asset].get_trades()


class MarketEnv:
    """`MarketEnv::<ASSETS>::new(start_time, tick_sizes, step_size, trading)` (market_env.rs:73-90) plus the shuffle
    seed the reference passes to `step` as an RNG (`Xoroshiro128StarStar::seed_from_u64(seed)`).

    `market` selects one of `n_markets` lockstep markets for the per-market calls (default 0).

    Which path: this class submits on the host (`place_order` / `submit` return ids at once and raise on an off-tick
    price; `step` synchronises), which suits scripted, order-by-order use and in-kernel agents (`run_agents`).  An
    RL-style loop that produces a fixed block of rows per market and step on the GPU should use
    `gym.MarketVectorEnv` instead: one launch per step, no host synchronisation, CUDA-graph capturable, same results."""

    def __init__(self, seed: int, start_time: int, tick_sizes: typing.Sequence[int], step_size: int, trading: bool = True, *,
                 n_markets: int = 1, **kw):
        ticks = [int(t) for t in tick_sizes]
        if not ticks:
            raise ValueError("at least one asset")
        if min(ticks) <= 0:
            raise ValueError("tick sizes must be > 0")
        self.n_assets, self.n_markets, self.tick_sizes = len(ticks), n_markets, ticks
        self.tick_size = math.gcd(*ticks)   # the handle's tick: every asset's tick is a multiple of it
        kw.setdefault("max_steps", 1 << 10)
        # assets=1 would mean "plain envs" to the library; a one-asset market is the same thing as an Env
        self._env = BatchedEnv(self.n_assets * n_markets, seed, start_time, self.tick_size, step_size, trading,
                               assets=self.n_assets if self.n_assets > 1 else 0, obs_words=abi.OBS_L2, **kw)
        if any(t != self.tick_size for t in ticks):   # (several assets: a one-asset market has one tick)
            try:
                self._env.set_tick_sizes(ticks)   # asset a's tick for book a of every market
            except Exception:
                self._env.close()
                raise

    def _book(self, asset: int, market: int = 0) -> int:
        if not 0 <= asset < self.n_assets:
            raise IndexError("asset index out of range")
        return market * self.n_assets + asset

    # ------------------------------------------------------------------ instructions (queued until step)
    def place_order(self, asset: int, bid: bool, vol: int, trader_id: int, price: typing.Optional[int] = None,
                    market: int = 0) -> MarketOrderId:
        """market_env.rs:163-176; `price=None` is a market order.  Raises ValueError on a tick-size violation."""
        out = self._env.submit([abi.ACT_NEW], side=[bid], vol=[vol], trader=[trader_id], price=[price or 0],
                               env=[self._book(asset, market)], flags=[abi.F_MARKET if price is None else abi.F_HAS_PRICE])
        return (asset, int(out[0]))

    def cancel_order(self, order_id: MarketOrderId, market: int = 0):
        self._env.submit([abi.ACT_CANCEL], order_id=[order_id[1]], env=[self._book(order_id[0], market)])

    def modify_order(self, order_id: MarketOrderId, new_price: typing.Optional[int] = None, new_vol: typing.Optional[int] = None,
                     market: int = 0):
        f = (abi.F_HAS_PRICE if new_price is not None else 0) | (abi.F_HAS_VOL if new_vol is not None else 0)
        self._env.submit([abi.ACT_MODIFY], order_id=[order_id[1]], price=[new_price or 0], vol=[new_vol or 0],
                         env=[self._book(order_id[0], market)], flags=[f])

    def submit(self, action, asset, side=None, vol=None, trader=None, price=None, order_id=None, market=None, flags=None):
        """Vectorised form over many (market, asset) pairs; rows are queued in array order (that order is the
        market's transaction queue before the shuffle).  Returns the u64 ids (NO_ID where none is created)."""
        asset = np.asarray(asset, dtype=np.uint32)
        market = np.zeros_like(asset) if market is None else np.asarray(market, dtype=np.uint32)
        return self._env.submit(action, side=side, vol=vol, trader=trader, price=price, order_id=order_id,
                                env=market * np.uint32(self.n_assets) + asset, flags=flags)

    def step(self, n_steps: int = 1): self._env.step(n_steps)
    def enable_trading(self): self._env.set_trading(True)
    def disable_trading(self): self._env.set_trading(False)

    # ------------------------------------------------------------------ reads
    def time(self, market: int = 0) -> int: return self._env.time(self._book(0, market))

    def level_2_data(self, market: int = 0) -> np.ndarray:
        """`MarketEnv::level_2_data` (market_env.rs:331): the cached end-of-step data of every asset, `[ASSETS, 45]` in the
        StepEnvNumpy.level_2_data layout."""
        d = self._env.level_2_data()
        return d[market * self.n_assets:(market + 1) * self.n_assets].copy()

    def bid_asks(self, market: int = 0) -> typing.List[typing.Tuple[int, int]]:
        """`Market::bid_asks` of the LIVE books (market.rs:189-191)."""
        return [tuple(int(x) for x in self._env.book_level_1(self._book(a, market))[:2]) for a in range(self.n_assets)]

    def get_level_2_data_history(self, asset: int, market: int = 0) -> np.ndarray:
        return self._env.history(self._book(asset, market))

    def get_prices(self, asset: int, market: int = 0):
        h = self.get_level_2_data_history(asset, market); return h[:, 1].copy(), h[:, 2].copy()

    def get_volumes(self, asset: int, market: int = 0):
        h = self.get_level_2_data_history(asset, market); return h[:, 4].copy(), h[:, 3].copy()

    def get_touch_volumes(self, asset: int, market: int = 0):
        h = self.get_level_2_data_history(asset, market); return h[:, 5].copy(), h[:, 7].copy()

    def get_touch_order_counts(self, asset: int, market: int = 0):
        h = self.get_level_2_data_history(asset, market); return h[:, 6].copy(), h[:, 8].copy()

    def get_trade_vols(self, asset: int, market: int = 0):
        return self.get_level_2_data_history(asset, market)[:, 0].copy()

    def get_orders(self, asset: int, market: int = 0): return self._env.get_orders(self._book(asset, market))
    def get_trades(self, asset: int, market: int = 0): return self._env.get_trades(self._book(asset, market))

    def order_status(self, order_id: MarketOrderId, market: int = 0) -> int:
        return self._env.order_status(order_id[1], self._book(order_id[0], market))

    def env_errors(self) -> np.ndarray: return self._env.env_errors()

    # ------------------------------------------------------------------ in-kernel agents (market_sim_runner)
    def set_agents(self, agents: typing.Sequence["_MarketAgentGroup"]):
        """The fields of a `#[derive(MarketAgentSet)]` struct, in declaration order (crates/step_sim/src/agents/mod.rs:238-258)."""
        self._env.set_agents([a.group for a in agents], assets=[a.asset for a in agents])

    def run_agents(self, n_steps: int, seed: int):
        """`n_steps` of `{ agents.update(env, rng); env.step(rng) }` for every market inside one kernel launch
        (runner.rs:107-131).  Draws are Philox-keyed per (seed; market, step, agent) — DESIGN.md "RNG contract"."""
        self._env.run_agents(n_steps, seed)

    def stats(self) -> dict: return self._env.stats()


# ---------------------------------------------------------------------- the *Market agent twins
class _MarketAgentGroup:
    asset: int
    group: np.void


class RandomMarketAgents(_MarketAgentGroup):
    """`RandomMarketAgents::new(asset, n_agents, tick_range, vol_range, tick_size, activity_rate)`
    (crates/step_sim/src/agents/random_agent.rs:173-202)."""

    def __init__(self, asset: int, n_agents: int, tick_range: typing.Tuple[int, int], vol_range: typing.Tuple[int, int],
                 tick_size: int, activity_rate: float):
        from .core import random_group
        self.asset, self.group = asset, random_group(n_agents, tick_range, vol_range, tick_size, activity_rate)


class MomentumParams(typing.NamedTuple):
    """crates/step_sim/src/agents/momentum_agent.rs:16-35 (same field order)."""
    tick_size: int
    p_cancel: float
    trade_vol: int
    decay: float
    demand: float
    scale: float
    order_ratio: float
    price_dist_mu: float
    price_dist_sigma: float


class MomentumMarketAgent(_MarketAgentGroup):
    """`MomentumMarketAgent::new(agent_id_start, n_agents, asset, params)` (momentum_agent.rs:294-325)."""

    def __init__(self, agent_id_start: int, n_agents: int, asset: int, params: MomentumParams):
        from .core import momentum_group
        self.asset = asset
        self.group = momentum_group(agent_id_start, n_agents, params.tick_size, params.p_cancel, params.trade_vol, params.decay,
                                    params.demand, params.scale, params.order_ratio, params.price_dist_mu, params.price_dist_sigma)


class NoiseAgentParams(typing.NamedTuple):
    """crates/step_sim/src/agents/noise_agent.rs:14-29 (same field order)."""
    tick_size: int
    p_limit: float
    p_market: float
    p_cancel: float
    trade_vol: int
    price_dist_mu: float
    price_dist_sigma: float


class NoiseMarketAgent(_MarketAgentGroup):
    """`NoiseMarketAgent::new(asset, agent_id_start, n_agents, params)` (noise_agent.rs:236-258)."""

    def __init__(self, asset: int, agent_id_start: int, n_agents: int, params: NoiseAgentParams):
        from .core import noise_group
        self.asset = asset
        self.group = noise_group(agent_id_start, n_agents, params.tick_size, params.p_limit, params.p_market, params.p_cancel,
                                 params.trade_vol, params.price_dist_mu, params.price_dist_sigma)


def market_sim_runner(env: MarketEnv, agents: typing.Sequence[_MarketAgentGroup], seed: int, n_steps: int,
                      show_progress: bool = False):
    """`bourse_de::market_sim_runner(env, agents, seed, n_steps, show_progress)` (crates/step_sim/src/runner.rs:107-131)."""
    env.set_agents(agents)
    env.run_agents(n_steps, seed)
