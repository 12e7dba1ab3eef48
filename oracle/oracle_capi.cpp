// ORACLE — TEST INFRASTRUCTURE ONLY (see oracle/rng.hpp header).
//
// Flat C entry points over the CPU restatement so that pytest (ctypes) and bench.py's cpu_baseline /
// `--impl reference` legs can drive it.  Array layouts mirror the reference's Python surface:
//   rust/src/types.rs:4-31             PyTrade / PyOrder tuple field order
//   rust/src/step_sim_numpy.rs:300-368 level_1_data (9) / level_2_data (45) array layout
//   rust/src/step_sim.rs:381-395       StepEnv.level_1_data_array (8, no trade_vol)
// The instruction record `orc_instr` and the agent-group record `orc_group` share their byte layout
// with `bb_instr` / `bb_agent_group` of include/bourse_b200.h so that one numpy array drives both
// the CUDA path and this checker.
#include <atomic>
#include <chrono>
#include <cstring>
#include <thread>

#include "env.hpp"

using namespace oracle;

// message of the last PriceError an agent run stopped at (orc_sim_run, orc_sim_agents_update, orc_market_run)
static thread_local std::string last_error;

extern "C" {

const char* orc_last_error(void) { return last_error.c_str(); }

struct orc_instr {  // 32 bytes, == bb_instr
    uint64_t t;
    uint32_t op_flags;  // low 8 bits: op; bits 8..: flags
    uint32_t order_id;
    uint32_t price;
    uint32_t vol;
    uint32_t trader;
    uint32_t aux;
};
enum { OP_NOOP = 0, OP_NEW = 1, OP_CANCEL = 2, OP_MODIFY = 3, OP_SET_TRADING = 4 };
enum { F_BID = 1u << 8, F_MARKET = 1u << 9, F_HAS_PRICE = 1u << 10, F_HAS_VOL = 1u << 11, F_EMIT = 1u << 12 };

struct orc_group {  // 80 bytes, == bb_agent_group
    uint32_t kind;      // 0 RandomAgents, 1 MomentumAgent, 2 NoiseAgent
    uint32_t n_agents;
    uint32_t tick_lo, tick_hi;  // random: tick range;  momentum: tick_lo = agent_id_start
    uint32_t vol_lo, vol_hi;    // random: vol range;   momentum: vol_lo = trade_vol
    uint32_t tick_size;
    float rate;                 // random: activity_rate; momentum: p_cancel
    double decay, demand, scale, order_ratio, mu, sigma;
};

struct SimHandle {
    Sim sim;
    Xoroshiro128StarStar rng;
    SimHandle(uint64_t seed, Nanos start, Price tick, Nanos step, bool trading)
        : sim(start, tick, step, trading), rng(Xoroshiro128StarStar::seed_from_u64(seed)) {}
};

// ---------------------------------------------------------------- OrderBook (immediate mode)
void* orc_book_new(uint64_t start_time, uint32_t tick_size, int trading) {
    return new OrderBook(start_time, tick_size, trading != 0);
}
void orc_book_free(void* b) { delete (OrderBook*)b; }
void orc_book_set_time(void* b, uint64_t t) { ((OrderBook*)b)->set_time(t); }
uint64_t orc_book_time(void* b) { return ((OrderBook*)b)->get_time(); }
void orc_book_set_trading(void* b, int on) { on ? ((OrderBook*)b)->enable_trading() : ((OrderBook*)b)->disable_trading(); }

// returns 0 ok, -1 price error
int orc_book_create(void* b, int bid, uint32_t vol, uint32_t trader, int has_price, uint32_t price, uint64_t* out_id) {
    try {
        *out_id = ((OrderBook*)b)->create_order(bid ? BID : ASK, vol, trader, has_price != 0, price);
        return 0;
    } catch (const PriceError&) {
        return -1;
    }
}
int orc_book_place_id(void* b, uint64_t id) {
    OrderBook* ob = (OrderBook*)b;
    if (id >= ob->orders.size()) return -2;
    ob->place_order(id);
    return 0;
}
int orc_book_place(void* b, int bid, uint32_t vol, uint32_t trader, int has_price, uint32_t price, uint64_t* out_id) {
    try {
        *out_id = ((OrderBook*)b)->create_and_place_order(bid ? BID : ASK, vol, trader, has_price != 0, price);
        return 0;
    } catch (const PriceError&) {
        return -1;
    }
}
int orc_book_cancel(void* b, uint64_t id) {
    OrderBook* ob = (OrderBook*)b;
    if (id >= ob->orders.size()) return -2;  // the reference panics (orderbook.rs:642)
    ob->cancel_order(id);
    return 0;
}
int orc_book_modify(void* b, uint64_t id, int has_price, uint32_t price, int has_vol, uint32_t vol) {
    OrderBook* ob = (OrderBook*)b;
    if (id >= ob->orders.size()) return -2;  // index panic in the reference (orderbook.rs:749)
    ob->modify_order(id, has_price != 0, price, has_vol != 0, vol);
    return 0;
}
int orc_book_order_status(void* b, uint64_t id) {
    OrderBook* ob = (OrderBook*)b;
    if (id >= ob->orders.size()) return -2;
    return (int)ob->orders[id].order.status;
}
uint32_t orc_book_trade_vol(void* b) { return ((OrderBook*)b)->get_trade_vol(); }
double orc_book_mid_price(void* b) { return ((OrderBook*)b)->mid_price(); }

// Level1Data in struct order (types.rs:252-269):
// bid_price, ask_price, bid_vol, ask_vol, bid_touch_vol, ask_touch_vol, bid_touch_orders, ask_touch_orders
void orc_book_l1(void* b, uint32_t* out) {
    const Level1Data d = ((OrderBook*)b)->level_1_data();
    out[0] = d.bid_price; out[1] = d.ask_price; out[2] = d.bid_vol; out[3] = d.ask_vol;
    out[4] = d.bid_touch_vol; out[5] = d.ask_touch_vol; out[6] = d.bid_touch_orders; out[7] = d.ask_touch_orders;
}

static void l2_to_array(const Level2Data& d, uint32_t trade_vol, uint32_t* out) {  // step_sim_numpy.rs:351-368
    out[0] = trade_vol; out[1] = d.bid_price; out[2] = d.ask_price; out[3] = d.ask_vol; out[4] = d.bid_vol;
    for (int i = 0; i < LEVELS; ++i) {
        out[5 + 4 * i + 0] = d.bid_price_levels[i].first;
        out[5 + 4 * i + 1] = d.bid_price_levels[i].second;
        out[5 + 4 * i + 2] = d.ask_price_levels[i].first;
        out[5 + 4 * i + 3] = d.ask_price_levels[i].second;
    }
}
void orc_book_l2(void* b, uint32_t* out) {
    OrderBook* ob = (OrderBook*)b;
    l2_to_array(ob->level_2_data(), ob->get_trade_vol(), out);
}
uint64_t orc_book_n_orders(void* b) { return ((OrderBook*)b)->orders.size(); }
uint64_t orc_book_n_trades(void* b) { return ((OrderBook*)b)->trades.size(); }
// PyOrder field order (rust/src/types.rs:19-31); order_id == index
void orc_book_orders(void* b, uint8_t* side_is_bid, uint8_t* status, uint64_t* arr, uint64_t* end, uint32_t* vol,
                     uint32_t* start_vol, uint32_t* price, uint32_t* trader) {
    OrderBook* ob = (OrderBook*)b;
    for (size_t i = 0; i < ob->orders.size(); ++i) {
        const Order& o = ob->orders[i].order;
        side_is_bid[i] = o.side == BID; status[i] = (uint8_t)o.status; arr[i] = o.arr_time; end[i] = o.end_time;
        vol[i] = o.vol; start_vol[i] = o.start_vol; price[i] = o.price; trader[i] = o.trader_id;
    }
}
// PyTrade field order (rust/src/types.rs:4-17)
void orc_book_trades(void* b, uint64_t* t, uint8_t* side_is_bid, uint32_t* price, uint32_t* vol, uint64_t* active,
                     uint64_t* passive) {
    OrderBook* ob = (OrderBook*)b;
    for (size_t i = 0; i < ob->trades.size(); ++i) {
        const Trade& x = ob->trades[i];
        t[i] = x.t; side_is_bid[i] = x.side == BID; price[i] = x.price; vol[i] = x.vol;
        active[i] = x.active_order_id; passive[i] = x.passive_order_id;
    }
}

// Replay a packed instruction stream through the immediate-mode book (SURVEY.md 3.5 / config C2).
// Every instruction first sets the book time to `t`.  Instructions flagged F_EMIT append one
// 45-word L2 record (trade_vol first) to `obs_out`; returns the number of records written, or a
// negative error (-1 price error at instruction *err_at, -2 bad id).
int64_t orc_book_replay(void* b, const orc_instr* ins, uint64_t n, uint32_t* obs_out, uint64_t obs_cap, uint64_t* err_at) {
    OrderBook* ob = (OrderBook*)b;
    uint64_t n_obs = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const orc_instr& x = ins[i];
        const uint32_t op = x.op_flags & 0xFF;
        ob->set_time(x.t);
        try {
            switch (op) {
                case OP_NEW:
                    ob->create_and_place_order((x.op_flags & F_BID) ? BID : ASK, x.vol, x.trader, !(x.op_flags & F_MARKET), x.price);
                    break;
                case OP_CANCEL:
                    if (x.order_id >= ob->orders.size()) { if (err_at) *err_at = i; return -2; }
                    ob->cancel_order(x.order_id);
                    break;
                case OP_MODIFY:
                    if (x.order_id >= ob->orders.size()) { if (err_at) *err_at = i; return -2; }
                    ob->modify_order(x.order_id, (x.op_flags & F_HAS_PRICE) != 0, x.price, (x.op_flags & F_HAS_VOL) != 0, x.vol);
                    break;
                case OP_SET_TRADING:
                    x.vol ? ob->enable_trading() : ob->disable_trading();
                    break;
                default: break;
            }
        } catch (const PriceError&) {
            if (err_at) *err_at = i;
            return -1;
        }
        if ((x.op_flags & F_EMIT) && n_obs < obs_cap) {
            l2_to_array(ob->level_2_data(), ob->get_trade_vol(), obs_out + 45 * n_obs);
            ++n_obs;
        }
    }
    return (int64_t)n_obs;
}

// ---------------------------------------------------------------- Env / Sim
void* orc_sim_new(uint64_t seed, uint64_t start_time, uint32_t tick_size, uint64_t step_size, int trading) {
    return new SimHandle(seed, start_time, tick_size, step_size, trading != 0);
}
void orc_sim_free(void* s) { delete (SimHandle*)s; }
void* orc_sim_book(void* s) { return &((SimHandle*)s)->sim.env.book; }  // borrowed; use with orc_book_* getters
void orc_sim_keep_records(void* s, int on) { ((SimHandle*)s)->sim.env.keep_records = on != 0; }

int orc_sim_place(void* s, int bid, uint32_t vol, uint32_t trader, int has_price, uint32_t price, uint64_t* out_id) {
    try {
        *out_id = ((SimHandle*)s)->sim.env.place_order(bid ? BID : ASK, vol, trader, has_price != 0, price);
        return 0;
    } catch (const PriceError&) {
        return -1;
    }
}
void orc_sim_cancel(void* s, uint64_t id) { ((SimHandle*)s)->sim.env.cancel_order(id); }
void orc_sim_modify(void* s, uint64_t id, int has_price, uint32_t price, int has_vol, uint32_t vol) {
    ((SimHandle*)s)->sim.env.modify_order(id, has_price != 0, price, has_vol != 0, vol);
}
// returns 0, or -2 when a queued instruction named an id that does not exist (reference: panic)
int orc_sim_step(void* s) {
    SimHandle* h = (SimHandle*)s;
    try {
        h->sim.env.step(h->rng);
    } catch (const std::out_of_range&) {
        return -2;
    }
    return 0;
}
uint64_t orc_sim_n_queued(void* s) { return ((SimHandle*)s)->sim.env.transactions.size(); }
void orc_sim_set_trading(void* s, int on) { orc_book_set_trading(orc_sim_book(s), on); }
// cached end-of-step L2 (env.rs:132, 293-295) in the 45-word array layout, live trade_vol in slot 0
void orc_sim_l2(void* s, uint32_t* out) {
    SimHandle* h = (SimHandle*)s;
    l2_to_array(h->sim.env.level_2_data, h->sim.env.book.get_trade_vol(), out);
}
uint64_t orc_sim_n_steps(void* s) { return ((SimHandle*)s)->sim.env.trade_vols.size(); }
// history as [steps][45] in the level_2_data array layout, slot 0 = that step's trade volume
void orc_sim_history(void* s, uint32_t* out) {
    SimHandle* h = (SimHandle*)s;
    const Level2DataRecords& r = h->sim.env.records;
    const size_t n = h->sim.env.trade_vols.size();
    for (size_t k = 0; k < n; ++k) {
        uint32_t* o = out + 45 * k;
        o[0] = h->sim.env.trade_vols[k]; o[1] = r.bid_price[k]; o[2] = r.ask_price[k]; o[3] = r.ask_vol[k]; o[4] = r.bid_vol[k];
        for (int i = 0; i < LEVELS; ++i) {
            o[5 + 4 * i + 0] = r.bid_vol_at[i][k]; o[5 + 4 * i + 1] = r.bid_n_at[i][k];
            o[5 + 4 * i + 2] = r.ask_vol_at[i][k]; o[5 + 4 * i + 3] = r.ask_n_at[i][k];
        }
    }
}

static void add_groups(Sim& sim, const orc_group* g, uint32_t n_groups) {
    for (uint32_t i = 0; i < n_groups; ++i) {
        if (g[i].kind == 0) {
            sim.add_random(RandomAgentsParams{g[i].n_agents, g[i].tick_lo, g[i].tick_hi, g[i].vol_lo, g[i].vol_hi,
                                              g[i].tick_size, g[i].rate});
        } else if (g[i].kind == 1) {
            sim.add_momentum(MomentumParams{g[i].tick_lo, g[i].n_agents, g[i].tick_size, g[i].rate, g[i].vol_lo, g[i].decay,
                                            g[i].demand, g[i].scale, g[i].order_ratio, g[i].mu, g[i].sigma});
        } else {  // NoiseAgent: p_limit / p_market travel in the decay / demand slots
            sim.add_noise(NoiseParams{g[i].tick_lo, g[i].n_agents, g[i].tick_size, (float)g[i].decay, (float)g[i].demand, g[i].rate,
                                      g[i].vol_lo, g[i].mu, g[i].sigma});
        }
    }
}
void orc_sim_set_groups(void* s, const orc_group* g, uint32_t n_groups) { add_groups(((SimHandle*)s)->sim, g, n_groups); }
// keyed != 0: Philox contract (what the CUDA path mirrors);  keyed == 0: reference-style shared stream
// 0, or -1 when an agent's limit price was off its book's tick: the reference agents unwrap create_order's PriceError
// (orderbook.rs:367-383) and panic.  The env stays as it was at the throw (completed steps' records
// readable, the failing step's instructions queued); orc_last_error() gives the reference's message.
int orc_sim_run(void* s, int keyed, uint64_t seed, uint32_t env_id, uint64_t n_steps) {
    SimHandle* h = (SimHandle*)s;
    try {
        if (keyed) h->sim.run_keyed(seed, env_id, n_steps); else h->sim.run_stream(seed, n_steps);
    } catch (const PriceError& e) {
        last_error = e.what();
        return -1;
    }
    return 0;
}
uint64_t orc_sim_n_instructions(void* s) { return ((SimHandle*)s)->sim.n_instructions; }
// the two halves of one keyed step (instructions queued in between take part in the step's shuffle)
int orc_sim_agents_update(void* s, uint64_t seed, uint32_t env_id) {  // 0, or -1 as orc_sim_run
    try {
        ((SimHandle*)s)->sim.agents_update_keyed(seed, env_id);
    } catch (const PriceError& e) {
        last_error = e.what();
        return -1;
    }
    return 0;
}
int orc_sim_step_keyed(void* s, uint64_t seed, uint32_t env_id) {
    try {
        ((SimHandle*)s)->sim.step_keyed(seed, env_id);
    } catch (const std::out_of_range&) {
        return -2;
    }
    return 0;
}

// ---------------------------------------------------------------- MarketEnv (multi-asset)
struct MarketHandle {
    MarketSim sim;
    MarketEnv& env;
    Xoroshiro128StarStar rng;
    MarketHandle(uint64_t seed, Nanos start, const std::vector<Price>& ticks, Nanos step, bool trading)
        : sim(start, ticks, step, trading), env(sim.env), rng(Xoroshiro128StarStar::seed_from_u64(seed)) {}
};
void* orc_market_new(uint64_t seed, uint64_t start_time, const uint32_t* tick_sizes, uint32_t n_assets, uint64_t step_size, int trading) {
    return new MarketHandle(seed, start_time, std::vector<Price>(tick_sizes, tick_sizes + n_assets), step_size, trading != 0);
}
void orc_market_free(void* m) { delete (MarketHandle*)m; }
void* orc_market_book(void* m, uint32_t asset) { return &((MarketHandle*)m)->env.books[asset]; }  // borrowed, for orc_book_* getters
int orc_market_place(void* m, uint32_t asset, int bid, uint32_t vol, uint32_t trader, int has_price, uint32_t price, uint64_t* out_id) {
    try {
        *out_id = ((MarketHandle*)m)->env.place_order(asset, bid ? BID : ASK, vol, trader, has_price != 0, price);
        return 0;
    } catch (const PriceError&) {
        return -1;
    }
}
void orc_market_cancel(void* m, uint32_t asset, uint64_t id) { ((MarketHandle*)m)->env.cancel_order(asset, id); }
void orc_market_modify(void* m, uint32_t asset, uint64_t id, int has_price, uint32_t price, int has_vol, uint32_t vol) {
    ((MarketHandle*)m)->env.modify_order(asset, id, has_price != 0, price, has_vol != 0, vol);
}
int orc_market_step(void* m) {
    try {
        MarketHandle* h = (MarketHandle*)m;
        h->env.step(h->rng);
        return 0;
    } catch (const std::out_of_range&) {
        return -2;
    }
}
uint64_t orc_market_n_steps(void* m, uint32_t asset) { return ((MarketHandle*)m)->env.trade_vols[asset].size(); }
void orc_market_history(void* m, uint32_t asset, uint32_t* out) {  // [n_steps][45], StepEnvNumpy.level_2_data layout
    MarketHandle* h = (MarketHandle*)m;
    const Level2DataRecords& r = h->env.records[asset];
    const std::vector<Vol>& tv = h->env.trade_vols[asset];
    for (size_t k = 0; k < tv.size(); ++k) {
        uint32_t* o = out + 45 * k;
        o[0] = tv[k]; o[1] = r.bid_price[k]; o[2] = r.ask_price[k]; o[3] = r.ask_vol[k]; o[4] = r.bid_vol[k];
        for (int i = 0; i < LEVELS; ++i) {
            o[5 + 4 * i + 0] = r.bid_vol_at[i][k]; o[5 + 4 * i + 1] = r.bid_n_at[i][k];
            o[5 + 4 * i + 2] = r.ask_vol_at[i][k]; o[5 + 4 * i + 3] = r.ask_n_at[i][k];
        }
    }
}

// market agent twins: group i trades asset assets[i] (RandomMarketAgents / MomentumMarketAgent / NoiseMarketAgent)
static void add_market_groups(MarketSim& sim, const orc_group* g, const uint32_t* assets, uint32_t n_groups) {
    for (uint32_t i = 0; i < n_groups; ++i) {
        if (g[i].kind == 0) {
            sim.add_random(assets[i], RandomAgentsParams{g[i].n_agents, g[i].tick_lo, g[i].tick_hi, g[i].vol_lo, g[i].vol_hi,
                                                         g[i].tick_size, g[i].rate});
        } else if (g[i].kind == 1) {
            sim.add_momentum(assets[i], MomentumParams{g[i].tick_lo, g[i].n_agents, g[i].tick_size, g[i].rate, g[i].vol_lo,
                                                       g[i].decay, g[i].demand, g[i].scale, g[i].order_ratio, g[i].mu, g[i].sigma});
        } else {
            sim.add_noise(assets[i], NoiseParams{g[i].tick_lo, g[i].n_agents, g[i].tick_size, (float)g[i].decay, (float)g[i].demand,
                                                 g[i].rate, g[i].vol_lo, g[i].mu, g[i].sigma});
        }
    }
}
void orc_market_set_groups(void* m, const orc_group* g, const uint32_t* assets, uint32_t n_groups) {
    add_market_groups(((MarketHandle*)m)->sim, g, assets, n_groups);
}
// keyed != 0: Philox contract keyed by market id (what the CUDA path mirrors); keyed == 0: market_sim_runner's shared stream
// 0, or -1 as orc_sim_run
int orc_market_run(void* m, int keyed, uint64_t seed, uint32_t market_id, uint64_t n_steps) {
    MarketHandle* h = (MarketHandle*)m;
    try {
        if (keyed) h->sim.run_keyed(seed, market_id, n_steps); else h->sim.run_stream(seed, n_steps);
    } catch (const PriceError& e) {
        last_error = e.what();
        return -1;
    }
    return 0;
}
uint64_t orc_market_n_instructions(void* m) { return ((MarketHandle*)m)->sim.n_instructions; }

// `n_markets` agent-driven markets across `n_threads` threads; out[0] = instructions, out[1] = trades, out[2] = book-steps
double orc_bench_market_agents(uint32_t n_markets, uint32_t n_threads, uint64_t n_steps, uint64_t seed, int keyed, uint64_t start_time,
                               const uint32_t* tick_sizes, uint32_t n_assets, uint64_t step_size, const orc_group* g,
                               const uint32_t* assets, uint32_t n_groups, uint64_t* out) {
    std::atomic<uint32_t> next(0);
    std::atomic<uint64_t> n_ins(0), n_tr(0);
    const std::vector<Price> ticks(tick_sizes, tick_sizes + n_assets);
    auto worker = [&]() {
        for (;;) {
            const uint32_t e = next.fetch_add(1);
            if (e >= n_markets) break;
            MarketSim sim(start_time, ticks, step_size, true);
            add_market_groups(sim, g, assets, n_groups);
            if (keyed) sim.run_keyed(seed, e, n_steps); else sim.run_stream(seed + e, n_steps);
            n_ins += sim.n_instructions;
            for (auto& b : sim.env.books) n_tr += b.trades.size();
        }
    };
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> th;
    for (uint32_t i = 0; i < n_threads; ++i) th.emplace_back(worker);
    for (auto& x : th) x.join();
    const auto t1 = std::chrono::steady_clock::now();
    out[0] = n_ins; out[1] = n_tr; out[2] = (uint64_t)n_markets * n_assets * n_steps;
    return std::chrono::duration<double>(t1 - t0).count();
}

// ---------------------------------------------------------------- CPU baseline
// Runs `n_envs` independent agent-driven markets, one env per host thread at a time, `n_threads`
// threads (SURVEY.md 8d "one env per host core across all cores").  Env `e` uses seed `seed + e`
// in stream mode (each env its own reference-style sim_runner) or the Philox key (seed, env e).
// out[0] = instructions processed, out[1] = trades, out[2] = env-steps; returns elapsed seconds.
double orc_bench_agents(uint32_t n_envs, uint32_t n_threads, uint64_t n_steps, uint64_t seed, int keyed,
                        uint64_t start_time, uint32_t tick_size, uint64_t step_size, const orc_group* g,
                        uint32_t n_groups, uint64_t* out) {
    std::atomic<uint32_t> next(0);
    std::atomic<uint64_t> n_ins(0), n_tr(0);
    auto worker = [&]() {
        for (;;) {
            const uint32_t e = next.fetch_add(1);
            if (e >= n_envs) break;
            Sim sim(start_time, tick_size, step_size, true);
            add_groups(sim, g, n_groups);
            if (keyed) sim.run_keyed(seed, e, n_steps); else sim.run_stream(seed + e, n_steps);
            n_ins += sim.n_instructions;
            n_tr += sim.env.book.trades.size();
        }
    };
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> th;
    for (uint32_t i = 0; i < n_threads; ++i) th.emplace_back(worker);
    for (auto& x : th) x.join();
    const auto t1 = std::chrono::steady_clock::now();
    out[0] = n_ins; out[1] = n_tr; out[2] = (uint64_t)n_envs * n_steps;
    return std::chrono::duration<double>(t1 - t0).count();
}

// Replays `n_books` copies of one instruction stream (config C2 style) across threads.
double orc_bench_replay(uint32_t n_books, uint32_t n_threads, uint32_t tick_size, const orc_instr* ins, uint64_t n, uint64_t* out) {
    std::atomic<uint32_t> next(0);
    std::atomic<uint64_t> n_tr(0);
    auto worker = [&]() {
        for (;;) {
            const uint32_t e = next.fetch_add(1);
            if (e >= n_books) break;
            OrderBook ob(0, tick_size, true);
            orc_book_replay(&ob, ins, n, nullptr, 0, nullptr);
            n_tr += ob.trades.size();
        }
    };
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> th;
    for (uint32_t i = 0; i < n_threads; ++i) th.emplace_back(worker);
    for (auto& x : th) x.join();
    const auto t1 = std::chrono::steady_clock::now();
    out[0] = (uint64_t)n_books * n; out[1] = n_tr;
    return std::chrono::duration<double>(t1 - t0).count();
}

// Deep-book variant (config C5): every thread first replays the untimed prefix ins[0, n_pre) (the resting book),
// all threads then start the timed suffix ins[n_pre, n) together; returns the slowest thread's suffix time.
double orc_bench_replay_suffix(uint32_t n_threads, uint32_t tick_size, const orc_instr* ins, uint64_t n_pre, uint64_t n, uint64_t* out) {
    std::atomic<uint32_t> ready(0);
    std::atomic<uint64_t> n_tr(0);
    std::vector<double> secs(n_threads, 0.0);
    auto worker = [&](uint32_t i) {
        OrderBook ob(0, tick_size, true);
        orc_book_replay(&ob, ins, n_pre, nullptr, 0, nullptr);
        const uint64_t tr0 = ob.trades.size();
        ready.fetch_add(1);
        while (ready.load() < n_threads) std::this_thread::yield();
        const auto t0 = std::chrono::steady_clock::now();
        orc_book_replay(&ob, ins + n_pre, n - n_pre, nullptr, 0, nullptr);
        secs[i] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        n_tr += ob.trades.size() - tr0;
    };
    std::vector<std::thread> th;
    for (uint32_t i = 0; i < n_threads; ++i) th.emplace_back(worker, i);
    for (auto& x : th) x.join();
    out[0] = (uint64_t)n_threads * (n - n_pre); out[1] = n_tr;
    double mx = 0;
    for (double x : secs) mx = x > mx ? x : mx;
    return mx;
}

// Vectorised-loop baseline (bourse_b200.gym.VectorEnv's workload): `n_envs` Envs, each fed `rows` instruction rows per
// step for `n_steps` steps from a cyclic table of `n_blocks` action blocks laid out [block][env][row] (the array the GPU
// path reads from device memory), with the submit-then-step semantics of StepEnvNumpy.submit_instructions + step
// (rust/src/step_sim_numpy.rs:233-275).  out[0] = rows queued, out[1] = trades, out[2] = env-steps; returns seconds.
double orc_bench_env_rows(uint32_t n_envs, uint32_t n_threads, uint64_t n_steps, uint32_t rows, const orc_instr* blocks,
                          uint32_t n_blocks, uint32_t block_envs, uint64_t seed, uint32_t tick_size, uint64_t step_size, uint64_t* out) {
    std::atomic<uint32_t> next(0);
    std::atomic<uint64_t> n_q(0), n_tr(0);
    auto worker = [&]() {
        for (;;) {
            const uint32_t e = next.fetch_add(1);
            if (e >= n_envs) break;
            Env env(0, tick_size, step_size, true);
            env.keep_records = false;
            Xoroshiro128StarStar rng = Xoroshiro128StarStar::seed_from_u64(seed + e);
            uint64_t q = 0;
            for (uint64_t s = 0; s < n_steps; ++s) {
                const orc_instr* r = blocks + ((size_t)(s % n_blocks) * block_envs + (e % block_envs)) * rows;
                for (uint32_t k = 0; k < rows; ++k) {
                    const uint32_t op = r[k].op_flags & 0xFF;
                    try {
                        if (op == OP_NEW) {
                            env.place_order((r[k].op_flags & F_BID) ? BID : ASK, r[k].vol, r[k].trader, !(r[k].op_flags & F_MARKET), r[k].price);
                            ++q;
                        } else if (op == OP_CANCEL) {
                            if (r[k].order_id < env.book.orders.size()) { env.cancel_order(r[k].order_id); ++q; }
                        } else if (op == OP_MODIFY) {
                            if (r[k].order_id < env.book.orders.size()) {
                                env.modify_order(r[k].order_id, (r[k].op_flags & F_HAS_PRICE) != 0, r[k].price, (r[k].op_flags & F_HAS_VOL) != 0, r[k].vol);
                                ++q;
                            }
                        }
                    } catch (const PriceError&) {
                    }
                }
                env.step(rng);
            }
            n_q += q;
            n_tr += env.book.trades.size();
        }
    };
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> th;
    for (uint32_t i = 0; i < n_threads; ++i) th.emplace_back(worker);
    for (auto& x : th) x.join();
    const auto t1 = std::chrono::steady_clock::now();
    out[0] = n_q; out[1] = n_tr; out[2] = (uint64_t)n_envs * n_steps;
    return std::chrono::duration<double>(t1 - t0).count();
}

// ---------------------------------------------------------------- RNG probes for the known-answer tests
void orc_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
    const Philox4 r = philox4x32_10(c0, c1, c2, c3, k0, k1);
    memcpy(out, r.v, 16);
}
void orc_xoroshiro(uint64_t seed, uint32_t n, uint64_t* out) {
    Xoroshiro128StarStar r = Xoroshiro128StarStar::seed_from_u64(seed);
    for (uint32_t i = 0; i < n; ++i) out[i] = r.next_u64();
}
// the generator from an explicit state (rand_xoshiro's from_seed): u64 outputs and the u32 / f32 / range draws derived from them
void orc_xoroshiro_state(uint64_t s0, uint64_t s1, uint32_t n, uint64_t* out64, uint32_t* out32, float* outf, uint32_t range,
                         uint32_t* out_range) {
    Xoroshiro128StarStar a, b, c, d;
    a.s0 = b.s0 = c.s0 = d.s0 = s0;
    a.s1 = b.s1 = c.s1 = d.s1 = s1;
    for (uint32_t i = 0; i < n; ++i) {
        out64[i] = a.next_u64();
        out32[i] = b.next_u32();
        outf[i] = gen_f32(c);
        out_range[i] = gen_range_u32(d, 0, range);
    }
}
void orc_shuffle_perm(uint64_t seed, uint32_t n, uint32_t* out) {
    Xoroshiro128StarStar r = Xoroshiro128StarStar::seed_from_u64(seed);
    std::vector<uint32_t> v(n);
    for (uint32_t i = 0; i < n; ++i) v[i] = i;
    shuffle(r, v);
    memcpy(out, v.data(), 4 * n);
}
uint32_t orc_round_price(double p, double tick, int up) { return up ? round_price_up(p, tick) : round_price_down(p, tick); }

}  // extern "C"
