/* bourse_b200 — C ABI of the B200-native batched limit-order-book simulator.
 *
 * This is the drop-in boundary for the reference's hot path (SURVEY.md section 8b): the calls
 * below are what a binding for `bourse.core` (PyO3 module, /root/reference/rust/src/lib.rs:7-15)
 * or a Rust `extern "C"` host would bind instead of `bourse_book::OrderBook` /
 * `bourse_de::{Env, sim_runner}`.  Plain pointers and sizes only; no torch / numpy types.
 *
 * One handle owns `n_envs` independent books ("envs") on ONE CUDA device plus everything the
 * reference keeps per `Env`: order table, trade log, transaction queue, per-step level-2 history.
 * All pointer arguments are HOST pointers unless the function name ends in `_device`.
 * Every function returns BB_OK (0) or a negative bb_status; bb_last_error() gives the text.
 * A handle is not thread-safe.  Calls are synchronous unless stated otherwise.
 *
 * There is no CPU fallback: bb_create fails with BB_ECUDA when no sm_100 device is usable.
 */
#ifndef BOURSE_B200_H
#define BOURSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BB_ABI_VERSION 1

typedef struct bb_handle bb_handle;

typedef enum {
    BB_OK = 0,
    BB_EPRICE = -1,   /* price not a multiple of tick size: OrderError::PriceError, orderbook.rs:127-142 */
    BB_EBADID = -2,   /* order id does not exist: the reference panics, orderbook.rs:642 / :749 */
    BB_ECAP = -3,     /* a configured capacity (orders / trades / queue / pages / steps) was exceeded */
    BB_ECUDA = -4,    /* CUDA runtime error or no usable device */
    BB_EINVAL = -5,   /* bad argument */
    BB_EDEVICE = -6   /* the device flagged an env error during the call; see bb_env_errors */
} bb_status;

/* per-env sticky error bits reported by bb_env_errors */
#define BB_ERR_CAP_ORDERS 0x01u
#define BB_ERR_CAP_TRADES 0x02u
#define BB_ERR_CAP_PAGES  0x04u
#define BB_ERR_CAP_QUEUE  0x08u
#define BB_ERR_BAD_ID     0x10u
#define BB_ERR_GRANULE    0x20u  /* a resting price was not a multiple of price_granule, or an agent's limit price not one of its book's tick */
#define BB_ERR_CAP_STEPS  0x40u
#define BB_ERR_CAP_LIVE   0x80u  /* MomentumAgent live-order list / dense engine's resting-order slots overflow */
#define BB_ERR_TIME_ORDER 0x100u /* dense engine: a resting order arrived out of time order at its price level */
#define BB_ERR_PRICE 0x200u      /* bb_step_device: a NEW row's limit price was not a multiple of its env's tick (row dropped) */
#define BB_ERR_ROW_OP 0x400u     /* bb_run_agents_with_rows: a MODIFY row or a trader id >= 2^19 (row dropped) */
#define BB_ERR_LOCKED 0x800u     /* deep engine: both sides would rest at one price level (trading disabled) */

#define BB_OBS_L1 9u   /* StepEnvNumpy.level_1_data layout, rust/src/step_sim_numpy.rs:300-318 */
#define BB_OBS_L2 45u  /* StepEnvNumpy.level_2_data layout, rust/src/step_sim_numpy.rs:351-368 */
#define BB_LEVELS 10u  /* hard-wired in the reference's Python surface, rust/src/step_sim.rs:438 */

#define BB_NO_ID UINT64_MAX  /* id returned for rows that create nothing, step_sim_numpy.rs:256-267 */
#define BB_ALL_ENVS 0xFFFFFFFFu

/* Replaces the constructor arguments of OrderBook::new (orderbook.rs:158-171), Env::new
 * (crates/step_sim/src/env.rs:84-95) and StepEnv/StepEnvNumpy::new (rust/src/step_sim.rs:63-75),
 * batched over n_envs, plus the capacities a preallocating device implementation needs. */
typedef struct {
    uint32_t struct_size;   /* sizeof(bb_config) */
    int32_t device;         /* CUDA device ordinal */
    uint32_t n_envs;        /* books owned by this handle (this rank's shard) */
    uint32_t env_id_base;   /* global id of env 0: keeps agent RNG invariant to the sharding */
    uint64_t start_time;    /* Nanos */
    uint64_t step_size;     /* Nanos advanced per Env::step */
    uint64_t seed;          /* env e shuffles with Xoroshiro128**(seed + env_id_base + e) (step_sim.rs:73) */
    uint32_t tick_size;     /* > 0; every book's tick until bb_set_tick_sizes gives books their own */
    uint32_t price_granule; /* ladder granularity; 0 => tick_size.  Every resting price must be a multiple */
    uint32_t trading;       /* initial trading flag */
    uint32_t obs_words;     /* BB_OBS_L1 or BB_OBS_L2: record written to the history each step */
    uint32_t max_orders;    /* per env */
    uint32_t max_trades;    /* per env; 0 disables the trade log (trade_vol is still tracked) */
    uint32_t max_steps;     /* per env history records (steps, or emitted snapshots in replay mode) */
    uint32_t max_queue;     /* per env instructions per step (bb_reserve_queue grows it) */
    uint32_t pages_smem;    /* 32-level price pages per book resident in shared memory; 0 => default */
    uint32_t pages_total;   /* total pages per book (the rest live in HBM); 0 => default */
    /* Dense-window engine for shallow books (the layout BASELINE.json's north_star names: a dense tick-indexed
     * ladder in shared memory with non-empty-level bitmaps, resting orders in shared-memory slots).  Selected
     * when win_levels > 0; requires price_granule == 1.  Every resting price must lie in
     * [win_lo, win_lo + win_levels) and at most live_cap orders may rest per book at any time, else the env flags
     * BB_ERR_CAP_PAGES / BB_ERR_CAP_LIVE; resting orders must arrive in non-decreasing time per price level (always
     * true in Env mode and for replay streams with increasing time), else BB_ERR_TIME_ORDER.  Within those limits
     * results are bit-identical to the paged engine (win_levels == 0), which has none of these limits. */
    uint32_t win_lo;        /* price of ladder level 0 */
    uint32_t win_levels;    /* number of price levels; rounded up to a multiple of 32; 0 => paged engine */
    uint32_t live_cap;      /* resident resting orders per book, <= 254; 0 => 128 */
    /* Multi-asset markets (bourse_book::Market crates/order_book/src/market.rs:59-95, bourse_de::MarketEnv
     * crates/step_sim/src/market_env.rs:47-135): books [m * assets, (m + 1) * assets) form market m.  The books stay
     * independent; what a market shares is ONE transaction queue per step, shuffled as a whole, with event i of the
     * shuffled queue executing at time start + i on its asset's book (market_env.rs:108-121).  n_envs must be a
     * multiple of assets; market m shuffles with Xoroshiro128**(seed + env_id_base / assets + m).  0 or 1 => every
     * book is its own Env.  In-kernel agents on a multi-asset handle are defined with bb_set_agents_market. */
    uint32_t assets;
    /* Deep-book engine (csrc/deep.cuh, csrc/deepw.cuh) for books with up to millions of resting orders, replayed instruction
     * streams (bb_replay / bb_replay_device; BASELINE config C5): one CTA per book — a fetch warp that prefetches the records
     * cancels / modifies name, a chain warp that keeps the price ladder (shared memory) in event order and writes per-level
     * micro-ops, a replay warp that applies them to the array (chunked) price-time queues in HBM one lane per price level and
     * places the trades with a warp prefix sum, a retire warp that streams the order-record updates out.  Selected when
     * deep_chunks > 0, together with the window fields above: win_levels <= 8192 price levels starting at win_lo,
     * price_granule == 1; deep_chunks = 256-byte queue chunks per book (31 entries each; one per resting order in the
     * worst case, ~ resting orders / 31 + win_levels + entries appended during a launch / 31 in practice).  Preconditions
     * beyond the window: strictly increasing time between resting inserts (BB_ERR_TIME_ORDER) and one side per price
     * level (BB_ERR_LOCKED: only reachable while trading is disabled).  Env mode and in-kernel agents are
     * not available on a deep handle (BB_EINVAL). */
    uint32_t deep_chunks;
} bb_config;

/* One instruction, 32 bytes; replaces Event<OrderId> (crates/order_book/src/types.rs:229-249) plus
 * the creation arguments of create_order (orderbook.rs:356-396).  Streams of these are what the
 * replay kernel bulk-copies from HBM. */
typedef struct {
    uint64_t t;        /* replay mode: book time this instruction executes at (OrderBook::set_time) */
    uint32_t op_flags; /* BB_OP_* | BB_F_* */
    uint32_t order_id; /* CANCEL / MODIFY target */
    uint32_t price;    /* NEW: limit price; MODIFY: new price when BB_F_HAS_PRICE */
    uint32_t vol;      /* NEW: volume; MODIFY: new volume when BB_F_HAS_VOL; SET_TRADING: 0 / 1 */
    uint32_t trader;   /* NEW: trader id */
    uint32_t aux;      /* reserved, 0 (the library keeps a market's submission order here while instructions are queued) */
} bb_instr;

#define BB_OP_NOOP 0u
#define BB_OP_NEW 1u          /* create_and_place_order, orderbook.rs:411-421 */
#define BB_OP_CANCEL 2u       /* cancel_order, orderbook.rs:622-644 */
#define BB_OP_MODIFY 3u       /* modify_order, orderbook.rs:743-772 */
#define BB_OP_SET_TRADING 4u  /* enable/disable_trading, orderbook.rs:188-198 */
#define BB_OP_RESTORE 5u      /* internal: re-insert an Active order from its record (bb_load_book) */
#define BB_OP_MASK 0xFFu
#define BB_F_BID (1u << 8)
#define BB_F_MARKET (1u << 9)     /* price == None */
#define BB_F_HAS_PRICE (1u << 10)
#define BB_F_HAS_VOL (1u << 11)
#define BB_F_EMIT (1u << 12)      /* replay mode: append a level-2 record to the history afterwards */

/* Actions of StepEnvNumpy.submit_instructions (rust/src/step_sim_numpy.rs:254-268) */
#define BB_ACT_NOOP 0u
#define BB_ACT_NEW 1u
#define BB_ACT_CANCEL 2u
#define BB_ACT_MODIFY 3u /* extension: Env::modify_order (env.rs:208-219) through the array call */

/* One built-in agent group, 80 bytes; groups are updated in array order each step, as the fields
 * of a #[derive(AgentSet)] struct are (crates/macros/src/lib.rs:57-72).
 *  kind 0 RandomAgents::new(n_agents, (tick_lo,tick_hi), (vol_lo,vol_hi), tick_size, rate)
 *         crates/step_sim/src/agents/random_agent.rs:66-81
 *  kind 1 MomentumAgent::new(agent_id_start = tick_lo, n_agents, MomentumParams{tick_size,
 *         p_cancel = rate, trade_vol = vol_lo, decay, demand, scale, order_ratio, mu, sigma})
 *         crates/step_sim/src/agents/momentum_agent.rs:16-35, 118-134
 *  kind 2 NoiseAgent::new(agent_id_start = tick_lo, n_agents, NoiseAgentParams{tick_size, p_limit = decay,
 *         p_market = demand, p_cancel = rate, trade_vol = vol_lo, mu, sigma})
 *         crates/step_sim/src/agents/noise_agent.rs:14-44, 98-114
 *  kinds 1 and 2: vol_hi = capacity of the agent's list of resting limit orders (the reference's Vec<OrderId>,
 *         momentum_agent.rs:99-102; common.rs:56-75 prunes it every step); 0 => 254.  A list that would outgrow it flags
 *         BB_ERR_CAP_LIVE.  The population's largest request sizes every group's list (4 bytes per entry per env). */
typedef struct {
    uint32_t kind;
    uint32_t n_agents;
    uint32_t tick_lo, tick_hi;
    uint32_t vol_lo, vol_hi;
    uint32_t tick_size;
    float rate;
    double decay, demand, scale, order_ratio, mu, sigma;
} bb_agent_group;

#define BB_GROUP_RANDOM 0u
#define BB_GROUP_MOMENTUM 1u
#define BB_GROUP_NOISE 2u

typedef struct {
    uint64_t instructions;   /* events that reached process_event (New + Cancel + Modify) */
    uint64_t orders_created;
    uint64_t trades;
    uint64_t traded_volume;
    uint64_t env_steps;
    uint64_t transitions;    /* order state changes after creation (place, fill, cancel, modify) */
    uint64_t error_envs;     /* envs with a non-zero error word */
    uint64_t l1_checksum;    /* FNV-1a over every env's current 9-word level-1 record */
} bb_stats_t;

/* ---- lifetime ------------------------------------------------------------------------------ */
int bb_abi_version(void);
int bb_create(const bb_config* cfg, bb_handle** out);
int bb_destroy(bb_handle* h);
int bb_reset(bb_handle* h); /* back to the freshly created state (same config, same agents); asynchronous */
/* Grow (never shrink) the per-env order table, trade log and history to at least these capacities, keeping their contents.
 * The reference's Vec<OrderEntry> / Vec<Trade> / Level2DataRecords grow without bound (orderbook.rs:113-115, data.rs:9-57);
 * a host that cannot size a run up front calls this when usage nears a capacity (the Python OrderBook / StepEnv /
 * StepEnvNumpy classes do).  Synchronous; costs one device-to-device copy of the slab that grows. */
int bb_reserve(bb_handle* h, uint32_t max_orders, uint32_t max_trades, uint32_t max_steps);
/* Grow (never shrink) max_queue, the number of transactions one env may queue for ONE step.  The reference's
 * Env::transactions is an unbounded Vec (crates/step_sim/src/env.rs:93-96, 121); here a step's queue is shuffled in shared
 * memory, so it is bounded by what fits there next to the book image (BB_ECAP beyond that, nothing changed).  bb_step refuses
 * a step whose queue exceeds max_queue with BB_ECAP BEFORE applying anything (the transactions stay queued), so a host can
 * call this and step again; the Python StepEnv / StepEnvNumpy classes reserve ahead of need.  Synchronous. */
int bb_reserve_queue(bb_handle* h, uint32_t max_queue);
/* Forget the per-step records (Level2DataRecords, data.rs:9-57) of every env: the history restarts at record 0, the books,
 * order tables and trade logs are untouched.  For open-ended loops that consume each step's observation as it is produced
 * (bb_step_device / bb_run_agents_with_rows) and would otherwise run into max_steps.  Asynchronous. */
int bb_clear_history(bb_handle* h);
/* Per-book tick sizes (MarketEnv::new(start_time, tick_sizes, step_size, trading), crates/step_sim/src/market_env.rs:73-90,
 * gives each asset's OrderBook its own tick).  n == n_envs: ticks[e] is env e's tick; on a multi-asset handle n == assets
 * gives asset a's tick to book a of every market.  Each book then checks create_order prices against its own tick
 * (bb_submit, bb_replay, bb_step_device, bb_run_agents_with_rows rows, RandomAgents / MomentumAgent / NoiseAgent prices;
 * not bb_replay_device) and lays out its level-2
 * record at its own tick offsets; until this is called every book has bb_config.tick_size.  Refused with BB_EINVAL, the
 * handle unchanged, for a NULL array, a wrong n, a tick of 0 or one that is not a multiple of the price granule, and while
 * any env holds orders or queued transactions (a reference book gets its tick at creation only; bb_reset first).  The ticks
 * survive bb_reset.  On the paged engine a book whose tick is k x the granule spreads its levels k times more thinly over the
 * 32-price pages and may need a larger pages_total; the dense and deep engines (granule 1) are unaffected.  Synchronous. */
int bb_set_tick_sizes(bb_handle* h, const uint32_t* ticks, uint32_t n);
const char* bb_last_error(const bb_handle* h /* may be NULL */);
/* run on a caller-owned CUDA stream (cudaStream_t); NULL restores the handle's own stream */
int bb_set_stream(bb_handle* h, void* cuda_stream);
int bb_synchronize(bb_handle* h);

/* ---- Env mode: queued instructions + step (crates/step_sim/src/env.rs:116-219) ---------------- */
/* Replaces Env::place_order / cancel_order / modify_order and StepEnvNumpy.submit_limit_orders /
 * submit_cancellations / submit_instructions (rust/src/step_sim_numpy.rs:147-275) for a batch of
 * rows over many envs.  Rows are processed in order; ids are assigned per env in row order.
 * On a tick error at row r the call returns BB_EPRICE, *n_done = r, rows < r stay queued (the
 * reference's lazy map short-circuits the same way) and bb_last_error() holds the reference's
 * message.  `flags` may be NULL (=> limit orders, BB_F_HAS_PRICE|BB_F_HAS_VOL for modifies);
 * otherwise BB_F_MARKET / BB_F_HAS_PRICE / BB_F_HAS_VOL per row.  `env` may be NULL when n_envs==1.
 * out_ids[r] = new order id, or BB_NO_ID for rows that create nothing. */
int bb_submit(bb_handle* h, uint64_t n, const uint32_t* env, const uint32_t* action, const uint8_t* side_is_bid,
              const uint32_t* vol, const uint32_t* trader, const uint32_t* price, const uint64_t* order_id,
              const uint32_t* flags, uint64_t* out_ids, uint64_t* n_done);
/* Env::step for every env, n_steps times (queued instructions are consumed by the first). */
int bb_step(bb_handle* h, uint32_t n_steps);

/* Vectorised Env loop with DEVICE-resident actions (SURVEY.md 8f rank 4; the array call it batches is
 * StepEnvNumpy.submit_instructions + step, rust/src/step_sim_numpy.rs:233-275, :139-145): the step's rows for every env
 * are already in device memory (d_env_offsets[n_envs + 1] delimits each env's slice of d_instrs, bb_instr::t is ignored)
 * and never visit the host.  Per env, in row order, exactly what submission would have done: BB_OP_NEW rows create the
 * next order ids (d_out_ids[row], BB_NO_ID for every other row; may be NULL), BB_OP_CANCEL / BB_OP_MODIFY rows are queued,
 * BB_OP_NOOP and unknown codes queue nothing; then ONE Env::step.  A NEW row whose limit price is off the tick grid is
 * dropped, as when create_order returns PriceError, and flags the env with BB_ERR_PRICE (the next synchronous call
 * reports BB_EPRICE).  d_obs_out (device, [n_envs][obs_words], may be NULL) receives every env's end-of-step
 * observation record from the same launch — what StepEnvNumpy.level_1_data / level_2_data would return next.
 * Asynchronous on the handle's stream: one kernel launch and no host synchronisation, so the call may be recorded into a
 * CUDA graph together with the caller's own kernels (stream capture on the stream given to bb_set_stream). */
int bb_step_device(bb_handle* h, const bb_instr* d_instrs, const uint64_t* d_env_offsets, uint64_t n_rows, uint64_t* d_out_ids,
                   uint32_t* d_obs_out);
/* bb_level2 / bb_level1 into DEVICE memory: d_out[n_envs][45] / d_out[n_envs][9].  Asynchronous. */
int bb_level2_device(bb_handle* h, uint32_t* d_out);
int bb_level1_device(bb_handle* h, uint32_t* d_out);
/* Device buffers for callers without a CUDA allocator of their own (numpy-only hosts); any device pointer works above.
 * bb_memcpy kind: 1 host to device, 2 device to host, 3 device to device; synchronous on the handle's stream. */
int bb_device_alloc(bb_handle* h, uint64_t bytes, void** d_ptr);
int bb_device_free(bb_handle* h, void* d_ptr);
int bb_memcpy(bb_handle* h, void* dst, const void* src, uint64_t bytes, int kind);

/* ---- immediate mode: OrderBook API / replayed streams (orderbook.rs:411-792) ------------------ */
/* env_offsets[n_envs + 1] delimits each env's slice of `instrs`.  Every instruction executes at its
 * own `t`.  NEW rows get ids in stream order.  Rows flagged BB_F_EMIT append a level-2 record.  A limit NEW whose price
 * is not a multiple of its env's tick (create_order's PriceError, orderbook.rs:367-383) refuses the whole call with
 * BB_EPRICE before any env changes; bb_last_error() names the env, the row and the reference's message.  MODIFY prices
 * are not checked, as in the reference. */
int bb_replay(bb_handle* h, const bb_instr* instrs, const uint64_t* env_offsets);
/* same with both arrays already resident in device memory (asynchronous on the handle's stream).  The stream never visits
 * the host and is not tick-checked: the caller guarantees that every limit NEW is on its env's tick. */
int bb_replay_device(bb_handle* h, const bb_instr* d_instrs, const uint64_t* d_env_offsets);

/* ---- built-in agents: sim_runner (crates/step_sim/src/runner.rs:46-69) ------------------------ */
/* Defines the agent set (resets agent state).  Groups run in array order. */
int bb_set_agents(bb_handle* h, const bb_agent_group* groups, uint32_t n_groups);
/* Multi-asset handles (bb_config.assets = 2..4): the *Market twins of the built-in agents — RandomMarketAgents
 * (crates/step_sim/src/agents/random_agent.rs:165-247), MomentumMarketAgent (momentum_agent.rs:282-409),
 * NoiseMarketAgent (noise_agent.rs:226-345) — as fields of a #[derive(MarketAgentSet)] struct: group i is the same
 * bb_agent_group as above and trades asset asset[i] of every market.  bb_run_agents then runs market_sim_runner
 * (crates/step_sim/src/runner.rs:107-131): all groups update in array order, the market's queue is shuffled as a
 * whole and event i executes at start + i on its asset's book (market_env.rs:108-121).  The RNG unit is the market:
 * Philox key (seed; global market id = (env_id_base + env) / assets, step, agent slot counted over all groups). */
int bb_set_agents_market(bb_handle* h, const bb_agent_group* groups, const uint32_t* asset, uint32_t n_groups);
/* n_steps of { agents.update(env); env.step() } for every env inside one persistent kernel.
 * Draws are Philox4x32-10 keyed (seed; global env id, step, agent) — DESIGN.md "RNG contract".
 * Asynchronous on the handle's stream; pair with bb_synchronize or any read call. */
int bb_run_agents(bb_handle* h, uint64_t seed, uint32_t n_steps);
/* ONE env-step of { agents.update(env); <the caller's rows>; env.step() } with the rows already in DEVICE memory: the loop of a
 * learning agent trading against the built-in background agents (SURVEY.md 8f rank 4).  Rows are laid out as for
 * bb_step_device and submitted after the agents' updates, in row order: BB_OP_NEW (ids in d_out_ids, BB_NO_ID elsewhere;
 * may be NULL) and BB_OP_CANCEL; no-op rows queue nothing; BB_OP_MODIFY rows are refused (BB_ERR_ROW_OP).  Everything
 * takes part in the step's one Philox-keyed shuffle.  d_obs_out ([n_envs][obs_words], may be NULL) receives the
 * end-of-step records from the same launch.  Asynchronous on the handle's stream. */
int bb_run_agents_with_rows(bb_handle* h, uint64_t seed, const bb_instr* d_instrs, const uint64_t* d_env_offsets, uint64_t n_rows,
                            uint64_t* d_out_ids, uint32_t* d_obs_out);
/* Same run, with every env-step's observation record (Level2DataRecords, crates/step_sim/src/data.rs:9-57; the
 * arrays StepEnvNumpy.get_market_data returns, rust/src/step_sim_numpy.rs:448-516) streamed to HOST memory while
 * the simulation runs: the steps are launched in chunks of chunk_steps (0 = a geometric schedule: half of what is
 * left, at least 32) and chunk k is copied out on a second stream while chunk k+1 is simulated.  host_out[n_envs][n_steps][obs_words], pinned memory
 * recommended.  Synchronous. */
int bb_run_agents_to_host(bb_handle* h, uint64_t seed, uint32_t n_steps, uint32_t chunk_steps, uint32_t* host_out);

/* ---- reads ---------------------------------------------------------------------------------- */
/* cached end-of-step data of every env + live trade_vol in slot 0 (N7/N8 of SURVEY.md):
 * out[n_envs][9] / out[n_envs][45] */
int bb_level1(bb_handle* h, uint32_t* out);
int bb_level2(bb_handle* h, uint32_t* out);
/* live book of one env, OrderBook::level_1_data field order (types.rs:252-269): 8 words */
int bb_book_level1(bb_handle* h, uint32_t env, uint32_t* out8);
/* live book of one env in the 45-word layout */
int bb_book_level2(bb_handle* h, uint32_t env, uint32_t* out45);
int bb_n_steps(bb_handle* h, uint32_t env, uint32_t* n);
/* history records [first, first+n) of one env: out[n][obs_words] (Level2DataRecords, data.rs:9-57) */
int bb_history(bb_handle* h, uint32_t env, uint32_t first, uint32_t n, uint32_t* out);
/* first n_steps records of every env: out[n_envs][n_steps][obs_words]; one strided D2H copy */
int bb_history_all(bb_handle* h, uint32_t n_steps, uint32_t* out);
int bb_n_orders(bb_handle* h, uint32_t env, uint64_t* n);
int bb_n_trades(bb_handle* h, uint32_t env, uint64_t* n);
/* PyOrder columns (rust/src/types.rs:19-31); order_id == row index.  Any column may be NULL. */
int bb_orders(bb_handle* h, uint32_t env, uint64_t first, uint64_t n, uint8_t* side_is_bid, uint8_t* status,
              uint64_t* arr_time, uint64_t* end_time, uint32_t* vol, uint32_t* start_vol, uint32_t* price,
              uint32_t* trader);
/* PyTrade columns (rust/src/types.rs:4-17) */
int bb_trades(bb_handle* h, uint32_t env, uint64_t first, uint64_t n, uint64_t* t, uint8_t* side_is_bid,
              uint32_t* price, uint32_t* vol, uint64_t* active_id, uint64_t* passive_id);
/* Bulk export of EVERY env's order table / trade log in the device record layout (one strided copy each): what
 * sim_runner leaves in host memory on the reference (orderbook.rs:113-115).  out[n_envs][cap_per_env] records, row e holds
 * env e's first min(count, cap_per_env) records; counts[n_envs] = records the env has.  bb_order_rec.meta: bits 0-2 Status
 * (types.rs:51-75), bit 3 side is bid; `link` words are engine-private. */
typedef struct {
    uint32_t price, vol, link0, link1;
    uint64_t key_time;
    uint32_t meta, start_vol;
    uint64_t arr_time, end_time;
    uint32_t trader, pad[3];
} bb_order_rec; /* 64 bytes */
typedef struct {
    uint64_t t;
    uint32_t price, vol, active_id, passive_id, side_is_bid, pad;
} bb_trade_rec; /* 32 bytes */
int bb_orders_all(bb_handle* h, uint32_t cap_per_env, bb_order_rec* out, uint32_t* counts);
int bb_trades_all(bb_handle* h, uint32_t cap_per_env, bb_trade_rec* out, uint32_t* counts);
/* time component of each order's queue key (OrderEntry.key.2, orderbook.rs:36-44); 0 for orders that never rested */
int bb_order_keys(bb_handle* h, uint32_t env, uint64_t first, uint64_t n, uint64_t* key_time);
int bb_order_status(bb_handle* h, uint32_t env, uint64_t order_id, uint8_t* status);
int bb_time(bb_handle* h, uint32_t env, uint64_t* t);
int bb_set_time(bb_handle* h, uint32_t env, uint64_t t);
int bb_set_trading(bb_handle* h, uint32_t env /* or BB_ALL_ENVS */, int on);
/* Per-env STICKY error words (BB_ERR_* bits raised by any call since creation / bb_reset / bb_clear_errors).  A call reports
 * (through its return code) only the errors raised by that call: after a refused instruction — e.g. a cancel of an unknown
 * id, where the reference panics before mutating anything (orderbook.rs:642) — the handle stays usable. */
int bb_env_errors(bb_handle* h, uint32_t* out /* [n_envs] */);
int bb_clear_errors(bb_handle* h); /* zero every env's sticky error word; asynchronous */
int bb_stats(bb_handle* h, bb_stats_t* out);
/* Replaces `impl TryFrom<OrderBookState> for OrderBook` (orderbook.rs:891-918, the load half of the JSON
 * snapshot): overwrite env's book with the given order table and trade log, then rebuild both sides by
 * re-inserting every Active order under its stored key (side, price, key_time).  Column layout as in
 * bb_orders / bb_trades.  The env must have no queued instructions. */
int bb_load_book(bb_handle* h, uint32_t env, uint64_t t, uint32_t trade_vol, int trading, uint64_t n_orders,
                 const uint8_t* side_is_bid, const uint8_t* status, const uint64_t* arr_time, const uint64_t* end_time,
                 const uint32_t* vol, const uint32_t* start_vol, const uint32_t* price, const uint32_t* trader,
                 const uint64_t* key_time, uint64_t n_trades, const uint64_t* tr_t, const uint8_t* tr_side_is_bid,
                 const uint32_t* tr_price, const uint32_t* tr_vol, const uint64_t* tr_active, const uint64_t* tr_passive);
/* device pointer + strides of the history ring, for zero-copy consumers (DLPack at the Python edge) */
int bb_history_device(bb_handle* h, void** d_ptr, uint64_t* env_stride_words, uint32_t* obs_words);

/* ---- multi-GPU (SURVEY.md 8e) ------------------------------------------------------------------ */
/* Books share no state (crates/step_sim/src/env.rs:58-71: an Env owns its OrderBook, queue and records), so a job shards
 * its envs over GPUs — one bb_handle per device, contiguous blocks of global env ids (bb_config.env_id_base keeps the agent
 * RNG invariant to the sharding) — and runs them with NO per-step collective.  The one exchange is the end-of-run
 * all-gather of every shard's statistics, over NCCL (NVLink 5 / NVSwitch).  NCCL is loaded at run time (libnccl.so.2);
 * these calls fail with BB_ECUDA where it is absent, everything above works without it.
 *   one process per GPU (torchrun, MPI, ...): rank 0 calls bb_comm_unique_id, the host hands the 128 bytes to every rank
 *     by whatever means it has, each rank calls bb_comm_init_rank with its own device;
 *   one process driving several GPUs: bb_comm_init_all (ncclCommInitAll), rank i == devices[i]. */
typedef struct bb_comm bb_comm;
#define BB_COMM_ID_BYTES 128
int bb_comm_unique_id(unsigned char* out_id /* [BB_COMM_ID_BYTES] */);
int bb_comm_init_rank(const unsigned char* id, int n_ranks, int rank, int device, bb_comm** out);
int bb_comm_init_all(int n_dev, const int* devices /* NULL => 0..n_dev-1 */, bb_comm** out);
int bb_comm_n_ranks(const bb_comm* c);
int bb_comm_destroy(bb_comm* c);
const char* bb_comm_last_error(void);
/* bb_stats of every local shard, all-gathered: handles[n_local] = this process's handles in local-rank order (n_local == 1
 * after bb_comm_init_rank, == n_dev after bb_comm_init_all); elapsed_ms[n_local] (may be NULL) travels with the counters so
 * that the caller can take the max over ranks.  out_stats[n_ranks], out_elapsed_ms[n_ranks] (may be NULL), rank order. */
int bb_gather_stats(bb_comm* c, bb_handle* const* handles, uint32_t n_local, const double* elapsed_ms, bb_stats_t* out_stats,
                    double* out_elapsed_ms);

#ifdef __cplusplus
}
#endif
#endif /* BOURSE_B200_H */
