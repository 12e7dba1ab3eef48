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
typedef struct bb_store bb_store; /* device-resident book snapshots of a handle (bb_store_create) */

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
#define BB_ERR_ROW_OP 0x400u     /* bb_run_agents_with_rows(_market): a MODIFY row or a trader id >= 2^19 (row dropped); markets: a row's aux names no asset */
#define BB_ERR_LOCKED 0x800u     /* deep engine: both sides would rest at one price level (trading disabled) */
#define BB_ERR_SLOT 0x1000u      /* bb_restore_device: the slot was empty, out of range, or saved from a book of another tick */
#define BB_ERR_PARAMS 0x2000u    /* bb_set_agent_params_device: a unit's parameter row broke the declared population (row not applied) */

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
     * level (BB_ERR_LOCKED: only reachable while trading is disabled).  Env steps run through bb_step_device (device
     * rows; step_size >= max_queue keeps the time precondition, since event i of a step runs at start + i), and so do
     * in-kernel agents (bb_set_agents, bb_run_agents(_with_rows): every RandomAgents price must lie in the window); the
     * host-queued Env calls (bb_submit / bb_step) are not available on a deep handle (BB_EINVAL). */
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
    uint32_t aux;      /* bb_step_device_market: the row's asset; elsewhere reserved, 0 (the library keeps a market's
                          submission order here while instructions are queued) */
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
 * call this and step again; the Python StepEnv / StepEnvNumpy classes reserve ahead of need.  On a deep-book handle it
 * regrows the staging stream of bb_step_device (n_envs x (max_queue + 1) instructions), which always fits.  Synchronous. */
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
 * reports BB_EPRICE).  Only the first max_queue rows of an env's slice are submitted: the rows past them create and queue
 * nothing (BB_NO_ID) and the env is flagged BB_ERR_CAP_QUEUE.  d_obs_out (device, [n_envs][obs_words], may be NULL) receives every env's end-of-step
 * observation record from the same launch — what StepEnvNumpy.level_1_data / level_2_data would return next.
 * Asynchronous on the handle's stream: one kernel launch and no host synchronisation, so the call may be recorded into a
 * CUDA graph together with the caller's own kernels (stream capture on the stream given to bb_set_stream).
 * Deep-book handles (bb_config.deep_chunks) take the same rows with the same results, in two launches and with no
 * allocation: the first submits and shuffles each env's rows into a staging stream sized by max_queue, the second
 * replays it through the deep engine.  Its preconditions apply: a resting limit price outside the window flags
 * BB_ERR_CAP_PAGES, and BB_ERR_TIME_ORDER is flagged where resting orders of one step would reuse key times of an earlier
 * one, which step_size >= max_queue rules out. */
int bb_step_device(bb_handle* h, const bb_instr* d_instrs, const uint64_t* d_env_offsets, uint64_t n_rows, uint64_t* d_out_ids,
                   uint32_t* d_obs_out);
/* The same device-resident loop for multi-asset markets (bb_config.assets >= 2; no upper limit on assets here).  One call
 * does, for every market m, what MarketEnv::place_order / cancel_order / modify_order for each of the market's rows, in row
 * order, then one MarketEnv::step(rng) would do (crates/step_sim/src/market_env.rs:108-121, 163-219).
 * d_market_offsets[n_markets + 1] (device) delimits market m's slice of d_instrs; bb_instr::t is ignored and bb_instr::aux
 * is the row's asset (0 .. assets - 1).  BB_OP_NEW rows with an on-tick limit price or BB_F_MARKET create the next order id
 * of their asset's book (ids are per book, MarketOrderId = (asset, id), market.rs:270-280) in d_out_ids[row];
 * BB_OP_CANCEL / BB_OP_MODIFY rows target (aux, order_id); no-ops and unknown codes queue nothing.  A limit price off the
 * asset's own tick creates and queues nothing and flags that asset's book BB_ERR_PRICE; a row with aux >= assets queues
 * nothing and flags book 0 of its market BB_ERR_ROW_OP.  Every row that creates nothing gets BB_NO_ID.  The market's queue
 * is shuffled as a whole with the same Xoroshiro128** stream bb_step uses for it (seed + env_id_base / assets + m), event i
 * of the shuffled queue runs at start + i on its asset's book, and every book then advances by step_size and appends one
 * record.  A market with more than assets * max_queue rows flags BB_ERR_CAP_QUEUE on each of its books, applies none of
 * its rows and hands out no ids; its books still step.  On the dense engine BB_ERR_TIME_ORDER follows the rule of
 * bb_step for the same queue.  d_obs_out ([n_envs][obs_words], may be NULL) receives every book's end-of-step record;
 * book m * assets + a is asset a of market m.  In-kernel agents do not run.  bb_step and this call may be interleaved
 * freely on one handle.  Asynchronous: one kernel launch, no host synchronisation, and it may be recorded into a CUDA graph
 * on a freshly created or reset handle or after an earlier bb_step_device_market; right after a bb_step that shuffled,
 * capture is refused with BB_EINVAL (call it once outside the capture first).  Refused with BB_EINVAL on a single-asset
 * handle (use bb_step_device), on the deep engine, while host-queued instructions are pending, and for NULL arguments.
 * n_rows sizes the internal id buffer when d_out_ids is NULL. */
int bb_step_device_market(bb_handle* h, const bb_instr* d_instrs, const uint64_t* d_market_offsets, uint64_t n_rows,
                          uint64_t* d_out_ids, uint32_t* d_obs_out);
/* The same market loop with the built-in market agents (bb_set_agents_market) trading in every market: ONE step of
 * market_sim_runner (crates/step_sim/src/runner.rs:107-131) with the caller's calls between the agents' update and the
 * step — `agents.update(&mut env, rng); env.place_order(..) / env.cancel_order(..) for each row; env.step(rng)`
 * (market_env.rs:108-121, 163-219).  For every market m, in one launch:
 *   1. all agent groups update in array order, each on its own asset's book, with bb_run_agents' Philox key (seed; global
 *      market id (env_id_base + book) / assets, step, agent slot counted over all groups);
 *   2. the market's rows (d_market_offsets and bb_instr::aux as for bb_step_device_market) are submitted in row order:
 *      BB_OP_NEW with an on-tick limit price or BB_F_MARKET creates the next id of its asset's book (after the ids the
 *      agents took) in d_out_ids[row] (may be NULL); BB_OP_CANCEL targets (aux, order_id); no-ops queue nothing; every
 *      row that creates nothing gets BB_NO_ID;
 *   3. the market's queue — every group's instructions in array order, then the queued rows in row order — is shuffled
 *      as a whole with bb_run_agents' Philox-keyed Fisher-Yates, event i runs at start + i on its asset's book, and every
 *      book advances by step_size and appends one record; d_obs_out ([n_envs][obs_words], may be NULL) receives it.
 * Row errors are sticky per-book bits, and no row fails silently: a limit NEW off its asset's tick is dropped without
 * taking an id (BB_ERR_PRICE on that asset's book); a row with aux >= assets queues nothing (BB_ERR_ROW_OP on book 0 of
 * the market); a MODIFY row, or a NEW with a trader id >= 2^19, is dropped (the in-kernel queue carries NEW and CANCEL
 * only; BB_ERR_ROW_OP on the row's book); a cancel of an id its book has not issued by the end of submission flags
 * BB_ERR_BAD_ID on that book.  Queue capacity: a book whose own events (its groups' instructions plus its rows) exceed
 * max_queue is flagged BB_ERR_CAP_QUEUE and its results are unspecified; a market whose whole queue exceeds
 * assets * max_queue flags BB_ERR_CAP_QUEUE on every book and processes no event that step (ids are still taken and the
 * books still step).  Refused with BB_EINVAL on a single-asset handle (use bb_run_agents_with_rows), before
 * bb_set_agents_market, on the deep engine, while host-queued instructions are pending, for NULL arguments, and inside a
 * stream capture (as every agent launch).  Asynchronous on the handle's stream. */
int bb_run_agents_with_rows_market(bb_handle* h, uint64_t seed, const bb_instr* d_instrs, const uint64_t* d_market_offsets,
                                   uint64_t n_rows, uint64_t* d_out_ids, uint32_t* d_obs_out);
/* bb_level2 / bb_level1 into DEVICE memory: d_out[n_envs][45] / d_out[n_envs][9].  Asynchronous. */
int bb_level2_device(bb_handle* h, uint32_t* d_out);
int bb_level1_device(bb_handle* h, uint32_t* d_out);
/* Order records by id for a whole batch of device-resident queries: get_orders()[id] / order_status(id) of the reference
 * (rust/src/step_sim_numpy.rs, rust/src/types.rs:19-31) for every env at once.  A unit is an env on a single-asset handle and
 * a market on a multi-asset one; d_ids is [units][n_per_unit], the shape of the id block bb_step_device(_market) returns.
 * Query q of unit u reads book u, or book u * assets + d_assets[q] on a multi-asset handle (d_assets [units][n_per_unit];
 * it must be NULL on a single-asset handle and non-NULL on a multi-asset one).  Output q of every non-NULL column (each
 * [units][n_per_unit], columns as in bb_orders) is that order's field.  A BB_NO_ID query writes BB_STATUS_NONE and zeros
 * and flags nothing, so a padded block is legal input.  An id without a record (>= the book's order count, or >= max_orders
 * after BB_ERR_CAP_ORDERS) writes the same and flags BB_ERR_BAD_ID on its book (the reference panics); an asset >= assets
 * writes the same and flags BB_ERR_ROW_OP on book 0 of the market.  Those sticky bits are all the call changes.  Every
 * engine, deep included.  Refused with BB_EINVAL for a NULL d_ids, for more than 2^39 - 256 queries, and while host-queued
 * instructions are pending (their ids have no record yet).  Asynchronous on the handle's stream: one launch, no host synchronisation and no allocation,
 * so the call may be recorded into a CUDA graph.  Outputs are ordered after every earlier launch on the stream. */
#define BB_STATUS_NONE 0xFFu /* status written for a query that names no order */
int bb_orders_device(bb_handle* h, const uint64_t* d_ids, const uint32_t* d_assets, uint64_t n_per_unit, uint8_t* d_side_is_bid,
                     uint8_t* d_status, uint64_t* d_arr_time, uint64_t* d_end_time, uint32_t* d_vol, uint32_t* d_start_vol,
                     uint32_t* d_price, uint32_t* d_trader);
/* Per book, the trades logged since a caller-owned cursor: the entries get_trades() (rust/src/types.rs:4-17) gained since the
 * last read, for every book at once.  d_cursor[n_envs] (device) is read and written.  For book b, with
 * logged = min(trades, max_trades): d_count[b] = logged - d_cursor[b] (may exceed cap), the first min(count, cap) of those
 * trades go to row b of the [n_envs][cap] columns in log order, and d_cursor[b] advances by the number written, so a small
 * cap loses nothing: the rest come with the next call.  Unused slots of a row hold active_id = passive_id = BB_NO_ID and
 * zeros elsewhere, so the id columns can be passed straight to bb_orders_device (book b of a market handle is asset
 * b % assets of market b / assets).  A cursor at or past `logged` gives count 0 and is left as it is; after bb_reset the
 * caller zeroes its cursors.  Trades the full log could not hold are not reported (the book's BB_ERR_CAP_TRADES says they
 * happened); nothing past max_trades is read.  (A log that overflowed and was then grown with bb_reserve has no records in
 * the slots between its old capacity and its trade count: they read as whatever the slab holds there, as with bb_trades;
 * bb_reset before growing a log that overflowed.)  Ids are widened to u64 to compare directly with the vector loops' ids.
 * d_count and every column may be NULL.  Every engine, deep included; changes nothing but d_cursor and the outputs.
 * Refused with BB_EINVAL for a NULL d_cursor, while host-queued instructions are pending, and on a handle with
 * max_trades == 0.  Asynchronous on the handle's stream: one launch, no host synchronisation and no allocation, so the
 * call may be recorded into a CUDA graph. */
int bb_trades_device(bb_handle* h, uint32_t* d_cursor, uint32_t cap, uint32_t* d_count, uint64_t* d_t, uint8_t* d_side_is_bid,
                     uint32_t* d_price, uint32_t* d_vol, uint64_t* d_active_id, uint64_t* d_passive_id);
/* Per-unit reset for the device-resident loops: end the episodes of some envs (a unit is an env on a single-asset handle and
 * a market of `assets` books on a multi-asset one, as in bb_orders_device) while the others keep running — gymnasium's
 * per-env autoreset, with the done mask computed on the device.  All pointers are device pointers.
 *   d_mask [units] (required): a non-zero entry resets the unit.  Every book of a reset unit returns to what bb_reset makes
 *     it: an empty book at start_time with the config's trading flag; order count, trade log and history count at 0; sticky
 *     error word and header counters zeroed; its in-kernel agents' state cleared (RandomAgents held ids, MomentumAgent /
 *     NoiseAgent state and live lists).  It keeps its tick size, the agent groups and all else bb_reset keeps.  So a
 *     book's order table and trade log start again from slot 0: each env recycles max_orders / max_trades at its own
 *     episode boundary.  Books of units whose entry is 0 are not touched.
 *   d_seeds [units] or NULL: the unit's random streams.  NULL: they continue — the Xoroshiro128** shuffle state and the
 *     step counter (the `step` word of every agent's Philox draw) keep their values, so the next episode draws the shuffles
 *     and agent draws the unit would have drawn without the reset.  Non-NULL: the unit's shuffle stream becomes
 *     Xoroshiro128StarStar::seed_from_u64(d_seeds[u]) (every book of a market gets the market's stream) and its step
 *     counter restarts at 0.  A unit re-seeded with its creation seed (seed + env_id_base + e; markets
 *     seed + env_id_base / assets + m) is therefore bit-identical from then on to that unit of a freshly created handle.
 *     The agents' Philox key is (launch seed, global env / market id, step): a seeded reset replays the creation-time agent
 *     draws as well, fresh agent draws come from an unseeded reset (or a new launch seed).
 *   d_obs_out [n_envs][obs_words] or NULL: the rows of reset books receive the fresh book's record, what bb_level1_device /
 *     bb_level2_device return for them right after the reset; other rows are not written.
 *   d_cursor [n_envs] or NULL: a bb_trades_device cursor array; the entries of reset books are zeroed, so the next read
 *     reports the new episode's trades from log index 0.
 * Order ids a caller holds for a reset book are void: a later CANCEL of one flags BB_ERR_BAD_ID as any unknown id does.
 * bb_stats counts from the reset on for reset books (their counters restart at 0); its env_steps is the sum of the step
 * counters, so it keeps an unseeded unit's steps and drops a seeded unit's.  bb_n_steps of a reset book is 0, so the envs'
 * history counts differ afterwards: bb_run_agents_to_host, which streams every env's records from one common index, needs
 * a bb_clear_history first.
 * On a multi-asset handle right after a bb_step that shuffled, a seeded reset first copies the host's streams of the
 * markets to the books (synchronous); inside a stream capture that case is refused with BB_EINVAL.  An unseeded reset
 * leaves every market's stream where it is.  Every engine: paged, dense and deep (the deep engine has no shuffle or agents:
 * only d_mask, d_obs_out and d_cursor matter there).  Refused with BB_EINVAL, the handle unchanged, for a NULL handle or
 * d_mask, while host-queued instructions are pending, and in the capture case above.  Asynchronous on the handle's stream:
 * one launch, no host synchronisation and no allocation, so the call may be recorded into a CUDA graph with the steps. */
int bb_reset_device(bb_handle* h, const uint8_t* d_mask, const uint64_t* d_seeds, uint32_t* d_obs_out, uint32_t* d_cursor);
/* Device-resident book snapshots for the vector loops: save the full state of some units into the slots of a device store,
 * and restore any units from any slots (one slot into many units included) — episodes that start from a warm book,
 * branching rollouts, replays from a midpoint.  A unit is an env, or a market of `assets` books on a multi-asset handle, as
 * in bb_reset_device; a slot holds one unit.
 *
 * bb_store_create: a store of n_slots slots, sized from the handle's current capacities; every slot starts empty.
 *   *out_bytes (may be NULL) receives its size in bytes; with out == NULL the call only reports that size and allocates
 *   nothing.  An allocation failure returns BB_ECUDA with the size in the message.  The store belongs to the handle:
 *   bb_destroy frees every store not yet destroyed (its pointer is then invalid).
 * bb_store_destroy: frees a store (synchronises the handle's stream).  NULL is a no-op.
 *
 * What a slot holds, per book: the blob (header, page directory and pages; the dense window; or the deep image), the order
 * table prefix [0, min(n_orders, max_orders)), the trade log prefix [0, min(n_trades, max_trades)), the in-kernel agents'
 * state of the book (RandomAgents held ids, MomentumAgent / NoiseAgent state and live lists), on the deep engine the chunk
 * pool prefix up to its allocator's bump, and the book's tick.  The per-step history is not saved.
 *
 * bb_save_device: d_units [n_slots] (device): slot k receives unit d_units[k]; BB_NO_SLOT leaves slot k as it is, and a
 *   unit index >= units marks slot k empty.  The handle is not changed.
 * bb_restore_device: d_slots [units] (device): unit u takes the state of slot d_slots[u]; BB_NO_SLOT leaves the unit
 *   untouched; many units may name one slot.  A restored book is the saved book — book, order table, trade log, time,
 *   trading flag, sticky error word, header counters and agent state — with a history count (bb_n_steps) of 0.
 *   d_seeds [units] or NULL: NULL gives the book the slot's Xoroshiro128** shuffle state and Philox step counter, so a unit
 *   restored from its own saved state continues bit-identically under the same actions (agent draws are keyed by the global
 *   env / market id as well: another unit restored from that slot draws other agent instructions; rows-only units restored
 *   from one slot continue identically).  Non-NULL: the unit's shuffle stream becomes
 *   Xoroshiro128StarStar::seed_from_u64(d_seeds[u]), as bb_reset_device seeds it; the step counter is the slot's.
 *   d_obs_out [n_envs][obs_words] or NULL: the rows of restored books receive what bb_level1_device / bb_level2_device
 *   return for them right after the restore (a second launch); other rows are not written.
 *   d_cursor [n_envs] or NULL: a bb_trades_device cursor; the entries of restored books are set to the restored log's
 *   logged count, so the next read reports only trades made after the restore.
 *   A unit that names a slot >= n_slots, an empty slot, or a slot whose saved tick differs from that of the book it would
 *   restore (checked per book, so per-env ticks work) is left untouched and each of its books is flagged BB_ERR_SLOT; all
 *   books of a market share the outcome.  Order ids a caller holds for a restored book now name the slot's orders.
 *
 * Both calls work on every engine; on the deep engine a unit is a book, and d_seeds re-seeds the stream its
 * bb_step_device steps shuffle with.  On a multi-asset handle
 * right after a bb_step that shuffled, both first copy the host's streams of the markets to the books (synchronous), which
 * is refused inside a stream capture.  Refused with BB_EINVAL, the handle and the store unchanged, for NULL arguments, a
 * store created by another handle, a store created before a later bb_reserve that grew a capacity or a later
 * bb_set_agents / bb_set_agents_market / bb_set_tick_sizes, while host-queued instructions are pending, and in the
 * capture case above.  Asynchronous on the handle's stream, with no host synchronisation and no allocation, so both may be
 * recorded into a CUDA graph with the steps. */
#define BB_NO_SLOT 0xFFFFFFFFu
int bb_store_create(bb_handle* h, uint32_t n_slots, bb_store** out, uint64_t* out_bytes);
int bb_store_destroy(bb_store* s);
int bb_save_device(bb_handle* h, bb_store* s, const uint32_t* d_units);
int bb_restore_device(bb_handle* h, bb_store* s, const uint32_t* d_slots, const uint64_t* d_seeds, uint32_t* d_obs_out,
                      uint32_t* d_cursor);
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
/* Defines the agent set (resets agent state).  Groups run in array order.  On a deep-book handle (bb_config.deep_chunks) the
 * prices of every RandomAgents group, [tick_lo * tick_size, (tick_hi - 1) * tick_size], must lie in the window
 * [win_lo, win_lo + win_levels): otherwise BB_EINVAL and the previous population stays.  MomentumAgent / NoiseAgent quotes
 * follow the book and cannot be bounded up front; one that would rest outside the window flags BB_ERR_CAP_PAGES. */
int bb_set_agents(bb_handle* h, const bb_agent_group* groups, uint32_t n_groups);
/* Multi-asset handles (bb_config.assets = 2..4): the *Market twins of the built-in agents — RandomMarketAgents
 * (crates/step_sim/src/agents/random_agent.rs:165-247), MomentumMarketAgent (momentum_agent.rs:282-409),
 * NoiseMarketAgent (noise_agent.rs:226-345) — as fields of a #[derive(MarketAgentSet)] struct: group i is the same
 * bb_agent_group as above and trades asset asset[i] of every market.  bb_run_agents then runs market_sim_runner
 * (crates/step_sim/src/runner.rs:107-131): all groups update in array order, the market's queue is shuffled as a
 * whole and event i executes at start + i on its asset's book (market_env.rs:108-121).  The RNG unit is the market:
 * Philox key (seed; global market id = (env_id_base + env) / assets, step, agent slot counted over all groups). */
int bb_set_agents_market(bb_handle* h, const bb_agent_group* groups, const uint32_t* asset, uint32_t n_groups);
/* Per-unit agent parameters and Philox keys for the population bb_set_agents / bb_set_agents_market declared.  A unit is an
 * env, or a market on a multi-asset handle.  Every unit whose d_mask byte is non-zero (d_mask NULL: every unit) takes its row
 * d_params[u][0 .. n_groups) and / or its key d_keys[u]; d_params NULL keeps the units' records, d_keys NULL their keys.
 * From then on every agent launch of the handle (bb_run_agents, bb_run_agents_to_host, bb_run_agents_with_rows(_market))
 * runs group gi of unit u with record d_params[u][gi], and draws with key seed ^ key[u] (a 64-bit XOR): every RandomAgents,
 * MomentumAgent and NoiseAgent draw and the step's shuffle.  Unit u with key k draws what it would draw with seed ^ k;
 * keys start at 0.  The shuffle streams that bb_reset_device re-seeds (device-row steps, bb_step) are not affected.
 *   The declared population is the envelope: what bb_set_agents sized from the groups (agent state, trader ids, live
 * lists, the dense window) stays valid.  A record r for group gi, declared as d, is valid only if r.kind, r.n_agents and
 * r.tick_size equal d's and
 *   - RandomAgents: d.tick_lo <= r.tick_lo < r.tick_hi <= d.tick_hi and d.vol_lo <= r.vol_lo < r.vol_hi <= d.vol_hi; rate free;
 *   - MomentumAgent / NoiseAgent: r.tick_lo == d.tick_lo (agent_id_start) and r.vol_hi == d.vol_hi (live-list capacity);
 *     rate, vol_lo (trade_vol), decay, demand, scale, order_ratio, mu and sigma free.
 * Validation happens on the device: a unit with any invalid record changes nothing, its key included, and every book of it
 * is flagged BB_ERR_PARAMS; the other units are applied.
 *   Lifetime: the first call allocates [units][n_groups] records and [units] keys, filled from the declared groups and zero
 * keys, then applies the call.  bb_set_agents(_market) drops both (shared parameters and zero keys again); bb_reset,
 * bb_reset_device and bb_restore_device keep them (they are configuration, not state: store slots do not hold them);
 * bb_destroy frees them.  With the tables, agent launches run variants that read each unit's row from memory.
 *   One launch on the handle's stream, no host synchronisation (the first call also allocates).  BB_EINVAL, handle
 * unchanged: no population, or d_params and d_keys both NULL. */
int bb_set_agent_params_device(bb_handle* h, const bb_agent_group* d_params /* [units][n_groups] or NULL */,
                               const uint64_t* d_keys /* [units] or NULL */, const uint8_t* d_mask /* [units] or NULL = all */);
/* n_steps of { agents.update(env); env.step() } for every env inside one persistent kernel.
 * Draws are Philox4x32-10 keyed (seed; global env id, step, agent) — DESIGN.md "RNG contract".
 * Asynchronous on the handle's stream; pair with bb_synchronize or any read call.
 * Deep-book handles run the same steps with the same results in two launches per step: the first runs the agents'
 * updates, submits the rows (bb_run_agents_with_rows) and shuffles each book's queue into the staging stream, the second
 * replays it through the deep engine.  Their preconditions apply as for bb_step_device (step_size >= max_queue; a resting
 * price outside the window flags BB_ERR_CAP_PAGES), and max_queue is limited to 57856 there (BB_ECAP). */
int bb_run_agents(bb_handle* h, uint64_t seed, uint32_t n_steps);
/* ONE env-step of { agents.update(env); <the caller's rows>; env.step() } with the rows already in DEVICE memory: the loop of a
 * learning agent trading against the built-in background agents (SURVEY.md 8f rank 4).  Rows are laid out as for
 * bb_step_device and submitted after the agents' updates, in row order: BB_OP_NEW (ids in d_out_ids, BB_NO_ID elsewhere;
 * may be NULL) and BB_OP_CANCEL; no-op rows queue nothing; BB_OP_MODIFY rows, and BB_OP_NEW rows whose trader id is >= 2^19,
 * are dropped (BB_NO_ID, no id taken) and flag the env BB_ERR_ROW_OP.  Everything
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
