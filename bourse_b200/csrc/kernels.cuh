// Kernels of the batched simulator (sm_100a).  One warp owns one book for the whole launch; a CTA is
// just `WPB` independent warps sharing an SM's shared memory, so there is no __syncthreads anywhere.
//
//   k_apply<MODE_REPLAY>  immediate-mode instruction streams (OrderBook API, config C2)
//                         reference: orderbook.rs:411-421, 583-792 driven at explicit times
//   k_apply<MODE_ENV>     Env::step over host-queued instructions (crates/step_sim/src/env.rs:116-135)
//   k_apply<MODE_ENV_MKT> MarketEnv::step over device-resident rows, one slice per market (market_env.rs:108-121)
//   k_sim                 persistent { agents.update; env.step } x n_steps (runner.rs:46-69) with the
//                         built-in RandomAgents / MomentumAgent generated in-kernel
//   k_snapshot            live level-1 / level-2 / touch data of every book (orderbook.rs:287-324)
//   k_orders_gather       order records by id for a batch of queries (bb_orders_device)
//   k_trades_window       each book's trades since a caller-owned cursor (bb_trades_device)
#pragma once
#include "../../include/bourse_b200.h"
#include "book.cuh"
#include "philox.cuh"
#include "tma.cuh"
#include "deep.cuh"

namespace bb {

#define MODE_REPLAY 0
#define MODE_ENV 1
#define MODE_ENV_MKT 2  // bb_step_device_market: MarketEnv::step over device-resident rows, one slice per market
#define MAX_GROUPS 8
#define LIVE_CAP 254  // default capacity of a MomentumAgent / NoiseAgent live-order list (per group per env)
// env-steps of observation records staged in shared memory per bulk store: 8 level-1 records (288 B) or 4 level-2
// records (720 B); both are multiples of 16 bytes and keep the staging area under 1.5 KB per book
#define OBS_STAGE_STEPS(obs_words) ((obs_words) > 9u ? 4u : 8u)

// The reference keeps the ids of a MomentumAgent's resting limit orders in a Vec (momentum_agent.rs:99-102, common.rs:56-75).
// Here the list is an array of KParams::mom_live_cap entries (the largest capacity any group of the population asked for,
// bb_agent_group::vol_hi; 254 by default) behind a 24-byte header; records are KParams::mom_stride bytes apart.
struct MomState {
    double momentum, last_price;
    u32 has_last, n_live;
    u32 live[2];  // [mom_live_cap]
};
#define MOM_HDR_BYTES 24u
static_assert(sizeof(MomState) == MOM_HDR_BYTES + 8, "MomState layout");

struct KParams {
    unsigned char* blobs;
    u64 blob_stride;
    OrderRec* ord;
    TradeRec* tr;
    u32* hist;
    u32* err_flag;
    u64 step_size;
    u64 hist_env_stride;  // words
    u32 blob_smem_bytes;
    u32 n_envs, env_id_base;
    Geo geo;  // p_total, p_smem, granule, max_orders, max_trades, per-env ticks
    u32 max_steps, max_queue, obs_words;
    u32 warp_smem_bytes, off_perm, off_obs, off_instr, off_bar, off_q, off_ag;
    // k_apply
    const bb_instr* instrs;
    const u64* offsets;
    u32 n_steps;
    u32 host_order;  // MODE_ENV: instructions arrive in processing order with their time offset in bb_instr::t (markets)
    // MODE_ENV, bb_step_device: rows come straight from the caller's device buffer — ids are assigned here in row order
    // (create_order at submission, env.rs:173), rows that queue nothing (no-ops, tick errors) are left out of the shuffle
    u32 assign_ids;
    u64* out_ids;    // [total rows]: the id each row created, BB_NO_ID for rows that create nothing
    u32* obs_out;    // [n_envs][obs_words] or null: the step's observation record, also written here (bb_step_device)
    // k_sim
    u32 n_groups, agents_per_env, mom_groups_per_env;
    u32 mom_stride, mom_live_cap;  // bytes between MomState records; entries in each live list
    u32 chip_agents;  // dense engine: capacity of the on-chip agent tables (agents_per_env; markets: the largest per-asset count)
    u32* rslot;
    MomState* mom;
    uint4* scratch;  // [resident warps][max_queue]
    u32 seed_lo, seed_hi;
    bb_agent_group groups[MAX_GROUPS];
    // k_sim<.., MKT = true>: multi-asset markets with in-kernel agents (bb_set_agents_market)
    u32 assets;                   // books per market; the market's books are consecutive warps of one CTA
    u32 off_mkt;                  // per-warp offset of the market's shared words (used in the market's first warp only)
    u32 group_asset[MAX_GROUPS];  // asset each agent group trades
    // k_deep (deep.cuh): shared-memory offsets, chunk pools [n_envs][dp_chunks] x 256 B
    DeepOff dp;
    unsigned char* dp_pool;
    u32 dp_chunks;
    u32 dp_fast;  // k_deepw: 1 = batch-parallel passes enabled (0: every event through the serial path; debugging)
    // k_sim, bit gi: RandomAgents group gi trades a book whose tick does not divide the group's tick_size, so the queued
    // prices are checked against the book's tick (the host derives it from the groups and the tick table).  Last, so that
    // the other kernels' parameter offsets stay where they were
    u32 rand_tick_mask;
    // k_sim<.., PU = true> (bb_set_agent_params_device): each unit's own group records, [units][n_groups], read in place of
    // `groups`, and its Philox key, [units], XORed into (seed_lo, seed_hi) for every draw of the unit.  After
    // rand_tick_mask for the same reason
    const bb_agent_group* unit_groups;
    const u64* unit_keys;
};

// Values the optimiser would otherwise rematerialise at every use (S2R for the lane id, cvta + multiply
// for the shared base, a 64-bit multiply-add for the order slab) are passed through an opaque move so they
// stay in registers: profiles/r01_v4 showed ~35 warp instructions per event spent recomputing them.
__device__ __forceinline__ u32 keep32(u32 v) {
    u32 r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
    return r;
}
__device__ __forceinline__ u64 keep64(u64 v) {
    u64 r;
    asm volatile("mov.u64 %0, %1;" : "=l"(r) : "l"(v));
    return r;
}

// page lookup cache of the generic paged geometry: every entry must name a valid slot (0 is always one)
template <class G> __device__ __forceinline__ void pcache_init(const G& g, u32 sb, u32 lane) {
    if constexpr (!G::FAST && !G::DENSE) {
        sts(sb + g.pc_off + 4u * lane, 0u);
        __syncwarp();
    }
}

__device__ __forceinline__ void make_book(Book& b, const KParams& p, u32 sb, u32 env, u32 lane) {
    b.sb = sb;
    b.tag_lane = keep32(sb + 128u + 4u * lane);
    b.oh = keep64((u64)(p.ord + (size_t)env * p.geo.max_orders));
    b.env = env;
    b.blob = keep64((u64)(p.blobs + (size_t)env * p.blob_stride));
    b.lane = lane;
}

// bulk-load the shared-memory image of a book (header, page directory, resident pages)
__device__ __forceinline__ bool blob_load(const KParams& p, u32 sb, u32 env, u32 bar, u32& phase, u32 lane) {
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        mbar_expect_tx_a(bar, p.blob_smem_bytes);
        bulk_g2s_a(sb, p.blobs + (size_t)env * p.blob_stride, p.blob_smem_bytes, bar);
    }
    const bool ok = mbar_wait_a(bar, phase);
    phase ^= 1u;
    return ok;
}
__device__ __forceinline__ void blob_store(const KParams& p, u32 sb, u32 env, u32 lane) {
    __syncwarp();
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        bulk_s2g_a(p.blobs + (size_t)env * p.blob_stride, sb, p.blob_smem_bytes);
        bulk_commit();
        bulk_wait_all<0>();
    }
    __syncwarp();
}

// append one observation record to the env's history (Level2DataRecords::append_record, data.rs:44-56)
template <class G> __device__ __forceinline__ void emit_obs_direct(const G& g, Book& b, const KParams& p, u32 env) {
    u32 w0, w1;
    book_obs(g, b, p.obs_words, &w0, &w1);
    if (p.obs_out) {  // the caller's device buffer gets the record too: one launch per vectorised step, no snapshot pass
        u32* o = p.obs_out + (size_t)env * p.obs_words;
        if (b.lane < p.obs_words) o[b.lane] = w0;
        if (b.lane + 32u < p.obs_words) o[b.lane + 32u] = w1;
    }
    const u32 n = lds(b.sb + HDR_NSTEPS);
    __syncwarp();  // every lane has read the count before lane 0 bumps it
    if (n < p.max_steps) {
        const u64 dst = (u64)(p.hist + (size_t)env * p.hist_env_stride + (size_t)n * p.obs_words);
        if (b.lane < p.obs_words) stg32(dst + 4u * b.lane, w0);
        if (b.lane + 32u < p.obs_words) stg32(dst + 4u * (b.lane + 32u), w1);
        if (b.lane == 0u) sts(b.sb + HDR_NSTEPS, n + 1);
    } else {
        b.err |= ERR_CAP_STEPS;
    }
    __syncwarp();
}

// one decoded instruction against the book (process_event, orderbook.rs:782-792)
template <bool CT, class G> __device__ __forceinline__ void apply_instr(const G& g, Book& b, u32 op_flags, u32 order_id, u32 price,
                                                                        u32 vol, u32 trader, u64 t, bool assign_id) {
    const u32 op = op_flags & BB_OP_MASK;
    if (op == BB_OP_SET_TRADING) {
        b.flags = vol ? (b.flags | FL_TRADING) : (b.flags & ~FL_TRADING);
        return;
    }
    if (op == BB_OP_RESTORE) {
        if constexpr (G::DENSE) {
            d_restore(g, b, order_id);
            return;
        }
        // bb_load_book: the record is already in HBM; an Active order goes back on its side under its stored key
        // (BTreeMap re-insertion of orderbook.rs:898-905, equal keys overwrite as on the reference)
        const u64 ra = b.oh + (u64)order_id * ORD_STRIDE;
        const uint4 a = ldg128(ra), c = ldg128(ra + 16u);
        if (order_id + 1 > b.n_orders) b.n_orders = order_id + 1;
        if ((c.z & META_STATUS_MASK) == ST_ACTIVE) {
            u32 prev, next;
            const u64 kt = ((u64)c.y << 32) | c.x;
            book_insert(g, b, (c.z & META_BID) ? 1u : 0u, a.x, kt, order_id, a.y, &prev, &next);
            stg32(ra + OH_NEXT, next);
            stg32(ra + OH_PREV, prev);
            stg32(ra + OH_META, c.z & ~META_GHOST);
        }
        return;
    }
    if (op < BB_OP_NEW || op > BB_OP_MODIFY) return;
    b.d_instr += 1;
    if (op == BB_OP_NEW) {
        const u32 side = (op_flags & BB_F_BID) ? 1u : 0u;
        if (op_flags & BB_F_MARKET) price = side ? 0xFFFFFFFFu : 0u;  // types.rs:160-172, 213-225
        u32 id = order_id;
        if (assign_id) {
            id = b.n_orders;
            b.n_orders = id + 1;
        }
        // two inlined copies, each constant-folded for its side (no per-use `side ? bid : ask` selects)
        if (side) book_apply<true, CT>(g, b, EV_NEW, id, 1u, price, vol, trader, false, false, t);
        else book_apply<true, CT>(g, b, EV_NEW, id, 0u, price, vol, trader, false, false, t);
    } else {
        // BB_OP_CANCEL / MODIFY == EV_CANCEL / EV_MODIFY
        book_apply<false, CT>(g, b, op, order_id, 0u, price, vol, trader, (op_flags & BB_F_HAS_PRICE) != 0,
                          (op_flags & BB_F_HAS_VOL) != 0, t);
    }
}

// Submission of a caller's device-resident rows: what Env / MarketEnv::place_order, cancel_order and modify_order do
// (env.rs:173, market_env.rs:163-219), warp-wide in row order over the slice p.instrs[off, off + m), for book `b`.  Only
// the first n_acc rows are submitted; the others create, queue and flag nothing (each kernel keeps its own queue-capacity
// policy).  A NEW row takes the next id of its book; a limit price off the tick of the row's book is create_order's
// PriceError (orderbook.rs:367-383): nothing is created or queued and the book is flagged ERR_PRICE.  Every row gets its id,
// or BB_NO_ID, in out_ids from the book it belongs to.
//   MKT   the slice is a market's and bb_instr::aux the row's asset; b is asset mk_a of the market.  Every book walks the
//         whole slice.  Rows naming no asset of the market queue nothing and flag book 0, which writes their ids.
//   SIMQ  k_sim's queue carries NEW and CANCEL only: a MODIFY row, or a NEW whose trader id does not fit 19 bits, is dropped
//         with ERR_ROW_OP.  A cancel of an id its book has not issued by the end of submission is the reference's panic
//         (orderbook.rs:642): ERR_BAD_ID.  Without SIMQ (k_apply) MODIFY rows are queued and each new id's order record is
//         published with status New, as create_order does at submission.
// c.next is the book's next id, c.n counts this book's queued rows, c.n_mkt (MKT) the market's.  Every queued row is handed
// to sink(j, x, y, mine, is_new, id, pos, pos_mkt): the row's two 16-byte halves, whether it is this book's, whether it took
// id `id` of this book, and its positions among this book's and the market's queued rows.
struct RowCount {
    u32 next, n, n_mkt;
};
template <bool MKT, bool SIMQ, class G, class Sink>
__device__ __forceinline__ void submit_rows(const G& g, const KParams& p, Book& b, u64 off, u32 m, u32 n_acc, u32 mk_a, RowCount& c,
                                            Sink sink) {
    const bb_instr* ins = p.instrs + off;
    const u32 book0 = b.env - mk_a, tick = MKT ? 0u : __ldg(g.ticks + book0), below = (1u << b.lane) - 1u;
    u32 max_cancel = 0;  // SIMQ: 1 + the largest id a cancel row of this book names
    for (u32 j0 = 0; j0 < n_acc; j0 += 32) {
        const u32 j = j0 + b.lane;
        // x: (t), op_flags, order_id; y: price, vol, trader, aux — loaded field by field, so that a caller that needs only
        // some of them (k_apply: op_flags, price, aux) loads only those
        uint4 x = make_uint4(0u, 0u, 0u, 0u), y = x;
        if (j < n_acc) {
            x.z = ins[j].op_flags;
            x.w = ins[j].order_id;
            y = make_uint4(ins[j].price, ins[j].vol, ins[j].trader, ins[j].aux);
        }
        const u32 op = x.z & BB_OP_MASK, asset = MKT ? y.w : 0u;
        const bool ok = !MKT || asset < p.assets;  // (a lane past the slice holds a no-op row)
        const bool own = !MKT || (ok ? asset == mk_a : mk_a == 0u);
        const bool bad_tick = ok && op == BB_OP_NEW && !(x.z & BB_F_MARKET) && (y.x % (MKT ? __ldg(g.ticks + book0 + asset) : tick) != 0u);
        const bool bad_op = SIMQ && ok && (op == BB_OP_MODIFY || (op == BB_OP_NEW && y.z >= (1u << 19)));
        const bool is_new = ok && op == BB_OP_NEW && !bad_tick && !bad_op;
        const bool queued = is_new || (ok && (op == BB_OP_CANCEL || (!SIMQ && op == BB_OP_MODIFY)));
        const u32 nm = __ballot_sync(BB_FULL, is_new && own), om = __ballot_sync(BB_FULL, queued && own);
        const u32 qm = MKT ? __ballot_sync(BB_FULL, queued) : om;
        const u32 id = c.next + __popc(nm & below), pos = c.n + __popc(om & below);
        if (j < n_acc && own) {
            p.out_ids[off + j] = is_new ? (u64)id : BB_NO_ID;
            if (!SIMQ && is_new && id < g.max_orders) stg32(b.oh + (u64)id * ORD_STRIDE + OH_META, ST_NEW | ((x.z & BB_F_BID) ? META_BID : 0u));
        }
        if (queued) sink(j, x, y, own, is_new && own, id, pos, MKT ? c.n_mkt + __popc(qm & below) : pos);
        if (SIMQ && own && ok && op == BB_OP_CANCEL) max_cancel = max(max_cancel, x.w == 0xFFFFFFFFu ? x.w : x.w + 1u);
        if (__any_sync(BB_FULL, bad_tick && own)) b.err |= ERR_PRICE;
        if ((MKT || SIMQ) && __any_sync(BB_FULL, (bad_op && own) || (MKT && !ok && mk_a == 0u))) b.err |= ERR_ROW_OP;
        c.next += __popc(nm);
        c.n += __popc(om);
        if (MKT) c.n_mkt += __popc(qm);
    }
    if (SIMQ && __reduce_max_sync(BB_FULL, max_cancel) > c.next) b.err |= ERR_BAD_ID;
#pragma unroll 1
    for (u32 j = n_acc + b.lane; j < m; j += 32) {  // (kept rolled: it runs only for a slice over the cap)
        const u32 asset = MKT ? ins[j].aux : 0u;
        if (!MKT || (asset < p.assets ? asset == mk_a : mk_a == 0u)) p.out_ids[off + j] = BB_NO_ID;
    }
}

// the generic paged geometry is shared-memory limited to <= 5 CTAs per SM anyway: give it the registers
template <int MODE, int ENG> __global__ void __launch_bounds__(128, (ENG == ENG_PAGED || ENG == ENG_PAGED_RES) ? 5 : 7) k_apply(const __grid_constant__ KParams p) {
    typedef GeoT<ENG> G;
    extern __shared__ __align__(128) unsigned char smem[];
    const u32 lane = keep32(threadIdx.x & 31u), warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const u32 sb = keep32(smem_u32(smem) + warp * p.warp_smem_bytes);
    const u32 bar = sb + p.off_bar;      // three 8-byte mbarriers
    const u32 perm = sb + p.off_perm;    // u16 [max_queue]
    const u32 chunk = sb + p.off_instr;  // two 1 KB instruction batches
    const GeoT<ENG>& g = static_cast<const GeoT<ENG>&>(p.geo);
    if (lane == 0) {
        mbar_init_a(bar, 1);
        mbar_init_a(bar + 8u, 1);
        mbar_init_a(bar + 16u, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_proxy_async();
    __syncwarp();
    u32 ph_blob = 0, ph_c0 = 0, ph_c1 = 0;
    pcache_init(g, sb, lane);

    for (u32 env = blockIdx.x * wpb + warp; env < p.n_envs; env += gridDim.x * wpb) {
        Book b;
        make_book(b, p, sb, env, lane);
        if (lane == 0) prefetch_l1((u64)(g.ticks + env));  // the tick is read at the row checks and level-2 records
        if (!blob_load(p, sb, env, bar, ph_blob, lane)) {
            if (lane == 0) atomicOr(p.err_flag, 0x80000000u);
            return;
        }
        book_from_header(g, b);
        // MODE_ENV_MKT: the offsets delimit markets; this book is asset mk_a of market env / assets
        constexpr bool MK = MODE == MODE_ENV_MKT;
        const u32 mk_a = MK ? env % p.assets : 0u;
        const u32 slice = MK ? env / p.assets : env;
        const u64 off = p.offsets[slice];
        const u32 n = (u32)(p.offsets[slice + 1] - off);
        const bb_instr* ins = p.instrs + off;

        if (MODE == MODE_REPLAY) {
            // stream the env's instruction slice through two 1 KB shared-memory batches with bulk copies
            auto issue = [&](u32 i0, u32 buf) {
                const u32 cnt = min(32u, n - i0);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    mbar_expect_tx_a(bar + 8u + 8u * buf, cnt * 32u);
                    bulk_g2s_a(chunk + buf * 1024u, ins + i0, cnt * 32u, bar + 8u + 8u * buf);
                }
            };
            if (n) issue(0, 0);
            for (u32 i0 = 0, buf = 0; i0 < n; i0 += 32, buf ^= 1u) {
                if (i0 + 32 < n) issue(i0 + 32, buf ^ 1u);
                u32& ph = buf ? ph_c1 : ph_c0;
                if (!mbar_wait_a(bar + 8u + 8u * buf, ph)) {
                    if (lane == 0) atomicOr(p.err_flag, 0x80000000u);
                    return;
                }
                ph ^= 1u;
                const u32 cnt = min(32u, n - i0);
                if constexpr (!G::DENSE) {
                    // one lane per instruction of the batch: start pulling the order record a cancel / modify targets
                    // towards L2 now, so that its DRAM latency overlaps the events queued ahead of it
                    if (lane < cnt) {
                        const u64 w = lds64(chunk + buf * 1024u + 32u * lane + 8u);  // op_flags | order_id << 32
                        const u32 op = (u32)w & BB_OP_MASK, tid = (u32)(w >> 32);
                        if ((op == BB_OP_CANCEL || op == BB_OP_MODIFY) && tid < g.max_orders) prefetch_l2(b.oh + (u64)tid * ORD_STRIDE);
                    }
                }
                for (u32 k = 0; k < cnt; ++k) {
                    const uint4 x = lds128(chunk + buf * 1024u + 32u * k), y = lds128(chunk + buf * 1024u + 32u * k + 16u);
                    const u64 t = ((u64)x.y << 32) | x.x;
                    b.t = t;
                    apply_instr<true>(g, b, x.z, x.w, y.x, y.y, y.z, t, true);
                    if (x.z & BB_F_EMIT) emit_obs_direct(g, b, p, env);
                }
                __syncwarp();
            }
        } else {
            for (u32 s = 0; s < p.n_steps; ++s) {
                const u64 start = b.t;
                b.trade_vol = 0;  // env.rs:117-118
                const u32 m = (s == 0) ? n : 0u;
                u32 nv;  // transactions in the queue
                // device-submitted rows (bb_step_device, bb_step_device_market): the queue is a permutation of row indices
                // (a market's: every book keeps the whole market's queue)
                auto to_perm = [&](u32 j, uint4, uint4, bool, bool, u32, u32, u32 pos_mkt) { sts16(perm + 2u * pos_mkt, j); };
                if constexpr (MK) {
                    const bool drop = m > p.assets * p.max_queue;  // the whole market's queue must fit the permutation
                    if (drop) b.err |= ERR_CAP_QUEUE;
                    RowCount c{b.n_orders, 0u, 0u};
                    submit_rows<true, false>(g, p, b, off, m, drop ? 0u : m, mk_a, c, to_perm);
                    b.n_orders = c.next;
                    nv = c.n_mkt;
                    // the host-ordered path's rule, over this book's share of the queue
                    if constexpr (G::DENSE) {
                        if (c.n > p.step_size || (start <= b.max_key_time && (b.flags & (FL_HAS_ASK | FL_HAS_BID)))) b.err |= ERR_TIME_ORDER;
                    }
                } else {
                    if (m > p.max_queue) b.err |= ERR_CAP_QUEUE;
                    if constexpr (G::DENSE) {  // the dense engine relies on t = start + i being new, increasing key times
                        if (m > p.step_size || (start <= b.max_key_time && (b.flags & (FL_HAS_ASK | FL_HAS_BID)))) b.err |= ERR_TIME_ORDER;
                    }
                    const u32 mm = min(m, p.max_queue);  // the first max_queue rows run
                    nv = mm;
                    if (p.assign_ids) {
                        RowCount c{b.n_orders, 0u, 0u};
                        submit_rows<false, false>(g, p, b, off, m, mm, 0u, c, to_perm);
                        b.n_orders = c.next;
                        nv = c.n;
                    } else {
                        // (a) create_order happened at submission (env.rs:173): publish status New for the new ids
                        u32 max_id = 0;
                        for (u32 j = lane; j < mm; j += 32) {
                            const u32 of = ins[j].op_flags, id = ins[j].order_id;
                            if ((of & BB_OP_MASK) == BB_OP_NEW && id < g.max_orders) {
                                stg32(b.oh + (u64)id * ORD_STRIDE + OH_META, ST_NEW | ((of & BB_F_BID) ? META_BID : 0u));
                                max_id = max(max_id, id + 1);
                            }
                            sts16(perm + 2u * j, j);
                        }
                        max_id = __reduce_max_sync(BB_FULL, max_id);
                        if (max_id > b.n_orders) b.n_orders = max_id;
                    }
                }
                __syncwarp();
                // (b) transactions.shuffle(rng) (env.rs:121): Fisher-Yates from the back.  Multi-asset markets shuffle
                // one queue across their books (market_env.rs:114-115): on the host-ordered path the host did that and the
                // slice is in order; in MODE_ENV_MKT every book of the market shuffles the whole queue with its own copy
                // of the market's Xoroshiro state (all copies advance alike)
                if (!p.host_order && lane == 0u) {  // a serial chain: one lane applies it (see the swap loop of k_sim)
                    u64 s0 = lds64(b.sb + HDR_RNG0), s1 = lds64(b.sb + HDR_RNG1);
                    for (u32 i = nv; i > 1; --i) {
                        const u32 j = xoroshiro_range(s0, s1, i);
                        const u32 x = lds16(perm + 2u * (i - 1)), y = lds16(perm + 2u * j);
                        sts16(perm + 2u * (i - 1), y);
                        sts16(perm + 2u * j, x);
                    }
                    sts64(b.sb + HDR_RNG0, s0);
                    sts64(b.sb + HDR_RNG1, s1);
                }
                __syncwarp();
                // (c) process in shuffled order at t = start + i (env.rs:123-127)
                for (u32 i0 = 0; i0 < nv; i0 += 32) {
                    u32 cnt = min(32u, nv - i0);
                    if constexpr (MK) {
                        // this book's events of the batch, in queue order, each with its position in the shuffled market
                        // queue (its time offset) in bb_instr::t; the NEW ids were written by this warp above
                        bool mine = false;
                        uint4 x0, x1;
                        if (lane < cnt) {
                            const u32 pj = lds16(perm + 2u * (i0 + lane));
                            const uint4* src = reinterpret_cast<const uint4*>(ins + pj);
                            x0 = src[0];
                            x1 = src[1];
                            mine = x1.w == mk_a;
                            if (mine && (x0.z & BB_OP_MASK) == BB_OP_NEW) x0.w = (u32)p.out_ids[off + pj];
                            x0.x = i0 + lane;
                            x0.y = 0u;
                        }
                        const u32 mm = __ballot_sync(BB_FULL, mine);
                        if (mine) {
                            const u32 pos = __popc(mm & ((1u << lane) - 1u));
                            sts128(chunk + 32u * pos, x0);
                            sts128(chunk + 32u * pos + 16u, x1);
                        }
                        cnt = __popc(mm);
                    } else if (lane < cnt) {
                        const u32 pj = lds16(perm + 2u * (i0 + lane));
                        const uint4* src = reinterpret_cast<const uint4*>(ins + pj);
                        uint4 x0 = src[0];
                        if (p.assign_ids && (x0.z & BB_OP_MASK) == BB_OP_NEW) x0.w = (u32)p.out_ids[off + pj];
                        sts128(chunk + 32u * lane, x0);
                        sts128(chunk + 32u * lane + 16u, src[1]);
                    }
                    __syncwarp();
                    for (u32 k = 0; k < cnt; ++k) {
                        const uint4 x = lds128(chunk + 32u * k), y = lds128(chunk + 32u * k + 16u);
                        const u64 t = start + ((MK || p.host_order) ? (((u64)x.y << 32) | x.x) : (u64)(i0 + k));
                        b.t = t;
                        apply_instr<false>(g, b, x.z, x.w, y.x, y.y, y.z, t, false);
                    }
                    __syncwarp();
                }
                b.t = start + p.step_size;  // env.rs:129
                if (lane == 0u) sts(b.sb + HDR_STEPCTR, lds(b.sb + HDR_STEPCTR) + 1u);
                emit_obs_direct(g, b, p, env);  // env.rs:132-134
            }
        }
        if (b.err && lane == 0) atomicOr(p.err_flag, b.err);
        book_to_header(g, b);
        blob_store(p, sb, env, lane);
    }
}

// ---------------------------------------------------------------------------------------------------
// In-kernel agents
struct Emit {  // running state of one env-step's transaction queue
    u32 n;      // instructions queued so far
    u32 next_id;
};

__device__ __forceinline__ void queue_push(const KParams& p, uint4* q, Emit& e, bool has, u32 op_flags, u32 id, u32 price,
                                           u32 vol, u32 lane) {
    const u32 m = __ballot_sync(BB_FULL, has);
    const u32 pos = e.n + __popc(m & ((1u << lane) - 1u));
    if (has) {
        if (pos < p.max_queue) q[pos] = make_uint4(op_flags, id, price, vol);
    }
    e.n += __popc(m);
}

__device__ __forceinline__ bool order_is_active(const Geo& g, const Book& b, u32 id) {
    return id < g.max_orders && (ldg32(b.oh + (u64)id * ORD_STRIDE + OH_META) & META_STATUS_MASK) == ST_ACTIVE;
}

// the Philox key halves of an agent draw: the unit's effective key (k_sim<.., PU>: seed ^ unit key, in key_l / key_h), else the
// launch's seed read where it is used, so that the other variants compile as they did before per-unit keys existed
template <bool PU> __device__ __forceinline__ u32 key_lo(const KParams& p, u32 key_l) {
    if constexpr (PU) return key_l;
    else return p.seed_lo;
}
template <bool PU> __device__ __forceinline__ u32 key_hi(const KParams& p, u32 key_h) {
    if constexpr (PU) return key_h;
    else return p.seed_hi;
}
// k_sim<.., PU>: the key halves of unit `unit`, the launch's seed XOR the unit's key
__device__ __forceinline__ void unit_key(const KParams& p, u32 unit, u32& key_l, u32& key_h) {
    const u64 key = __ldg(p.unit_keys + unit);
    key_l = p.seed_lo ^ (u32)key;
    key_h = p.seed_hi ^ (u32)(key >> 32);
}

// RandomAgents::update (crates/step_sim/src/agents/random_agent.rs:85-119), one lane per agent
template <bool PU>
__device__ __forceinline__ void random_agents_update(const KParams& p, const bb_agent_group& ag, const Book& b, uint4* q,
                                                     Emit& e, u32* slots, u32 env_g, u32 step, u32 slot_base, u32 key_l, u32 key_h) {
    for (u32 a0 = 0; a0 < ag.n_agents; a0 += 32) {
        const u32 a = a0 + b.lane;
        const bool valid = a < ag.n_agents;
        const uint4 r = philox4x32_10(env_g, step, slot_base + a, 0, key_lo<PU>(p, key_l), key_hi<PU>(p, key_h));
        const bool active = valid && (u32_to_f32_unit(r.x) < ag.rate);
        u32 held = BB_NIL;
        if (valid) held = slots[slot_base + a];
        bool live = false;
        if (active) live = order_is_active(p.geo, b, held);
        const bool do_cancel = active && live;
        const bool do_new = active && !live;
        const u32 new_mask = __ballot_sync(BB_FULL, do_new);
        const u32 id = e.next_id + __popc(new_mask & ((1u << b.lane) - 1u));
        const u32 side_bid = r.y >> 31;
        const u32 tick = ag.tick_lo + mulhi_range(r.z, ag.tick_hi - ag.tick_lo);
        const u32 vol = ag.vol_lo + mulhi_range(r.w, ag.vol_hi - ag.vol_lo);
        const u32 of = do_cancel ? 0u : (1u | (side_bid << 1) | (a << 13));  // bit0 NEW, bit1 bid, trader << 13
        queue_push(p, q, e, active, of, do_cancel ? held : id, tick * ag.tick_size, vol, b.lane);
        e.next_id += __popc(new_mask);
        if (active) slots[slot_base + a] = do_cancel ? BB_NIL : id;
    }
}

// Dense-engine variant: the agents' held order ids (u32 [A] at `agh`) and the slot each one was last seen resting
// in (u8 [A + 1] at Book::ags, entry 0 unused) live in shared memory for the whole launch, so "is my order still
// Active" is a shared-memory compare of the slot's id instead of a gather from the HBM order table, and the
// emitted instructions carry the hints described at d_apply (dense.cuh).
// `chip_base`: index of the group's first agent in the on-chip tables (== slot_base except in markets, whose books keep
// only their own groups' agents on chip).
template <class G, bool PU>
__device__ __forceinline__ void random_agents_update_dense(const KParams& p, const bb_agent_group& ag, const Book& b, u32 qs, Emit& e,
                                                           u32 agh, u32 env_g, u32 step, u32 slot_base, u32 chip_base, u32 key_l,
                                                           u32 key_h) {
    for (u32 a0 = 0; a0 < ag.n_agents; a0 += 32) {
        const u32 a = a0 + b.lane;
        const bool valid = a < ag.n_agents;
        const u32 ai = valid ? chip_base + a : 0u;
        const uint4 r = philox4x32_10(env_g, step, slot_base + a, 0, key_lo<PU>(p, key_l), key_hi<PU>(p, key_h));
        const bool active = valid && (u32_to_f32_unit(r.x) < ag.rate);
        const u32 held = lds(agh + 4u * ai);
        const u32 hs = lds8(b.ags + 1u + ai);
        const bool live = held != BB_NIL && lds(b.sb + G::DL::OFF_ID + 4u * hs) == held;
        const bool do_cancel = active && live;
        const bool do_new = active && !live;
        const u32 new_mask = __ballot_sync(BB_FULL, do_new);
        const u32 act_mask = __ballot_sync(BB_FULL, active);
        const u32 below = (1u << b.lane) - 1u;
        const u32 id = e.next_id + __popc(new_mask & below);
        const u32 side_bid = r.y >> 31;
        const u32 tick = ag.tick_lo + mulhi_range(r.z, ag.tick_hi - ag.tick_lo);
        const u32 vol = ag.vol_lo + mulhi_range(r.w, ag.vol_hi - ag.vol_lo);
        // x: bit 0 NEW, bit 1 bid, bits 2..12 hint (NEW: 1 + agent index; CANCEL: 1 + slot), bits 13.. trader id;
        // w: a cancel's is 0 (the journaled event loop marks the cancels that take effect there)
        const u32 of = do_cancel ? ((hs + 1u) << 2) : (1u | (side_bid << 1) | ((ai + 1u) << 2) | (a << 13));
        const u32 pos = e.n + __popc(act_mask & below);
        if (active) {
            if (pos < p.max_queue) sts128(qs + 16u * pos, make_uint4(of, do_cancel ? held : id, tick * ag.tick_size, do_cancel ? 0u : vol));
            sts(agh + 4u * ai, do_cancel ? BB_NIL : id);
        }
        e.n += __popc(act_mask);
        e.next_id += __popc(new_mask);
    }
}

// create_order's tick check (orderbook.rs:367-383) on the step's queued agent NEWs, q[0, n): an off-tick limit price is
// ERR_GRANULE, in the step at which the reference agent unwraps the PriceError.  It runs once per step over the queue,
// after all groups' updates, not inside the RandomAgents draw loop.  A bid market order's price is the sentinel
// 0xFFFFFFFF (types.rs:160-172) and is skipped; MomentumAgent / NoiseAgent limit prices were already checked at their
// draw, so scanning them again flags nothing new.  The dense engine's queue is in shared memory at `qs`, the others' in
// global scratch at `q`.
template <bool DENSE>
__device__ __forceinline__ void agent_tick_check(const uint4* q, u32 qs, u32 book_tick, u32 n, u32 lane, u32& err) {
    __syncwarp();
    bool bad = false;
    for (u32 i = lane; i < n; i += 32) {
        const u32 of = DENSE ? lds(qs + 16u * i) : q[i].x, price = DENSE ? lds(qs + 16u * i + 8u) : q[i].z;
        bad |= (of & 1u) && price != 0xFFFFFFFFu && price % book_tick != 0u;
    }
    if (__any_sync(BB_FULL, bad)) err |= ERR_GRANULE;
}

__device__ __forceinline__ u32 warp_excl_scan(u32 v, u32 lane, u32* total) {
    u32 x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 y = __shfl_up_sync(BB_FULL, x, d);
        if (lane >= (u32)d) x += y;
    }
    *total = __shfl_sync(BB_FULL, x, 31);
    return x - v;
}

// common.rs:21-41
__device__ __forceinline__ u32 round_price(double x, double tick, bool up) {
    x = (up ? ceil(x / tick) : floor(x / tick)) * tick;
    x = fmin(fmax(x, 0.0), 4294967295.0);
    return (u32)x;
}

// MomentumAgent::update (crates/step_sim/src/agents/momentum_agent.rs:145-209)
struct MomOut {
    u32 n, next_id, err;
};
template <bool PU>
__device__ __noinline__ MomOut momentum_agent_update(const KParams& p, const bb_agent_group& ag, u64 oh, u32 book_tick, u32 bid,
                                                     u32 ask, uint4* q, u32 e_n, u32 e_next_id, MomState* ms, u32 env_g,
                                                     u32 step, u32 gi, u32 slot_base) {
    // (`book_tick`, the tick of the book the group trades, takes the argument slot of the lane id, which is recomputed here:
    // one more argument costs the momentum k_sim variants spill traffic; for the same reason PU reads the unit's key here:
    // env_g is the unit's id plus the launch's first, and env_id_base is a multiple of assets)
    const u32 lane = threadIdx.x & 31u;
    u32 key_l = 0, key_h = 0;
    if constexpr (PU) unit_key(p, env_g - p.env_id_base / p.assets, key_l, key_h);
    Emit e;
    e.n = e_n;
    e.next_id = e_next_id;
    u32 err = 0;
    // (1) cancel_live_orders (common.rs:56-75): position-indexed draws, survivors compacted in place
    const u32 n_live = ms->n_live;
    u32 n_keep = 0;
    for (u32 k0 = 0; k0 < n_live; k0 += 32) {
        const u32 k = k0 + lane;
        const bool valid = k < n_live;
        u32 id = BB_NIL;
        bool active = false;
        if (valid) {
            id = ms->live[k];
            active = id < p.geo.max_orders && (ldg32(oh + (u64)id * ORD_STRIDE + OH_META) & META_STATUS_MASK) == ST_ACTIVE;
        }
        const uint4 r = philox4x32_10(env_g, step, PHILOX_SLOT_CANCEL | gi, k >> 2, key_lo<PU>(p, key_l), key_hi<PU>(p, key_h));
        const u32 word = (k & 3u) == 0 ? r.x : (k & 3u) == 1 ? r.y : (k & 3u) == 2 ? r.z : r.w;
        const bool keep = active && (u32_to_f32_unit(word) > ag.rate);
        const bool cancel = active && !keep;
        queue_push(p, q, e, cancel, 0u, id, 0, 0, lane);
        const u32 km = __ballot_sync(BB_FULL, keep);
        __syncwarp();
        if (keep) ms->live[n_keep + __popc(km & ((1u << lane) - 1u))] = id;
        n_keep += __popc(km);
        __syncwarp();
    }
    // (2) mid price of the live book (orderbook.rs:272-276; u32 spread wraps as in a release build)
    const double mid = (double)bid + 0.5 * (double)(u32)(ask - bid);
    const bool noise = ag.kind == BB_GROUP_NOISE;  // NoiseAgent::update, noise_agent.rs:126-177
    // (3) momentum and order probabilities
    double m = 0.0, p_market = 0.0;
    if (!noise && ms->has_last) {
        m = ms->momentum * (1.0 - ag.decay) + ag.decay * (mid - ms->last_price);
        p_market = ag.demand * tanh(ag.scale * m) / (double)ag.n_agents;
    }
    const double p_limit = ag.order_ratio * p_market;
    const double tick = (double)ag.tick_size;
    // (4) per trader: limit order then market order
    for (u32 j0 = 0; j0 < ag.n_agents; j0 += 32) {
        const u32 j = j0 + lane;
        const bool valid = j < ag.n_agents;
        const uint4 ra = philox4x32_10(env_g, step, slot_base + j, 0, key_lo<PU>(p, key_l), key_hi<PU>(p, key_h));
        const uint4 rb = philox4x32_10(env_g, step, slot_base + j, 1, key_lo<PU>(p, key_l), key_hi<PU>(p, key_h));
        const bool dir = (m > 0.0) || (m < 0.0);
        bool do_limit = valid && dir && (u64_to_f64_unit(ra.x, ra.y) < p_limit);
        bool do_market = valid && dir && (u64_to_f64_unit(ra.z, ra.w) < p_market);
        bool limit_bid = m > 0.0, market_bid = m > 0.0;
        if (noise) {  // fixed probabilities (f32 compares), a fair coin per order for the side
            do_limit = valid && (u32_to_f32_unit(ra.x) < (float)ag.decay);
            limit_bid = (ra.y >> 31) != 0;
            do_market = valid && (u32_to_f32_unit(ra.z) < (float)ag.demand);
            market_bid = (ra.w >> 31) != 0;
        }
        u32 price = 0;
        if (do_limit) {
            double u1 = u64_to_f64_unit(rb.x, rb.y);
            const double u2 = u64_to_f64_unit(rb.z, rb.w);
            if (u1 < 1e-300) u1 = 1e-300;
            const double nrm = sqrt(-2.0 * log(u1)) * cos(6.283185307179586476925 * u2);
            const double dist = fabs(exp(ag.mu + ag.sigma * nrm));
            price = limit_bid ? round_price(mid - dist, tick, false) : round_price(mid + dist, tick, true);
            if (price % book_tick != 0) err |= ERR_GRANULE;  // the reference unwraps a PriceError here
        }
        u32 total;
        const u32 cnt = (do_limit ? 1u : 0u) + (do_market ? 1u : 0u);
        const u32 before = warp_excl_scan(cnt, lane, &total);
        const u32 trader = ag.tick_lo + j;
        const u32 lm = __ballot_sync(BB_FULL, do_limit);
        const u32 id_l = e.next_id + before;
        const u32 id_m = id_l + (do_limit ? 1u : 0u);
        if (do_limit) {
            const u32 pos = e.n + before;
            if (pos < p.max_queue) q[pos] = make_uint4(1u | (limit_bid ? 2u : 0u) | (trader << 13), id_l, price, ag.vol_lo);
            const u32 lpos = n_keep + __popc(lm & ((1u << lane) - 1u));
            if (lpos < p.mom_live_cap) ms->live[lpos] = id_l; else err |= ERR_CAP_LIVE;
        }
        if (do_market) {
            const u32 pos = e.n + before + (do_limit ? 1u : 0u);
            // market order: the sentinel price IS the encoding (types.rs:160-172, 213-225)
            if (pos < p.max_queue)
                q[pos] = make_uint4(1u | (market_bid ? 2u : 0u) | (trader << 13), id_m, market_bid ? 0xFFFFFFFFu : 0u, ag.vol_lo);
        }
        n_keep = min(n_keep + __popc(lm), p.mom_live_cap);
        e.n += total;
        e.next_id += total;
    }
    __syncwarp();
    if (lane == 0) {
        if (!noise) {
            ms->momentum = m;
            ms->last_price = mid;
            ms->has_last = 1;
        }
        ms->n_live = n_keep;
    }
    __syncwarp();
    MomOut out;
    out.n = e.n;
    out.next_id = e.next_id;
    // the capacity / tick checks above are per lane (per trader): every lane must report them, lane 0 writes the header
    out.err = __reduce_or_sync(BB_FULL, err);
    return out;
}

// The step's shuffle (k_sim, k_env_agents_stage): Fisher-Yates from the back over the nq queued events, one Philox word per
// position (counter (env_g, step, PHILOX_SLOT_SHUFFLE, block of 4)), the draws made lane-parallel into jarr (u16 [nq]).
// The swaps are one serial chain: lane 0 applies them alone (32 lanes storing the same 16 bytes are 4 L1 wavefronts
// instead of 1, and the tools rightly flag unsynchronised same-address traffic between lanes).  The chain permutes perm
// (u16 [nq], built here from the identity) or, with QSWAP (the dense engine's on-chip queue at qs), the 16-byte events.
template <bool PU, bool QSWAP>
__device__ __forceinline__ void shuffle_queue(const KParams& p, u32 perm, u32 jarr, u32 qs, u32 nq, u32 env_g, u32 step, u32 key_l,
                                              u32 key_h, u32 lane) {
    if constexpr (!QSWAP)
        for (u32 i = lane; i < nq; i += 32) sts16(perm + 2u * i, i);
    for (u32 b0 = 0; b0 * 4u < nq; b0 += 32) {
        const u32 blk = b0 + lane;
        if (blk * 4u < nq) {
            const uint4 r = philox4x32_10(env_g, step, PHILOX_SLOT_SHUFFLE, blk, key_lo<PU>(p, key_l), key_hi<PU>(p, key_h));
            const u32 i = blk * 4u;
            // 4 consecutive u16 slots are always in bounds: the array is padded to a multiple of 8 bytes
            const u32 j0 = mulhi_range(r.x, i + 1), j1 = mulhi_range(r.y, i + 2);
            const u32 j2 = mulhi_range(r.z, i + 3), j3 = mulhi_range(r.w, i + 4);
            sts(jarr + 2u * i, j0 | (j1 << 16));
            sts(jarr + 2u * i + 4u, j2 | (j3 << 16));
        }
    }
    __syncwarp();
    if (lane != 0u) {
    } else if constexpr (QSWAP) {  // the queue is on chip: swap the 16-byte instructions themselves
        for (u32 i = nq; i > 1; --i) {
            const u32 j = lds16(jarr + 2u * (i - 1));
            const uint4 x = lds128(qs + 16u * (i - 1)), y = lds128(qs + 16u * j);
            sts128(qs + 16u * (i - 1), y);
            sts128(qs + 16u * j, x);
        }
    } else {
        for (u32 i = nq; i > 1; --i) {
            const u32 j = lds16(jarr + 2u * (i - 1));
            const u32 x = lds16(perm + 2u * (i - 1)), y = lds16(perm + 2u * j);
            sts16(perm + 2u * (i - 1), y);
            sts16(perm + 2u * j, x);
        }
    }
    __syncwarp();
}

// A caller's queued row as an event of the agents' queue (k_sim<.., EXT>, k_env_agents_stage): bit 0 NEW, bit 1 bid, no
// hint, trader id above bit 13; a market order carries the sentinel price (types.rs:160-172, 213-225)
__device__ __forceinline__ uint4 row_event(uint4 x, uint4 y, bool is_new, u32 id) {
    const bool bid = (x.z & BB_F_BID) != 0u;
    const u32 price = (x.z & BB_F_MARKET) ? (bid ? 0xFFFFFFFFu : 0u) : y.x;
    return make_uint4(is_new ? (1u | (bid ? 2u : 0u) | (y.z << 13)) : 0u, is_new ? id : x.w, price, y.y);
}

// named barrier over the warps of one market (bar.sync with an explicit thread count)
// Barrier ids are immediates (a CTA holds at most two markets): with a register id ptxas reserves all 16 hardware
// barriers for the CTA, which caps residency at 4 CTAs per SM.
__device__ __forceinline__ void market_bar_sync(u32 id, u32 n_threads) {
    if (id == 1u) asm volatile("bar.sync 1, %0;" ::"r"(n_threads) : "memory");
    else asm volatile("bar.sync 2, %0;" ::"r"(n_threads) : "memory");
}

// MKT: multi-asset markets with in-kernel agents — market_sim_runner (runner.rs:107-131) over the *Market agent twins
// (RandomMarketAgents random_agent.rs:165-247, MomentumMarketAgent momentum_agent.rs:282-409, NoiseMarketAgent
// noise_agent.rs:226-345).  The A books of a market are A consecutive warps of one CTA.  Every agent group trades one asset,
// so each warp runs the groups of its own book; what a market shares is the step's transaction queue
// (market_env.rs:108-121): all groups' instructions in declaration order, shuffled as a whole, event i of the shuffled
// queue executing at start + i on its asset's book.  The warps exchange their per-group instruction counts through
// shared memory (one named barrier per step), each then derives the same market-wide permutation from the market's
// Philox key and pulls out its own events together with their positions in it.
// EXT (bb_run_agents_with_rows; always with MOM): after the built-in agents' updates the caller's own rows for the env —
// already in device memory, the action block of an RL-style loop — are submitted in row order, exactly as
// `agents.update(env); env.place_order(..) / env.cancel_order(..); env.step()` would: NEW rows take the next ids, rows
// that queue nothing are skipped, and everything takes part in the step's one shuffle.
// MKT + EXT (bb_run_agents_with_rows_market): the rows are the market's slice, bb_instr::aux the row's asset.  Every book
// walks the whole slice (as k_apply<MODE_ENV_MKT> does), so every warp knows the market's queued-row count and which of
// those rows are its own: the queued rows follow all groups' instructions in the market's queue, and each book appends
// its own after its agents' events.  A per-warp bitmask over the market's queued rows (with per-word prefix counts) maps a
// shuffled position back to the book's own list; it sits behind jarr, in a layout only this variant uses.
// PU (bb_set_agent_params_device; always with MOM): every unit (env, or market) draws with its own group records and Philox
// key, p.unit_groups / p.unit_keys, instead of the launch's p.groups and (seed_lo, seed_hi).  The records stay inside the
// declared population (bb_set_agents sized everything from p.groups: n_agents, agent ids, live-list capacities, the dense
// window), so only the draws' parameters and key differ; n_agents is still read from p.groups.
template <int ENG, bool MOM, bool MKT = false, bool EXT = false, bool PU = false>
__global__ void __launch_bounds__(128, ENG == ENG_PAGED ? 5 : 7) k_sim(const __grid_constant__ KParams p) {
    static_assert(!EXT || MOM, "external rows ride on the unhinted (MOM) variants");
    static_assert(!PU || MOM, "per-unit parameters ride on the unhinted (MOM) variants");
    typedef GeoT<ENG> G;
    extern __shared__ __align__(128) unsigned char smem[];
    const u32 lane = keep32(threadIdx.x & 31u), warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const u32 sb = keep32(smem_u32(smem) + warp * p.warp_smem_bytes);
    const u32 bar = sb + p.off_bar;
    const u32 perm = sb + p.off_perm;          // u16 [max_queue]
    // u16 [max_queue] (the dense engine has no perm array); markets: perm and jarr hold the whole market's queue.  jarr
    // starts 8-byte aligned (the shuffle stores its draws as u32 pairs; an odd max_queue would misalign them), inside the
    // 16 bytes of slack make_layout reserves behind the two arrays
    const u32 jarr = perm + (MKT ? 2u * ((p.assets * p.max_queue + 7u) & ~7u) : G::DENSE ? 0u : 2u * ((p.max_queue + 3u) & ~3u));
    const u32 stage = sb + p.off_obs;          // u32 [2][OBS_STAGE_STEPS * obs_words]
    const u32 mk_a = MKT ? warp % p.assets : 0u;                           // the asset this warp's book is
    const u32 mk_sb = MKT ? sb - mk_a * p.warp_smem_bytes + p.off_mkt : 0u;  // u32 [2][MAX_GROUPS] in the market's first warp
    const u32 mk_bar = MKT ? 1u + warp / p.assets : 0u;
    // MKT + EXT: u32 [mk_words] mask of this book's rows among the market's queued rows, then u32 [mk_words] prefix counts
    const u32 mk_words = MKT && EXT ? (p.assets * p.max_queue + 31u) >> 5 : 0u;
    const u32 mk_rm = MKT && EXT ? perm + 4u * ((p.assets * p.max_queue + 7u) & ~7u) + 16u : 0u;
    u32 mk_phase = 0;
    // the step's transaction queue: L2-resident global scratch, or (dense engine) shared memory so that the event
    // loop fetches each instruction with one broadcast ld.shared.v4 instead of a gather + four shuffles
    const u32 qs = sb + p.off_q;
    uint4* q = G::DENSE ? reinterpret_cast<uint4*>(smem + (size_t)warp * p.warp_smem_bytes + p.off_q)
                                : p.scratch + (size_t)(blockIdx.x * wpb + warp) * p.max_queue;
    const u64 qa = (u64)q;
    const GeoT<ENG>& g = static_cast<const GeoT<ENG>&>(p.geo);
    if (lane == 0) {
        mbar_init_a(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_proxy_async();
    __syncwarp();
    u32 ph_blob = 0;
    const u32 stage_steps = OBS_STAGE_STEPS(p.obs_words), stage_words = stage_steps * p.obs_words;
    pcache_init(g, sb, lane);

    for (u32 env = blockIdx.x * wpb + warp; env < p.n_envs; env += gridDim.x * wpb) {
        Book b;
        make_book(b, p, sb, env, lane);
        if (!blob_load(p, sb, env, bar, ph_blob, lane)) {
            if (lane == 0) atomicOr(p.err_flag, 0x80000000u);
            if (MKT) __trap();  // leaving would strand the market's other warps at their barrier
            return;
        }
        book_from_header(g, b);
        // the RNG unit: the env, or the whole market (agent slots and the shuffle are market-wide)
        const u32 env_g = MKT ? (p.env_id_base + env) / p.assets : p.env_id_base + env;
        // PU: the unit's Philox key halves and group records
        u32 key_l = 0, key_h = 0;
        const bb_agent_group* urow = nullptr;
        if constexpr (PU) {
            const u32 unit = MKT ? env / p.assets : env;
            unit_key(p, unit, key_l, key_h);
            urow = p.unit_groups + (size_t)unit * p.n_groups;
        }
        u32* slots = p.rslot + (size_t)env * p.agents_per_env;
        const u32 agh = sb + p.off_ag;  // dense engine: held order id per agent, u32 [agents_per_env]
        if constexpr (G::DENSE) {
            // bring the agents' held ids on chip and find the slot each one rests in (one pass over the slot table);
            // markets keep only the agents of this book's own groups on chip, packed in declaration order
            b.ags = agh + 4u * p.chip_agents;
            u32 gbase = 0, cbase = 0;
            for (u32 gi = 0; gi < (MKT ? p.n_groups : 1u); ++gi) {
                const u32 ng = MKT ? p.groups[gi].n_agents : p.agents_per_env;
                if (!MKT || p.group_asset[gi] == mk_a) {
                    for (u32 a0 = 0; a0 < ng; a0 += 32) {
                        const u32 a = a0 + lane;
                        const u32 held = a < ng ? slots[gbase + a] : BB_NIL;
                        u32 hs = 0;
                        for (u32 s4 = 0; s4 < G::DL::LP; s4 += 4) {
                            const uint4 v = lds128(b.sb + G::DL::OFF_ID + 4u * s4);
                            hs = v.x == held ? s4 : v.y == held ? s4 + 1u : v.z == held ? s4 + 2u : v.w == held ? s4 + 3u : hs;
                        }
                        if (a < ng) {
                            sts(agh + 4u * (cbase + a), held);
                            sts8(b.ags + 1u + cbase + a, hs);
                        }
                    }
                    cbase += ng;
                }
                gbase += ng;
            }
            __syncwarp();
        }
        u32* hist_env = p.hist + (size_t)env * p.hist_env_stride;
        const u32 hist0 = lds(b.sb + HDR_NSTEPS);
        const bool staged = (hist0 & 3u) == 0;  // bulk stores need 16-byte aligned record groups
        u32 sbuf = 0, sfill = 0, sbase = hist0;
        u32 step = lds(b.sb + HDR_STEPCTR);

        for (u32 s = 0; s < p.n_steps; ++s, ++step) {
            // ---- agents.update(env, rng) in declaration order (crates/macros/src/lib.rs:57-72)
            Emit e;
            e.n = 0;
            e.next_id = b.n_orders;
            const u32 id0 = b.n_orders;
            u32 slot_base = 0, chip_base = 0, mi = 0;
            u32 mk_cnt = 0;  // markets: lane gi holds the number of instructions group gi queued (own groups only)
            for (u32 gi = 0; gi < p.n_groups; ++gi) {
                const bb_agent_group& ag = PU ? urow[gi] : p.groups[gi];  // PU: the unit's row in global memory, read through L1
                const bool mine = !MKT || p.group_asset[gi] == mk_a;
                const u32 n_before = e.n;
                if (!MOM || ag.kind == BB_GROUP_RANDOM) {
                    if (mine) {
                        if constexpr (G::DENSE) random_agents_update_dense<G, PU>(p, ag, b, qs, e, agh, env_g, step, slot_base, chip_base, key_l, key_h);
                        else random_agents_update<PU>(p, ag, b, q, e, slots, env_g, step, slot_base, key_l, key_h);
                    }
                } else {
                    if (mine) {
                        const MomOut mo = momentum_agent_update<PU>(p, ag, b.oh, __ldg(g.ticks + env), best_price(g, b, 1), best_price(g, b, 0), q, e.n,
                                                                e.next_id, (MomState*)((char*)p.mom + ((size_t)env * p.mom_groups_per_env + mi) * p.mom_stride), env_g,
                                                                step, gi, slot_base);
                        e.n = mo.n;
                        e.next_id = mo.next_id;
                        b.err |= mo.err;
                    }
                    ++mi;
                }
                if (MKT && lane == gi) mk_cnt = e.n - n_before;
                slot_base += ag.n_agents;
                if (mine) chip_base += ag.n_agents;
            }
            u32 mk_nr = 0;  // MKT + EXT: the market's queued rows (every book of the market counts the same)
            if constexpr (EXT) {
                // the caller's rows belong to the launch's first step; markets: the market's slice, every book walks it all
                const u32 unit = MKT ? env / p.assets : env;
                const u64 off = p.offsets[unit];
                const u32 m = s == 0 ? (u32)(p.offsets[unit + 1] - off) : 0u;
                const u32 cap = p.assets * p.max_queue;  // MKT: queued rows beyond it drop the market's step (below)
                const u32 nw = MKT ? min((m + 31u) >> 5, mk_words) : 0u;  // mask words the slice can touch
                if constexpr (MKT) {
                    for (u32 w = lane; w < nw; w += 32) sts(mk_rm + 4u * w, 0u);
                    __syncwarp();
                }
                // this book's rows join its queue as in-kernel events (row_event); markets also mark each one's index among
                // the market's queued rows in the mask
                auto to_queue = [&](u32, uint4 x, uint4 y, bool mine, bool is_new, u32 id, u32 pos, u32 pos_mkt) {
                    if (!mine) return;
                    if (pos < p.max_queue) {
                        const uint4 ev = row_event(x, y, is_new, id);
                        if constexpr (G::DENSE) sts128(qs + 16u * pos, ev);
                        else q[pos] = ev;
                    }
                    if (MKT && pos_mkt < cap) asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(mk_rm + 4u * (pos_mkt >> 5)), "r"(1u << (pos_mkt & 31u)) : "memory");
                };
                RowCount rows{e.next_id, e.n, 0u};
                submit_rows<MKT, true>(g, p, b, off, m, m, mk_a, rows, to_queue);
                e.next_id = rows.next;
                e.n = rows.n;
                mk_nr = rows.n_mkt;
                __syncwarp();
                if constexpr (MKT) {
                    // prefix counts: own queued rows in the words before each mask word
                    u32 run = 0;
                    for (u32 w0 = 0; w0 < nw; w0 += 32) {
                        const u32 w = w0 + lane;
                        u32 tot;
                        const u32 c = w < nw ? __popc(lds(mk_rm + 4u * w)) : 0u;
                        const u32 ex = warp_excl_scan(c, lane, &tot);
                        if (w < nw) sts(mk_rm + 4u * (mk_words + w), run + ex);
                        run += tot;
                    }
                    __syncwarp();
                }
            }
            if (e.n > p.max_queue) b.err |= ERR_CAP_QUEUE;
            u32 n = min(e.n, p.max_queue);
            // a RandomAgents group in rand_tick_mask can draw off its book's tick: the host runs such a population on the MOM
            // variants, so the hot RandomAgents-only kernels carry no check.  (The caller's rows are in the queue too: their
            // off-tick limit NEWs were dropped above.)
            if constexpr (MOM) {
                if (p.rand_tick_mask) agent_tick_check<G::DENSE>(q, qs, __ldg(g.ticks + env), n, lane, b.err);
            }
            b.n_orders = e.next_id;  // create_order at submission (env.rs:173)
            if constexpr (G::DENSE) {  // ids and slots are validated once per step (d_apply trusts hinted events)
                if (e.next_id > g.max_orders) {
                    b.err |= ERR_CAP_ORDERS;
                    n = 0;
                }
                // every new order of the step could rest: with fewer free slots than new orders the step is dropped
                // (flagged) rather than run with per-insert checks; a population of one-order agents never gets here
                if (e.next_id - id0 > b.free_top) {
                    b.err |= ERR_CAP_LIVE;
                    n = 0;
                }
            }
            __syncwarp();

            // ---- Env::step (env.rs:116-135)
            const u64 start = b.t;
            b.trade_vol = 0;
            if constexpr (G::DENSE) {  // the dense engine relies on t = start + i being new, increasing key times
                if (n > p.step_size || (start <= b.max_key_time && (b.flags & (FL_HAS_ASK | FL_HAS_BID)))) b.err |= ERR_TIME_ORDER;
            }
            // markets: exchange the per-group counts; `nq` is the length of the queue that gets shuffled
            u32 nq = n, mk_off = 0, mk_loc = 0, mk_all = 0, mk_ag = 0, mk_ag_mine = 0;
            if constexpr (MKT) {
                const u32 cb = mk_sb + 4u * MAX_GROUPS * (mk_phase & 1u);  // double-buffered: one barrier per step is enough
                mk_phase += 1;
                const bool own = lane < p.n_groups && p.group_asset[lane] == mk_a;
                if (own) sts(cb + 4u * lane, mk_cnt);
                market_bar_sync(mk_bar, 32u * p.assets);
                mk_all = lane < p.n_groups ? lds(cb + 4u * lane) : 0u;
                u32 total, total_mine;
                mk_off = warp_excl_scan(mk_all, lane, &total);            // first queue position of each group
                mk_loc = warp_excl_scan(own ? mk_all : 0u, lane, &total_mine);  // ... and its first entry in this book's list
                nq = total;
                if constexpr (EXT) {  // the queued rows follow every group's instructions; this book's after its agents'
                    mk_ag = total;
                    mk_ag_mine = total_mine;
                    nq = total + mk_nr;
                }
                if (nq > p.assets * p.max_queue) {  // some book overflowed its queue (flagged there): drop the step everywhere
                    b.err |= ERR_CAP_QUEUE;
                    nq = 0;
                }
                if constexpr (G::DENSE) {
                    if (nq > p.step_size) b.err |= ERR_TIME_ORDER;
                }
            }
            shuffle_queue<PU, G::DENSE && !MKT>(p, perm, jarr, qs, nq, env_g, step, key_l, key_h, lane);
            if constexpr (MKT) {
                // pull this book's events out of the market-wide permutation, in queue order: (index in the book's own
                // list, position in the shuffled queue = time offset), one u32 each, over the consumed draw array
                u32 n_mine = 0;
                for (u32 i0 = 0; i0 < nq; i0 += 32) {
                    const u32 i = i0 + lane;
                    const u32 gq = i < nq ? lds16(perm + 2u * i) : 0xFFFFFFFFu;
                    bool is_mine = false;
                    u32 li = 0;
                    for (u32 k = 0; k < p.n_groups; ++k) {
                        const u32 o = __shfl_sync(BB_FULL, mk_off, k), c = __shfl_sync(BB_FULL, mk_all, k);
                        const u32 lo = __shfl_sync(BB_FULL, mk_loc, k);
                        if (gq - o < c && p.group_asset[k] == mk_a) {
                            is_mine = true;
                            li = lo + (gq - o);
                        }
                    }
                    if constexpr (EXT) {
                        const u32 x = gq - mk_ag;  // index among the market's queued rows
                        if (gq < nq && gq >= mk_ag) {
                            const u32 wd = lds(mk_rm + 4u * (x >> 5));
                            if ((wd >> (x & 31u)) & 1u) {
                                is_mine = true;
                                li = mk_ag_mine + lds(mk_rm + 4u * (mk_words + (x >> 5))) + __popc(wd & ((1u << (x & 31u)) - 1u));
                            }
                        }
                    }
                    const u32 m = __ballot_sync(BB_FULL, is_mine);
                    const u32 pos = n_mine + __popc(m & ((1u << lane) - 1u));
                    if (is_mine && pos < p.max_queue) sts(jarr + 4u * pos, min(li, p.max_queue - 1u) | (i << 16));
                    n_mine += __popc(m);
                }
                n = min(n, n_mine);  // equal unless the step was dropped
                __syncwarp();
            }
            // process in shuffled order at t = start + i
            if constexpr (G::DENSE && !MOM && !MKT) {
                // Journaled: lane 0 runs the events alone (see below) and keeps only the book itself; the order records,
                // the trade log and the trade counters are written by all lanes after it (d_flush).  The trade journal
                // fills the queue entries past the step's events: when it is full, lane 0 stops, the warp flushes, and
                // lane 0 goes on from the suspended event with the volume it had left.
                const u32 nt0 = b.n_trades;
                const u32 jb = qs + 16u * n, jend = qs + 16u * (p.max_queue + 2u);
                u32 done = 0, rv = 0;  // events already written out; volume left of the suspended event `done`
                for (;;) {
                    u32 stop = n;
                    if (lane == 0) {
                        b.jp = jb;
                        b.jend = jend;
                        // two inlined handler copies on alternating prefetched quads, as on the write-through path
                        auto handle = [&](const uint4& ev, u32 i) -> u32 {
                            const u32 hint = (ev.x >> 2) & 0x7FFu;
                            b.ev = qs + 16u * i;
                            if (ev.x & 1u) {
                                if (ev.x & 2u) return d_apply<true, false, 1, true>(g, b, EV_NEW, ev.y, 1u, ev.z, ev.w, 0u, false, false, 0ull, hint);
                                return d_apply<true, false, 1, true>(g, b, EV_NEW, ev.y, 0u, ev.z, ev.w, 0u, false, false, 0ull, hint);
                            }
                            return d_apply<false, false, 1, true>(g, b, EV_CANCEL, ev.y, 0u, 0u, 0u, 0u, false, false, 0ull, hint);
                        };
                        uint4 e0 = lds128(qs + 16u * done);
                        if (rv) e0.w = rv;
                        for (u32 i = done; i < n; i += 2) {
                            const uint4 e1 = lds128(qs + 16u * i + 16u);  // (the queue is padded by two entries)
                            if ((rv = handle(e0, i))) {
                                stop = i;
                                break;
                            }
                            if (i + 1 >= n) break;
                            e0 = lds128(qs + 16u * i + 32u);
                            if ((rv = handle(e1, i + 1))) {
                                stop = i + 1;
                                break;
                            }
                        }
                    }
                    __syncwarp();
                    stop = __shfl_sync(BB_FULL, stop, 0);
                    rv = __shfl_sync(BB_FULL, rv, 0);
                    const u32 nj = (__shfl_sync(BB_FULL, b.jp, 0) - jb) >> 4;
                    b.vol_ask = __shfl_sync(BB_FULL, b.vol_ask, 0);
                    b.vol_bid = __shfl_sync(BB_FULL, b.vol_bid, 0);
                    b.bq_ask = __shfl_sync(BB_FULL, b.bq_ask, 0);
                    b.bq_bid = __shfl_sync(BB_FULL, b.bq_bid, 0);
                    b.flags = __shfl_sync(BB_FULL, b.flags, 0);
                    b.d_trans = __shfl_sync(BB_FULL, b.d_trans, 0);
                    b.free_top = __shfl_sync(BB_FULL, b.free_top, 0);
                    b.err = __shfl_sync(BB_FULL, b.err, 0);
                    d_flush(g, b, qs, agh, start, done, stop, jb, nj);
                    done = stop;
                    if (stop == n) break;
                }
                // transitions of the step: one per placed order and per fill (cancels counted theirs); traded volume
                b.d_trans += (b.n_trades - nt0) + (n ? e.next_id - id0 : 0u);
                b.d_volume += b.trade_vol;
            } else if constexpr (G::DENSE) {
                constexpr int H = MOM ? 2 : 1;  // RandomAgents always hint, MomentumAgent / NoiseAgent never do
                // With every event hinted the matching path has no lane-parallel step left, so it runs on LANE 0 ALONE:
                // a warp-uniform ld/st moves 32 copies of the same bytes through the L1 data pipe (4 wavefronts for a
                // 16-byte store), and that pipe, not instruction issue, was the busiest unit of the all-lane version
                // (78 % vs 70 %, profiles/r01_s5_summary.md).  The book registers are re-broadcast after the loop.
                const u32 nt0 = b.n_trades;
                if (MOM || lane == 0) {
                    // events are fetched one ahead into alternating register quads (two inlined copies of the handler:
                    // a single copy makes the compiler shuffle the prefetched quad through 6 moves per event)
                    auto handle = [&](const uint4& ev) {
                        const u32 hint = (ev.x >> 2) & 0x7FFu;
                        if (ev.x & 1u) {
                            if (ev.x & 2u) book_apply<true, false, G, H>(g, b, EV_NEW, ev.y, 1u, ev.z, ev.w, ev.x >> 13, false, false, b.t, hint);
                            else book_apply<true, false, G, H>(g, b, EV_NEW, ev.y, 0u, ev.z, ev.w, ev.x >> 13, false, false, b.t, hint);
                        } else {
                            book_apply<false, false, G, H>(g, b, EV_CANCEL, ev.y, 0u, 0u, 0u, 0u, false, false, b.t, hint);
                        }
                        b.t += 1;
                    };
                    if constexpr (MKT) {
                        for (u32 k = 0; k < n; ++k) {
                            const u32 w = lds(jarr + 4u * k);
                            const uint4 ev = lds128(qs + 16u * (w & 0xFFFFu));
                            b.t = start + (u64)(w >> 16);
                            handle(ev);
                        }
                    } else {
                    uint4 e0 = lds128(qs);
                    for (u32 i = 0; i < n; i += 2) {
                        const uint4 e1 = lds128(qs + 16u * i + 16u);  // (the queue is padded by two entries)
                        handle(e0);
                        if (i + 1 >= n) break;
                        e0 = lds128(qs + 16u * i + 32u);
                        handle(e1);
                    }
                    }
                }
                if constexpr (!MOM) {
                    __syncwarp();
                    b.max_key_time = __shfl_sync(BB_FULL, b.max_key_time, 0);
                    b.n_trades = __shfl_sync(BB_FULL, b.n_trades, 0);
                    b.trade_vol = __shfl_sync(BB_FULL, b.trade_vol, 0);
                    b.vol_ask = __shfl_sync(BB_FULL, b.vol_ask, 0);
                    b.vol_bid = __shfl_sync(BB_FULL, b.vol_bid, 0);
                    b.bq_ask = __shfl_sync(BB_FULL, b.bq_ask, 0);
                    b.bq_bid = __shfl_sync(BB_FULL, b.bq_bid, 0);
                    b.flags = __shfl_sync(BB_FULL, b.flags, 0);
                    b.err = __shfl_sync(BB_FULL, b.err, 0);
                    b.d_trans = __shfl_sync(BB_FULL, b.d_trans, 0);
                    b.d_volume = __shfl_sync(BB_FULL, b.d_volume, 0);
                    b.free_top = __shfl_sync(BB_FULL, b.free_top, 0);
                    b.tr_ptr = __shfl_sync(BB_FULL, b.tr_ptr, 0);
                }
                // transitions of the step: one per placed order and per fill (cancels counted theirs); traded volume
                b.d_trans += (b.n_trades - nt0) + (n ? e.next_id - id0 : 0u);
                b.d_volume += b.trade_vol;
            } else
            for (u32 i0 = 0; i0 < n; i0 += 32) {
                const u32 cnt = min(32u, n - i0);
                uint4 mine = make_uint4(0, 0, 0, 0);
                u32 toff = 0;
                if (lane < cnt) {
                    if constexpr (MKT) {
                        const u32 w = lds(jarr + 4u * (i0 + lane));
                        mine = ldg128(qa + 16u * (w & 0xFFFFu));
                        toff = w >> 16;
                    } else {
                        mine = ldg128(qa + 16u * lds16(perm + 2u * (i0 + lane)));
                    }
                }
                for (u32 k = 0; k < cnt; ++k) {
                    if constexpr (MKT) b.t = start + (u64)__shfl_sync(BB_FULL, toff, k);
                    const u32 of = __shfl_sync(BB_FULL, mine.x, k), id = __shfl_sync(BB_FULL, mine.y, k);
                    const u32 price = __shfl_sync(BB_FULL, mine.z, k), vol = __shfl_sync(BB_FULL, mine.w, k);
                    if (of & 1u) {
                        // NEW: one constant-folded copy of the placement path per side — except with MomentumAgent /
                        // NoiseAgent compiled in, where the kernel is instruction-fetch bound (25 % of the stall samples
                        // were "no instruction", profiles/r01_s7_summary.md) and ONE side-generic copy is 7 % faster
                        if constexpr (MOM) book_apply<true, false>(g, b, EV_NEW, id, (of >> 1) & 1u, price, vol, of >> 13, false, false, b.t);
                        else if (of & 2u) book_apply<true, false>(g, b, EV_NEW, id, 1u, price, vol, of >> 13, false, false, b.t);
                        else book_apply<true, false>(g, b, EV_NEW, id, 0u, price, vol, of >> 13, false, false, b.t);
                    } else {
                        book_apply<false, false>(g, b, EV_CANCEL, id, 0u, 0u, 0u, 0u, false, false, b.t);
                    }
                    b.t += 1;
                }
            }
            b.d_instr += n;
            b.t = start + p.step_size;
            __syncwarp();

            // ---- observation record: staged in shared memory, flushed with bulk stores
            if (staged) {
                u32 w0, w1;
                book_obs(g, b, p.obs_words, &w0, &w1);
                if (EXT && p.obs_out && s + 1 == p.n_steps) {  // the caller's observation buffer gets the last record too
                    u32* o = p.obs_out + (size_t)env * p.obs_words;
                    if (lane < p.obs_words) o[lane] = w0;
                    if (lane + 32u < p.obs_words) o[lane + 32u] = w1;
                }
                const u32 dst = stage + 4u * (sbuf * stage_words + sfill * p.obs_words);
                if (lane < p.obs_words) sts(dst + 4u * lane, w0);
                if (lane + 32u < p.obs_words) sts(dst + 4u * (lane + 32u), w1);
                if (++sfill == stage_steps) {
                    __syncwarp();
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        bulk_s2g_a(hist_env + (size_t)sbase * p.obs_words, stage + 4u * (sbuf * stage_words), stage_words * 4u);
                        bulk_commit();
                        // the other buffer's previous flush has released its source; markets stage in ONE buffer (shared
                        // memory is what limits their occupancy) and wait for this flush's reads, ~1 us per 4 steps
                        if (MKT) bulk_wait_read<0>(); else bulk_wait_read<1>();
                    }
                    __syncwarp();
                    sbase += stage_steps;
                    sfill = 0;
                    if (!MKT) sbuf ^= 1u;
                }
            } else {
                emit_obs_direct(g, b, p, env);
            }
        }
        // tail of the staging buffer
        if (staged) {
            __syncwarp();
            const u32 words = sfill * p.obs_words;
            u32* dst = hist_env + (size_t)sbase * p.obs_words;
            const u32 src = stage + 4u * (sbuf * stage_words);
            for (u32 i = lane; i < words; i += 32) dst[i] = lds(src + 4u * i);
            sts(b.sb + HDR_NSTEPS, hist0 + p.n_steps);
        }
        sts(b.sb + HDR_STEPCTR, step);
        if constexpr (G::DENSE) {
            __syncwarp();
            u32 gbase = 0, cbase = 0;
            for (u32 gi = 0; gi < (MKT ? p.n_groups : 1u); ++gi) {
                const u32 ng = MKT ? p.groups[gi].n_agents : p.agents_per_env;
                if (!MKT || p.group_asset[gi] == mk_a) {
                    for (u32 a = lane; a < ng; a += 32) slots[gbase + a] = lds(agh + 4u * (cbase + a));
                    cbase += ng;
                }
                gbase += ng;
            }
        }
        if (lane == 0) bulk_wait_all<0>();
        if (b.err && lane == 0) atomicOr(p.err_flag, b.err);
        book_to_header(g, b);
        blob_store(p, sb, env, lane);
    }
}

// ---------------------------------------------------------------------------------------------------
// Deep-book replay (deep.cuh, deepw.cuh): the fetch warp and the retire warp of k_deepw.
// Immediate-mode instruction streams (OrderBook API at explicit times, orderbook.rs:411-792), configs C5 / C2.
// pre-decoded flag bits the fetch warp adds to op_flags (above the public BB_F_* bits)
#define DPF_MARKET (1u << 16)      // the order takes the market path: BB_F_MARKET, or a limit price equal to the sentinel (N3)
#define DPF_CAP_ORDERS (1u << 17)  // a NEW row whose id would not fit the order table

// ENV (bb_step_device): a NEW row carries the id submission gave it (k_env_deep_stage) instead of taking the next one.
template <u32 RB, bool NAP = false, bool ENV = false>
__device__ __forceinline__ void dp_fetch_warp(const KParams& p, const DeepOff& o, u32 sb, u32 lane, const bb_instr* ins, u32 n, u64 oh,
                                              u32 next_id) {
    const u32 ctl = sb + o.ctl;
    const u32 nb = (n + 31u) >> 5;
    for (u32 b = 0; b < nb; ++b) {
        const u32 slot = b & (RB - 1u);
        if (b >= RB) {
            if (!dp_wait<NAP>(ctl, [&] { return ld_acq(ctl + CT_EV_CONSUMED) + RB > b; }, 1)) return;
        }
        const u32 cnt = min(32u, n - 32u * b);
        const u32 ia = sb + o.ev_ins + 1024u * slot, bar = sb + o.bar + 8u + 8u * slot;
        fence_proxy_async();
        __syncwarp();
        if (lane == 0u) {
            mbar_expect_tx_a(bar, cnt * 32u);
            bulk_g2s_a(ia, ins + 32u * (size_t)b, cnt * 32u, bar);
        }
        {
            DP_T0
            if (!mbar_wait_a(bar, (b / RB) & 1u)) {
                st_rel(ctl + CT_ABORT, 1u);
                return;
            }
            if (lane == 0u) { DP_ADD(2) }
        }
        // the record writes of every event below this index are performed and fenced: sampled BEFORE the loads below
        const u32 rf = ld_acq(ctl + CT_EV_RETIRED);
        uint4 x = make_uint4(0, 0, 0, 0), y = make_uint4(0, 0, 0, 0);
        if (lane < cnt) {
            x = lds128(ia + 32u * lane);
            y = lds128(ia + 32u * lane + 16u);
        }
        const u32 op = x.z & BB_OP_MASK;
        // ---- everything about an event that does not depend on the book is settled here, one lane per event:
        // NEW rows get their ids (create_order hands them out in stream order, orderbook.rs:356-396), the market
        // sentinel price (types.rs:160-172, 213-225), and the write-once half of their record goes straight to HBM
        const u32 new_mask = __ballot_sync(BB_FULL, op == BB_OP_NEW);
        if (op == BB_OP_NEW) {
            const u32 id = ENV ? x.w : next_id + __popc(new_mask & ((1u << lane) - 1u));
            const u32 side = (x.z >> 8) & 1u;
            const u32 price = (x.z & BB_F_MARKET) ? (side ? 0xFFFFFFFFu : 0u) : y.x;
            const bool market = side ? (price == 0xFFFFFFFFu) : (price == 0u);
            u32 of = x.z | (market ? DPF_MARKET : 0u);
            if (id >= p.geo.max_orders) {
                of |= DPF_CAP_ORDERS;
            } else {
                const u64 ra = oh + (u64)id * ORD_STRIDE;
                stg128(ra, price, y.y, 0u, BB_NIL);
                stg128(ra + 16u, 0u, 0u, ST_NEW | (side ? META_BID : 0u), y.y);
                stg128(ra + 32u, x.x, x.y, 0xFFFFFFFFu, 0xFFFFFFFFu);
                stg128(ra + 48u, y.z, 0u, 0u, 0u);
            }
            sts128(ia + 32u * lane, make_uint4(x.x, x.y, of, id));
            sts(ia + 32u * lane + 16u, price);
        } else if ((op == BB_OP_CANCEL || op == BB_OP_MODIFY) && x.w < p.geo.max_orders) {
            u64 src = oh + (u64)x.w * ORD_STRIDE;
            // a true data dependency on `rf` (always adds 0): the loads cannot be issued before rf was read
            asm volatile("{\n\t.reg .u64 z;\n\tcvt.u64.u32 z, %1;\n\tshr.u64 z, z, 32;\n\tadd.u64 %0, %0, z;\n\t}" : "+l"(src) : "r"(rf));
            const u32 ra = sb + o.ev_rec + 1024u * slot + 32u * lane;
            cp_async16(ra, src);
            cp_async16(ra + 16u, src + 16u);
        }
        next_id += __popc(new_mask);
        if (next_id > p.geo.max_orders) next_id = p.geo.max_orders;  // (later NEW rows fail the same way)
        {
            DP_T0
            cp_async_wait_all();
            if (new_mask) __threadfence();  // the record halves are in place before anything can name these ids
            __syncwarp();
            if (lane == 0u) { DP_ADD(3) }
        }
        if (lane == 0u) {
            sts(sb + o.ev_rf + 4u * slot, rf);
            st_rel(ctl + CT_EV_READY, b + 1u);
        }
    }
}

// TRADES: fill entries also append to the trade log in ring order (deep.cuh); k_deepw's book warp writes the log itself
template <u32 RCAP, bool TRADES, bool NAP = false>
__device__ __forceinline__ void dp_retire_warp(const KParams& p, const DeepOff& o, u32 sb, u32 lane, u64 oh, u64 tr, u32 n_tr0) {
    const u32 ctl = sb + o.ctl;
    u32 head = 0, n_tr = n_tr0, err = 0, ev_pub = 0;
    for (;;) {
        u32 tail = 0, q_ev = 0;
        bool fin = false;
        const bool ok = dp_wait<NAP>(ctl, [&] {
            fin = ld_acq(ctl + CT_FIN) != 0u;  // read before the tail: FIN is set after the last tail update
            q_ev = ld_acq(ctl + CT_Q_EV);      // ... and the event count before the tail it is covered by
            tail = ld_acq(ctl + CT_RET_TAIL);
            // nothing to drain: everything up to `tail` is out and fenced, so is every event counted before it was read
            // (events whose last entry was already drained when their count appeared must not wait for the next entry)
            if (tail == head && q_ev != ev_pub && lane == 0u) {
                ev_pub = q_ev;
                st_rel(ctl + CT_EV_RETIRED, q_ev);
            }
            return tail != head || fin;
        }, lane == 0u ? 10 : 31);
        if (!ok || (tail == head && fin)) break;
        const u32 n = min(32u, tail - head);
        // entry: a = {kind | side << 8 | status << 12 | filled << 16, order id, ., .}, b = {t lo, t hi, ., .}
        uint4 a = make_uint4(0, 0, 0, 0), b = make_uint4(0, 0, 0, 0);
        if (lane < n) {
            const u32 ea = sb + o.ret + DP_RENT * ((head + lane) & (RCAP - 1u));
            a = lds128(ea);
            b = lds128(ea + 16u);
        }
        const u64 t = ((u64)b.y << 32) | b.x;
        const u32 kind = a.x & 0xFFu, side_bit = ((a.x >> 8) & 1u) ? META_BID : 0u, status = (a.x >> 12) & 7u;
        const u32 fm = __ballot_sync(BB_FULL, kind == RK_FILL);
        // entries of one order are applied in ring order: lanes naming the same id take turns
        const u32 grp = __match_any_sync(BB_FULL, lane < n ? a.y : (0xFFFFFF00u | lane));
        const u32 rank = __popc(grp & ((1u << lane) - 1u));
        const u32 rounds = __reduce_max_sync(BB_FULL, rank) + 1u;
        const u64 ra = oh + (u64)a.y * ORD_STRIDE;
        if (TRADES && kind == RK_FILL) {  // {., passive id, traded vol, passive vol left} {t, price, active id}
            const u32 ti = n_tr + __popc(fm & ((1u << lane) - 1u));
            if (ti < p.geo.max_trades) {
                const u64 ta = tr + (u64)ti * 32u;
                stg128_cs(ta, b.x, b.y, b.z, a.z);
                stg128_cs(ta + 16u, b.w, a.y, (a.x >> 8) & 1u, 0u);
            } else if (p.geo.max_trades) {
                err |= ERR_CAP_TRADES;
            }
        }
        for (u32 r = 0; r < rounds; ++r) {
            if (lane < n && rank == r) {
                if (kind == RK_NEW) {  // {., id, vol left, queue position}: the fetch warp wrote the rest of the record
                    stg32(ra + OH_VOL, a.z);
                    stg32(ra + OH_META, status | side_bit);
                    if (status == ST_ACTIVE) {
                        stg32(ra + OH_NEXT, a.w);
                        stg64(ra + OH_KEYT, t);
                    } else {
                        stg64(ra + OC_END, t);
                    }
                } else if (kind == RK_REPLACE) {  // {., id, vol left, queue position} {t, new price}
                    stg128(ra, b.z, a.z, a.w, BB_NIL);
                    stg32(ra + OH_META, status | side_bit);
                    stg64(ra + (status == ST_FILLED ? OC_END : OH_KEYT), t);
                } else if (kind == RK_FILL) {
                    stg32(ra + OH_VOL, a.w);
                    if (a.x & 0x10000u) {
                        stg32(ra + OH_META, ST_FILLED | side_bit);
                        stg64(ra + OC_END, t);
                    }
                } else if (kind == RK_CANCEL) {
                    stg32(ra + OH_META, ST_CANCELLED | side_bit);
                    stg64(ra + OC_END, t);
                } else if (kind == RK_REDUCE) {  // {., id, new vol}
                    stg32(ra + OH_VOL, a.z);
                }
            }
            __syncwarp();
        }
        n_tr += __popc(fm);
        head += n;
        {
            DP_T0
            __threadfence();
            __syncwarp();
            if (lane == 0u) { DP_ADD(11) }
        }
#ifdef DP_PROF
        if (lane == 0u && blockIdx.x == 0) atomicAdd(&g_dp_prof[12], (unsigned long long)n);
#endif
        if (lane == 0u) {
            st_rel(ctl + CT_RET_DONE, head);
            // every entry up to the tail read above is out: so is everything of the events counted before that tail
            if (head == tail) {
                ev_pub = q_ev;
                st_rel(ctl + CT_EV_RETIRED, q_ev);
            }
        }
    }
    err = __reduce_or_sync(BB_FULL, err);
    if (lane == 0u) sts(ctl + CT_RERR, err);
}

}  // namespace bb
#include "deepw.cuh"
namespace bb {

// ---------------------------------------------------------------------------------------------------
// Deep-book replay kernel, batch-parallel (deepw.cuh): one CTA per book; warp 0 = the book (a batch of 32 events, one lane
// each), warp 1 = fetch, warp 2 = retire.  Same blob image, chunk pool, order records and trade log as k_deep.
// ROOMY: at most two books per SM — the staleness filters take their (larger) sizes from the launch; otherwise they are
// compile-time constants and the kernel is the compact one the four-books-per-SM case needs (its instruction cache is the limiter).
// ENV: the second launch of bb_step_device — the slices k_env_deep_stage staged (p.offsets holds {begin, end} per book), NEW
// rows with their ids, trade_vol from 0 (env.rs:117-118), and the closing record also written to p.obs_out.
template <bool ROOMY, bool ENV = false>
__global__ void __launch_bounds__(128, ROOMY ? 2 : 4) k_deepw(const __grid_constant__ KParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    // The four roles rotate with the wave a CTA belongs to (CTAs go round the 148 SMs of a B200, so the up-to-four CTAs that
    // share an SM are 148 apart): the four busy chain warps of an SM then sit on four different schedulers, not on one.
    const u32 lane = threadIdx.x & 31u, warp = ((threadIdx.x >> 5) + blockIdx.x / 148u) & 3u;
    const u32 sb = smem_u32(smem);
    const DeepOff& o = p.dp;
    const u32 ctl = sb + o.ctl;
    const u32 env = blockIdx.x;
    if (env >= p.n_envs) return;
    const u64 oh = (u64)(p.ord + (size_t)env * p.geo.max_orders);
    const u64 tr = (u64)(p.tr + (size_t)env * p.geo.max_trades);
    const u64 off = p.offsets[ENV ? 2u * env : env];
    const u32 n = (u32)(p.offsets[ENV ? 2u * env + 1u : env + 1u] - off);
    const bb_instr* ins = p.instrs + off;
    // ---- set-up: barriers, control words, cache tags, filter; then the book image (one bulk copy)
    if (threadIdx.x == 0) {
        for (u32 i = 0; i <= DW_RB; ++i) mbar_init_a(sb + o.bar + 8u * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // (CT_TICK: the book's tick, read by the level-2 records; loaded once here, off the record path)
    for (u32 i = threadIdx.x; i < CT_WORDS; i += blockDim.x) sts(ctl + 4u * i, 4u * i == CT_TICK ? __ldg(p.geo.ticks + env) : 0u);
    for (u32 i = threadIdx.x; i < (ROOMY ? o.dirty_n : DW_DIRTY); i += blockDim.x) sts(sb + o.dirty + 4u * i, 0u);
    for (u32 i = threadIdx.x; i < (ROOMY ? o.swept_n : DW_SWEPT); i += blockDim.x) sts(sb + (ROOMY ? o.swept : o.scratch + SC_SWEPT) + 4u * i, 0u);
    fence_proxy_async();
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx_a(sb + o.bar, o.smem_image);
        bulk_g2s_a(sb, p.blobs + (size_t)env * p.blob_stride, o.smem_image, sb + o.bar);
        if (!mbar_wait_a(sb + o.bar, 0u)) st_rel(ctl + CT_ABORT, 1u);
    }
    __syncthreads();
    const u32 n_tr0 = min((u32)lds64(sb + HDR_NTRADES_TOTAL), p.geo.max_trades);
#ifdef DP_PROF
    const long long dp_k0 = clock64();
#endif

    BkReg r;
    r.lvol = dp_keep32(sb + o.lvol);
    r.lcnt = dp_keep64((u64)(p.blobs + (size_t)env * p.blob_stride + o.lcnt));  // (the queues' counts / heads / tails stay in the blob)
    r.lht = dp_keep64((u64)(p.blobs + (size_t)env * p.blob_stride + o.lht));
    r.bma = dp_keep32(sb + o.bm);
    r.bmb = dp_keep32(sb + o.bm + 4u * (p.geo.d_levels >> 5));
    r.sma = dp_keep32(sb + o.sm);
    r.smb = dp_keep32(sb + o.sm + 4u * DP_NS);
    r.scr = dp_keep32(sb + o.scratch);
    r.ret = dp_keep32(sb + o.ret);
    r.dirty = dp_keep32(sb + o.dirty);
    r.swept = ROOMY ? dp_keep32(sb + o.swept) : r.scr + SC_SWEPT;  // (compact: a constant offset from the scratch base, no register)
    r.dirty_mask = ROOMY ? o.dirty_n - 1u : DW_DIRTY - 1u;
    r.swept_mask = ROOMY ? o.swept_n - 1u : DW_SWEPT - 1u;
    r.ctl = dp_keep32(ctl);
    r.fs = dp_keep32(sb + DP_OFF_FS);
    r.win_lo = p.geo.d_win_lo; r.W = p.geo.d_levels; r.max_orders = p.geo.max_orders;
    r.n_chunks = p.dp_chunks; r.max_trades = p.geo.max_trades;
    r.oh = dp_keep64(oh);
    r.chunks = dp_keep64((u64)(p.dp_pool + (size_t)env * p.dp_chunks * DP_CHUNK_BYTES));
    r.tr = dp_keep64(tr);
    if (threadIdx.x == 0) {  // the replay warp's scalars, at rest
        sts(ctl + RS_BUMP, lds(sb + DP_OFF_BUMP));
        sts(ctl + RS_NFREE, lds(sb + DP_OFF_NFREE));
        sts(ctl + RS_NTR, n_tr0);
        sts(ctl + RS_RET_TAIL, 0u);
    }
    __syncthreads();
    if (warp == 1u) {
        dp_fetch_warp<DW_RB, true, ENV>(p, o, sb, lane, ins, n, oh, lds(sb + HDR_NORDERS));
    } else if (warp == 2u) {
        dp_retire_warp<DW_RCAP, false, true>(p, o, sb, lane, oh, tr, n_tr0);
    } else if (warp == 3u) {
        bk_replay_warp(r, lane, n_tr0);
    } else if (warp == 0u) {
        // ---- the chain warp ---------------------------------------------------------------------------------------
        const u32 ev_ins = dp_keep32(sb + o.ev_ins), ev_rec = dp_keep32(sb + o.ev_rec);
        BkSt s;
        s.t = lds64(sb + HDR_T);
        s.max_key_time = lds64(sb + HDR_MAXKT);
        s.n_orders = lds(sb + HDR_NORDERS);
        s.trade_vol = ENV ? 0u : lds(sb + HDR_TRADEVOL);
        s.vol_ask = lds(sb + HDR_SIDEVOL);
        s.vol_bid = lds(sb + HDR_SIDEVOL + 4u);
        s.bq_ask = lds(sb + HDR_BESTQ);
        s.bq_bid = lds(sb + HDR_BESTQ + 4u);
        s.flags = (lds(sb + HDR_TRADING) ? FL_TRADING : 0u) | (lds(sb + HDR_HASBEST) ? FL_HAS_ASK : 0u) |
                  (lds(sb + HDR_HASBEST + 4u) ? FL_HAS_BID : 0u);
        s.err = 0u;
        s.d_instr = s.d_applied = 0u;
        s.zv = lds(sb + HDR_FREETOP);
        s.bump = s.n_free = 0u;  // (the queues' scalars are the replay warp's; bk_borrow brings them over)
        s.n_tr = n_tr0;
        s.ret_tail = s.ret_pub = s.ret_room = 0u;
        s.n_emit = s.done_seen = s.drain_seq = 0u;
#ifdef DP_PROF
        s.pf_flush = s.pf_rounds = s.pf_mops = s.pf_ser = 0u;
        for (int i = 0; i < 8; ++i) s.pf_reason[i] = 0u;
#endif
        const u32 n_orders0 = s.n_orders, trade_vol0 = s.trade_vol;
        const u32 fast = p.dp_fast;
        u32 lane_err = 0u;
        bool aborted = false;
        const u32 nb = (n + 31u) >> 5;
        for (u32 b = 0; b < nb && !aborted; ++b) {
            const u32 bslot = b & (DW_RB - 1u);
            if (!bk_wait(r, lane, [&] { return ld_acq(r.ctl + CT_EV_READY) > b; }, 6)) { aborted = true; break; }
            const u32 rf = lds(sb + o.ev_rf + 4u * bslot);
            const u32 cnt = min(32u, n - 32u * b);
            uint4 x = make_uint4(0, 0, 0, 0), y = x, a = x, c = x;
            if (lane < cnt) {
                const u32 eo = 1024u * bslot + 32u * lane;
                x = lds128(ev_ins + eo);
                y = lds128(ev_ins + eo + 16u);
                a = lds128(ev_rec + eo);
                c = lds128(ev_rec + eo + 16u);
            }
            u32 pending = cnt >= 32u ? BB_FULL : ((1u << cnt) - 1u);
            while (pending) {
                u32 obs_lane = 32u;
                if (!bk_batch<!ROOMY, ENV>(r, s, lane, pending, x, y, a, c, 32u * b, rf, fast, lane_err, obs_lane)) { aborted = true; break; }
                if (obs_lane < 32u) {  // Level2DataRecords::append_record (data.rs:44-56) for a row flagged BB_F_EMIT
                    const u32 bid = (s.flags & FL_HAS_BID) ? r.win_lo + s.bq_bid : 0u;
                    const u32 ask = (s.flags & FL_HAS_ASK) ? r.win_lo + s.bq_ask : 0xFFFFFFFFu;
                    u32 w0, w1;
                    bk_obs(r, lds(r.ctl + CT_TICK), lane, s.trade_vol, bid, ask, s.vol_ask, s.vol_bid, &w0, &w1);
                    // (a level-1 record is the first 9 words of the level-2 one: words 5..8 are the touch level of each side)
                    if (ENV && p.obs_out) {  // the step's observation (bb_step_device's d_obs_out)
                        u32* ob = p.obs_out + (size_t)env * p.obs_words;
                        if (lane < p.obs_words) ob[lane] = w0;
                        if (lane + 32u < p.obs_words) ob[lane + 32u] = w1;
                    }
                    const u32 nrec = lds(sb + HDR_NSTEPS);
                    __syncwarp();
                    if (nrec < p.max_steps) {
                        const u64 dst = (u64)(p.hist + (size_t)env * p.hist_env_stride + (size_t)nrec * p.obs_words);
                        if (lane < p.obs_words) stg32(dst + 4u * lane, w0);
                        if (lane + 32u < p.obs_words) stg32(dst + 4u * (lane + 32u), w1);
                        if (lane == 0u) sts(sb + HDR_NSTEPS, nrec + 1u);
                    } else {
                        s.err |= ERR_CAP_STEPS;
                    }
                    __syncwarp();
                    bk_give_back(r, s, lane);  // (bk_batch came back with the queues still borrowed)
                }
            }
            if (lane == 0u) st_rel(r.ctl + CT_EV_CONSUMED, b + 1u);
        }
        // ---- the replay warp finishes and parks; the header goes back into the image; the retire warp drains what is left and
        // exits on FIN, the replay warp on FIN_L
        if (!aborted && !bk_borrow(r, s, lane)) aborted = true;
        lane_err = __reduce_or_sync(BB_FULL, lane_err);
        __syncwarp();
        if (lane == 0u) {
            if (!aborted) st_rel(r.ctl + CT_RET_TAIL, s.ret_tail);
            st_rel(r.ctl + CT_FIN, 1u);
            st_rel(r.ctl + CT_FIN_L, 1u);
            sts64(sb + HDR_T, s.t);
            sts64(sb + HDR_MAXKT, s.max_key_time);
            sts64(sb + HDR_NCREATED, lds64(sb + HDR_NCREATED) + (s.n_orders - n_orders0));
            sts(sb + HDR_NORDERS, s.n_orders);
            sts(sb + HDR_TRADEVOL, s.trade_vol);
            sts(sb + HDR_SIDEVOL, s.vol_ask);
            sts(sb + HDR_SIDEVOL + 4u, s.vol_bid);
            sts(sb + HDR_BESTQ, s.bq_ask);
            sts(sb + HDR_BESTQ + 4u, s.bq_bid);
            sts(sb + HDR_TRADING, (s.flags & FL_TRADING) ? 1u : 0u);
            sts(sb + HDR_HASBEST, (s.flags & FL_HAS_ASK) ? 1u : 0u);
            sts(sb + HDR_HASBEST + 4u, (s.flags & FL_HAS_BID) ? 1u : 0u);
            sts(sb + HDR_FREETOP, s.zv);
            sts(sb + DP_OFF_BUMP, s.bump);
            sts(sb + DP_OFF_NFREE, s.n_free);
            sts64(sb + HDR_NINSTR, lds64(sb + HDR_NINSTR) + s.d_instr);
            // traded volume: trade_vol is never reset in replay mode; transitions: one per applied event and one per fill
            sts64(sb + HDR_VOLUME, lds64(sb + HDR_VOLUME) + (u32)(s.trade_vol - trade_vol0));
            sts64(sb + HDR_NTRANS, lds64(sb + HDR_NTRANS) + s.d_applied + (s.n_tr - n_tr0));
            sts(ctl + CT_LERR, s.err | lane_err);
            sts(ctl + CT_QNTR, s.n_tr - n_tr0);
            if (aborted) st_rel(ctl + CT_ABORT, 1u);
#ifdef DP_PROF
            if (blockIdx.x == 0)
                printf("k_deepw chain warp: runs %u, serial events %u (emit %u state %u big %u doubt %u same-id %u "
                       "time %u zero %u other %u)\n", s.pf_flush, s.pf_ser, s.pf_reason[0], s.pf_reason[1], s.pf_reason[2],
                       s.pf_reason[3], s.pf_reason[4], s.pf_reason[5], s.pf_reason[6], s.pf_reason[7]);
#endif
        }
    }
    __syncthreads();
#ifdef DP_PROF
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const char* nm[16] = {"-", "F:wait_consumed", "F:tma", "F:cpasync+fence", "C:ring_room", "C:borrow", "C:wait_ev", "P:wait_work",
                              "P:ret_room", "-", "R:wait", "R:fence", "R:entries", "C:doubt", "C:late", "-"};
        printf("k_deepw prof: n=%u cycles=%lld\n", n, clock64() - dp_k0);
        for (int i = 1; i < 15; ++i) {
            if (nm[i][0] != '-') printf("  %-16s cycles %12llu  count %10llu\n", nm[i], g_dp_prof[i], g_dp_prof[32 + i]);
            g_dp_prof[i] = 0; g_dp_prof[32 + i] = 0;
        }
    }
#endif
    if (threadIdx.x == 0) {
        const u32 fills = lds(ctl + CT_QNTR);
        const u64 tt = lds64(sb + HDR_NTRADES_TOTAL) + fills;
        sts64(sb + HDR_NTRADES_TOTAL, tt);
        sts(sb + HDR_NTRADES, (u32)min(tt, (u64)p.geo.max_trades));
        u32 err = lds(ctl + CT_RERR) | lds(ctl + CT_LERR) | lds(ctl + RS_ERR);
        if (ld_acq(ctl + CT_ABORT)) err |= 0x80000000u;
        sts(sb + HDR_ERR, lds(sb + HDR_ERR) | (err & 0x7FFFFFFFu));
        if (err) atomicOr(p.err_flag, err);
        fence_proxy_async();
        bulk_s2g_a(p.blobs + (size_t)env * p.blob_stride, sb, o.smem_image);
        bulk_commit();
        bulk_wait_all<0>();
    }
}

// ---------------------------------------------------------------------------------------------------
// bb_step_device on the deep engine, first of its two launches (the second is k_deepw<.., ENV>): Env::step up to the
// processing of its events (env.rs:116-127), one warp per book.  The rows are submitted as on the other engines
// (submit_rows: ids in row order, status New published, off-tick prices and rows past max_queue flagged), the queue is
// shuffled with the book's Xoroshiro stream (Fisher-Yates from the back, as k_apply), and the result is written as a replay
// slice into the staging stream: row stage[book][i] is event i at start + i (a NEW with its id), then a no-op at
// start + step_size flagged BB_F_EMIT that appends the step's record.  stage_off[2 book], [2 book + 1]: the slice's bounds.
// The header takes the new order count, stream state and step counter.  Dynamic shared memory: the permutation, u16
// [max_queue].
__global__ void __launch_bounds__(32) k_env_deep_stage(const __grid_constant__ KParams p, bb_instr* stage, u64* stage_off) {
    extern __shared__ __align__(128) unsigned char smem[];
    const u32 lane = threadIdx.x, env = blockIdx.x, perm = smem_u32(smem);
    BookHdr* hdr = reinterpret_cast<BookHdr*>(p.blobs + (size_t)env * p.blob_stride);
    Book b;
    b.env = env;
    b.lane = lane;
    b.err = 0u;
    b.oh = (u64)(p.ord + (size_t)env * p.geo.max_orders);
    const u64 off = p.offsets[env];
    const u32 m = (u32)(p.offsets[env + 1] - off), mm = min(m, p.max_queue);  // the first max_queue rows run
    if (m > p.max_queue) b.err |= ERR_CAP_QUEUE;
    const u32 n0 = hdr->n_orders;
    const u64 start = hdr->t;
    RowCount c{n0, 0u, 0u};
    submit_rows<false, false>(p.geo, p, b, off, m, mm, 0u, c, [&](u32 j, uint4, uint4, bool, bool, u32, u32 pos, u32) { sts16(perm + 2u * pos, j); });
    __syncwarp();
    if (lane == 0u) {  // transactions.shuffle(rng) (env.rs:121)
        u64 s0 = hdr->rng_s0, s1 = hdr->rng_s1;
        for (u32 i = c.n; i > 1; --i) {
            const u32 j = xoroshiro_range(s0, s1, i);
            const u32 x = lds16(perm + 2u * (i - 1)), y = lds16(perm + 2u * j);
            sts16(perm + 2u * (i - 1), y);
            sts16(perm + 2u * j, x);
        }
        hdr->rng_s0 = s0;
        hdr->rng_s1 = s1;
        hdr->n_orders = c.next;
        hdr->n_created += c.next - n0;
        hdr->step_counter += 1u;
        if (b.err) {
            hdr->err |= b.err;
            atomicOr(p.err_flag, b.err);
        }
    }
    __syncwarp();
    const u64 base = (u64)env * (p.max_queue + 1u);
    uint4* dst = reinterpret_cast<uint4*>(stage + base);
    for (u32 i = lane; i < c.n; i += 32u) {
        const u32 j = lds16(perm + 2u * i);
        const uint4* src = reinterpret_cast<const uint4*>(p.instrs + off + j);
        uint4 x = src[0];
        const u64 t = start + i;
        x.x = (u32)t;
        x.y = (u32)(t >> 32);
        x.z &= ~BB_F_EMIT;
        if ((x.z & BB_OP_MASK) == BB_OP_NEW) x.w = (u32)p.out_ids[off + j];
        dst[2u * i] = x;
        dst[2u * i + 1u] = src[1];
    }
    if (lane == 0u) {
        const u64 t = start + p.step_size;  // env.rs:129-134
        dst[2u * c.n] = make_uint4((u32)t, (u32)(t >> 32), BB_OP_NOOP | BB_F_EMIT, 0u);
        dst[2u * c.n + 1u] = make_uint4(0u, 0u, 0u, 0u);
        stage_off[2u * env] = base;
        stage_off[2u * env + 1u] = base + c.n + 1u;
    }
}

// ---------------------------------------------------------------------------------------------------
// bb_run_agents(_with_rows) on the deep engine, first of the two launches of each step (the second is k_deepw<.., ENV>): one
// k_sim<.., MOM, EXT> step up to the processing of its events, one warp per book.  The groups update in declaration order
// exactly as in k_sim (held ids in p.rslot, Momentum / Noise state in p.mom, the touch from the header's has_best / best_q)
// into the book's queue in global scratch, p.scratch [n_envs][max_queue]; a launch given rows (p.offsets) submits them next
// (submit_rows: NEW and CANCEL only).  Past max_queue events the queue is truncated and flagged ERR_CAP_QUEUE; it is checked
// against the book's tick when rand_tick_mask is set, shuffled with k_sim's Philox draws (shuffle_queue), and written as a
// replay slice in k_env_deep_stage's layout: event i at start + i (a NEW with its id, trader and price; a market order keeps
// its sentinel price, which k_deepw routes to the market path), then the BB_F_EMIT no-op at start + step_size.  Every staged
// NEW's record is published with status New, as create_order does at submission.  The header takes the new order count
// and step counter; the Xoroshiro stream is not used.  Dynamic shared memory: the permutation, then the swap targets, u16
// [max_queue] each, 16-byte aligned.
template <bool PU>
__global__ void __launch_bounds__(32) k_env_agents_stage(const __grid_constant__ KParams p, bb_instr* stage, u64* stage_off) {
    extern __shared__ __align__(128) unsigned char smem[];
    const u32 lane = threadIdx.x, env = blockIdx.x, perm = smem_u32(smem), jarr = perm + ((2u * p.max_queue + 15u) & ~15u);
    BookHdr* hdr = reinterpret_cast<BookHdr*>(p.blobs + (size_t)env * p.blob_stride);
    Book b;
    b.env = env;
    b.lane = lane;
    b.err = 0u;
    b.oh = (u64)(p.ord + (size_t)env * p.geo.max_orders);
    uint4* q = p.scratch + (size_t)env * p.max_queue;
    const u32 env_g = p.env_id_base + env, step = hdr->step_counter, n0 = hdr->n_orders, tick = __ldg(p.geo.ticks + env);
    const u64 start = hdr->t;
    const u32 bid = hdr->has_best[1] ? p.geo.d_win_lo + hdr->best_q[1] : 0u;
    const u32 ask = hdr->has_best[0] ? p.geo.d_win_lo + hdr->best_q[0] : 0xFFFFFFFFu;
    u32 key_l = 0, key_h = 0;
    const bb_agent_group* urow = nullptr;
    if constexpr (PU) {
        unit_key(p, env, key_l, key_h);
        urow = p.unit_groups + (size_t)env * p.n_groups;
    }
    u32* slots = p.rslot + (size_t)env * p.agents_per_env;
    // ---- agents.update(env, rng) in declaration order (crates/macros/src/lib.rs:57-72)
    Emit e;
    e.n = 0;
    e.next_id = n0;
    u32 slot_base = 0, mi = 0;
    for (u32 gi = 0; gi < p.n_groups; ++gi) {
        const bb_agent_group& ag = PU ? urow[gi] : p.groups[gi];
        if (ag.kind == BB_GROUP_RANDOM) {
            random_agents_update<PU>(p, ag, b, q, e, slots, env_g, step, slot_base, key_l, key_h);
        } else {
            const MomOut mo = momentum_agent_update<PU>(p, ag, b.oh, tick, bid, ask, q, e.n, e.next_id,
                                                        (MomState*)((char*)p.mom + ((size_t)env * p.mom_groups_per_env + mi) * p.mom_stride),
                                                        env_g, step, gi, slot_base);
            e.n = mo.n;
            e.next_id = mo.next_id;
            b.err |= mo.err;
            ++mi;
        }
        slot_base += ag.n_agents;
    }
    if (p.offsets) {  // the caller's rows, after the agents' instructions
        const u64 off = p.offsets[env];
        const u32 m = (u32)(p.offsets[env + 1] - off);
        RowCount rows{e.next_id, e.n, 0u};
        submit_rows<false, true>(p.geo, p, b, off, m, m, 0u, rows, [&](u32, uint4 x, uint4 y, bool, bool is_new, u32 id, u32 pos, u32) {
            if (pos < p.max_queue) q[pos] = row_event(x, y, is_new, id);
        });
        e.next_id = rows.next;
        e.n = rows.n;
    }
    if (e.n > p.max_queue) b.err |= ERR_CAP_QUEUE;
    const u32 n = min(e.n, p.max_queue);
    if (p.rand_tick_mask) agent_tick_check<false>(q, 0u, tick, n, lane, b.err);
    __syncwarp();
    shuffle_queue<PU, false>(p, perm, jarr, 0u, n, env_g, step, key_l, key_h, lane);
    const u64 base = (u64)env * (p.max_queue + 1u);
    uint4* dst = reinterpret_cast<uint4*>(stage + base);
    for (u32 i = lane; i < n; i += 32u) {
        const uint4 ev = q[lds16(perm + 2u * i)];
        const bool is_new = (ev.x & 1u) != 0u, side_bid = (ev.x & 2u) != 0u;
        if (is_new && ev.y < p.geo.max_orders) stg32(b.oh + (u64)ev.y * ORD_STRIDE + OH_META, ST_NEW | (side_bid ? META_BID : 0u));
        const u64 t = start + i;
        dst[2u * i] = make_uint4((u32)t, (u32)(t >> 32), is_new ? (BB_OP_NEW | (side_bid ? BB_F_BID : 0u)) : BB_OP_CANCEL, ev.y);
        dst[2u * i + 1u] = make_uint4(ev.z, ev.w, is_new ? ev.x >> 13 : 0u, 0u);
    }
    if (lane == 0u) {
        const u64 t = start + p.step_size;  // env.rs:129-134
        dst[2u * n] = make_uint4((u32)t, (u32)(t >> 32), BB_OP_NOOP | BB_F_EMIT, 0u);
        dst[2u * n + 1u] = make_uint4(0u, 0u, 0u, 0u);
        stage_off[2u * env] = base;
        stage_off[2u * env + 1u] = base + n + 1u;
        hdr->n_orders = e.next_id;  // create_order at submission (env.rs:173)
        hdr->n_created += e.next_id - n0;
        hdr->step_counter = step + 1u;
        if (b.err) {
            hdr->err |= b.err;
            atomicOr(p.err_flag, b.err);
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Live market data of every book: out45[env][45] (level_2_data layout) and out8[env][8] =
// OrderBook::level_1_data field order (orderbook.rs:287-301, touch by the `volumes` map).
// `only` [n_books] or nullptr: write the rows of the books whose entry is non-zero (bb_restore_device's restored books)
template <int ENG> __global__ void __launch_bounds__(128) k_snapshot(const __grid_constant__ KParams p, u32* out45, u32* out8,
                                                                     u32 first_env, u32 n_out, u32 words = 45u,
                                                                     const uint8_t* only = nullptr) {
    extern __shared__ __align__(128) unsigned char smem[];
    const u32 lane = keep32(threadIdx.x & 31u), warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const u32 sb = keep32(smem_u32(smem) + warp * p.warp_smem_bytes);
    const u32 bar = sb + p.off_bar;
    const GeoT<ENG>& g = static_cast<const GeoT<ENG>&>(p.geo);
    if (lane == 0) {
        mbar_init_a(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_proxy_async();
    __syncwarp();
    u32 ph = 0;
    pcache_init(g, sb, lane);
    for (u32 i = blockIdx.x * wpb + warp; i < n_out; i += gridDim.x * wpb) {
        const u32 env = first_env + i;
        if (only && !only[env]) continue;
        Book b;
        make_book(b, p, sb, env, lane);
        if (!blob_load(p, sb, env, bar, ph, lane)) return;
        book_from_header(g, b);
        u32 w0, w1;
        book_obs(g, b, 45u, &w0, &w1);
        if (out45) {  // `words` = 45 (level-2 record) or 9 (its level-1 prefix, rows packed)
            if (lane < words) out45[(size_t)i * words + lane] = w0;
            if (lane + 32u < words) out45[(size_t)i * words + 32u + lane] = w1;
        }
        if (out8) {
            u32 bv, bc, av, ac;
            best_by_volumes(g, b, 1, &bv, &bc);
            best_by_volumes(g, b, 0, &av, &ac);
            const u32 bid = best_price(g, b, 1), ask = best_price(g, b, 0);
            const u32 v = lane == 0 ? bid : lane == 1 ? ask : lane == 2 ? b.vol_bid : lane == 3 ? b.vol_ask
                        : lane == 4 ? bv : lane == 5 ? av : lane == 6 ? bc : ac;
            if (lane < 8) out8[(size_t)i * 8u + lane] = v;
        }
        __syncwarp();
    }
}

// bb_reset_device: which units k_init / k_init_deep reset and what else the launch writes.  mask == nullptr: every book,
// from the handle's creation seeds (bb_create, bb_reset).  A unit is an env, or a market of `assets` books.
struct ResetArgs {
    const uint8_t* mask;  // [units]; 0 leaves the unit's books untouched
    const u64* seeds;     // [units] or nullptr: re-seed the unit's shuffle stream and restart its step counter, or keep both
    u32 assets;
    u32* obs;             // [n_envs][obs_words] or nullptr: the fresh book's record (bb_level1_device / bb_level2_device)
    u32 obs_words;
    u32* cursor;          // [n_envs] or nullptr: a bb_trades_device cursor, zeroed for reset books
};

// Xoroshiro128StarStar::seed_from_u64: two SplitMix64 outputs (as upload_seeds on the host)
__device__ __forceinline__ void seed_stream(BookHdr& h, u64 x) {
    u64 z[2];
    for (int i = 0; i < 2; ++i) {
        x += 0x9e3779b97f4a7c15ULL;
        u64 y = x;
        y = (y ^ (y >> 30)) * 0xbf58476d1ce4e5b9ULL;
        y = (y ^ (y >> 27)) * 0x94d049bb133111ebULL;
        z[i] = y ^ (y >> 31);
    }
    h.rng_s0 = z[0];
    h.rng_s1 = z[1];
}

// thread 0 of a book's CTA: the fresh header (OrderBook::new orderbook.rs:158-171 + Env::new env.rs:84-95) with its random
// streams.  A masked reset reads the old header's stream and step counter before the caller overwrites it.
__device__ __forceinline__ BookHdr fresh_hdr(const unsigned char* b, u32 env, u64 start_time, u32 trading, const u64* rng_seeds,
                                             const ResetArgs& r) {
    BookHdr h;
    memset(&h, 0, sizeof(h));
    h.t = start_time;
    h.trading = trading;
    if (!r.mask) {
        h.rng_s0 = rng_seeds[2 * env];
        h.rng_s1 = rng_seeds[2 * env + 1];
    } else if (r.seeds) {
        seed_stream(h, r.seeds[env / r.assets]);
    } else {
        const BookHdr* old = reinterpret_cast<const BookHdr*>(b);
        h.rng_s0 = old->rng_s0;
        h.rng_s1 = old->rng_s1;
        h.step_counter = old->step_counter;
    }
    return h;
}

// what a reset book's CTA writes besides its blob: the fresh record (an empty book: ask = 0xFFFFFFFF, every other word 0)
// and its trade cursor
__device__ __forceinline__ void reset_outputs(u32 env, const ResetArgs& r) {
    if (r.obs)
        for (u32 i = threadIdx.x; i < r.obs_words; i += blockDim.x) r.obs[(size_t)env * r.obs_words + i] = i == 2u ? 0xFFFFFFFFu : 0u;
    if (r.cursor && threadIdx.x == 0) r.cursor[env] = 0u;
}

// the agents' state of a fresh book (k_init, k_init_deep): no held orders, no momentum history, empty live-order lists
__device__ __forceinline__ void reset_agents(u32 env, u32* rslot, u32 agents_per_env, MomState* mom, u32 mom_per_env, u32 mom_stride) {
    if (rslot)
        for (u32 i = threadIdx.x; i < agents_per_env; i += blockDim.x) rslot[(size_t)env * agents_per_env + i] = BB_NIL;
    if (mom)
        for (u32 i = threadIdx.x; i < mom_per_env; i += blockDim.x) {
            MomState* m = (MomState*)((char*)mom + ((size_t)env * mom_per_env + i) * mom_stride);
            m->momentum = 0.0; m->last_price = 0.0; m->has_last = 0; m->n_live = 0;
        }
}

// fresh-book initialisation (OrderBook::new orderbook.rs:158-171 + Env::new env.rs:84-95), of every book or of the units
// r.mask selects
__global__ void k_init(unsigned char* blobs, u64 blob_stride, u32 n_envs, u32 p_total, u64 start_time, u32 trading,
                       const u64* rng_seeds, u32* rslot, u32 agents_per_env, MomState* mom, u32 mom_per_env, u32 mom_stride, Geo dense,
                       u32 dense_lp, u32 dense_nwmax, ResetArgs r) {
    const u32 env = blockIdx.x;
    if (env >= n_envs) return;
    if (r.mask && !r.mask[env / r.assets]) return;
    unsigned char* b = blobs + (size_t)env * blob_stride;
    if (threadIdx.x == 0) {
        BookHdr h = fresh_hdr(b, env, start_time, trading, rng_seeds, r);
        h.free_top = dense.d_live;
        *reinterpret_cast<BookHdr*>(b) = h;
    }
    reset_outputs(env, r);
    if (dense_lp) {  // dense engine (DenseLayout<dense_lp, dense_nwmax>): empty bitmaps, every slot free
        const u32 off_fs = 128u + 12u * dense_lp, off_bm = off_fs + dense_lp;
        u32* bm = reinterpret_cast<u32*>(b + off_bm);
        for (u32 i = threadIdx.x; i < 2 * dense_nwmax; i += blockDim.x) bm[i] = 0;
        u32* ids = reinterpret_cast<u32*>(b + 128);
        for (u32 i = threadIdx.x; i < dense_lp; i += blockDim.x) {
            ids[i] = BB_NIL;
            b[off_fs + i] = (unsigned char)(i < dense.d_live ? dense.d_live - 1 - i : 0xFF);
        }
    } else {
        u32* tag = reinterpret_cast<u32*>(b + 128);
        for (u32 i = threadIdx.x; i < p_total; i += blockDim.x) {
            tag[i] = BB_TAG_FREE;
            tag[p_total + i] = 0;
            tag[2 * p_total + i] = 0;
        }
    }
    reset_agents(env, rslot, agents_per_env, mom, mom_per_env, mom_stride);
}

// fresh deep book (deep.cuh image): header, empty bitmaps, chunk 0 reserved as a sink; its agents' state as k_init's
__global__ void k_init_deep(unsigned char* blobs, u64 blob_stride, u32 n_envs, u64 start_time, u32 trading, const u64* rng_seeds,
                            u32 off_bm, u32 bm_bytes, u32* rslot, u32 agents_per_env, MomState* mom, u32 mom_per_env, u32 mom_stride,
                            ResetArgs r) {
    const u32 env = blockIdx.x;
    if (env >= n_envs) return;
    if (r.mask && !r.mask[env / r.assets]) return;
    unsigned char* b = blobs + (size_t)env * blob_stride;
    reset_outputs(env, r);
    if (threadIdx.x == 0) {
        *reinterpret_cast<BookHdr*>(b) = fresh_hdr(b, env, start_time, trading, rng_seeds, r);
        *reinterpret_cast<u32*>(b + DP_OFF_BUMP) = 1u;
        *reinterpret_cast<u32*>(b + DP_OFF_NFREE) = 0u;
    }
    u32* bm = reinterpret_cast<u32*>(b + off_bm);
    for (u32 i = threadIdx.x; i < bm_bytes / 4u; i += blockDim.x) bm[i] = 0u;
    reset_agents(env, rslot, agents_per_env, mom, mom_per_env, mom_stride);
}

// live market data of deep books, read straight from the blobs in HBM (same outputs as k_snapshot)
__global__ void __launch_bounds__(128) k_snapshot_deep(const __grid_constant__ KParams p, u32* out45, u32* out8, u32 first_env, u32 n_out,
                                                       u32 words, const uint8_t* only = nullptr) {
    const u32 lane = threadIdx.x & 31u, i = blockIdx.x * 4u + (threadIdx.x >> 5);
    if (i >= n_out) return;
    const u32 env = first_env + i;
    if (only && !only[env]) return;
    const unsigned char* b = p.blobs + (size_t)env * p.blob_stride;
    const BookHdr* h = reinterpret_cast<const BookHdr*>(b);
    const u32 W = p.geo.d_levels, nw = W >> 5, lo = p.geo.d_win_lo;
    const u32* bm = reinterpret_cast<const u32*>(b + p.dp.bm);
    const u32* lvol = reinterpret_cast<const u32*>(b + p.dp.lvol);
    const u32* lcnt = reinterpret_cast<const u32*>(b + p.dp.lcnt);
    auto level_at = [&](u32 side, u32 price, u32* vol, u32* cnt) {
        *vol = *cnt = 0;
        const u32 q = price - lo;
        if (q >= W) return;
        if (!((bm[(side ? nw : 0u) + (q >> 5)] >> (q & 31u)) & 1u)) return;
        *vol = lvol[q];
        *cnt = lcnt[q];
    };
    const u32 bid = h->has_best[1] ? lo + h->best_q[1] : 0u, ask = h->has_best[0] ? lo + h->best_q[0] : 0xFFFFFFFFu;
    if (out45) {
        const u32 tick = __ldg(p.geo.ticks + env);
        for (u32 w = lane; w < words; w += 32u) {
            u32 val;
            if (w >= 5u) {
                const u32 k = (w - 5u) >> 2, f = (w - 5u) & 3u;
                u32 v, n;
                if (f < 2u) level_at(1u, bid - k * tick, &v, &n);
                else level_at(0u, ask + k * tick, &v, &n);
                val = (f & 1u) ? n : v;
            } else {
                val = w == 0 ? h->trade_vol : w == 1 ? bid : w == 2 ? ask : w == 3 ? h->side_vol[0] : h->side_vol[1];
            }
            out45[(size_t)i * words + w] = val;
        }
    }
    if (out8 && lane < 8u) {
        u32 bv, bc, av, ac;
        level_at(1u, bid, &bv, &bc);
        level_at(0u, ask, &av, &ac);
        out8[(size_t)i * 8u + lane] = lane == 0 ? bid : lane == 1 ? ask : lane == 2 ? h->side_vol[1] : lane == 3 ? h->side_vol[0]
                                      : lane == 4 ? bv : lane == 5 ? av : lane == 6 ? bc : ac;
    }
}

// bb_orders_device: the records of order ids named by a [units][n_per_unit] query block (get_orders()[id] / order_status(id),
// rust/src/step_sim_numpy.rs), one thread per query.  Query q of unit u reads book u, or book u * assets + asset[q] on a
// multi-asset handle.  The first 32-byte sector of a record (price, vol, links, key time, meta, start_vol) is always read;
// the second (arr_time, end_time, trader) only when one of its columns is requested.  A BB_NO_ID query, an id without a
// record (ERR_BAD_ID on its book) and an asset outside the market (ERR_ROW_OP on the market's book 0) write "no order":
// BB_STATUS_NONE and zeros.  Record and header layouts are shared by every engine, so one instantiation serves them all.
__global__ void __launch_bounds__(256) k_orders_gather(unsigned char* blobs, u64 blob_stride, const OrderRec* ord, u32 max_orders,
                                                       const u64* ids, const u32* asset, u32 assets, u64 n_per_unit, u64 n_queries,
                                                       uint8_t* side_is_bid, uint8_t* status, u64* arr_time, u64* end_time, u32* vol,
                                                       u32* start_vol, u32* price, u32* trader) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_queries) return;
    const u64 unit = q / n_per_unit, id = __ldg(ids + q);
    uint4 s0 = make_uint4(0u, 0u, 0u, 0u), s1 = s0, c0 = s0, c1 = s0;  // the record's two sectors, 16 bytes at a time
    u32 st = BB_STATUS_NONE;
    if (id != BB_NO_ID) {
        u64 book = unit;
        u32 bad = 0u;
        if (asset) {
            const u32 a = __ldg(asset + q);
            book = unit * assets + (a < assets ? a : 0u);
            if (a >= assets) bad = ERR_ROW_OP;
        }
        BookHdr* h = reinterpret_cast<BookHdr*>(blobs + book * blob_stride);
        if (!bad && (id >= __ldg(&h->n_orders) || id >= max_orders)) bad = ERR_BAD_ID;
        if (bad) {
            atomicOr(&h->err, bad);
        } else {
            const uint4* r = reinterpret_cast<const uint4*>(ord + book * max_orders + id);
            s0 = __ldg(r);
            s1 = __ldg(r + 1);
            if (arr_time || end_time || trader) {
                c0 = __ldg(r + 2);
                c1 = __ldg(r + 3);
            }
            st = s1.z & META_STATUS_MASK;
        }
    }
    if (side_is_bid) side_is_bid[q] = (s1.z & META_BID) ? 1u : 0u;
    if (status) status[q] = (uint8_t)st;
    if (arr_time) arr_time[q] = ((u64)c0.y << 32) | c0.x;
    if (end_time) end_time[q] = ((u64)c0.w << 32) | c0.z;
    if (vol) vol[q] = s0.y;
    if (start_vol) start_vol[q] = s1.w;
    if (price) price[q] = s0.x;
    if (trader) trader[q] = c1.x;
}

// bb_trades_device: per book, the trades logged since the caller's cursor (get_trades(), rust/src/types.rs:4-17), one warp
// per book.  Lanes copy consecutive 32-byte records of the log into row `book` of the [n_books][cap] columns and pad the
// rest of the row with (0, 0, 0, 0, BB_NO_ID, BB_NO_ID); lane 0 writes the count and the advanced cursor.  Nothing at or
// beyond min(n_trades, max_trades) is read.
__global__ void __launch_bounds__(256) k_trades_window(const unsigned char* blobs, u64 blob_stride, const TradeRec* tr, u32 max_trades,
                                                       u32 n_books, u32* cursor, u32 cap, u32* count, u64* t, uint8_t* side_is_bid,
                                                       u32* price, u32* vol, u64* active_id, u64* passive_id) {
    const u32 lane = threadIdx.x & 31u, book = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (book >= n_books) return;
    u32 c = 0u, logged = 0u;
    if (lane == 0u) {  // (one lane reads the cursor it alone writes back)
        c = cursor[book];
        logged = min(__ldg(&reinterpret_cast<const BookHdr*>(blobs + (u64)book * blob_stride)->n_trades), max_trades);
    }
    c = __shfl_sync(BB_FULL, c, 0);
    logged = __shfl_sync(BB_FULL, logged, 0);
    const u32 avail = c < logged ? logged - c : 0u, n = min(avail, cap);
    const uint4* src = reinterpret_cast<const uint4*>(tr + (u64)book * max_trades + c);
    const u64 row = (u64)book * cap;
    for (u32 i = lane; i < cap; i += 32u) {
        uint4 a = make_uint4(0u, 0u, 0u, 0u), b = a;
        u64 act = BB_NO_ID, pas = BB_NO_ID;
        if (i < n) {
            a = __ldg(src + 2u * i);      // t, price, vol
            b = __ldg(src + 2u * i + 1u);  // active, passive, side_bid
            act = b.x;
            pas = b.y;
        }
        if (t) t[row + i] = ((u64)a.y << 32) | a.x;
        if (side_is_bid) side_is_bid[row + i] = (uint8_t)b.z;
        if (price) price[row + i] = a.z;
        if (vol) vol[row + i] = a.w;
        if (active_id) active_id[row + i] = act;
        if (passive_id) passive_id[row + i] = pas;
    }
    if (lane == 0u) {
        if (count) count[book] = avail;
        if (n) cursor[book] = c + n;
    }
}

// bb_save_device / bb_restore_device.  A slot holds one unit (an env, or a market of `assets` books); slot book k =
// slot * assets + a sits at data + k * book_bytes: the blob, the order table, the trade log, the agents' rslot slice, their
// MomState slice and (deep engine) the chunk pool, each section at its capacity, and meta[k] = {valid, tick, 0, 0}.
#define ERR_SLOT 0x1000u  // == BB_ERR_SLOT
struct StoreCopy {
    unsigned char* blobs;
    u64 blob_stride;
    OrderRec* ord;
    TradeRec* tr;
    u32* rslot;
    unsigned char* mom;
    unsigned char* pool;
    const u32* tick;
    unsigned char* data;  // the store
    uint4* meta;
    uint8_t* restored;    // [n_envs]: 1 for the books a restore rewrote (the mask of its observation launch), else 0
    u64 book_bytes, off_ord, off_tr, off_rslot, off_mom, off_pool;
    u32 max_orders, max_trades, rslot_bytes, mom_bytes, pool_chunks /* 0: not the deep engine */, assets, n_units, n_slots;
};

// part `part` of `parts` of a CTA-strided copy: 16 bytes a thread and iteration where both ends and the length allow it (the
// blob, order and trade sections), 4 bytes otherwise (the agent slices, whose per-env offsets are multiples of 4 or 8)
__device__ __forceinline__ void store_copy_part(unsigned char* dst, const unsigned char* src, u64 bytes, u32 part, u32 parts) {
    const u64 i0 = (u64)part * blockDim.x + threadIdx.x, step = (u64)parts * blockDim.x;
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src) | bytes) & 15u) == 0) {
        uint4* d = reinterpret_cast<uint4*>(dst);
        const uint4* s = reinterpret_cast<const uint4*>(src);
        for (u64 i = i0; i < bytes / 16u; i += step) d[i] = s[i];
    } else {
        u32* d = reinterpret_cast<u32*>(dst);
        const u32* s = reinterpret_cast<const u32*>(src);
        for (u64 i = i0; i < bytes / 4u; i += step) d[i] = s[i];
    }
}

// One book of k_store_copy, part `part` of `parts`.  Save: book = slot book k, sel[slot] the unit to save (BB_NO_SLOT: slot
// untouched; >= n_units: slot marked empty).  Restore: book = the handle's book, sel[unit] the slot to restore from
// (BB_NO_SLOT: unit untouched); a slot out of range, empty, or saved at another tick than any book of the unit flags every
// book of the unit ERR_SLOT and changes nothing else.  Every CTA reads the prefix lengths from the source header, which no
// CTA of the launch writes, and evaluates the slot's validity the same way.  Part 0 writes the header: on restore the
// slot's, with the history count at 0 and, given seeds, the unit's shuffle stream re-seeded (the step counter stays the
// slot's; deep books included: their Env steps shuffle with the same stream).
template <bool RESTORE>
__device__ __forceinline__ void store_copy_book(const StoreCopy& c, u32 book, u32 part, u32 parts, const u32* sel, const u64* seeds,
                                                u32* cursor) {
    const u32 A = c.assets, unit = book / A, a = book % A;
    const bool lead = part == 0 && threadIdx.x == 0;
    u64 live, stored;  // book indices into the handle's arrays and the store
    if (RESTORE) {
        const u32 slot = sel[unit];
        if (slot == BB_NO_SLOT) {
            if (lead) c.restored[book] = 0u;
            return;
        }
        bool ok = slot < c.n_slots;
        for (u32 j = 0; ok && j < A; ++j) {
            const uint4 m = c.meta[(u64)slot * A + j];
            ok = m.x != 0u && m.y == c.tick[(u64)unit * A + j];
        }
        if (lead) c.restored[book] = ok ? 1u : 0u;
        if (!ok) {
            if (lead) atomicOr(&reinterpret_cast<BookHdr*>(c.blobs + (u64)book * c.blob_stride)->err, ERR_SLOT);
            return;
        }
        live = book;
        stored = (u64)slot * A + a;
    } else {
        const u32 u = sel[unit];
        if (u == BB_NO_SLOT) return;
        if (u >= c.n_units) {
            if (lead) c.meta[book] = make_uint4(0u, 0u, 0u, 0u);
            return;
        }
        live = (u64)u * A + a;
        stored = book;
    }
    unsigned char* rec = c.data + stored * c.book_bytes;
    unsigned char* blob = c.blobs + live * c.blob_stride;
    const BookHdr* src_hdr = reinterpret_cast<const BookHdr*>(RESTORE ? rec : blob);
    const u64 n_ord = min(src_hdr->n_orders, c.max_orders), n_tr = min(src_hdr->n_trades, c.max_trades);
    const u64 n_chunks = c.pool_chunks ? min(*reinterpret_cast<const u32*>((RESTORE ? rec : blob) + DP_OFF_BUMP), c.pool_chunks) : 0u;
    auto copy = [&](unsigned char* live_p, unsigned char* stored_p, u64 bytes) {
        if (RESTORE) store_copy_part(live_p, stored_p, bytes, part, parts);
        else store_copy_part(stored_p, live_p, bytes, part, parts);
    };
    copy(blob + sizeof(BookHdr), rec + sizeof(BookHdr), c.blob_stride - sizeof(BookHdr));
    copy(reinterpret_cast<unsigned char*>(c.ord + live * c.max_orders), rec + c.off_ord, n_ord * sizeof(OrderRec));
    if (c.max_trades) copy(reinterpret_cast<unsigned char*>(c.tr + live * c.max_trades), rec + c.off_tr, n_tr * sizeof(TradeRec));
    if (c.rslot_bytes) copy(reinterpret_cast<unsigned char*>(c.rslot) + live * c.rslot_bytes, rec + c.off_rslot, c.rslot_bytes);
    if (c.mom_bytes) copy(c.mom + live * c.mom_bytes, rec + c.off_mom, c.mom_bytes);
    if (n_chunks) copy(c.pool + live * c.pool_chunks * DP_CHUNK_BYTES, rec + c.off_pool, n_chunks * DP_CHUNK_BYTES);
    if (!lead) return;
    BookHdr h = *src_hdr;
    if (RESTORE) {
        h.n_steps = 0u;
        if (seeds) seed_stream(h, seeds[unit]);
        *reinterpret_cast<BookHdr*>(blob) = h;
        if (cursor) cursor[book] = (u32)n_tr;
    } else {
        *reinterpret_cast<BookHdr*>(rec) = h;
        c.meta[book] = make_uint4(1u, c.tick[live], 0u, 0u);
    }
}

// bb_save_device (n_books = slot books) / bb_restore_device (n_books = the handle's books).  Grid (x, part): part y of every
// book is copied by the CTAs of row y, which stride over the books, so a book with a long prefix is copied by gridDim.y
// CTAs and a launch that selects few units costs a read of `sel` per unselected book.
template <bool RESTORE>
__global__ void __launch_bounds__(256) k_store_copy(const __grid_constant__ StoreCopy c, u32 n_books, const u32* sel, const u64* seeds,
                                                    u32* cursor) {
    for (u32 book = blockIdx.x; book < n_books; book += gridDim.x)
        store_copy_book<RESTORE>(c, book, blockIdx.y, gridDim.y, sel, seeds, cursor);
}

// bb_set_agent_params_device: one warp per unit, lane gi checks the unit's record for group gi against the declared one
// (the envelope rule of include/bourse_b200.h).  The unit's verdict is the warp's ballot: a unit with any
// record outside the declared population keeps its records and key and every book of it is flagged ERR_PARAMS; a valid
// unit takes its row and / or key.  Units the mask leaves out are not read.
#define ERR_PARAMS 0x2000u  // == BB_ERR_PARAMS
struct AgentParamsArgs {
    bb_agent_group decl[MAX_GROUPS];  // the declared population (bb_set_agents / bb_set_agents_market)
    const bb_agent_group* src;        // [units][n_groups] or null: records stay
    const u64* src_keys;              // [units] or null: keys stay
    const uint8_t* mask;              // [units] or null: every unit
    bb_agent_group* dst;              // the handle's tables
    u64* dst_keys;
    unsigned char* blobs;
    u64 blob_stride;
    u32 n_groups, units, assets;
};

__device__ __forceinline__ bool agent_record_fits(const bb_agent_group& r, const bb_agent_group& d) {
    if (r.kind != d.kind || r.n_agents != d.n_agents || r.tick_size != d.tick_size) return false;
    if (d.kind == BB_GROUP_RANDOM)
        return d.tick_lo <= r.tick_lo && r.tick_lo < r.tick_hi && r.tick_hi <= d.tick_hi && d.vol_lo <= r.vol_lo && r.vol_lo < r.vol_hi &&
               r.vol_hi <= d.vol_hi;
    return r.tick_lo == d.tick_lo && r.vol_hi == d.vol_hi;  // agent_id_start, live-list capacity
}

__global__ void __launch_bounds__(256) k_agent_params(const __grid_constant__ AgentParamsArgs a) {
    const u32 lane = threadIdx.x & 31u, unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (unit >= a.units || (a.mask && !a.mask[unit])) return;  // (whole warps leave together)
    const bool mine = a.src && lane < a.n_groups;
    bb_agent_group r;
    if (mine) r = a.src[(size_t)unit * a.n_groups + lane];
    if (!__all_sync(BB_FULL, !mine || agent_record_fits(r, a.decl[lane]))) {
        if (lane < a.assets) atomicOr(&reinterpret_cast<BookHdr*>(a.blobs + ((u64)unit * a.assets + lane) * a.blob_stride)->err, ERR_PARAMS);
        return;
    }
    if (mine) a.dst[(size_t)unit * a.n_groups + lane] = r;
    if (a.src_keys && lane == 0) a.dst_keys[unit] = a.src_keys[unit];
}

// reduction of per-env counters for bb_stats
__global__ void k_stats(const unsigned char* blobs, u64 blob_stride, u32 n_envs, unsigned long long* out) {
    unsigned long long v[7] = {0, 0, 0, 0, 0, 0, 0};
    for (u32 env = blockIdx.x * blockDim.x + threadIdx.x; env < n_envs; env += gridDim.x * blockDim.x) {
        const BookHdr* h = reinterpret_cast<const BookHdr*>(blobs + (size_t)env * blob_stride);
        v[0] += h->n_instr; v[1] += h->n_created; v[2] += h->n_trades_total; v[3] += h->traded_volume;
        v[4] += h->step_counter; v[5] += h->n_transitions; v[6] += h->err ? 1 : 0;
    }
    for (int i = 0; i < 7; ++i) {
        for (int d = 16; d > 0; d >>= 1) v[i] += __shfl_down_sync(BB_FULL, v[i], d);
        if ((threadIdx.x & 31) == 0 && v[i]) atomicAdd(&out[i], v[i]);
    }
}

}  // namespace bb
