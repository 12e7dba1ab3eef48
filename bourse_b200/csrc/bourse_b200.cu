// Host side of the C ABI declared in include/bourse_b200.h: handle lifetime, the per-env transaction
// queues of Env mode (crates/step_sim/src/env.rs:166-219), launches, and the read-back calls that
// feed the Python `bourse.core` mirror.  All compute happens in kernels.cuh; nothing here touches
// book state on the CPU, and there is no fallback when CUDA is unavailable.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.cuh"

using namespace bb;

namespace {

thread_local std::string g_last_error;

struct SmemLayout {
    u32 warp_bytes, off_perm, off_obs, off_instr, off_bar, off_q, off_ag, off_pc, off_mkt;
};

constexpr u32 WPB = 4;  // warps (books) per CTA

inline u32 align_up(u32 x, u32 a) { return (x + a - 1) / a * a; }

// Books per CTA for a layout: 4 warps unless a book's shared-memory image is so large (deep books with every price page
// resident) that only 2 or 1 fit in the 227 KB a CTA may use.
inline u32 wpb_for(u32 warp_bytes) {
    const u32 limit = 232448u - 1024u;
    return 4u * warp_bytes <= limit ? 4u : 2u * warp_bytes <= limit ? 2u : 1u;
}

}  // namespace

struct bb_handle {
    bb_config cfg;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
    cudaEvent_t chunk_done = nullptr;
    long long recorded_host = 0;  // history records per env written so far; -1 = unknown (ask the device)
    // device
    unsigned char* blobs = nullptr;
    OrderRec* ord = nullptr;
    TradeRec* tr = nullptr;
    u32* hist = nullptr;
    u32* err_flag = nullptr;
    u64* d_offsets = nullptr;
    u64* d_seeds = nullptr;
    bb_instr* d_instrs = nullptr;
    size_t d_instrs_cap = 0;
    u32* d_snap = nullptr;  // [n_envs][45]
    u32* d_tick = nullptr;  // [n_envs] tick size of each env's book (bb_set_tick_sizes); tick[] is its host mirror
    std::vector<u32> tick;
    unsigned long long* d_stats = nullptr;
    u32* rslot = nullptr;
    MomState* mom = nullptr;
    u32 mom_cap = LIVE_CAP, mom_stride = MOM_HDR_BYTES + 4u * LIVE_CAP;  // live-list entries / bytes per MomState record
    uint4* scratch = nullptr;
    size_t scratch_warps = 0;
    u64* d_ids = nullptr;  // bb_step_device: ids assigned on the device when the caller does not ask for them
    size_t d_ids_cap = 0;
    // pinned host staging
    bb_instr* h_instrs = nullptr;
    size_t h_instrs_cap = 0;
    u64* h_offsets = nullptr;
    u32* h_snap = nullptr;  // [n_envs][45] pinned: snapshots come back as ONE contiguous copy and are compacted here
    // layout
    u64 blob_stride = 0;
    u32 blob_smem_bytes = 0, p_total = 0, p_smem = 0, granule = 0, max_steps_padded = 0;
    bool all_resident = false;  // generic geometry with pages_smem == pages_total
    int eng = ENG_PAGED;  // ENG_FAST: granule == 1, one 32-entry page directory, no HBM pages; ENG_DENSE: dense window; ENG_DEEP
    Geo dgeo{};           // dense-engine geometry (d_* fields), zero otherwise
    u32 dense_lp = 0, dense_nwmax = 0;  // DenseLayout parameters of the selected variant
    u64 hist_env_stride = 0;
    SmemLayout lay_apply{}, lay_sim{}, lay_snap{};
    // deep-book engine (deep.cuh): shared-memory offsets of k_deep, chunk pools [n_envs][dp_chunks] x 256 B
    DeepOff dp{};
    unsigned char* dp_pool = nullptr;
    u32 dp_chunks = 0;
    bool deep_attr_set = false;
    bool deep_serial = false;  // developer switch (BOURSE_B200_DEEP=serial): every event through k_deepw's serial path
    // agents
    std::vector<bb_agent_group> groups;
    u32 rand_tick_mask = 0;  // KParams::rand_tick_mask, kept current by set_agents_impl and bb_set_tick_sizes
    std::vector<u32> group_asset;  // bb_set_agents_market: asset each group trades (empty: single-asset agents)
    u32 agents_per_env = 0, mom_groups = 0;
    u32 chip_agents = 0;  // on-chip agent table capacity of the dense engine (markets: the largest per-asset agent count)
    // host mirrors for Env mode
    std::vector<std::vector<bb_instr>> queue;
    std::vector<u64> n_orders_host;  // ids handed out so far (includes queued NEW)
    bool mirror_dirty = false;
    // multi-asset markets (bb_config.assets > 1): per-market submission counter and host-side shuffle RNG
    u32 assets = 1;
    std::vector<u32> market_seq;
    std::vector<u64> market_rng;  // Xoroshiro128** state, two words per market
    // bb_order_status: status column of one env, valid until the next launch that can change a status
    bool status_valid = false;
    u32 status_env = 0;
    std::vector<uint8_t> status_cache;
    std::vector<OrderRec> status_rec;
    struct OccEntry { const void* fn; size_t smem; u32 wpb; int per_sm; };
    std::vector<OccEntry> occ_cache;  // resident CTAs per SM of the kernels launched so far (grid_for)
    std::string err;
};

namespace {

int fail(bb_handle* h, int code, const std::string& msg) {
    g_last_error = msg;
    if (h) h->err = msg;
    return code;
}
#define CUDA_TRY(h, expr)                                                                              \
    do {                                                                                               \
        cudaError_t e__ = (expr);                                                                      \
        if (e__ != cudaSuccess)                                                                        \
            return fail(h, BB_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));             \
    } while (0)

u64 splitmix_next(u64& x) {
    x += 0x9e3779b97f4a7c15ULL;
    u64 z = x;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}

// with_queue: k_sim on the dense engine keeps the step's transaction queue and the agents' held-order state on chip
// host mirror of the device's Xoroshiro128** range draw (philox.cuh xoroshiro_range): rand 0.8.5 gen_range(0..n)
u64 rotl64_h(u64 x, int k) { return (x << k) | (x >> (64 - k)); }
u32 xoroshiro_range_h(u64& s0, u64& s1, u32 range) {
    const u32 zone = (range << __builtin_clz(range)) - 1u;
    for (;;) {
        const u64 r = rotl64_h(s0 * 5ULL, 7) * 9ULL;
        const u64 t = s1 ^ s0;
        s0 = rotl64_h(s0, 24) ^ t ^ (t << 16);
        s1 = rotl64_h(t, 37);
        const u32 v = (u32)r;  // next_u32 = low half of next_u64 (rand_xoshiro 0.6.0)
        const u32 lo = v * range;
        if (lo <= zone) return (u32)(((u64)v * range) >> 32);
    }
}

void seed_markets(bb_handle* h) {
    const u32 n_markets = h->cfg.n_envs / h->assets;
    h->market_seq.assign(n_markets, 0);
    h->market_rng.resize(2 * (size_t)n_markets);
    for (u32 m = 0; m < n_markets; ++m) {
        u64 x = h->cfg.seed + h->cfg.env_id_base / h->assets + m;
        h->market_rng[2 * m] = splitmix_next(x);
        h->market_rng[2 * m + 1] = splitmix_next(x);
    }
}

SmemLayout make_layout(const bb_handle* h, bool with_obs, bool with_instr, bool with_queue = false, bool market = false) {
    SmemLayout l{};
    u32 off = align_up(h->blob_smem_bytes, 16);
    l.off_perm = off;
    // perm + jarr (u16 each) + slack for 8-byte jarr stores; the on-chip queue is shuffled in place and needs no perm.
    // Markets with in-kernel agents: every book derives the permutation of the WHOLE market's queue (k_sim<.., MKT>)
    if (market) off += 4u * align_up(h->assets * h->cfg.max_queue, 8) + 16u;
    else off += align_up((with_queue ? 2u : 4u) * h->cfg.max_queue + 16u, 16);
    l.off_obs = off;
    if (with_obs) off += align_up((market ? 1u : 2u) * OBS_STAGE_STEPS(h->cfg.obs_words) * h->cfg.obs_words * 4u, 16);
    l.off_instr = off;
    if (with_instr) off += 2048;
    l.off_q = off;
    if (with_queue) off += 16u * h->cfg.max_queue + 32u;  // + two entries of padding for the one-ahead fetch
    l.off_ag = off;
    if (with_queue) off += align_up(5u * h->chip_agents + 1u, 16);  // held id u32 [A], slot u8 [A + 1]
    l.off_bar = off;
    off += 32;
    l.off_mkt = off;  // u32 [2][MAX_GROUPS]: the market's per-group instruction counts, double-buffered
    if (market) off += 8u * MAX_GROUPS;
    l.off_pc = off;
    // page lookup cache of the generic geometry (book.cuh find_page); FAST handles run the generic k_snapshot too
    if (h->eng < ENG_DENSE) off += PCACHE_ENTRIES;
    l.warp_bytes = align_up(off, 128);
    return l;
}

void fill_params(const bb_handle* h, const SmemLayout& l, KParams& p) {
    memset(&p, 0, sizeof(p));
    p.blobs = h->blobs;
    p.blob_stride = h->blob_stride;
    p.ord = h->ord;
    p.tr = h->tr;
    p.hist = h->hist;
    p.err_flag = h->err_flag;
    p.step_size = h->cfg.step_size;
    p.hist_env_stride = h->hist_env_stride;
    p.blob_smem_bytes = h->blob_smem_bytes;
    p.n_envs = h->cfg.n_envs;
    p.env_id_base = h->cfg.env_id_base;
    p.geo.p_total = h->p_total;
    p.geo.p_smem = h->p_smem;
    p.geo.granule = h->granule;
    p.geo.ticks = h->d_tick;
    p.geo.max_orders = h->cfg.max_orders;
    p.geo.max_trades = h->cfg.max_trades;
    p.geo.tr_base = (u64)h->tr;
    p.geo.blobs_base = (u64)h->blobs;
    p.geo.blob_stride = h->blob_stride;
    p.geo.d_win_lo = h->dgeo.d_win_lo; p.geo.d_levels = h->dgeo.d_levels; p.geo.d_live = h->dgeo.d_live;
    p.off_q = l.off_q;
    p.off_ag = l.off_ag;
    p.geo.pc_off = l.off_pc;
    p.max_steps = h->max_steps_padded;
    p.max_queue = h->cfg.max_queue;
    p.obs_words = h->cfg.obs_words;
    p.warp_smem_bytes = l.warp_bytes;
    p.off_perm = l.off_perm;
    p.off_obs = l.off_obs;
    p.off_instr = l.off_instr;
    p.off_bar = l.off_bar;
    p.off_mkt = l.off_mkt;
    p.assets = h->assets;
    p.dp = h->dp;
    p.dp_pool = h->dp_pool;
    p.dp_chunks = h->dp_chunks;
}

// shared-memory map of k_deepw (deep.cuh, deepw.cuh) for a window of W levels; `roomy`: at most two books per SM, so the
// two staleness filters can be four times larger (fewer false doubts: events that wait for the pipeline to drain)
DeepOff deep_layout(u32 W, u32 roomy /* filter size multiplier: 1, 4, 8 */) {
    DeepOff o{};
    const u32 nw = W / 32;
    o.bm = DP_OFF_BM;
    o.sm = o.bm + 8u * nw;
    o.lvol = align_up(o.sm + 8u * DP_NS, 16);
    o.lcnt = o.lvol + 4u * W;
    o.lht = o.lcnt + 4u * W;
    o.image_bytes = align_up(o.lht + 8u * W, 128);
    o.smem_image = o.lcnt;  // (16-byte aligned: the bulk copy stops exactly where the counts begin; they stay in the blob)
    u32 off = align_up(o.smem_image, 128);
    o.scratch = off; off += DW_SCRATCH;
    o.ev_ins = off; off += 1024u * DW_RB;
    o.ev_rec = off; off += 1024u * DW_RB;
    o.ev_rf = off; off += 16u;
    o.ret = off; off += DP_RENT * DW_RCAP;
    o.dirty_n = roomy * DW_DIRTY;
    o.swept_n = roomy * DW_SWEPT;
    o.dirty = off; off += 4u * o.dirty_n;
    o.swept = off; off += roomy > 1u ? 4u * o.swept_n : 0u;  // (the compact filter sits inside the scratch block)
    o.ctl = off; off += 4u * CT_WORDS;
    o.bar = off; off += 8u * (DW_RB + 1u);
    o.total = align_up(off, 128);
    return o;
}

template <class K> int grid_for(bb_handle* h, K kernel, const SmemLayout& l, u32 n_items, int* grid_out, u32 wpb = WPB) {
    const size_t smem = (size_t)l.warp_bytes * wpb;
    // the attribute / occupancy queries cost several microseconds of host time: a per-step caller (bb_step_device in an
    // RL loop) would be bound by them, so the answer is remembered per (kernel, shared-memory size, CTA width)
    int per_sm = 0;
    for (const auto& c : h->occ_cache)
        if (c.fn == (const void*)kernel && c.smem == smem && c.wpb == wpb) per_sm = c.per_sm;
    if (!per_sm) {
        CUDA_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, wpb * 32, smem));
        if (per_sm < 1) return fail(h, BB_EINVAL, "configuration does not fit in shared memory (reduce pages_smem / max_queue)");
        h->occ_cache.push_back({(const void*)kernel, smem, wpb, per_sm});
    }
    const u32 want = (n_items + wpb - 1) / wpb;
    const u32 cap = (u32)per_sm * (u32)h->sm_count;
    *grid_out = (int)(want < cap ? want : cap);
    if (*grid_out < 1) *grid_out = 1;
    return BB_OK;
}

int upload_seeds(bb_handle* h) {
    const bb_config& c = h->cfg;
    std::vector<u64> seeds(2 * (size_t)c.n_envs);
    for (u32 e = 0; e < c.n_envs; ++e) {  // Xoroshiro128StarStar::seed_from_u64 (rand_xoshiro 0.6.0)
        u64 x = c.seed + c.env_id_base + e;
        seeds[2 * e] = splitmix_next(x);
        seeds[2 * e + 1] = splitmix_next(x);
    }
    CUDA_TRY(h, cudaMemcpyAsync(h->d_seeds, seeds.data(), seeds.size() * 8, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

// asynchronous on the handle's stream: one small kernel rewrites every book header and page directory
int init_books(bb_handle* h) {
    const bb_config& c = h->cfg;
    if (h->eng == ENG_DEEP) {
        k_init_deep<<<c.n_envs, 128, 0, h->stream>>>(h->blobs, h->blob_stride, c.n_envs, c.start_time, c.trading ? 1u : 0u, h->d_seeds,
                                                     h->dp.bm, h->dp.lht - h->dp.bm);  // bitmaps, summaries, level volumes and order counts start at zero
        CUDA_TRY(h, cudaGetLastError());
        CUDA_TRY(h, cudaMemsetAsync(h->err_flag, 0, 4, h->stream));
        h->status_valid = false;
        for (auto& q : h->queue) q.clear();
        std::fill(h->n_orders_host.begin(), h->n_orders_host.end(), 0);
        h->mirror_dirty = false;
        h->recorded_host = 0;
        return BB_OK;
    }
    k_init<<<c.n_envs, 64, 0, h->stream>>>(h->blobs, h->blob_stride, c.n_envs, h->p_total, c.start_time, c.trading ? 1u : 0u,
                                           h->d_seeds, h->rslot, h->agents_per_env, h->mom, h->mom_groups, h->mom_stride, h->dgeo, h->dense_lp, h->dense_nwmax);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemsetAsync(h->err_flag, 0, 4, h->stream));
    h->status_valid = false;
    for (auto& q : h->queue) q.clear();
    std::fill(h->n_orders_host.begin(), h->n_orders_host.end(), 0);
    h->mirror_dirty = false;
    h->recorded_host = 0;
    if (h->assets > 1) seed_markets(h);
    return BB_OK;
}

int refresh_mirror(bb_handle* h) {
    if (!h->mirror_dirty) return BB_OK;
    std::vector<u32> n(h->cfg.n_envs);
    CUDA_TRY(h, cudaMemcpy2DAsync(n.data(), 4, h->blobs + offsetof(BookHdr, n_orders), h->blob_stride, 4, h->cfg.n_envs,
                                  cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (u32 e = 0; e < h->cfg.n_envs; ++e) h->n_orders_host[e] = n[e] + [&] {
        u64 k = 0;
        for (auto& x : h->queue[e]) k += (x.op_flags & BB_OP_MASK) == BB_OP_NEW;
        return k;
    }();
    h->mirror_dirty = false;
    return BB_OK;
}

int check_device_errors(bb_handle* h) {
    u32 flag = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&flag, h->err_flag, 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (flag) {
        CUDA_TRY(h, cudaMemsetAsync(h->err_flag, 0, 4, h->stream));
        char buf[256];
        snprintf(buf, sizeof buf, "device flagged env errors 0x%x (0x1 orders 0x2 trades 0x4 pages/window 0x8 queue 0x10 bad id "
                                  "0x20 granule 0x40 steps 0x80 live slots 0x100 time order 0x200 tick size 0x400 unsupported row); see bb_env_errors", flag);
        return fail(h, (flag & ERR_BAD_ID) ? BB_EBADID : (flag & 0x80000000u) ? BB_ECUDA : (flag & ERR_PRICE) ? BB_EPRICE : (flag & ERR_ROW_OP) ? BB_EINVAL : BB_ECAP, buf);
    }
    return BB_OK;
}

int ensure_instr_capacity(bb_handle* h, size_t n) {
    if (n > h->d_instrs_cap) {
        if (h->d_instrs) cudaFree(h->d_instrs);
        h->d_instrs = nullptr;
        const size_t cap = n + n / 2 + 1024;
        CUDA_TRY(h, cudaMalloc(&h->d_instrs, cap * sizeof(bb_instr)));
        h->d_instrs_cap = cap;
    }
    if (n > h->h_instrs_cap) {
        if (h->h_instrs) cudaFreeHost(h->h_instrs);
        h->h_instrs = nullptr;
        const size_t cap = n + n / 2 + 1024;
        CUDA_TRY(h, cudaMallocHost(&h->h_instrs, cap * sizeof(bb_instr)));
        h->h_instrs_cap = cap;
    }
    return BB_OK;
}

int launch_apply(bb_handle* h, int mode, const bb_instr* d_instrs, const u64* d_offsets, u32 n_steps, bool host_order = false,
                 u64* d_out_ids = nullptr, u32* d_obs_out = nullptr) {
    KParams p;
    fill_params(h, h->lay_apply, p);
    p.instrs = d_instrs;
    p.offsets = d_offsets;
    p.n_steps = n_steps;
    h->status_valid = false;
    p.host_order = host_order ? 1u : 0u;
    p.assign_ids = d_out_ids ? 1u : 0u;
    p.out_ids = d_out_ids;
    p.obs_out = d_obs_out;
    if (h->eng == ENG_DEEP) {
        if (mode != MODE_REPLAY || d_out_ids || d_obs_out) return fail(h, BB_EINVAL, "the deep-book engine replays instruction streams only");
        if (!h->deep_attr_set) {
            CUDA_TRY(h, cudaFuncSetAttribute(k_deepw<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448 - 1024));
            CUDA_TRY(h, cudaFuncSetAttribute(k_deepw<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448 - 1024));
            h->deep_attr_set = true;
        }
        p.dp_fast = h->deep_serial ? 0u : 1u;
        if (h->dp.dirty_n > DW_DIRTY) k_deepw<true><<<h->cfg.n_envs, 128, h->dp.total, h->stream>>>(p);
        else k_deepw<false><<<h->cfg.n_envs, 128, h->dp.total, h->stream>>>(p);
        CUDA_TRY(h, cudaGetLastError());
        h->recorded_host = -1;
        return BB_OK;
    }
    int grid = 0, rc;
    const u32 wpb = wpb_for(h->lay_apply.warp_bytes);
    const size_t smem = (size_t)h->lay_apply.warp_bytes * wpb;
#define LAUNCH_APPLY(M, E)                                                                            \
    do {                                                                                              \
        if ((rc = grid_for(h, k_apply<M, E>, h->lay_apply, h->cfg.n_envs, &grid, wpb))) return rc;    \
        k_apply<M, E><<<grid, wpb * 32, smem, h->stream>>>(p);                                        \
    } while (0)
    if (mode == MODE_REPLAY) {
        if (h->eng == ENG_DENSE) LAUNCH_APPLY(MODE_REPLAY, ENG_DENSE);
        else if (h->eng == ENG_DENSE_L) LAUNCH_APPLY(MODE_REPLAY, ENG_DENSE_L);
        else if (h->eng == ENG_FAST) LAUNCH_APPLY(MODE_REPLAY, ENG_FAST);
        else if (h->all_resident) LAUNCH_APPLY(MODE_REPLAY, ENG_PAGED_RES);
        else LAUNCH_APPLY(MODE_REPLAY, ENG_PAGED);
    } else {
        if (h->eng == ENG_DENSE) LAUNCH_APPLY(MODE_ENV, ENG_DENSE);
        else if (h->eng == ENG_DENSE_L) LAUNCH_APPLY(MODE_ENV, ENG_DENSE_L);
        else if (h->eng == ENG_FAST) LAUNCH_APPLY(MODE_ENV, ENG_FAST);
        else if (h->all_resident) LAUNCH_APPLY(MODE_ENV, ENG_PAGED_RES);
        else LAUNCH_APPLY(MODE_ENV, ENG_PAGED);
    }
#undef LAUNCH_APPLY
    CUDA_TRY(h, cudaGetLastError());
    // a launch recorded into a CUDA graph (bb_step_device inside a captured RL loop) will run any number of times:
    // the host-side record count is unknown from here on and is re-read from the device when next needed
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(h->stream, &cap);
    if (mode == MODE_ENV && h->recorded_host >= 0 && cap == cudaStreamCaptureStatusNone) h->recorded_host += n_steps;
    else h->recorded_host = -1;
    return BB_OK;
}

int snapshot(bb_handle* h, u32 first_env, u32 n, u32* d45, u32* d8, u32 words = 45u) {
    KParams p;
    fill_params(h, h->lay_snap, p);
    if (h->eng == ENG_DEEP) {
        k_snapshot_deep<<<(n + 3) / 4, 128, 0, h->stream>>>(p, d45, d8, first_env, n, words);
        CUDA_TRY(h, cudaGetLastError());
        return BB_OK;
    }
    int grid = 0, rc;
    const u32 wpb = wpb_for(h->lay_snap.warp_bytes);
    const size_t smem = (size_t)h->lay_snap.warp_bytes * wpb;
    if (h->eng == ENG_DENSE) {
        if ((rc = grid_for(h, k_snapshot<ENG_DENSE>, h->lay_snap, n, &grid, wpb))) return rc;
        k_snapshot<ENG_DENSE><<<grid, wpb * 32, smem, h->stream>>>(p, d45, d8, first_env, n, words);
    } else if (h->eng == ENG_DENSE_L) {
        if ((rc = grid_for(h, k_snapshot<ENG_DENSE_L>, h->lay_snap, n, &grid, wpb))) return rc;
        k_snapshot<ENG_DENSE_L><<<grid, wpb * 32, smem, h->stream>>>(p, d45, d8, first_env, n, words);
    } else {
        if ((rc = grid_for(h, k_snapshot<ENG_PAGED>, h->lay_snap, n, &grid, wpb))) return rc;
        k_snapshot<ENG_PAGED><<<grid, wpb * 32, smem, h->stream>>>(p, d45, d8, first_env, n, words);
    }
    CUDA_TRY(h, cudaGetLastError());
    return BB_OK;
}

#define CHECK_H(h) \
    if (!(h)) return fail(nullptr, BB_EINVAL, "null handle")
#define CHECK_ENV(h, env) \
    if ((env) >= (h)->cfg.n_envs) return fail(h, BB_EINVAL, "env index out of range")

}  // namespace

extern "C" {

int bb_abi_version(void) { return BB_ABI_VERSION; }

const char* bb_last_error(const bb_handle* h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int bb_create(const bb_config* cfg, bb_handle** out) {
    if (!cfg || !out) return fail(nullptr, BB_EINVAL, "null argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(bb_config)) return fail(nullptr, BB_EINVAL, "bb_config.struct_size mismatch");
    if (cfg->tick_size == 0 || cfg->n_envs == 0) return fail(nullptr, BB_EINVAL, "tick_size and n_envs must be > 0");
    if (cfg->obs_words != BB_OBS_L1 && cfg->obs_words != BB_OBS_L2) return fail(nullptr, BB_EINVAL, "obs_words must be 9 or 45");
    if (cfg->max_orders == 0 || cfg->max_queue == 0 || cfg->max_queue > 65535 || cfg->max_steps == 0)
        return fail(nullptr, BB_EINVAL, "max_orders, max_steps must be > 0 and 0 < max_queue <= 65535");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
        return fail(nullptr, BB_ECUDA, "no CUDA device available: bourse_b200 has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= n_dev) return fail(nullptr, BB_EINVAL, "device ordinal out of range");
    cudaDeviceProp prop;
    CUDA_TRY(nullptr, cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return fail(nullptr, BB_ECUDA, std::string("device is ") + prop.name + " (sm_" + std::to_string(prop.major) +
                                           std::to_string(prop.minor) + "); this library is built for sm_100a only");
    CUDA_TRY(nullptr, cudaSetDevice(cfg->device));

    if (cfg->assets > 1 && (cfg->n_envs % cfg->assets != 0 || cfg->env_id_base % cfg->assets != 0))
        return fail(nullptr, BB_EINVAL, "n_envs and env_id_base must be multiples of assets (books per market)");
    bb_handle* h = new bb_handle();
    h->cfg = *cfg;
    h->assets = cfg->assets > 1 ? cfg->assets : 1u;
    h->sm_count = prop.multiProcessorCount;
    h->granule = cfg->price_granule ? cfg->price_granule : cfg->tick_size;
    h->p_smem = cfg->pages_smem ? cfg->pages_smem : 10u;
    const u32 usable = cfg->pages_total ? cfg->pages_total : h->p_smem;  // pages a book may hold
    if (h->p_smem > usable) h->p_smem = usable;
    h->p_total = align_up(usable, 32);
    h->eng = (h->granule == 1 && h->p_total == 32 && usable == h->p_smem) ? ENG_FAST : ENG_PAGED;
    h->all_resident = h->eng == ENG_PAGED && usable == h->p_smem;  // k_apply<.., ENG_PAGED_RES>: no HBM page variants
    h->blob_smem_bytes = 128u + 12u * h->p_total + 512u * h->p_smem;
    h->blob_stride = 128ull + 12ull * h->p_total + 512ull * h->p_total;
    if (cfg->win_levels && !cfg->deep_chunks) {  // dense-window engine (csrc/dense.cuh), two compiled size classes
        const u32 W = align_up(cfg->win_levels, 32), L = cfg->live_cap ? cfg->live_cap : 128u;
        if (h->granule != 1 || W > 32 * DenseLarge::NWMAX || L > 254 || (u64)cfg->win_lo + W > 0x100000000ull) {
            delete h;
            return fail(nullptr, BB_EINVAL, "dense engine needs price_granule == 1, win_levels <= 1024, live_cap <= 254 and "
                                            "win_lo + win_levels <= 2^32");
        }
        const bool small = L <= DenseSmall::LP && W <= 32 * DenseSmall::NWMAX;
        h->dgeo.d_win_lo = cfg->win_lo; h->dgeo.d_levels = W; h->dgeo.d_live = L;
        h->eng = small ? ENG_DENSE : ENG_DENSE_L;
        h->dense_lp = small ? DenseSmall::LP : DenseLarge::LP;
        h->dense_nwmax = small ? DenseSmall::NWMAX : DenseLarge::NWMAX;
        h->blob_smem_bytes = align_up(small ? DenseSmall::image_bytes(W) : DenseLarge::image_bytes(W), 16);
        h->blob_stride = align_up(h->blob_smem_bytes, 128);
        h->p_total = h->p_smem = 0;
    }
    if (cfg->deep_chunks) {  // deep-book engine (csrc/deep.cuh): the dense-window fields describe its ladder
        const u32 W = align_up(cfg->win_levels, 32);
        if (!cfg->win_levels || h->granule != 1 || W > 32u * 32u * DP_NS || (u64)cfg->win_lo + W > 0x100000000ull || h->assets > 1 ||
            cfg->deep_chunks < 2 || cfg->deep_chunks >= (1u << 27)) {
            delete h;
            return fail(nullptr, BB_EINVAL, "deep engine needs price_granule == 1, 0 < win_levels <= 8192, win_lo + win_levels <= 2^32, "
                                            "2 <= deep_chunks < 2^27 and single-asset envs");
        }
        h->eng = ENG_DEEP;
        h->dgeo.d_win_lo = cfg->win_lo; h->dgeo.d_levels = W; h->dgeo.d_live = 0;
        h->dense_lp = h->dense_nwmax = 0;
        if (const char* m = getenv("BOURSE_B200_DEEP")) h->deep_serial = !strcmp(m, "serial");
        // one book per SM: filters x8; two: x4 (while two CTAs still fit an SM); more: the compact sizes
        h->dp = deep_layout(W, cfg->n_envs <= 148u ? 8u : cfg->n_envs <= 2u * 148u ? 4u : 1u);
        if (cfg->n_envs > 148u && h->dp.total > 113u * 1024u) h->dp = deep_layout(W, 1u);  // (a wide window: keep two CTAs per SM possible)
        h->dp_chunks = cfg->deep_chunks;
        if (h->dp.total > 232448u - 1024u) {
            delete h;
            return fail(nullptr, BB_EINVAL, "deep engine: window does not fit in shared memory");
        }
        h->blob_smem_bytes = h->dp.image_bytes;
        h->blob_stride = h->dp.image_bytes;
        h->p_total = h->p_smem = 0;
    }
    h->max_steps_padded = align_up(cfg->max_steps, 4);
    h->hist_env_stride = (u64)h->max_steps_padded * cfg->obs_words;
    h->lay_apply = make_layout(h, false, true);
    h->lay_sim = make_layout(h, true, false, h->eng >= ENG_DENSE);
    h->lay_snap = make_layout(h, false, false);
    h->queue.resize(cfg->n_envs);
    h->n_orders_host.assign(cfg->n_envs, 0);

    auto bail = [&](int rc) {
        bb_destroy(h);
        return rc;
    };
#define TRY_ALLOC(expr)                                                                                   \
    do {                                                                                                  \
        cudaError_t e__ = (expr);                                                                         \
        if (e__ != cudaSuccess) return bail(fail(nullptr, BB_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__))); \
    } while (0)
    const size_t ne = cfg->n_envs;
    TRY_ALLOC(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    TRY_ALLOC(cudaMalloc(&h->blobs, ne * h->blob_stride));
    TRY_ALLOC(cudaMemsetAsync(h->blobs, 0, ne * h->blob_stride, h->stream));
    TRY_ALLOC(cudaMalloc(&h->ord, ne * cfg->max_orders * sizeof(OrderRec)));
    if (cfg->max_trades) TRY_ALLOC(cudaMalloc(&h->tr, ne * cfg->max_trades * sizeof(TradeRec)));
    TRY_ALLOC(cudaMalloc(&h->hist, ne * h->hist_env_stride * 4));
    if (h->eng == ENG_DEEP) TRY_ALLOC(cudaMalloc(&h->dp_pool, ne * (size_t)h->dp_chunks * DP_CHUNK_BYTES));
    TRY_ALLOC(cudaMalloc(&h->err_flag, 4));
    TRY_ALLOC(cudaMalloc(&h->d_offsets, (ne + 1) * 8));
    TRY_ALLOC(cudaMalloc(&h->d_seeds, ne * 16));
    TRY_ALLOC(cudaMalloc(&h->d_snap, ne * 45 * 4));
    TRY_ALLOC(cudaMalloc(&h->d_tick, ne * 4));
    h->tick.assign(ne, cfg->tick_size);
    TRY_ALLOC(cudaMemcpyAsync(h->d_tick, h->tick.data(), ne * 4, cudaMemcpyHostToDevice, h->stream));
    TRY_ALLOC(cudaMalloc(&h->d_stats, 8 * 8));
    TRY_ALLOC(cudaMallocHost(&h->h_offsets, (ne + 1) * 8));
    TRY_ALLOC(cudaMallocHost(&h->h_snap, ne * 45 * 4));
#undef TRY_ALLOC
    int rc = upload_seeds(h);
    if (!rc) rc = init_books(h);
    if (!rc && cudaStreamSynchronize(h->stream) != cudaSuccess) rc = fail(nullptr, BB_ECUDA, "init kernel failed");
    if (rc) return bail(rc);
    *out = h;
    return BB_OK;
}

int bb_destroy(bb_handle* h) {
    if (!h) return BB_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    cudaFree(h->blobs); cudaFree(h->ord); cudaFree(h->tr); cudaFree(h->hist); cudaFree(h->err_flag);
    cudaFree(h->d_offsets); cudaFree(h->d_seeds); cudaFree(h->d_instrs); cudaFree(h->d_snap); cudaFree(h->d_stats); cudaFree(h->d_tick);
    cudaFree(h->rslot); cudaFree(h->mom); cudaFree(h->scratch); cudaFree(h->d_ids); cudaFree(h->dp_pool);
    if (h->h_instrs) cudaFreeHost(h->h_instrs);
    if (h->h_offsets) cudaFreeHost(h->h_offsets);
    if (h->h_snap) cudaFreeHost(h->h_snap);
    if (h->chunk_done) cudaEventDestroy(h->chunk_done);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return BB_OK;
}

int bb_reset(bb_handle* h) {
    CHECK_H(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return init_books(h);
}

// KParams::rand_tick_mask: bit gi for a RandomAgents group that trades some book whose tick does not divide its tick_size.
// Only such groups can draw an off-tick limit price: a population with one runs on the k_sim variants that check the
// queued prices (run_agents_impl), on-grid populations keep the RandomAgents-only kernels, which carry no check.
static void update_rand_tick_mask(bb_handle* h) {
    h->rand_tick_mask = 0;
    for (size_t gi = 0; gi < h->groups.size(); ++gi) {
        if (h->groups[gi].kind != BB_GROUP_RANDOM) continue;
        for (u32 e = 0; e < h->cfg.n_envs; ++e)  // markets: env e is book e % assets of its market
            if ((h->group_asset.empty() || e % h->assets == h->group_asset[gi]) && h->groups[gi].tick_size % h->tick[e] != 0) {
                h->rand_tick_mask |= 1u << gi;
                break;
            }
    }
}

int bb_set_tick_sizes(bb_handle* h, const uint32_t* ticks, uint32_t n) {
    CHECK_H(h);
    const u32 ne = h->cfg.n_envs;
    if (!ticks) return fail(h, BB_EINVAL, "null tick array");
    if (n != ne && !(h->assets > 1 && n == h->assets))
        return fail(h, BB_EINVAL, "bb_set_tick_sizes: n must be n_envs (" + std::to_string(ne) + ")" +
                                      (h->assets > 1 ? " or assets (" + std::to_string(h->assets) + ")" : std::string()));
    for (u32 i = 0; i < n; ++i) {
        if (ticks[i] == 0) return fail(h, BB_EINVAL, "bb_set_tick_sizes: tick " + std::to_string(i) + " is 0");
        if (ticks[i] % h->granule != 0)
            return fail(h, BB_EINVAL, "bb_set_tick_sizes: tick " + std::to_string(ticks[i]) + " is not a multiple of the price granule " +
                                          std::to_string(h->granule));
    }
    // a reference book gets its tick at creation only (orderbook.rs:158-171): refuse while any book holds orders
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    std::vector<u32> n_ord(ne);
    CUDA_TRY(h, cudaMemcpy2DAsync(n_ord.data(), 4, h->blobs + offsetof(BookHdr, n_orders), h->blob_stride, 4, ne,
                                  cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (u32 e = 0; e < ne; ++e)
        if (n_ord[e] || !h->queue[e].empty())
            return fail(h, BB_EINVAL, "bb_set_tick_sizes: env " + std::to_string(e) + " has orders or queued transactions (bb_reset first)");
    std::vector<u32> t(ne);
    for (u32 e = 0; e < ne; ++e) t[e] = ticks[n == ne ? e : e % h->assets];  // market m's book a = env m * assets + a
    CUDA_TRY(h, cudaMemcpyAsync(h->d_tick, t.data(), (size_t)ne * 4, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->tick.swap(t);
    update_rand_tick_mask(h);
    return BB_OK;
}

int bb_set_stream(bb_handle* h, void* cuda_stream) {
    CHECK_H(h);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return BB_OK;
}

int bb_synchronize(bb_handle* h) {
    CHECK_H(h);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_submit(bb_handle* h, uint64_t n, const uint32_t* env, const uint32_t* action, const uint8_t* side_is_bid,
              const uint32_t* vol, const uint32_t* trader, const uint32_t* price, const uint64_t* order_id,
              const uint32_t* flags, uint64_t* out_ids, uint64_t* n_done) {
    CHECK_H(h);
    if (n_done) *n_done = 0;
    if (!action) return fail(h, BB_EINVAL, "action array is required");
    if (!env && h->cfg.n_envs != 1) return fail(h, BB_EINVAL, "env array is required when n_envs > 1");
    int rc = refresh_mirror(h);
    if (rc) return rc;
    for (uint64_t r = 0; r < n; ++r) {
        const u32 e = env ? env[r] : 0u;
        if (e >= h->cfg.n_envs) return fail(h, BB_EINVAL, "env index out of range at row " + std::to_string(r));
        const u32 f = flags ? flags[r] : (BB_F_HAS_PRICE | BB_F_HAS_VOL);
        bb_instr x{};
        uint64_t id_out = BB_NO_ID;
        switch (action[r]) {
            case BB_ACT_NEW: {
                const bool market = flags && (f & BB_F_MARKET);
                const u32 p = price ? price[r] : 0u;
                if (!market && p % h->tick[e] != 0) {  // create_order tick check against the env's tick, orderbook.rs:367-383
                    if (n_done) *n_done = r;
                    return fail(h, BB_EPRICE, "Price " + std::to_string(p) + " was not a multiple of tick-size " +
                                                  std::to_string(h->tick[e]));
                }
                if (h->n_orders_host[e] >= h->cfg.max_orders) {
                    if (n_done) *n_done = r;
                    return fail(h, BB_ECAP, "max_orders exceeded for env " + std::to_string(e));
                }
                id_out = h->n_orders_host[e]++;
                x.op_flags = BB_OP_NEW | ((side_is_bid && side_is_bid[r]) ? BB_F_BID : 0u) | (market ? BB_F_MARKET : 0u);
                x.order_id = (u32)id_out;
                x.price = p;
                x.vol = vol ? vol[r] : 0u;
                x.trader = trader ? trader[r] : 0u;
                break;
            }
            case BB_ACT_CANCEL:
            case BB_ACT_MODIFY: {
                const uint64_t id = order_id ? order_id[r] : 0;
                x.op_flags = action[r] == BB_ACT_CANCEL ? BB_OP_CANCEL : (BB_OP_MODIFY | (f & (BB_F_HAS_PRICE | BB_F_HAS_VOL)));
                // ids that do not fit 32 bits cannot exist; keep them out of range so the step flags BB_EBADID
                x.order_id = id > 0xFFFFFFFEull ? 0xFFFFFFFFu : (u32)id;
                x.price = price ? price[r] : 0u;
                x.vol = vol ? vol[r] : 0u;
                break;
            }
            default:  // BB_ACT_NOOP and unknown codes are no-ops (step_sim_numpy.rs:256, 267)
                if (out_ids) out_ids[r] = BB_NO_ID;
                if (n_done) *n_done = r + 1;
                continue;
        }
        if (h->assets > 1) x.aux = h->market_seq[e / h->assets]++;  // position in the market's transaction queue
        h->queue[e].push_back(x);
        if (out_ids) out_ids[r] = id_out;
        if (n_done) *n_done = r + 1;
    }
    return BB_OK;
}

int bb_step(bb_handle* h, uint32_t n_steps) {
    CHECK_H(h);
    if (h->eng == ENG_DEEP) return fail(h, BB_EINVAL, "the deep-book engine replays instruction streams only (bb_replay / bb_replay_device)");
    if (n_steps == 0) return BB_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const u32 ne = h->cfg.n_envs;
    size_t total = 0;
    for (u32 e = 0; e < ne; ++e) {
        h->h_offsets[e] = total;
        total += h->queue[e].size();
    }
    h->h_offsets[ne] = total;
    // A step's queue is shuffled in shared memory: a queue beyond max_queue is refused BEFORE anything is applied (the
    // transactions stay queued; bb_reserve_queue makes room) instead of being cut short on the device.
    if (h->assets <= 1)
        for (u32 e = 0; e < ne; ++e)
            if (h->queue[e].size() > h->cfg.max_queue)
                return fail(h, BB_ECAP, "env " + std::to_string(e) + " has " + std::to_string(h->queue[e].size()) +
                                            " transactions queued for this step, max_queue is " + std::to_string(h->cfg.max_queue) +
                                            " (bb_reserve_queue grows it)");
    int rc = ensure_instr_capacity(h, total + 1);
    if (rc) return rc;
    if (h->assets > 1) {
        // MarketEnv::step (market_env.rs:108-121): the market's queue, in submission order, is shuffled as a whole;
        // event i of the shuffled queue runs at start + i.  Each book receives its events in that order with the
        // offset i in bb_instr::t (k_apply's host_order path).
        const u32 A = h->assets;
        std::vector<bb_instr> all;
        std::vector<u32> book;
        std::vector<size_t> fill(A);
        for (u32 m = 0; m < ne / A; ++m) {
            const u32 n = h->market_seq[m];
            if (n) {
                all.assign(n, bb_instr{});
                book.assign(n, 0);
                for (u32 a = 0; a < A; ++a)
                    for (const bb_instr& x : h->queue[m * A + a]) {
                        all[x.aux] = x;
                        book[x.aux] = a;
                    }
                u64& s0 = h->market_rng[2 * m];
                u64& s1 = h->market_rng[2 * m + 1];
                for (u32 i = n; i > 1; --i) {  // SliceRandom::shuffle, rand 0.8.5
                    const u32 j = xoroshiro_range_h(s0, s1, i);
                    std::swap(all[i - 1], all[j]);
                    std::swap(book[i - 1], book[j]);
                }
                for (u32 a = 0; a < A; ++a) fill[a] = h->h_offsets[m * A + a];
                for (u32 i = 0; i < n; ++i) {
                    bb_instr x = all[i];
                    x.t = i;
                    x.aux = 0;
                    h->h_instrs[fill[book[i]]++] = x;
                }
            }
            for (u32 a = 0; a < A; ++a) h->queue[m * A + a].clear();
            h->market_seq[m] = 0;
        }
    } else
    for (u32 e = 0; e < ne; ++e) {
        if (!h->queue[e].empty())
            memcpy(h->h_instrs + h->h_offsets[e], h->queue[e].data(), h->queue[e].size() * sizeof(bb_instr));
        h->queue[e].clear();
    }
    if (total) CUDA_TRY(h, cudaMemcpyAsync(h->d_instrs, h->h_instrs, total * sizeof(bb_instr), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_offsets, h->h_offsets, (ne + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = launch_apply(h, MODE_ENV, h->d_instrs, h->d_offsets, n_steps, h->assets > 1))) return rc;
    return check_device_errors(h);
}

int bb_replay(bb_handle* h, const bb_instr* instrs, const uint64_t* env_offsets) {
    CHECK_H(h);
    if (!env_offsets) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const u32 ne = h->cfg.n_envs;
    const size_t total = env_offsets[ne];
    if (total && !instrs) return fail(h, BB_EINVAL, "null instruction array");
    // create_order's tick check (orderbook.rs:367-383) on every limit NEW, before anything is applied: a stream with an
    // off-tick price changes no env (MODIFY prices are not checked, as in the reference).  A tick of 1 takes every price,
    // so such an env's rows are not walked here (the pass would sit in front of the launch)
    for (u32 e = 0; e < ne; ++e) {
        if (h->tick[e] == 1) continue;
        for (size_t i = env_offsets[e]; i < env_offsets[e + 1]; ++i) {
            const bb_instr& x = instrs[i];
            if ((x.op_flags & BB_OP_MASK) == BB_OP_NEW && !(x.op_flags & BB_F_MARKET) && x.price % h->tick[e] != 0)
                return fail(h, BB_EPRICE, "bb_replay: env " + std::to_string(e) + " row " + std::to_string(i) + ": Price " +
                                              std::to_string(x.price) + " was not a multiple of tick-size " + std::to_string(h->tick[e]));
        }
    }
    int rc = refresh_mirror(h);
    if (rc) return rc;
    if ((rc = ensure_instr_capacity(h, total + 1))) return rc;
    if (total) memcpy(h->h_instrs, instrs, total * sizeof(bb_instr));
    memcpy(h->h_offsets, env_offsets, (ne + 1) * 8);
    if (total) CUDA_TRY(h, cudaMemcpyAsync(h->d_instrs, h->h_instrs, total * sizeof(bb_instr), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_offsets, h->h_offsets, (ne + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = launch_apply(h, MODE_REPLAY, h->d_instrs, h->d_offsets, 0))) return rc;
    for (u32 e = 0; e < ne; ++e)
        for (size_t i = env_offsets[e]; i < env_offsets[e + 1]; ++i)
            h->n_orders_host[e] += (instrs[i].op_flags & BB_OP_MASK) == BB_OP_NEW;
    return check_device_errors(h);
}

int bb_replay_device(bb_handle* h, const bb_instr* d_instrs, const uint64_t* d_env_offsets) {
    CHECK_H(h);
    if (!d_env_offsets) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    h->mirror_dirty = true;
    return launch_apply(h, MODE_REPLAY, d_instrs, d_env_offsets, 0);
}

static int set_agents_impl(bb_handle* h, const bb_agent_group* groups, const uint32_t* asset, uint32_t n_groups) {
    CHECK_H(h);
    if (h->eng == ENG_DEEP) return fail(h, BB_EINVAL, "the deep-book engine replays instruction streams only (no in-kernel agents)");
    if (n_groups > MAX_GROUPS) return fail(h, BB_EINVAL, "at most 8 agent groups");
    if (n_groups && !groups) return fail(h, BB_EINVAL, "null groups");
    if (asset) {
        if (h->assets < 2) return fail(h, BB_EINVAL, "bb_set_agents_market needs a handle created with assets > 1");
        if (h->assets > WPB) return fail(h, BB_EINVAL, "in-kernel market agents support at most 4 assets per market");
        if ((u64)h->assets * h->cfg.max_queue > 65535) return fail(h, BB_EINVAL, "assets * max_queue must stay below 65536");
        for (u32 i = 0; i < n_groups; ++i)
            if (asset[i] >= h->assets) return fail(h, BB_EINVAL, "agent group asset index out of range");
    }
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    u32 total = 0, mom = 0, mom_cap = LIVE_CAP;
    for (u32 i = 0; i < n_groups; ++i) {
        const bb_agent_group& g = groups[i];
        if (g.kind == BB_GROUP_RANDOM) {
            if (g.tick_hi <= g.tick_lo || g.vol_hi <= g.vol_lo) return fail(h, BB_EINVAL, "empty tick/vol range");
            if (g.n_agents >= (1u << 19)) return fail(h, BB_EINVAL, "too many agents in a group");
        } else if (g.kind == BB_GROUP_MOMENTUM || g.kind == BB_GROUP_NOISE) {
            if ((u64)g.tick_lo + g.n_agents >= (1u << 19)) return fail(h, BB_EINVAL, "momentum trader ids must stay below 2^19");
            if (g.tick_size == 0 || g.n_agents == 0) return fail(h, BB_EINVAL, "momentum group needs tick_size and n_agents > 0");
            if (g.vol_hi > (1u << 20)) return fail(h, BB_EINVAL, "live-order list capacity (vol_hi of a momentum / noise group) above 2^20");
            mom_cap = std::max(mom_cap, g.vol_hi);  // 0 = the default
            ++mom;
        } else {
            return fail(h, BB_EINVAL, "unknown agent group kind");
        }
        total += g.n_agents;
    }
    // every check happens before any allocation is touched: a refused population leaves the previous one intact
    if (h->eng >= ENG_DENSE && total > 2046) return fail(h, BB_EINVAL, "the dense engine supports at most 2046 agents per env");
    // agent state is (re)allocated only when the population's shape changes: cudaFree / cudaMalloc synchronise the
    // whole device and cost ~100 ms next to tens of GB of slabs, which used to dominate the end-to-end pass
    const size_t ne = h->cfg.n_envs;
    mom_cap = (mom_cap + 1u) & ~1u;  // (records stay 8-byte aligned)
    if (total != h->agents_per_env || mom != h->mom_groups || mom_cap != h->mom_cap || (total && !h->rslot) || (mom && !h->mom)) {
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        cudaFree(h->rslot); h->rslot = nullptr;
        cudaFree(h->mom); h->mom = nullptr;
        // from here until both tables exist the handle has NO agents: a failed allocation must not leave the old groups
        // pointing at freed (or wrongly sized) state
        h->groups.clear(); h->group_asset.clear();
        h->agents_per_env = h->mom_groups = h->chip_agents = 0;
        if (total) CUDA_TRY(h, cudaMalloc(&h->rslot, ne * total * 4));
        h->mom_cap = mom_cap;
        h->mom_stride = MOM_HDR_BYTES + 4u * mom_cap;
        if (mom) CUDA_TRY(h, cudaMalloc(&h->mom, ne * mom * (size_t)h->mom_stride));
    }
    h->groups.assign(groups, groups + n_groups);
    h->group_asset.clear();
    if (asset) h->group_asset.assign(asset, asset + n_groups);
    h->agents_per_env = total;
    h->chip_agents = total;
    if (asset) {
        h->chip_agents = 0;
        for (u32 a = 0; a < h->assets; ++a) {
            u32 n = 0;
            for (u32 i = 0; i < n_groups; ++i)
                if (asset[i] == a) n += groups[i].n_agents;
            h->chip_agents = std::max(h->chip_agents, n);
        }
    }
    h->mom_groups = mom;
    update_rand_tick_mask(h);
    h->lay_sim = make_layout(h, true, false, h->eng >= ENG_DENSE, asset != nullptr);  // the on-chip agent state depends on the population
    if (total) CUDA_TRY(h, cudaMemsetAsync(h->rslot, 0xFF, ne * total * 4, h->stream));
    if (mom) CUDA_TRY(h, cudaMemsetAsync(h->mom, 0, ne * mom * (size_t)h->mom_stride, h->stream));
    return BB_OK;
}

int bb_step_device(bb_handle* h, const bb_instr* d_instrs, const uint64_t* d_env_offsets, uint64_t n_rows, uint64_t* d_out_ids,
                   uint32_t* d_obs_out) {
    CHECK_H(h);
    if (!d_env_offsets || (n_rows && !d_instrs)) return fail(h, BB_EINVAL, "null argument");
    if (h->assets > 1) return fail(h, BB_EINVAL, "bb_step_device drives single-asset envs (multi-asset queues are ordered on the host)");
    if (h->eng == ENG_DEEP) return fail(h, BB_EINVAL, "the deep-book engine replays instruction streams only");
    for (auto& q : h->queue)
        if (!q.empty()) return fail(h, BB_EINVAL, "host-queued instructions pending: call bb_step first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (!d_out_ids) {  // the kernel needs somewhere to keep the ids between assignment and execution
        if (n_rows + 1 > h->d_ids_cap) {
            CUDA_TRY(h, cudaStreamSynchronize(h->stream));
            cudaFree(h->d_ids);
            h->d_ids = nullptr;
            h->d_ids_cap = n_rows + n_rows / 2 + 1024;
            CUDA_TRY(h, cudaMalloc(&h->d_ids, h->d_ids_cap * 8));
        }
        d_out_ids = h->d_ids;
    }
    h->mirror_dirty = true;  // ids were handed out on the device
    return launch_apply(h, MODE_ENV, d_instrs, d_env_offsets, 1, false, d_out_ids, d_obs_out);
}

int bb_level2_device(bb_handle* h, uint32_t* d_out) {
    CHECK_H(h);
    if (!d_out) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return snapshot(h, 0, h->cfg.n_envs, d_out, nullptr, 45u);
}

int bb_level1_device(bb_handle* h, uint32_t* d_out) {
    CHECK_H(h);
    if (!d_out) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    return snapshot(h, 0, h->cfg.n_envs, d_out, nullptr, 9u);
}

int bb_device_alloc(bb_handle* h, uint64_t bytes, void** d_ptr) {
    CHECK_H(h);
    if (!d_ptr) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMalloc(d_ptr, bytes ? bytes : 1));
    return BB_OK;
}

int bb_device_free(bb_handle* h, void* d_ptr) {
    CHECK_H(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, cudaFree(d_ptr));
    return BB_OK;
}

int bb_memcpy(bb_handle* h, void* dst, const void* src, uint64_t bytes, int kind) {
    CHECK_H(h);
    if (kind < 1 || kind > 3) return fail(h, BB_EINVAL, "kind must be 1 (host to device), 2 (device to host) or 3 (device to device)");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemcpyAsync(dst, src, bytes, (cudaMemcpyKind)kind, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_clear_history(bb_handle* h) {
    CHECK_H(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    // every env's record count back to zero (one strided memset over the book headers); the books are untouched
    CUDA_TRY(h, cudaMemset2DAsync(h->blobs + offsetof(BookHdr, n_steps), h->blob_stride, 0, 4, h->cfg.n_envs, h->stream));
    h->recorded_host = 0;
    return BB_OK;
}

int bb_reserve(bb_handle* h, uint32_t max_orders, uint32_t max_trades, uint32_t max_steps) {
    CHECK_H(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (h->copy_stream) CUDA_TRY(h, cudaStreamSynchronize(h->copy_stream));
    const size_t ne = h->cfg.n_envs;
    // one slab at a time: allocate the larger one, copy every env's rows across (2-D copy, old pitch -> new pitch), swap
    auto grow = [&](void** slab, size_t old_row, size_t new_row) -> int {
        void* fresh = nullptr;
        CUDA_TRY(h, cudaMalloc(&fresh, ne * new_row));
        if (*slab && old_row)
            CUDA_TRY(h, cudaMemcpy2DAsync(fresh, new_row, *slab, old_row, old_row, ne, cudaMemcpyDeviceToDevice, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        cudaFree(*slab);
        *slab = fresh;
        return BB_OK;
    };
    int rc;
    if (max_orders > h->cfg.max_orders) {
        if ((rc = grow((void**)&h->ord, (size_t)h->cfg.max_orders * sizeof(OrderRec), (size_t)max_orders * sizeof(OrderRec)))) return rc;
        h->cfg.max_orders = max_orders;
    }
    if (max_trades > h->cfg.max_trades && h->cfg.max_trades) {  // (0 = the trade log is disabled for this handle)
        if ((rc = grow((void**)&h->tr, (size_t)h->cfg.max_trades * sizeof(TradeRec), (size_t)max_trades * sizeof(TradeRec)))) return rc;
        h->cfg.max_trades = max_trades;
    }
    if (max_steps > h->cfg.max_steps) {
        const u32 padded = align_up(max_steps, 4);
        const u64 stride = (u64)padded * h->cfg.obs_words;
        if ((rc = grow((void**)&h->hist, h->hist_env_stride * 4, stride * 4))) return rc;
        h->cfg.max_steps = max_steps;
        h->max_steps_padded = padded;
        h->hist_env_stride = stride;
    }
    return BB_OK;
}

int bb_reserve_queue(bb_handle* h, uint32_t max_queue) {
    CHECK_H(h);
    if (max_queue <= h->cfg.max_queue || h->eng == ENG_DEEP) return BB_OK;  // (the deep-book engine has no Env-step queue)
    if (max_queue > 65535 || (h->assets > 1 && (u64)h->assets * max_queue > 65535))
        return fail(h, BB_EINVAL, "max_queue (times assets, for markets) must stay below 65536");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (h->copy_stream) CUDA_TRY(h, cudaStreamSynchronize(h->copy_stream));
    // the step's permutation (and, for the dense engine's in-kernel agents, the queue itself) lives in shared memory: the
    // layouts are rebuilt for the new capacity, and the request is refused while the Env-step kernel could not run one book
    // per CTA with it (k_sim's fit is checked at its launch, like at creation)
    const u32 old = h->cfg.max_queue;
    h->cfg.max_queue = max_queue;
    const SmemLayout la = make_layout(h, false, true);
    if (la.warp_bytes > 232448u - 1024u) {
        h->cfg.max_queue = old;
        return fail(h, BB_ECAP, "max_queue does not fit in shared memory next to the book image");
    }
    h->lay_apply = la;
    h->lay_sim = make_layout(h, true, false, h->eng >= ENG_DENSE, !h->group_asset.empty());
    h->lay_snap = make_layout(h, false, false);
    cudaFree(h->scratch);  // k_sim's global-memory queues are sized by max_queue: reallocated at the next agent launch
    h->scratch = nullptr;
    h->scratch_warps = 0;
    return BB_OK;
}

int bb_set_agents(bb_handle* h, const bb_agent_group* groups, uint32_t n_groups) {
    return set_agents_impl(h, groups, nullptr, n_groups);
}

int bb_set_agents_market(bb_handle* h, const bb_agent_group* groups, const uint32_t* asset, uint32_t n_groups) {
    if (n_groups && !asset) return fail(h, BB_EINVAL, "null asset array");
    return set_agents_impl(h, groups, asset, n_groups);
}

namespace {
struct ExtRows {  // bb_run_agents_with_rows: the caller's device-resident rows for the launch's first step
    const bb_instr* d_instrs;
    const u64* d_offsets;
    u64* d_out_ids;
    u32* d_obs_out;
};
int run_agents_impl(bb_handle* h, uint64_t seed, uint32_t n_steps, const ExtRows* ext);
}  // namespace

int bb_run_agents(bb_handle* h, uint64_t seed, uint32_t n_steps) { return run_agents_impl(h, seed, n_steps, nullptr); }

int bb_run_agents_with_rows(bb_handle* h, uint64_t seed, const bb_instr* d_instrs, const uint64_t* d_env_offsets, uint64_t n_rows,
                            uint64_t* d_out_ids, uint32_t* d_obs_out) {
    CHECK_H(h);
    if (!d_env_offsets || (n_rows && !d_instrs)) return fail(h, BB_EINVAL, "null argument");
    if (h->assets > 1) return fail(h, BB_EINVAL, "bb_run_agents_with_rows drives single-asset envs");
    const ExtRows ext{d_instrs, d_env_offsets, d_out_ids, d_obs_out};
    return run_agents_impl(h, seed, 1, &ext);
}

namespace {
int run_agents_impl(bb_handle* h, uint64_t seed, uint32_t n_steps, const ExtRows* ext) {
    CHECK_H(h);
    if (h->eng == ENG_DEEP) return fail(h, BB_EINVAL, "the deep-book engine replays instruction streams only");
    if (h->groups.empty()) return fail(h, BB_EINVAL, "bb_set_agents has not been called");
    const bool mkt = !h->group_asset.empty();
    if (h->assets > 1 && !mkt)
        return fail(h, BB_EINVAL, "single-asset agents on a multi-asset handle: use bb_set_agents_market");
    if (n_steps == 0) return BB_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    for (auto& q : h->queue)
        if (!q.empty()) return fail(h, BB_EINVAL, "host-queued instructions pending: call bb_step first");
    {   // k_sim stages its records without per-step capacity checks, so the count must be known on the host: no graph capture
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(h->stream, &cap);
        if (cap != cudaStreamCaptureStatusNone)
            return fail(h, BB_EINVAL, "agent launches cannot be captured into a CUDA graph (bb_step_device can)");
    }
    // history capacity is validated up front so the kernel can stage records without per-step checks
    if (h->recorded_host < 0) {  // after a replay the number of emitted records is only known to the device
        CUDA_TRY(h, cudaMemcpy2DAsync(h->h_offsets, 8, h->blobs + offsetof(BookHdr, n_steps), h->blob_stride, 4, 1,
                                      cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        h->recorded_host = *(u32*)h->h_offsets;
    }
    if ((u64)h->recorded_host + n_steps > h->max_steps_padded) return fail(h, BB_ECAP, "max_steps exceeded");
    KParams p;
    fill_params(h, h->lay_sim, p);
    p.n_steps = n_steps;
    p.n_groups = (u32)h->groups.size();
    p.agents_per_env = h->agents_per_env;
    p.chip_agents = h->chip_agents;
    p.mom_groups_per_env = h->mom_groups;
    p.mom_stride = h->mom_stride;
    p.mom_live_cap = h->mom_cap;
    p.rslot = h->rslot;
    p.mom = h->mom;
    p.seed_lo = (u32)seed;
    p.seed_hi = (u32)(seed >> 32);
    for (size_t i = 0; i < h->groups.size(); ++i) p.groups[i] = h->groups[i];
    p.rand_tick_mask = h->rand_tick_mask;
    for (size_t i = 0; i < h->group_asset.size(); ++i) p.group_asset[i] = h->group_asset[i];
    if (ext) {
        p.instrs = ext->d_instrs;
        p.offsets = ext->d_offsets;
        p.out_ids = ext->d_out_ids;
        p.obs_out = ext->d_obs_out;
    }
    int grid = 0, rc;
    // external rows carry no slot hints: they run on the variants that also serve MomentumAgent / NoiseAgent events.  So
    // does a RandomAgents group that can draw off its book's tick: only those variants check the queued prices
    const bool mom = h->mom_groups != 0 || ext != nullptr || h->rand_tick_mask != 0;
    // markets: the A books of a market are A consecutive warps of one CTA (a CTA holds as many whole markets as fit in 4 warps)
    const u32 wpb = mkt ? (WPB / h->assets) * h->assets : wpb_for(h->lay_sim.warp_bytes);
    const size_t sim_smem = (size_t)h->lay_sim.warp_bytes * wpb;
#define SIM_CASE(E, M)                                                                                     \
    if (h->eng == E && mom == M) {                                                                         \
        if (mkt) { if ((rc = grid_for(h, k_sim<E, M, true>, h->lay_sim, h->cfg.n_envs, &grid, wpb))) return rc; } \
        else if (ext) { if ((rc = grid_for(h, k_sim<E, true, false, true>, h->lay_sim, h->cfg.n_envs, &grid, wpb))) return rc; } \
        else if ((rc = grid_for(h, k_sim<E, M, false>, h->lay_sim, h->cfg.n_envs, &grid, wpb))) return rc;  \
    }
    SIM_CASE(ENG_FAST, false) SIM_CASE(ENG_FAST, true) SIM_CASE(ENG_PAGED, false) SIM_CASE(ENG_PAGED, true)
    SIM_CASE(ENG_DENSE, false) SIM_CASE(ENG_DENSE, true) SIM_CASE(ENG_DENSE_L, false) SIM_CASE(ENG_DENSE_L, true)
#undef SIM_CASE
    const size_t warps = (size_t)grid * wpb;
    if (h->eng < ENG_DENSE && warps > h->scratch_warps) {
        cudaFree(h->scratch);
        h->scratch = nullptr;
        CUDA_TRY(h, cudaMalloc(&h->scratch, warps * h->cfg.max_queue * sizeof(uint4)));
        h->scratch_warps = warps;
    }
    p.scratch = h->scratch;
#define SIM_LAUNCH(E, M)                                                                       \
    if (h->eng == E && mom == M) {                                                             \
        if (mkt) k_sim<E, M, true><<<grid, wpb * 32, sim_smem, h->stream>>>(p);                \
        else if (ext) k_sim<E, true, false, true><<<grid, wpb * 32, sim_smem, h->stream>>>(p); \
        else k_sim<E, M, false><<<grid, wpb * 32, sim_smem, h->stream>>>(p);                   \
    }
    SIM_LAUNCH(ENG_FAST, false) SIM_LAUNCH(ENG_FAST, true) SIM_LAUNCH(ENG_PAGED, false) SIM_LAUNCH(ENG_PAGED, true)
    SIM_LAUNCH(ENG_DENSE, false) SIM_LAUNCH(ENG_DENSE, true) SIM_LAUNCH(ENG_DENSE_L, false) SIM_LAUNCH(ENG_DENSE_L, true)
#undef SIM_LAUNCH
    CUDA_TRY(h, cudaGetLastError());
    h->mirror_dirty = true;
    h->status_valid = false;
    h->recorded_host += n_steps;
    return BB_OK;
}
}  // namespace

// Run n_steps env-steps and stream every env-step's observation record to HOST memory while the simulation runs:
// the steps are launched in chunks, and chunk k's records are copied out on a second stream while chunk k+1 is being
// simulated, so only the last chunk's copy is exposed.  host_out is [n_envs][n_steps][obs_words] u32 (pinned memory
// recommended).  Synchronous: on return the records are in host_out.
int bb_run_agents_to_host(bb_handle* h, uint64_t seed, uint32_t n_steps, uint32_t chunk_steps, uint32_t* host_out) {
    CHECK_H(h);
    if (!host_out) return fail(h, BB_EINVAL, "null argument");
    if (n_steps == 0) return BB_OK;
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (!h->copy_stream) CUDA_TRY(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    if (!h->chunk_done) CUDA_TRY(h, cudaEventCreateWithFlags(&h->chunk_done, cudaEventDisableTiming));
    // chunk_steps == 0: geometric schedule (half of what is left, at least 32 steps): few launches, and the last
    // chunk, whose copy cannot overlap anything, is small.  Chunk sizes are multiples of 8 so that every chunk's first
    // record stays 16-byte aligned for the bulk stores.
    const bool geometric = chunk_steps == 0;
    chunk_steps = align_up(chunk_steps, 8);
    const u32 w = h->cfg.obs_words;
    for (u32 first = 0, n = 0; first < n_steps; first += n) {
        const u32 left = n_steps - first;
        n = geometric ? align_up(left / 2 > 32 ? left / 2 : 32, 8) : chunk_steps;
        if (n > left) n = left;
        int rc = bb_run_agents(h, seed, n);
        if (rc) {  // do not return while earlier chunks are still being copied into the caller's buffer
            cudaStreamSynchronize(h->copy_stream);
            return rc;
        }
        const size_t rec0 = (size_t)h->recorded_host - n;  // first record of this chunk inside each env's history
        CUDA_TRY(h, cudaEventRecord(h->chunk_done, h->stream));
        CUDA_TRY(h, cudaStreamWaitEvent(h->copy_stream, h->chunk_done, 0));
        CUDA_TRY(h, cudaMemcpy2DAsync(host_out + (size_t)first * w, (size_t)n_steps * w * 4, h->hist + rec0 * w,
                                      h->hist_env_stride * 4, (size_t)n * w * 4, h->cfg.n_envs, cudaMemcpyDeviceToHost,
                                      h->copy_stream));
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->copy_stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_level2(bb_handle* h, uint32_t* out) {
    CHECK_H(h);
    if (!out) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = snapshot(h, 0, h->cfg.n_envs, h->d_snap, nullptr);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(out, h->d_snap, (size_t)h->cfg.n_envs * 45 * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_level1(bb_handle* h, uint32_t* out) {
    CHECK_H(h);
    if (!out) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = snapshot(h, 0, h->cfg.n_envs, h->d_snap, nullptr);
    if (rc) return rc;
    // one contiguous copy into pinned memory, compacted on the host: a strided 2-D copy of 36-byte rows costs the
    // copy engine ~0.3 us per row (1.2 ms for 4096 envs, measured), the contiguous 737 KB take ~30 us
    CUDA_TRY(h, cudaMemcpyAsync(h->h_snap, h->d_snap, (size_t)h->cfg.n_envs * 45 * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (size_t e = 0; e < h->cfg.n_envs; ++e) memcpy(out + 9 * e, h->h_snap + 45 * e, 36);
    return BB_OK;
}

int bb_book_level1(bb_handle* h, uint32_t env, uint32_t* out8) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = snapshot(h, env, 1, nullptr, h->d_snap);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(out8, h->d_snap, 32, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_book_level2(bb_handle* h, uint32_t env, uint32_t* out45) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = snapshot(h, env, 1, h->d_snap, nullptr);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(out45, h->d_snap, 180, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

static int read_hdr_u32(bb_handle* h, u32 env, size_t off, u32* v) {
    CUDA_TRY(h, cudaMemcpyAsync(v, h->blobs + (size_t)env * h->blob_stride + off, 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_n_steps(bb_handle* h, uint32_t env, uint32_t* n) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    return read_hdr_u32(h, env, offsetof(BookHdr, n_steps), n);
}

int bb_history(bb_handle* h, uint32_t env, uint32_t first, uint32_t n, uint32_t* out) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    if ((u64)first + n > h->max_steps_padded) return fail(h, BB_EINVAL, "history range out of bounds");
    if (n == 0) return BB_OK;
    const u32 w = h->cfg.obs_words;
    CUDA_TRY(h, cudaMemcpyAsync(out, h->hist + (size_t)env * h->hist_env_stride + (size_t)first * w, (size_t)n * w * 4,
                                cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_history_all(bb_handle* h, uint32_t n_steps, uint32_t* out) {
    CHECK_H(h);
    if (n_steps > h->max_steps_padded) return fail(h, BB_EINVAL, "history range out of bounds");
    if (n_steps == 0) return BB_OK;
    const size_t row = (size_t)n_steps * h->cfg.obs_words * 4;
    CUDA_TRY(h, cudaMemcpy2DAsync(out, row, h->hist, h->hist_env_stride * 4, row, h->cfg.n_envs, cudaMemcpyDeviceToHost,
                                  h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_history_device(bb_handle* h, void** d_ptr, uint64_t* env_stride_words, uint32_t* obs_words) {
    CHECK_H(h);
    if (d_ptr) *d_ptr = h->hist;
    if (env_stride_words) *env_stride_words = h->hist_env_stride;
    if (obs_words) *obs_words = h->cfg.obs_words;
    return BB_OK;
}

int bb_n_orders(bb_handle* h, uint32_t env, uint64_t* n) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    int rc = refresh_mirror(h);
    if (rc) return rc;
    *n = h->n_orders_host[env];
    return BB_OK;
}

int bb_n_trades(bb_handle* h, uint32_t env, uint64_t* n) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    u32 v = 0;
    int rc = read_hdr_u32(h, env, offsetof(BookHdr, n_trades), &v);
    *n = v;
    return rc;
}

int bb_orders(bb_handle* h, uint32_t env, uint64_t first, uint64_t n, uint8_t* side_is_bid, uint8_t* status,
              uint64_t* arr_time, uint64_t* end_time, uint32_t* vol, uint32_t* start_vol, uint32_t* price,
              uint32_t* trader) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    int rc = refresh_mirror(h);
    if (rc) return rc;
    if (first + n > h->n_orders_host[env]) return fail(h, BB_EBADID, "order range out of bounds");
    if (n == 0) return BB_OK;
    // ids below the device count are materialised records; the rest are still New in the host queue
    u64 n_queued_new = 0;
    for (auto& x : h->queue[env]) n_queued_new += (x.op_flags & BB_OP_MASK) == BB_OP_NEW;
    const u64 n_dev = h->n_orders_host[env] - n_queued_new;
    const u64 dev_n = first < n_dev ? std::min(n, n_dev - first) : 0;
    std::vector<OrderRec> rec(dev_n);
    if (dev_n)
        CUDA_TRY(h, cudaMemcpyAsync(rec.data(), h->ord + (size_t)env * h->cfg.max_orders + first, dev_n * sizeof(OrderRec),
                                    cudaMemcpyDeviceToHost, h->stream));
    u64 t_now = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&t_now, h->blobs + (size_t)env * h->blob_stride, 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (u64 i = 0; i < dev_n; ++i) {
        if (side_is_bid) side_is_bid[i] = (rec[i].meta & META_BID) ? 1 : 0;
        if (status) status[i] = (uint8_t)(rec[i].meta & META_STATUS_MASK);
        if (arr_time) arr_time[i] = rec[i].arr_time;
        if (end_time) end_time[i] = rec[i].end_time;
        if (vol) vol[i] = rec[i].vol;
        if (start_vol) start_vol[i] = rec[i].start_vol;
        if (price) price[i] = rec[i].price;
        if (trader) trader[i] = rec[i].trader;
    }
    for (auto& x : h->queue[env]) {
        if ((x.op_flags & BB_OP_MASK) != BB_OP_NEW) continue;
        if (x.order_id < first || x.order_id >= first + n) continue;
        const u64 i = x.order_id - first;
        const bool bid = x.op_flags & BB_F_BID;
        if (side_is_bid) side_is_bid[i] = bid;
        if (status) status[i] = ST_NEW;
        if (arr_time) arr_time[i] = t_now;  // create_order stamps the current book time (orderbook.rs:373)
        if (end_time) end_time[i] = ~0ULL;
        const u32 p = (x.op_flags & BB_F_MARKET) ? (bid ? 0xFFFFFFFFu : 0u) : x.price;
        if (vol) vol[i] = x.vol;
        if (start_vol) start_vol[i] = x.vol;
        if (price) price[i] = p;
        if (trader) trader[i] = x.trader;
    }
    return BB_OK;
}

int bb_trades(bb_handle* h, uint32_t env, uint64_t first, uint64_t n, uint64_t* t, uint8_t* side_is_bid, uint32_t* price,
              uint32_t* vol, uint64_t* active_id, uint64_t* passive_id) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    u32 have = 0;
    int rc = read_hdr_u32(h, env, offsetof(BookHdr, n_trades), &have);
    if (rc) return rc;
    if (first + n > have) return fail(h, BB_EINVAL, "trade range out of bounds");
    if (n == 0) return BB_OK;
    std::vector<TradeRec> rec(n);
    CUDA_TRY(h, cudaMemcpyAsync(rec.data(), h->tr + (size_t)env * h->cfg.max_trades + first, n * sizeof(TradeRec),
                                cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (u64 i = 0; i < n; ++i) {
        if (t) t[i] = rec[i].t;
        if (side_is_bid) side_is_bid[i] = (uint8_t)rec[i].side_bid;
        if (price) price[i] = rec[i].price;
        if (vol) vol[i] = rec[i].vol;
        if (active_id) active_id[i] = rec[i].active;
        if (passive_id) passive_id[i] = rec[i].passive;
    }
    return BB_OK;
}

static_assert(sizeof(bb_order_rec) == sizeof(OrderRec) && sizeof(bb_trade_rec) == sizeof(TradeRec), "public record layouts");

int bb_orders_all(bb_handle* h, uint32_t cap_per_env, bb_order_rec* out, uint32_t* counts) {
    CHECK_H(h);
    if (!out || !counts) return fail(h, BB_EINVAL, "null argument");
    for (auto& q : h->queue)
        if (!q.empty()) return fail(h, BB_EINVAL, "host-queued instructions pending: call bb_step first");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const u32 cap = std::min(cap_per_env, h->cfg.max_orders);
    CUDA_TRY(h, cudaMemcpy2DAsync(counts, 4, h->blobs + offsetof(BookHdr, n_orders), h->blob_stride, 4, h->cfg.n_envs,
                                  cudaMemcpyDeviceToHost, h->stream));
    if (cap)
        CUDA_TRY(h, cudaMemcpy2DAsync(out, (size_t)cap_per_env * sizeof(OrderRec), h->ord, (size_t)h->cfg.max_orders * sizeof(OrderRec),
                                      (size_t)cap * sizeof(OrderRec), h->cfg.n_envs, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_trades_all(bb_handle* h, uint32_t cap_per_env, bb_trade_rec* out, uint32_t* counts) {
    CHECK_H(h);
    if (!out || !counts) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    const u32 cap = std::min(cap_per_env, h->cfg.max_trades);
    CUDA_TRY(h, cudaMemcpy2DAsync(counts, 4, h->blobs + offsetof(BookHdr, n_trades), h->blob_stride, 4, h->cfg.n_envs,
                                  cudaMemcpyDeviceToHost, h->stream));
    if (cap)
        CUDA_TRY(h, cudaMemcpy2DAsync(out, (size_t)cap_per_env * sizeof(TradeRec), h->tr, (size_t)h->cfg.max_trades * sizeof(TradeRec),
                                      (size_t)cap * sizeof(TradeRec), h->cfg.n_envs, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_order_keys(bb_handle* h, uint32_t env, uint64_t first, uint64_t n, uint64_t* key_time) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    int rc = refresh_mirror(h);
    if (rc) return rc;
    if (first + n > h->n_orders_host[env]) return fail(h, BB_EBADID, "order range out of bounds");
    u64 n_queued_new = 0;
    for (auto& x : h->queue[env]) n_queued_new += (x.op_flags & BB_OP_MASK) == BB_OP_NEW;
    const u64 n_dev = h->n_orders_host[env] - n_queued_new;
    const u64 dev_n = first < n_dev ? std::min(n, n_dev - first) : 0;
    std::vector<OrderRec> rec(dev_n);
    if (dev_n) {
        CUDA_TRY(h, cudaMemcpyAsync(rec.data(), h->ord + (size_t)env * h->cfg.max_orders + first, dev_n * sizeof(OrderRec),
                                    cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    for (u64 i = 0; i < n; ++i) key_time[i] = i < dev_n ? rec[i].key_time : 0;
    return BB_OK;
}

int bb_load_book(bb_handle* h, uint32_t env, uint64_t t, uint32_t trade_vol, int trading, uint64_t n_orders,
                 const uint8_t* side_is_bid, const uint8_t* status, const uint64_t* arr_time, const uint64_t* end_time,
                 const uint32_t* vol, const uint32_t* start_vol, const uint32_t* price, const uint32_t* trader,
                 const uint64_t* key_time, uint64_t n_trades, const uint64_t* tr_t, const uint8_t* tr_side_is_bid,
                 const uint32_t* tr_price, const uint32_t* tr_vol, const uint64_t* tr_active, const uint64_t* tr_passive) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    if (!h->queue[env].empty()) return fail(h, BB_EINVAL, "env has queued instructions");
    if (n_orders > h->cfg.max_orders || n_trades > h->cfg.max_trades) return fail(h, BB_ECAP, "snapshot exceeds max_orders / max_trades");
    if (n_orders && !(side_is_bid && status && arr_time && end_time && vol && start_vol && price && trader && key_time))
        return fail(h, BB_EINVAL, "null order column");
    if (n_trades && !(tr_t && tr_side_is_bid && tr_price && tr_vol && tr_active && tr_passive))
        return fail(h, BB_EINVAL, "null trade column");
    // 1. fresh header + page directory for this env, keeping its shuffle stream
    BookHdr hdr;
    CUDA_TRY(h, cudaMemcpyAsync(&hdr, h->blobs + (size_t)env * h->blob_stride, sizeof(hdr), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    const u64 s0 = hdr.rng_s0, s1 = hdr.rng_s1;
    const u32 steps = hdr.n_steps, step_counter = hdr.step_counter;
    memset(&hdr, 0, sizeof(hdr));
    hdr.t = t;
    hdr.rng_s0 = s0;
    hdr.rng_s1 = s1;
    hdr.n_steps = steps;
    hdr.step_counter = step_counter;
    hdr.trade_vol = trade_vol;
    hdr.trading = trading ? 1u : 0u;
    hdr.n_trades = (u32)n_trades;
    hdr.n_trades_total = n_trades;
    std::vector<u32> dir;
    if (h->eng == ENG_DEEP) {  // the image k_init_deep writes: empty bitmaps, zero level volumes / counts, chunk 0 reserved
        dir.assign((h->dp.lht - 128) / 4, 0u);
        dir[(DP_OFF_BUMP - 128) / 4] = 1u;
    } else if (h->eng >= ENG_DENSE) {  // empty bitmaps, every slot free (same image k_init writes)
        const Geo& d = h->dgeo;
        hdr.free_top = d.d_live;
        dir.assign((h->blob_smem_bytes - 128) / 4, 0u);
        unsigned char* img = reinterpret_cast<unsigned char*>(dir.data()) - 128;
        const u32 off_fs = 128u + 12u * h->dense_lp;
        for (u32 i = 0; i < h->dense_lp; ++i) {
            reinterpret_cast<u32*>(img + 128)[i] = BB_NIL;
            img[off_fs + i] = (unsigned char)(i < d.d_live ? d.d_live - 1 - i : 0xFF);
        }
    } else {
        dir.assign(3 * (size_t)h->p_total, 0u);
        std::fill(dir.begin(), dir.begin() + h->p_total, BB_TAG_FREE);
    }
    CUDA_TRY(h, cudaMemcpyAsync(h->blobs + (size_t)env * h->blob_stride, &hdr, sizeof(hdr), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->blobs + (size_t)env * h->blob_stride + 128, dir.data(), dir.size() * 4, cudaMemcpyHostToDevice,
                                h->stream));
    // 2. order table and trade log straight into their slabs
    std::vector<OrderRec> rec(n_orders);
    for (u64 i = 0; i < n_orders; ++i) {
        OrderRec& r = rec[i];
        r.price = price[i]; r.vol = vol[i]; r.next = BB_NIL; r.prev = BB_NIL;
        r.key_time = key_time[i];
        r.meta = (status[i] & META_STATUS_MASK) | (side_is_bid[i] ? META_BID : 0u);
        r.start_vol = start_vol[i]; r.arr_time = arr_time[i]; r.end_time = end_time[i];
        r.trader = trader[i]; r.pad0 = r.pad1 = r.pad2 = 0;
    }
    std::vector<TradeRec> tr(n_trades);
    for (u64 i = 0; i < n_trades; ++i) {
        tr[i].t = tr_t[i]; tr[i].price = tr_price[i]; tr[i].vol = tr_vol[i];
        tr[i].active = (u32)tr_active[i]; tr[i].passive = (u32)tr_passive[i];
        tr[i].side_bid = tr_side_is_bid[i] ? 1u : 0u; tr[i].pad = 0;
    }
    if (n_orders)
        CUDA_TRY(h, cudaMemcpyAsync(h->ord + (size_t)env * h->cfg.max_orders, rec.data(), n_orders * sizeof(OrderRec),
                                    cudaMemcpyHostToDevice, h->stream));
    if (n_trades)
        CUDA_TRY(h, cudaMemcpyAsync(h->tr + (size_t)env * h->cfg.max_trades, tr.data(), n_trades * sizeof(TradeRec),
                                    cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    // 3. rebuild the sides on the device: one RESTORE instruction per order, in id order
    std::vector<bb_instr> ins(n_orders);
    std::vector<u32> order(n_orders);
    for (u64 i = 0; i < n_orders; ++i) order[i] = (u32)i;
    // the dense and deep engines only append to their queues: feed them the orders by key time (ties keep id order)
    if (h->eng >= ENG_DENSE)
        std::stable_sort(order.begin(), order.end(), [&](u32 a, u32 b) { return key_time[a] < key_time[b]; });
    for (u64 i = 0; i < n_orders; ++i) {
        memset(&ins[i], 0, sizeof(bb_instr));
        ins[i].t = t;
        ins[i].op_flags = BB_OP_RESTORE;
        ins[i].order_id = order[i];
    }
    std::vector<u64> offs(h->cfg.n_envs + 1, 0);
    for (u32 e = env + 1; e <= h->cfg.n_envs; ++e) offs[e] = n_orders;
    int rc = ensure_instr_capacity(h, n_orders + 1);
    if (rc) return rc;
    if (n_orders) memcpy(h->h_instrs, ins.data(), n_orders * sizeof(bb_instr));
    memcpy(h->h_offsets, offs.data(), offs.size() * 8);
    if (n_orders) CUDA_TRY(h, cudaMemcpyAsync(h->d_instrs, h->h_instrs, n_orders * sizeof(bb_instr), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_offsets, h->h_offsets, offs.size() * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = launch_apply(h, MODE_REPLAY, h->d_instrs, h->d_offsets, 0))) return rc;
    if ((rc = check_device_errors(h))) return rc;
    // the replay left hdr.t at the last instruction's time == t; counters restored below
    h->n_orders_host[env] = n_orders;
    return BB_OK;
}

int bb_order_status(bb_handle* h, uint32_t env, uint64_t order_id, uint8_t* status) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    int rc = refresh_mirror(h);
    if (rc) return rc;
    if (order_id >= h->n_orders_host[env])
        return fail(h, BB_EBADID, "No order with id " + std::to_string(order_id) + " exists");
    for (auto& x : h->queue[env])
        if ((x.op_flags & BB_OP_MASK) == BB_OP_NEW && x.order_id == order_id) {
            *status = ST_NEW;
            return BB_OK;
        }
    // Statuses only change inside launches: the first query after one brings the env's whole status column to the host
    // (one contiguous copy of its order records) and later queries are served from it.  The reference's Python agents
    // ask for the status of every held order each step (src/bourse/step_sim/agents/random_agent.py:77-91); one device
    // round trip per query made that loop 4x slower than it needs to be.
    if (!(h->status_valid && h->status_env == env && order_id < h->status_cache.size())) {
        u64 n_queued_new = 0;
        for (auto& x : h->queue[env]) n_queued_new += (x.op_flags & BB_OP_MASK) == BB_OP_NEW;
        const u64 n_dev = h->n_orders_host[env] - n_queued_new;
        if (order_id >= n_dev) return fail(h, BB_EBADID, "No order with id " + std::to_string(order_id) + " exists");
        h->status_rec.resize(n_dev);
        CUDA_TRY(h, cudaMemcpyAsync(h->status_rec.data(), h->ord + (size_t)env * h->cfg.max_orders, n_dev * sizeof(OrderRec),
                                    cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        h->status_cache.resize(n_dev);
        for (u64 i = 0; i < n_dev; ++i) h->status_cache[i] = (uint8_t)(h->status_rec[i].meta & META_STATUS_MASK);
        h->status_env = env;
        h->status_valid = true;
    }
    *status = h->status_cache[order_id];
    return BB_OK;
}

int bb_time(bb_handle* h, uint32_t env, uint64_t* t) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    CUDA_TRY(h, cudaMemcpyAsync(t, h->blobs + (size_t)env * h->blob_stride, 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_set_time(bb_handle* h, uint32_t env, uint64_t t) {
    CHECK_H(h);
    CHECK_ENV(h, env);
    CUDA_TRY(h, cudaMemcpyAsync(h->blobs + (size_t)env * h->blob_stride, &t, 8, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_set_trading(bb_handle* h, uint32_t env, int on) {
    CHECK_H(h);
    const u32 first = env == BB_ALL_ENVS ? 0 : env, cnt = env == BB_ALL_ENVS ? h->cfg.n_envs : 1;
    if (env != BB_ALL_ENVS) CHECK_ENV(h, env);
    std::vector<u32> v(cnt, on ? 1u : 0u);
    CUDA_TRY(h, cudaMemcpy2DAsync(h->blobs + (size_t)first * h->blob_stride + offsetof(BookHdr, trading), h->blob_stride,
                                  v.data(), 4, 4, cnt, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_env_errors(bb_handle* h, uint32_t* out) {
    CHECK_H(h);
    CUDA_TRY(h, cudaMemcpy2DAsync(out, 4, h->blobs + offsetof(BookHdr, err), h->blob_stride, 4, h->cfg.n_envs,
                                  cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return BB_OK;
}

int bb_clear_errors(bb_handle* h) {
    CHECK_H(h);
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemset2DAsync(h->blobs + offsetof(BookHdr, err), h->blob_stride, 0, 4, h->cfg.n_envs, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->err_flag, 0, 4, h->stream));
    return BB_OK;
}

int bb_stats(bb_handle* h, bb_stats_t* out) {
    CHECK_H(h);
    if (!out) return fail(h, BB_EINVAL, "null argument");
    CUDA_TRY(h, cudaSetDevice(h->cfg.device));
    CUDA_TRY(h, cudaMemsetAsync(h->d_stats, 0, 64, h->stream));
    k_stats<<<(h->cfg.n_envs + 255) / 256, 256, 0, h->stream>>>(h->blobs, h->blob_stride, h->cfg.n_envs, h->d_stats);
    CUDA_TRY(h, cudaGetLastError());
    unsigned long long v[8];
    CUDA_TRY(h, cudaMemcpyAsync(v, h->d_stats, 64, cudaMemcpyDeviceToHost, h->stream));
    std::vector<u32> l1((size_t)h->cfg.n_envs * 9);
    int rc = bb_level1(h, l1.data());
    if (rc) return rc;
    u64 fnv = 0xcbf29ce484222325ULL;
    const unsigned char* b = (const unsigned char*)l1.data();
    for (size_t i = 0; i < l1.size() * 4; ++i) fnv = (fnv ^ b[i]) * 0x100000001b3ULL;
    out->instructions = v[0];
    out->orders_created = v[1];
    out->trades = v[2];
    out->traded_volume = v[3];
    out->env_steps = v[4];
    out->transitions = v[5];
    out->error_envs = v[6];
    out->l1_checksum = fnv;
    return BB_OK;
}

}  // extern "C"
