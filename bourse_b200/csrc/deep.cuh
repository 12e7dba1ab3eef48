// Deep-book engine, shared definitions (included by kernels.cuh): the shared-memory map of a deep book, the control words its
// warps talk through, the retire-ring entry kinds, acquire / release and async-copy helpers, the bounded spin.  The engine itself
// is deepw.cuh (book side: decode / ladder chain / queue replay) and kernels.cuh (fetch warp, retire warp, k_deepw).
//
// Same reference semantics as the other engines (side.rs:36-143, orderbook.rs:429-772), built for books with ~10^6 resting
// orders (BASELINE config C5): ONE CTA PER BOOK.
//
// Price-time queues are ARRAYS, not linked lists: a level's FIFO is a chain of 256-byte chunks in HBM (31 entries of
// {order id, remaining volume} + a link).  An order remembers the position of its entry, so a cancel writes a tombstone
// there and never touches its neighbours, and a sweep reads consecutive entries.
//
// The fetch warp runs ahead of the book, so the order record it prefetches for a cancel / modify may be older than a write
// that is still on its way to HBM.  The record may be used only if no event that touched the order (its own events, or a
// sweep that filled it) was still in the pipeline when it was read: a filter of recently touched order ids (and of recently
// swept levels) answers that, and the doubtful case waits for the pipeline to drain and reads the record again.
//
// Preconditions (violations set a per-env error bit and never change results silently):
//   * resting prices inside [d_win_lo, d_win_lo + d_levels)                                     else ERR_CAP_PAGES
//   * strictly increasing time between resting inserts (no equal-(price, time) keys, N1)         else ERR_TIME_ORDER
//   * a price level holds one side at a time (true while trading is enabled and volumes are > 0)  else ERR_LOCKED
//   * chunk pool not exhausted                                                                   else ERR_CAP_PAGES
#pragma once

namespace bb {

#define ERR_LOCKED 0x800u  // deep engine: both sides resting at one price (trading disabled, or a crossing zero-volume order)

// ---- shared-memory image of a deep book (persisted in the book blob between launches) -------------------------------
//   0     BookHdr (128 B; free_top doubles as the "a zero-volume order has rested" flag)
//   128   chunk_bump u32 (next never-used chunk id; chunk 0 is a sink), n_free u32 (entries on the free-chunk stack)
//   192   free-chunk stack u32 [DP_FS_CAP]                                                     (queue warp)
//   1216  bitmap ask [NW], bitmap bid [NW]   bit q set <=> level q holds resting orders of that side   (ladder warp)
//         summary ask [8], summary bid [8]   bit w set <=> bitmap word w is non-zero                   (ladder warp)
//         lvol [W] u32   resting volume per price level                                                (ladder warp)
//         lcnt [W] u32   resting orders per price level                                                (queue warp)
//         lht  [W] u64   {head, tail} of the level's queue: chunk id << 5 | entry index (tail: next free entry)  (queue warp)
#define DP_OFF_BUMP 128u
#define DP_OFF_NFREE 132u
#define DP_OFF_FS 192u
#define DP_FS_CAP 256u
#define DP_OFF_BM (DP_OFF_FS + 4u * DP_FS_CAP)
#define DP_NS 8u  // summary words per side: up to 8192 levels
#define DP_CHUNK_BYTES 256u
#define DP_CHUNK_ENTRIES 31u
// scratch (not persisted), relative to the end of the image
#define DP_RENT 32u
struct DeepOff {             // byte offsets from the CTA's shared-memory base, filled by the host
    u32 bm, sm, lvol, lcnt, lht, image_bytes;
    u32 smem_image;  // bytes of the image that live in shared memory during a launch (k_deepw: up to lcnt; its queues' counts / heads / tails stay in the blob)
    u32 scratch, ev_ins, ev_rec, ev_rf, ret, dirty, swept, ctl, bar, total;
    u32 dirty_n, swept_n;  // filter sizes (powers of two): larger when few books share an SM (fewer false doubts)
};
// control words (u32 each, at DeepOff::ctl)
#define CT_EV_READY 0u      // fetch: batches published
#define CT_EV_CONSUMED 4u   // ladder: batches it is done with
#define CT_CMD_TAIL 8u      // ladder: commands produced
#define CT_CMD_DONE 12u     // queue: commands fully processed
#define CT_RET_TAIL 16u     // queue: retire entries produced
#define CT_RET_DONE 20u     // retire: entries whose stores are performed and fenced
#define CT_Q_EV 24u         // queue: events whose commands are all processed (published after CT_RET_TAIL)
#define CT_EV_RETIRED 28u   // retire: events whose record writes are all performed and fenced
#define CT_FIN_L 32u        // ladder: no more commands will come
#define CT_FIN 36u          // queue: no more retire entries will come
#define CT_ABORT 40u        // any warp: a bounded wait ran out (the launch flags 0x80000000 and unwinds)
#define CT_RERR 44u         // retire warp's error bits
#define CT_QERR 48u         // queue warp's error bits
#define CT_LERR 52u         // ladder warp's error bits
#define CT_QNTR 56u         // queue warp: trades made in this launch
// k_deepw (deepw.cuh): chain warp <-> replay warp
#define CT_MOP_TAIL 64u     // chain: micro-ops published
#define CT_MOP_DONE 68u     // replay: micro-ops replayed
#define CT_DRAIN 72u        // chain: odd = "finish what is published, then park" (even: run)
#define CT_PARKED 76u       // replay: the CT_DRAIN value it has parked for
#define RS_BUMP 80u         // the replay warp's scalars, at rest here between rounds (the chain warp borrows them while the
#define RS_NFREE 84u        // replay warp is parked: complex events run on the chain warp)
#define RS_NTR 88u
#define RS_RET_TAIL 92u
#define RS_ERR 96u
#define CT_TICK 100u        // the book's tick (level-2 records), written at set-up
#define CT_WORDS 32u

// retire entry kinds
#define RK_NEW 1u
#define RK_REPLACE 2u
#define RK_FILL 3u
#define RK_CANCEL 4u
#define RK_REDUCE 5u

__device__ __forceinline__ u32 ld_acq(u32 a) {
    u32 v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void st_rel(u32 a, u32 v) { asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u64 ldg64_cg(u64 a) {
    u64 v;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint4 ldg128_cg(u64 a) {
    uint4 v;
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(a) : "memory");
    return v;
}
__device__ __forceinline__ void cp_async16(u32 smem_dst, u64 gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
// Developer profiling (-DDP_PROF): cycles book 0's warps spend in each kind of wait, printed at the end of the launch.
#ifdef DP_PROF
__device__ unsigned long long g_dp_prof[64];
#define DP_T0 const long long dp_t0_ = clock64();
#define DP_ADD(slot)                                                                  \
    if (blockIdx.x == 0) {                                                            \
        atomicAdd(&g_dp_prof[slot], (unsigned long long)(clock64() - dp_t0_));        \
        atomicAdd(&g_dp_prof[32 + (slot)], 1ull);                                     \
    }
#else
#define DP_T0
#define DP_ADD(slot)
#endif
// bounded spin on a control word; returns false when the wait ran out or another warp aborted
#define DP_SPIN_MAX (1u << 25)
// NAP: the waiting warp sleeps between polls (producers / consumers that are far ahead: their polling would otherwise take
// issue slots and shared-memory bandwidth from the book warps of the SM)
template <bool NAP = false, class F> __device__ __forceinline__ bool dp_wait(u32 ctl, F cond, int prof_slot = 0) {
    DP_T0
    for (u32 spin = 0; spin < DP_SPIN_MAX; ++spin) {
        if (cond()) {
            DP_ADD(prof_slot)
            return true;
        }
        if (NAP && spin >= 4u) __nanosleep(spin < 64u ? 100u : 400u);
        if ((spin & 255u) == 255u && ld_acq(ctl + CT_ABORT)) return false;
    }
    st_rel(ctl + CT_ABORT, 1u);
    return false;
}
__device__ __forceinline__ u32 dp_keep32(u32 v) {
    u32 r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
    return r;
}
__device__ __forceinline__ u64 dp_keep64(u64 v) {
    u64 r;
    asm volatile("mov.u64 %0, %1;" : "=l"(r) : "l"(v));
    return r;
}

}  // namespace bb
