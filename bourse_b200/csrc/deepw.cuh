// Deep-book engine, the book side: chain warp and replay warp (included by kernels.cuh after deep.cuh; kernel k_deepw).
//
// Reference semantics: side.rs:36-143, orderbook.rs:429-772.  Data structures (deep.cuh): dense tick-indexed level volumes +
// per-side bitmaps in shared memory, chunked array queues in HBM, fetch warp in front, retire warp behind.  The first version of
// this engine ran one event at a time on lane 0 of two warps (ladder, queue): ~200 dependent instructions each per event, 1250
// cycles per event on a B200 SM (profiles/r02_summary.md) — a single thread of a GPU is a slow CPU.  Here an event's work is
// cut along its data, and only the true recurrence stays serial.  Two warps, a ring of micro-ops between them:
//
// CHAIN WARP
//
//   decode    (32 events, one lane each) everything about an event that does not depend on the book: what kind of
//             instruction it is, whether the order record the fetch warp prefetched can be trusted (not touched by an event
//             still on its way to HBM, not named twice in the batch), where the order it names rests.  Anything unusual —
//             a market-data record, a zero-volume order, a doubtful record, trading switched off, time standing still —
//             makes the event COMPLEX: it runs alone through the whole reference algorithm (bk_serial);
//   chain     the price ladder, strictly in event order but nothing else: level volumes, bitmaps, best bid / ask.  It
//             decides how much an aggressive order takes from each level it crosses and where an order rests, and writes
//             that down as MICRO-OPS, each on ONE price level: T(ake) q volume, A(ppend) q order, R(emove) q position,
//             D(ecrease) q position volume.  Lane 0 runs it alone (plain loads / stores, side-specialised code) and writes
//             16-byte records; all lanes then turn them into self-contained 32-byte micro-ops in the ring.
// REPLAY WARP
//   replay    (32 micro-ops, one lane each) the price-time queues.  Levels are independent, so the micro-ops are grouped
//             by level (__match_any_sync) and the first lane of every group walks its level's FIFO through the group's
//             micro-ops in order — all levels of the round at the same time.  Fills are staged with their (micro-op, rank)
//             key; a warp prefix sum over the fill counts then gives every trade its place in the trade log and in the
//             retire ring in event order, one trade per passive order in queue order (orderbook.rs:429-454, 843-870).
//
// Queue entries are read with ordinary (L1-cached) loads: only this CTA ever touches its book's chunk pool, the head
// chunks of the levels around the touch stay in L1 (latency close to shared memory), and a lane can walk its level alone.
// Trades go to the trade log straight from the replay warp (their order in the log is the event order = the ring order);
// order-record updates go through the retire ring to the retire warp.  Complex events run on the chain warp while the replay
// warp is parked (bk_borrow / bk_give_back: the queues' scalars change hands through the control block).
#pragma once

namespace bb {

#define DW_RB 4u        // event-ring depth in batches of 32
#define DW_RCAP 256u    // retire-ring entries
#define DW_DIRTY 2048u  // touched-order filter buckets (by order id) / DW_SWEPT swept-level filter buckets (by level): the sizes
#define DW_SWEPT 256u   // for launches with more than two books per SM; 8192 / 1024 otherwise (DeepOff::dirty_n, swept_n)
#define DW_MOPS 128u    // micro-op ring (32 bytes each) between the chain warp and the replay warp; a replay round takes up to 32
#define DW_COUT 64u     // the chain's output list per run (16 bytes each)
#define DW_FILLS 192u   // fills staged per flush (16 bytes each): also the largest volume one flush may take
// scratch block (byte offsets from BkReg::scr)
#define SC_MOP 0u
#define SC_EVD (SC_MOP + 32u * DW_MOPS)      // decoded events, 48 bytes per lane
#define SC_FILL (SC_EVD + 48u * 32u)         // staged fills {micro-op | rank << 8, passive id, traded volume, passive volume left}
#define SC_NFILL (SC_FILL + 16u * DW_FILLS)  // per micro-op of the round: fills made
#define SC_POS (SC_NFILL + 4u * 32u)         // ... position of the appended entry
#define SC_SPARE (SC_POS + 4u * 32u)         // ... a fresh chunk (bit 31: used)
#define SC_FREED (SC_SPARE + 4u * 32u)       // ... up to two chunks it emptied
#define SC_FCOUNT (SC_FREED + 8u * 32u)
#define SC_SWEPT (SC_FCOUNT + 16u)           // the swept-level filter at its compact size (DW_SWEPT buckets; larger ones live elsewhere)
#define SC_COUT (SC_SWEPT + 4u * DW_SWEPT)   // the chain's output: one 16-byte record per micro-op
#define DW_SCRATCH (SC_COUT + 16u * DW_COUT)

__device__ __forceinline__ void reds_max(u32 a, u32 v) { asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u32 atoms_add(u32 a, u32 v) {
    u32 o;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory");
    return o;
}

struct BkReg {  // launch-invariant addresses and limits (pinned in registers)
    u32 lvol, bma, bmb, sma, smb, scr, ret, dirty, swept, ctl, fs;
    u32 dirty_mask, swept_mask;
    u32 win_lo, W, max_orders, n_chunks, max_trades;
    u64 oh, chunks, tr;
    u64 lcnt, lht;  // per level, in the book's blob (global memory, L1-cached: only this CTA touches them): resting orders;
                    // {head, tail} of the level's queue: chunk id << 5 | entry index (tail: next free entry)
};
struct BkSt {  // the book's scalar state: warp-uniform (every lane holds the same values)
    u64 t, max_key_time;
    u32 n_orders, trade_vol, vol_ask, vol_bid, bq_ask, bq_bid, flags, err;
    u32 d_instr, d_applied, zv;
    u32 bump, n_free;       // chunk allocator
    u32 n_tr;               // next trade-log index
    u32 ret_tail, ret_room, ret_pub;
    u32 n_emit, done_seen;  // chain warp: micro-ops written to the ring, (a lower bound of) those the replay warp has finished
    u32 drain_seq;          // chain warp: the CT_DRAIN value last written
#ifdef DP_PROF
    u32 pf_flush, pf_rounds, pf_mops, pf_ser, pf_reason[8];
#endif
};
__device__ __forceinline__ u32 bk_bm(const BkReg& r, u32 side, u32 w) { return (side ? r.bmb : r.bma) + 4u * w; }
__device__ __forceinline__ u32 bk_sm(const BkReg& r, u32 side, u32 w) { return (side ? r.smb : r.sma) + 4u * w; }
__device__ __forceinline__ bool bk_has_best(const BkSt& s, u32 side) { return (s.flags >> (1u + side)) & 1u; }
__device__ __forceinline__ u32 bk_best_q(const BkSt& s, u32 side) { return side ? s.bq_bid : s.bq_ask; }
__device__ __forceinline__ void bk_add_side(BkSt& s, u32 side, u32 dv) {
    if (side) s.vol_bid += dv; else s.vol_ask += dv;
}

// lane 0 polls a control word until cond() holds; the outcome is broadcast so that the warp stays uniform
template <class F> __device__ __forceinline__ bool bk_wait(const BkReg& r, u32 lane, F cond, int prof_slot) {
    u32 ok = 1u;
    if (lane == 0u) ok = dp_wait(r.ctl, cond, prof_slot) ? 1u : 0u;
    return __shfl_sync(BB_FULL, ok, 0) != 0u;
}

// ---- retire ring ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool bk_ret_space(const BkReg& r, BkSt& s, u32 lane, u32 n) {
    if (s.ret_tail + n <= s.ret_room) return true;
    u32 room = 0u;
    __syncwarp();  // (the other lanes' ring entries are ordered before lane 0's release)
    if (lane == 0u && s.ret_pub != s.ret_tail) st_rel(r.ctl + CT_RET_TAIL, s.ret_tail);  // what waits to be drained must be visible
    s.ret_pub = s.ret_tail;
    const u32 tail = s.ret_tail;
    const bool ok = bk_wait(r, lane, [&] {
        room = ld_acq(r.ctl + CT_RET_DONE) + DW_RCAP;
        return tail + n <= room;
    }, 8);
    s.ret_room = __shfl_sync(BB_FULL, room, 0);
    return ok;
}
__device__ __forceinline__ void bk_ret_write(const BkReg& r, u32 idx, uint4 a, uint4 b) {
    const u32 ea = r.ret + DP_RENT * (idx & (DW_RCAP - 1u));
    sts128(ea, a);
    sts128(ea + 16u, b);
}
// one entry, written by lane 0
__device__ __forceinline__ bool bk_ret1(const BkReg& r, BkSt& s, u32 lane, uint4 a, uint4 b) {
    if (!bk_ret_space(r, s, lane, 1u)) return false;
    if (lane == 0u) bk_ret_write(r, s.ret_tail, a, b);
    s.ret_tail += 1;
    return true;
}
// everything produced so far becomes visible to the retire warp; `ev_done` events are complete
__device__ __forceinline__ void bk_publish(const BkReg& r, BkSt& s, u32 lane, u32 ev_done) {
    __syncwarp();
    if (lane == 0u) {
        if (s.ret_pub != s.ret_tail) st_rel(r.ctl + CT_RET_TAIL, s.ret_tail);
        st_rel(r.ctl + CT_Q_EV, ev_done);
    }
    s.ret_pub = s.ret_tail;
}

// ---- trade log (types.rs:105-118), written by the lane that found the fill ---------------------------------------------
__device__ __forceinline__ void bk_trade(const BkReg& r, BkSt& s, u32 ti, u32 t_lo, u32 t_hi, u32 price, u32 vol, u32 active, u32 passive,
                                         u32 passive_bid, u32& err) {
    if (ti < r.max_trades) {
        const u64 ta = r.tr + (u64)ti * 32u;
        stg128_cs(ta, t_lo, t_hi, price, vol);
        stg128_cs(ta + 16u, active, passive, passive_bid, 0u);
    } else if (r.max_trades) {
        err |= ERR_CAP_TRADES;
    }
}

// ---- chunk pool (warp-uniform; lane 0 stores) --------------------------------------------------------------------------
__device__ __forceinline__ u64 bk_chunk(const BkReg& r, u32 c) { return r.chunks + (u64)c * DP_CHUNK_BYTES; }
__device__ __forceinline__ u32 bk_alloc(const BkReg& r, BkSt& s, u32 lane) {
    u32 c;
    if (s.n_free) {
        s.n_free -= 1;
        c = lds(r.fs + 4u * s.n_free);
    } else if (s.bump < r.n_chunks) {
        c = s.bump++;
    } else {
        s.err |= ERR_CAP_PAGES;
        return 0u;  // chunk 0 is never handed out: a safe sink
    }
    if (lane == 0u) stg32(bk_chunk(r, c) + 8u * DP_CHUNK_ENTRIES, BB_NIL);
    return c;
}
__device__ __forceinline__ void bk_free_chunk(const BkReg& r, BkSt& s, u32 lane, u32 c) {
    if (c != 0u && s.n_free < DP_FS_CAP) {
        if (lane == 0u) sts(r.fs + 4u * s.n_free, c);
        s.n_free += 1;
        __syncwarp();
    }
}

// level q of `side` just became empty (its bitmap bit is still set): clear it and, if it was the touch, find the next one
// SOLO: called by lane 0 alone (the chain): plain program order, no warp synchronisation.
template <bool SOLO = false>
__device__ __forceinline__ void bk_level_gone(const BkReg& r, BkSt& s, u32 lane, u32 side, u32 q) {
    const u32 w = q >> 5;
    const u32 ba = bk_bm(r, side, w);
    const u32 m = lds(ba) & ~(1u << (q & 31u));
    const u32 sa = bk_sm(r, side, w >> 5);
    const u32 sv = lds(sa);
    if (!SOLO) __syncwarp();
    if (SOLO || lane == 0u) {
        sts(ba, m);
        if (m == 0u) sts(sa, sv & ~(1u << (w & 31u)));
    }
    if (!SOLO) __syncwarp();
    if (!(bk_has_best(s, side) && bk_best_q(s, side) == q)) return;
    // q was the best level: every other level of this side lies on the far side of it
    if (side == 0u) {
        if (m) { s.bq_ask = (w << 5) + (u32)__ffs(m) - 1u; return; }
        u32 sw = w >> 5;
        u32 ms = lds(bk_sm(r, 0u, sw)) & ~((2u << (w & 31u)) - 1u);  // summary bits above word w
        while (ms == 0u) {
            if (++sw >= DP_NS) { s.flags &= ~FL_HAS_ASK; return; }
            ms = lds(bk_sm(r, 0u, sw));
        }
        const u32 w2 = (sw << 5) + (u32)__ffs(ms) - 1u;
        s.bq_ask = (w2 << 5) + (u32)__ffs(lds(bk_bm(r, 0u, w2))) - 1u;
    } else {
        if (m) { s.bq_bid = (w << 5) + 31u - (u32)__clz(m); return; }
        u32 sw = w >> 5;
        u32 ms = lds(bk_sm(r, 1u, sw)) & ((1u << (w & 31u)) - 1u);  // summary bits below word w
        while (ms == 0u) {
            if (sw == 0u) { s.flags &= ~FL_HAS_BID; return; }
            --sw;
            ms = lds(bk_sm(r, 1u, sw));
        }
        const u32 w2 = (sw << 5) + 31u - (u32)__clz(ms);
        s.bq_bid = (w2 << 5) + 31u - (u32)__clz(lds(bk_bm(r, 1u, w2)));
    }
}

// insert_order's queue half (side.rs:54-66), one order, warp-uniform: append to the level's chunk chain -> entry position
__device__ __forceinline__ u32 bk_append(const BkReg& r, BkSt& s, u32 lane, u32 q, u32 id, u32 vol) {
    const u32 cnt = ldg32(r.lcnt + 4u * q);
    const u32 tail = ldg32(r.lht + 8u * q + 4u);
    __syncwarp();
    u32 pos;
    if (cnt == 0u) {
        const u32 c = bk_alloc(r, s, lane);
        pos = c << 5;
        if (lane == 0u) stg64(r.lht + 8u * q, ((u64)(pos + 1u) << 32) | pos);
    } else {
        u32 c = tail >> 5, idx = tail & 31u;
        if (idx == DP_CHUNK_ENTRIES) {  // tail chunk full: link a new one
            const u32 c2 = bk_alloc(r, s, lane);
            if (lane == 0u) stg32(bk_chunk(r, c) + 8u * DP_CHUNK_ENTRIES, c2);
            c = c2;
            idx = 0u;
        }
        pos = (c << 5) | idx;
        if (lane == 0u) stg32(r.lht + 8u * q + 4u, pos + 1u);
    }
    if (lane == 0u) {
        stg32(r.lcnt + 4u * q, cnt + 1u);
        stg64(bk_chunk(r, pos >> 5) + 8u * (pos & 31u), ((u64)vol << 32) | id);
    }
    __syncwarp();
    return pos;
}
// remove_order's queue half (side.rs:75-84): tombstone the entry
__device__ __forceinline__ void bk_remove(const BkReg& r, BkSt& s, u32 lane, u32 q, u32 pos) {
    const u32 cnt = ldg32(r.lcnt + 4u * q);
    const u64 ht = ldg64(r.lht + 8u * q);
    __syncwarp();
    if (lane == 0u) {
        stg32(bk_chunk(r, pos >> 5) + 8u * (pos & 31u), BB_NIL);
        stg32(r.lcnt + 4u * q, cnt <= 1u ? 0u : cnt - 1u);
    }
    if (cnt <= 1u && ((u32)ht >> 5) == ((u32)(ht >> 32) >> 5)) bk_free_chunk(r, s, lane, (u32)ht >> 5);  // a longer all-dead chain is left to the pool
    __syncwarp();
}

// ---- match_orders over one level (orderbook.rs:843-870), the whole warp: a prefix sum over the FIFO ------------------------
// Takes `take` volume from the head of level q's queue — and, with `exhaust`, every order left there afterwards (the
// aggressor still had volume, so it also trades, at volume 0, with the zero-volume orders behind: `while order.vol > 0`,
// orderbook.rs:436).  Lanes load consecutive queue entries of the head chunk, an inclusive scan over the resting volumes
// tells every lane whether its order is reached and whether it is filled completely; one trade per passive order, in queue
// order.  `mark`: the value the touched orders' filter buckets get.
__device__ __forceinline__ bool bk_sweep(const BkReg& r, BkSt& s, u32 lane, u32 q, u32 opp, u32 take, bool exhaust, u32 id, u32 t_lo, u32 t_hi,
                                         u32 price, u32 mark, u32& lane_err) {
    for (u32 guard = 0; guard < (1u << 22); ++guard) {
        const u32 cnt0 = ldg32(r.lcnt + 4u * q);
        if (!((take > 0u || exhaust) && cnt0 > 0u)) break;
        const u64 ht = ldg64(r.lht + 8u * q);
        const u32 head = (u32)ht, tail = (u32)(ht >> 32);
        const u32 c = head >> 5, idx = head & 31u, tc = tail >> 5;
        const u32 end = (c == tc) ? (tail & 31u) : DP_CHUNK_ENTRIES;
        const u64 e = ldg64(bk_chunk(r, c) + 8u * lane);  // the head chunk: one coalesced 256-byte load (L1)
        const u32 nc = __shfl_sync(BB_FULL, (u32)e, 31);   // (its last 8 bytes are the link)
        const u32 pid = (u32)e, pvol = (u32)(e >> 32);
        const bool live = lane >= idx && lane < end && pid != BB_NIL;
        const u32 v = live ? pvol : 0u;
        u32 incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 y = __shfl_up_sync(BB_FULL, incl, d);
            if (lane >= (u32)d) incl += y;
        }
        const u32 excl = incl - v;
        const bool reached = live && (excl < take || exhaust);
        const bool full = reached && incl <= take;
        const u32 mr = __ballot_sync(BB_FULL, reached), mf = __ballot_sync(BB_FULL, full);
        const u32 mp = mr & ~mf;
        const u32 nr = __popc(mr);
        const u32 total = __shfl_sync(BB_FULL, incl, 31);
        const u32 traded = min(take, total);
        if (!bk_ret_space(r, s, lane, nr)) return false;
        if (reached) {
            const u32 tv = full ? pvol : take - excl;
            const u32 pv = pvol - tv;
            const u32 k = __popc(mr & ((1u << lane) - 1u));
            // trade: side / price are the passive order's (orderbook.rs:853-862)
            bk_ret_write(r, s.ret_tail + k, make_uint4(RK_FILL | (opp << 8) | (pv == 0u ? 0x10000u : 0u), pid, tv, pv), make_uint4(t_lo, t_hi, price, id));
            bk_trade(r, s, s.n_tr + k, t_lo, t_hi, price, tv, id, pid, opp, lane_err);
            reds_max(r.dirty + 4u * (pid & r.dirty_mask), mark);
            if (!full) stg32(bk_chunk(r, c) + 8u * lane + 4u, pv);  // the partially filled order stays at the head of its level
        }
        take -= traded;
        s.ret_tail += nr;
        s.n_tr += nr;
        const u32 cnt = cnt0 - __popc(mf);
        __syncwarp();
        bool done = false;
        if (cnt == 0u) {  // the level is gone
            if (c == tc) bk_free_chunk(r, s, lane, c);
            if (lane == 0u) stg32(r.lcnt + 4u * q, 0u);
        } else {
            u32 nh = 0u;
            bool bad = false;
            if (mp) {
                nh = (c << 5) | ((u32)__ffs(mp) - 1u);
                done = true;
            } else if (take == 0u && !exhaust) {  // ended exactly on an order boundary
                nh = (c << 5) | (mf ? 32u - (u32)__clz(mf) : idx);
                done = true;
            } else if (c != tc) {  // this chunk is used up: follow the link
                bk_free_chunk(r, s, lane, c);
                if (nc < r.n_chunks) nh = nc << 5; else bad = true;  // broken chain: only after an earlier capacity error
            } else {  // live orders counted but none found: only after an earlier capacity error
                bad = true;
            }
            if (bad) s.err |= ERR_CAP_PAGES;
            if (lane == 0u) {
                stg32(r.lcnt + 4u * q, bad ? 0u : cnt);
                if (!bad) stg32(r.lht + 8u * q, nh);
            }
        }
        __syncwarp();
        if (done) break;
    }
    return true;
}

// (vol, count) of `side` at an arbitrary price: per-lane
__device__ __forceinline__ void bk_level_at(const BkReg& r, u32 side, u32 price, u32* vol, u32* cnt) {
    *vol = 0;
    *cnt = 0;
    const u32 q = price - r.win_lo;
    if (q >= r.W) return;
    if (!((lds(bk_bm(r, side, q >> 5)) >> (q & 31u)) & 1u)) return;
    *vol = lds(r.lvol + 4u * q);
    *cnt = ldg32(r.lcnt + 4u * q);
}
// observation words of the book: lane l owns words l and l + 32 (layout: book_obs in book.cuh)
__device__ __forceinline__ void bk_obs(const BkReg& r, u32 tick, u32 lane, u32 trade_vol, u32 bid, u32 ask, u32 vol_ask, u32 vol_bid, u32* w0,
                                       u32* w1) {
    u32 out[2];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const u32 w = lane + 32u * half;
        u32 val = 0;
        if (w >= 5u && w < 45u) {
            const u32 i = (w - 5u) >> 2, f = (w - 5u) & 3u;
            u32 v, n;
            if (f < 2u) bk_level_at(r, 1u, bid - i * tick, &v, &n);
            else bk_level_at(r, 0u, ask + i * tick, &v, &n);
            val = (f & 1u) ? n : v;
        } else if (w < 5u) {
            val = w == 0 ? trade_vol : w == 1 ? bid : w == 2 ? ask : w == 3 ? vol_ask : vol_bid;
        }
        out[half] = val;
    }
    *w0 = out[0];
    *w1 = out[1];
}

// =====================================================================================================================
// One event through the whole reference algorithm, warp-uniformly (x, y: the pre-decoded instruction; a, c: the prefetched
// order record of a cancel / modify).  `ev_done`: events complete once this one is; `rf`: events whose record writes were
// in HBM when the record was fetched.  Returns false when a bounded wait ran out.
// ENV (bb_step_device): a NEW carries the id submission gave it, and the order count is already the post-submission one.
template <bool ENV = false>
__device__ __forceinline__ bool bk_serial(const BkReg& r, BkSt& s, u32 lane, uint4 x, uint4 y, uint4 a, uint4 c, u32 ev_done, u32 rf, u32& lane_err) {
    s.t = ((u64)x.y << 32) | x.x;
    const u32 op = x.z & BB_OP_MASK;
    // the order that goes through matching (NEW, or the second half of a replace)
    u32 kind = 0u, side = 0u, price = 0u, vol = 0u, id = 0u;
    bool market = false;
    if (op == BB_OP_NEW) {  // (id, sentinel price and the market flag were settled by the fetch warp)
        s.d_instr += 1;
        if (x.z & DPF_CAP_ORDERS) {
            s.err |= ERR_CAP_ORDERS;
        } else {
            id = x.w;
            if (!ENV) s.n_orders = id + 1u;
            kind = RK_NEW;
            side = (x.z >> 8) & 1u;  // BB_F_BID
            price = y.x;
            market = (x.z & DPF_MARKET) != 0u;
            vol = y.y;
        }
    } else if (op == BB_OP_CANCEL || op == BB_OP_MODIFY) {
        s.d_instr += 1;
        id = x.w;
        if (id >= s.n_orders || id >= r.max_orders) {
            s.err |= ERR_BAD_ID;  // the reference panics (orderbook.rs:642, :749)
        } else {
            // The order's record as the fetch warp saw it: usable iff every write to it was in HBM by then, i.e. no event that
            // touched the order (its own, or a sweep that filled it) was still in the pipeline.
            const u32 dv = lds(r.dirty + 4u * (id & r.dirty_mask));
            if (dv > rf) {  // doubtful: let the pipeline drain up to that event, read again
                bk_publish(r, s, lane, ev_done - 1u);
                if (!bk_wait(r, lane, [&] { return ld_acq(r.ctl + CT_EV_RETIRED) >= dv; }, 13)) return false;
                a = ldg128_cg(r.oh + (u64)id * ORD_STRIDE);
                c = ldg128_cg(r.oh + (u64)id * ORD_STRIDE + 16u);
            }
            if ((c.z & META_STATUS_MASK) == ST_ACTIVE) {
                const u32 oside = (c.z & META_BID) ? 1u : 0u;
                const bool has_p = (x.z & BB_F_HAS_PRICE) != 0u, has_v = (x.z & BB_F_HAS_VOL) != 0u;
                const u32 q = a.x - r.win_lo;
                const bool reduce = op == BB_OP_MODIFY && !has_p && has_v && y.y < a.y;
                if (op == BB_OP_MODIFY && !has_p && !has_v) {
                } else if (q >= r.W) {  // never rested (flagged when it was placed)
                } else if (reduce) {  // reduce in place: priority kept (orderbook.rs:755-757)
                    const u32 la = r.lvol + 4u * q;
                    const u32 lv = lds(la);
                    __syncwarp();
                    if (lane == 0u) {
                        sts(la, lv - (a.y - y.y));
                        stg32(bk_chunk(r, a.z >> 5) + 8u * (a.z & 31u) + 4u, y.y);
                    }
                    bk_add_side(s, oside, y.y - a.y);
                    if (y.y == 0u) s.zv = 1u;
                    if (!bk_ret1(r, s, lane, make_uint4(RK_REDUCE, id, y.y, 0u), make_uint4(x.x, x.y, 0u, 0u))) return false;
                    if (lane == 0u) reds_max(r.dirty + 4u * (id & r.dirty_mask), ev_done);
                    s.d_applied += 1;
                } else {  // cancel_order (orderbook.rs:622-644), or the remove half of replace_order (:679-723)
                    const bool cancel = op == BB_OP_CANCEL;
                    const u32 la = r.lvol + 4u * q;
                    const u32 nv = lds(la) - a.y;
                    __syncwarp();
                    if (lane == 0u) sts(la, nv);
                    bk_add_side(s, oside, 0u - a.y);
                    bk_remove(r, s, lane, q, a.z);
                    if (cancel && !bk_ret1(r, s, lane, make_uint4(RK_CANCEL | (oside << 8), id, 0u, 0u), make_uint4(x.x, x.y, 0u, 0u))) return false;
                    if (nv == 0u && (!s.zv || ldg32(r.lcnt + 4u * q) == 0u)) bk_level_gone(r, s, lane, oside, q);
                    if (lane == 0u) reds_max(r.dirty + 4u * (id & r.dirty_mask), ev_done);
                    if (cancel) {
                        s.d_applied += 1;
                    } else {  // never a market order (N4)
                        kind = RK_REPLACE;
                        side = oside;
                        price = has_p ? y.x : a.x;
                        vol = has_v ? y.y : a.y;
                    }
                }
            }
        }
    } else if (op == BB_OP_SET_TRADING) {
        s.flags = y.y ? (s.flags | FL_TRADING) : (s.flags & ~FL_TRADING);
    } else if (op == BB_OP_RESTORE) {
        // bb_load_book: put an Active order read from its HBM record back on its side (orderbook.rs:898-905).  The host feeds
        // the orders by key time, so appending rebuilds every level's FIFO; equal keys on one level are the N1 collision.
        id = x.w;
        if (id < r.max_orders) {
            const uint4 ra = ldg128_cg(r.oh + (u64)id * ORD_STRIDE), rc = ldg128_cg(r.oh + (u64)id * ORD_STRIDE + 16u);
            if (id + 1u > s.n_orders) s.n_orders = id + 1u;
            if ((rc.z & META_STATUS_MASK) == ST_ACTIVE) {
                const u32 rside = (rc.z & META_BID) ? 1u : 0u, q = ra.x - r.win_lo, rvol = ra.y;
                const u64 kt = ((u64)rc.y << 32) | rc.x;
                if (q >= r.W) {
                    s.err |= ERR_CAP_PAGES;
                } else {
                    const u32 ba = bk_bm(r, rside, q >> 5), bit = 1u << (q & 31u);
                    const u32 la = r.lvol + 4u * q;
                    const u32 bw = lds(ba), lv = lds(la);
                    const u32 sa = bk_sm(r, rside, q >> 10);
                    const u32 sv = lds(sa);
                    const bool locked = !(bw & bit) && ((lds(bk_bm(r, rside ^ 1u, q >> 5)) & bit) != 0u);
                    __syncwarp();
                    if (locked) {
                        s.err |= ERR_LOCKED;
                    } else {
                        if (!(bw & bit)) {
                            if (lane == 0u) {
                                sts(la, rvol);
                                sts(ba, bw | bit);
                                if (bw == 0u) sts(sa, sv | (1u << ((q >> 5) & 31u)));
                            }
                            if (!bk_has_best(s, rside) || (rside ? q > s.bq_bid : q < s.bq_ask)) {
                                if (rside) s.bq_bid = q; else s.bq_ask = q;
                                s.flags |= FL_HAS_ASK << rside;
                            }
                        } else {
                            if (kt <= s.max_key_time) s.err |= ERR_TIME_ORDER;
                            if (lane == 0u) sts(la, lv + rvol);
                        }
                        __syncwarp();
                        bk_add_side(s, rside, rvol);
                        if (kt > s.max_key_time) s.max_key_time = kt;
                        if (rvol == 0u) s.zv = 1u;
                        const u32 pos = bk_append(r, s, lane, q, id, rvol);
                        if (lane == 0u) stg32(r.oh + (u64)id * ORD_STRIDE + OH_NEXT, pos);  // (the rest of the record is the snapshot's)
                    }
                }
            }
        } else {
            s.err |= ERR_CAP_ORDERS;
        }
    }
    if (kind) {
        // ---- match_bid / match_ask (orderbook.rs:429-487): level by level from the touch
        u32 rem = vol;
        const u32 opp = side ^ 1u;
        if (s.flags & FL_TRADING) {
            while (rem > 0u && bk_has_best(s, opp)) {
                const u32 bq = bk_best_q(s, opp);
                const u32 bprice = r.win_lo + bq;
                if (side ? (price < bprice) : (price > bprice)) break;
                const u32 la = r.lvol + 4u * bq;
                const u32 lv = lds(la);
                const u32 take = min(rem, lv), nv = lv - take;
                rem -= take;
                const bool exhaust = rem > 0u;  // the aggressor goes on: it takes every order left on this level
                __syncwarp();
                if (lane == 0u) sts(la, nv);
                s.trade_vol += take;
                bk_add_side(s, opp, 0u - take);
                if (!bk_sweep(r, s, lane, bq, opp, take, exhaust, id, x.x, x.y, bprice, ev_done, lane_err)) return false;
                if (nv == 0u && (exhaust || !s.zv || ldg32(r.lcnt + 4u * bq) == 0u)) bk_level_gone(r, s, lane, opp, bq);
            }
        }
        // ---- rest or finish (orderbook.rs:495-531, 699-722)
        const bool filled = vol != 0u && rem == 0u;
        u32 status = filled ? ST_FILLED : market ? ((s.flags & FL_TRADING) ? ST_CANCELLED : ST_REJECTED) : ST_ACTIVE;
        u32 pos = 0u;
        bool rests = false;
        if (status == ST_ACTIVE) {  // insert_order (side.rs:54-66)
            const u32 q = price - r.win_lo;
            if (q >= r.W) {
                s.err |= ERR_CAP_PAGES;
            } else {
                const u32 ba = bk_bm(r, side, q >> 5), bit = 1u << (q & 31u);
                const u32 la = r.lvol + 4u * q;
                const u32 bw = lds(ba);
                const u32 lv = lds(la);
                bool ok = true;
                if (!(bw & bit)) {
                    // the level array is shared by the two sides.  While trading is enabled an order only rests where the other
                    // side is empty, with one exception the reference allows: a ZERO-volume order never matches
                    // (orderbook.rs:436) and rests wherever its price says (SURVEY N5)
                    if (lds(bk_bm(r, opp, q >> 5)) & bit) {
                        s.err |= ERR_LOCKED;
                        ok = false;
                    } else {
                        const u32 sa = bk_sm(r, side, q >> 10);
                        const u32 sv = lds(sa);
                        __syncwarp();
                        if (lane == 0u) {
                            sts(la, rem);
                            sts(ba, bw | bit);
                            if (bw == 0u) sts(sa, sv | (1u << ((q >> 5) & 31u)));
                        }
                        const bool better = !bk_has_best(s, side) || (side ? q > s.bq_bid : q < s.bq_ask);
                        if (better) {
                            if (side) s.bq_bid = q; else s.bq_ask = q;
                            s.flags |= FL_HAS_ASK << side;
                        }
                    }
                } else {
                    if (s.t <= s.max_key_time) s.err |= ERR_TIME_ORDER;
                    __syncwarp();
                    if (lane == 0u) sts(la, lv + rem);
                }
                __syncwarp();
                if (ok) {
                    bk_add_side(s, side, rem);
                    if (s.t > s.max_key_time) s.max_key_time = s.t;
                    if (rem == 0u) s.zv = 1u;
                    pos = bk_append(r, s, lane, q, id, rem);
                    rests = true;
                }
            }
        }
        // the order's record: resting -> position and key time; ended -> final status and end time (an order that could not
        // rest — flagged above — keeps status Active in its record and is not on the book)
        if (!bk_ret1(r, s, lane, make_uint4(kind | (side << 8) | (status << 12), id, rem, rests ? pos : 0u), make_uint4(x.x, x.y, price, 0u)))
            return false;
        if (lane == 0u) reds_max(r.dirty + 4u * (id & r.dirty_mask), ev_done);
        s.d_applied += 1;
    }
    bk_publish(r, s, lane, ev_done);
    return true;
}

// =====================================================================================================================
// Micro-ops (32 bytes, in shared memory): w0 = level | kind << 13 | exhaust << 16, w1 = order id (T: the aggressor),
// w2 / w3 = arguments, w4 / w5 = event time, w6 = the event's order-record entry when this is its last micro-op
// (retire kind | side << 8 | status << 12; 0 = none), w7 = the event's filter mark (events complete once it is).
//   MK_T  w2 = volume to take, exhaust: and every order left on the level; w3 = the entry's third word
//   MK_A  w2 = volume
//   MK_R  w2 = entry position
//   MK_D  w2 = entry position, w3 = new volume
//   MK_N  nothing to do on the book (carries an entry only)
// The entry's words: RK_NEW {kind, id, volume left, position}, RK_REPLACE {kind, id, volume left, position} + price,
// RK_CANCEL {kind, id}, RK_REDUCE {kind, id, new volume}; `position` comes from the A micro-op, `volume left` is w2 of an
// A micro-op and w3 otherwise, a replace's price is the level's (A) or w3's high... see bk_own_entry.
#define MK_T 0u
#define MK_A 1u
#define MK_R 2u
#define MK_D 3u
#define MK_N 4u

// decoded event flags (SC_EVD word 0)
#define EF_REM 1u
#define EF_RED 2u
#define EF_PLACE 4u
#define EF_PSIDE 8u
#define EF_OSIDE 16u
#define EF_REPLACE 32u
#define EF_INSTR 64u
#define EF_NEW 128u
#define EF_MARKET 256u

// ---- replay: one round = up to 32 micro-ops from the ring (starting at `head`), one lane each -------------------------------
// (`rhead`: ring index of its first micro-op.)  Returns the number of micro-ops done (0 when a bounded wait ran out).  `s` is the REPLAY warp's state: chunk allocator, trade
// count, retire ring.  A round stops short of 32 where the volume its takes may fill would overflow the fill staging area.
__device__ __forceinline__ u32 bk_replay_round(const BkReg& r, BkSt& s, u32 lane, u32 rhead, u32 avail, u32& lane_err) {
    const u32 lt = (1u << lane) - 1u;
    {
        const u32 ma = r.scr + SC_MOP + 32u * ((rhead + lane) & (DW_MOPS - 1u));
        uint4 w = make_uint4(0, 0, 0, 0), v = w;
        if (lane < avail) {
            w = lds128(ma);
            v = lds128(ma + 16u);
        }
        // the round: the longest prefix whose takes fit the staging area (each take alone does)
        u32 cum = (lane < avail && ((w.x >> 13) & 7u) == MK_T) ? w.z : 0u;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const u32 a = __shfl_up_sync(BB_FULL, cum, k);
            if (lane >= (u32)k) cum += a;
        }
        const u32 n_round = __popc(__ballot_sync(BB_FULL, lane < avail && cum <= DW_FILLS));
        const bool valid = lane < n_round;
#ifdef DP_PROF
        s.pf_rounds += 1;
        s.pf_mops += n_round;
#endif
        const u32 q = w.x & 0x1FFFu, kind = (w.x >> 13) & 7u;
        // a fresh chunk for every append (it needs at most one); what is not used goes back below
        const bool is_a = valid && kind == MK_A;
        const u32 am = __ballot_sync(BB_FULL, is_a);
        if (am) {
            const u32 na = __popc(am), rank = __popc(am & lt);
            const u32 from_stack = min(na, s.n_free);
            u32 sp = 0u;
            if (is_a) {
                if (rank < from_stack) sp = lds(r.fs + 4u * (s.n_free - 1u - rank));
                else if (s.bump + (rank - from_stack) < r.n_chunks) sp = s.bump + (rank - from_stack);
                else lane_err |= ERR_CAP_PAGES;  // (chunk 0 is a safe sink)
                sts(r.scr + SC_SPARE + 4u * lane, sp);
            }
            s.n_free -= from_stack;
            s.bump = min(s.bump + (na - from_stack), r.n_chunks);
        }
        if (valid) {
            sts(r.scr + SC_NFILL + 4u * lane, 0u);
            sts64(r.scr + SC_FREED + 8u * lane, 0ull);
        }
        if (lane == 0u) sts(r.scr + SC_FCOUNT, 0u);
        __syncwarp();
        // ---- one lane per level: the level's micro-ops in order --------------------------------------------------------
        const u32 mg = __match_any_sync(BB_FULL, (valid && kind != MK_N) ? q : (0xFFFFFF00u | lane));
        if (valid && kind != MK_N && (mg & lt) == 0u) {
            u32 cnt = ldg32(r.lcnt + 4u * q);
            const u64 ht = ldg64(r.lht + 8u * q);
            u32 head = (u32)ht, tail = (u32)(ht >> 32);
            for (u32 mm = mg; mm; mm &= mm - 1u) {
                const u32 j = (u32)__ffs(mm) - 1u;
                const uint4 x = lds128(r.scr + SC_MOP + 32u * ((rhead + j) & (DW_MOPS - 1u)));
                const u32 kj = (x.x >> 13) & 7u;
                if (kj == MK_A) {  // insert_order's queue half (side.rs:54-66)
                    if (cnt == 0u || (tail & 31u) == DP_CHUNK_ENTRIES) {
                        const u32 sa = r.scr + SC_SPARE + 4u * j;
                        const u32 c = lds(sa);
                        sts(sa, c | 0x80000000u);
                        stg32(bk_chunk(r, c) + 8u * DP_CHUNK_ENTRIES, BB_NIL);
                        if (cnt == 0u) head = c << 5;
                        else stg32(bk_chunk(r, tail >> 5) + 8u * DP_CHUNK_ENTRIES, c);
                        tail = c << 5;
                    }
                    stg64(bk_chunk(r, tail >> 5) + 8u * (tail & 31u), ((u64)x.z << 32) | x.y);
                    sts(r.scr + SC_POS + 4u * j, tail);
                    tail += 1;
                    cnt += 1;
                } else if (kj == MK_R) {  // remove_order's queue half (side.rs:75-84): a tombstone
                    stg32(bk_chunk(r, x.z >> 5) + 8u * (x.z & 31u), BB_NIL);
                    if (cnt <= 1u) {
                        cnt = 0u;
                        if ((head >> 5) == (tail >> 5)) sts(r.scr + SC_FREED + 8u * j, head >> 5);  // a longer all-dead chain is left to the pool
                    } else {
                        cnt -= 1;
                    }
                } else if (kj == MK_D) {
                    stg32(bk_chunk(r, x.z >> 5) + 8u * (x.z & 31u) + 4u, x.w);
                } else {  // MK_T: match_orders over this level (orderbook.rs:843-870), entry by entry from the head
                    u32 take = x.z, nf = 0u, nfree = 0u;
                    const bool exhaust = (x.x >> 16) & 1u;
                    while ((take > 0u || exhaust) && cnt > 0u) {
                        const u32 c = head >> 5, idx = head & 31u, tc = tail >> 5;
                        const u32 end = (c == tc) ? (tail & 31u) : DP_CHUNK_ENTRIES;
                        if (idx >= end) {  // this chunk is used up: follow the link
                            const u32 nc = ldg32(bk_chunk(r, c) + 8u * DP_CHUNK_ENTRIES);
                            if (c == tc || nc >= r.n_chunks) {  // live orders counted but none found: only after an earlier capacity error
                                lane_err |= ERR_CAP_PAGES;
                                cnt = 0u;
                                break;
                            }
                            if (nfree < 2u) sts(r.scr + SC_FREED + 8u * j + 4u * nfree, c);
                            nfree += 1;
                            head = nc << 5;
                            continue;
                        }
                        const u64 e = ldg64(bk_chunk(r, c) + 8u * idx);
                        const u32 pid = (u32)e, pvol = (u32)(e >> 32);
                        if (pid == BB_NIL) {  // tombstone
                            head += 1;
                            continue;
                        }
                        const u32 tv = min(take, pvol), pv = pvol - tv;
                        take -= tv;
                        const u32 f = atoms_add(r.scr + SC_FCOUNT, 1u);
                        if (f < DW_FILLS) sts128(r.scr + SC_FILL + 16u * f, make_uint4(j | (nf << 8), pid, tv, pv));
                        else lane_err |= 0x80000000u;  // (cannot happen: a flush takes at most DW_FILLS volume)
                        nf += 1;
                        if (pv != 0u) {  // partially filled: stays at the head; the aggressor is done
                            stg32(bk_chunk(r, c) + 8u * idx + 4u, pv);
                            break;
                        }
                        head += 1;
                        cnt -= 1;
                    }
                    if (cnt == 0u && (head >> 5) == (tail >> 5) && nfree < 2u) sts(r.scr + SC_FREED + 8u * j + 4u * nfree, head >> 5);  // the level is gone
                    sts(r.scr + SC_NFILL + 4u * j, nf);
                }
            }
            stg32(r.lcnt + 4u * q, cnt);
            stg64(r.lht + 8u * q, ((u64)tail << 32) | head);
        }
        __syncwarp();
        // ---- places in the retire ring and in the trade log: event order, i.e. micro-op order ---------------------------------
        const u32 nf = valid ? lds(r.scr + SC_NFILL + 4u * lane) : 0u;
        const u32 own = valid ? v.z : 0u;
        u32 ci = nf + (own ? 1u : 0u), fi = nf;  // inclusive prefix sums: ring entries, fills
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const u32 a = __shfl_up_sync(BB_FULL, ci, k), b = __shfl_up_sync(BB_FULL, fi, k);
            if (lane >= (u32)k) { ci += a; fi += b; }
        }
        const u32 n_ring = __shfl_sync(BB_FULL, ci, 31), n_fill = __shfl_sync(BB_FULL, fi, 31);
        if (!bk_ret_space(r, s, lane, n_ring)) return 0u;
        const u32 ring0 = s.ret_tail + ci - (nf + (own ? 1u : 0u)), tr0 = s.n_tr + fi - nf;  // this micro-op's first ring slot / trade
        // the fills, 32 at a time: trade record + the passive order's record update
        for (u32 f0 = 0; f0 < n_fill; f0 += 32u) {
            const u32 f = f0 + lane;
            uint4 g = make_uint4(0, 0, 0, 0);
            if (f < n_fill) g = lds128(r.scr + SC_FILL + 16u * f);
            const u32 j = g.x & 31u, k = g.x >> 8;
            const u32 jr = __shfl_sync(BB_FULL, ring0, j), jt = __shfl_sync(BB_FULL, tr0, j);
            const u32 jq = __shfl_sync(BB_FULL, q, j), jid = __shfl_sync(BB_FULL, w.y, j);
            const u32 jlo = __shfl_sync(BB_FULL, v.x, j), jhi = __shfl_sync(BB_FULL, v.y, j), jmark = __shfl_sync(BB_FULL, v.w, j);
            const u32 jopp = __shfl_sync(BB_FULL, (w.x >> 17) & 1u, j);
            if (f < n_fill) {
                const u32 price = r.win_lo + jq;
                // trade: side / price are the passive order's (orderbook.rs:853-862)
                bk_ret_write(r, jr + k, make_uint4(RK_FILL | (jopp << 8) | (g.w == 0u ? 0x10000u : 0u), g.y, g.z, g.w), make_uint4(jlo, jhi, price, jid));
                bk_trade(r, s, jt + k, jlo, jhi, price, g.z, jid, g.y, jopp, lane_err);
                reds_max(r.dirty + 4u * (g.y & r.dirty_mask), jmark);
            }
        }
        // the events' own record entries
        if (own) {
            const u32 ek = own & 0xFFu;
            uint4 ea = make_uint4(own, w.y, 0u, 0u), eb = make_uint4(v.x, v.y, 0u, 0u);
            if (kind == MK_A) {  // the order rests: volume left, queue position; a replace also carries its new price
                ea.z = w.z;
                ea.w = lds(r.scr + SC_POS + 4u * lane);
                eb.z = r.win_lo + q;
            } else if (ek == RK_REDUCE) {
                ea.z = w.w;
            } else if (ek == RK_NEW) {  // ended without resting: volume left (a market order's unfilled rest)
                ea.z = w.w;
            } else if (ek == RK_REPLACE) {  // filled: its new price
                eb.z = w.w;
            }
            bk_ret_write(r, ring0 + nf, ea, eb);
            reds_max(r.dirty + 4u * (w.y & r.dirty_mask), v.w);
        }
        s.ret_tail += n_ring;
        s.n_tr += n_fill;
        // ---- chunks: unused spares and emptied chunks go back on the free stack, in lane order ---------------------------------
        {
            u32 c0 = 0u, c1 = 0u, c2 = 0u;
            if (valid) {
                if (is_a) {
                    const u32 sp = lds(r.scr + SC_SPARE + 4u * lane);
                    if (!(sp & 0x80000000u)) c0 = sp;
                }
                const u64 fr = lds64(r.scr + SC_FREED + 8u * lane);
                c1 = (u32)fr;
                c2 = (u32)(fr >> 32);
            }
            u32 n = (c0 ? 1u : 0u) + (c1 ? 1u : 0u) + (c2 ? 1u : 0u), incl = n;
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) {
                const u32 a = __shfl_up_sync(BB_FULL, incl, k);
                if (lane >= (u32)k) incl += a;
            }
            const u32 tot = __shfl_sync(BB_FULL, incl, 31);
            if (tot) {
                u32 at = s.n_free + incl - n;
                if (c0 && at < DP_FS_CAP) sts(r.fs + 4u * at++, c0);
                if (c1 && at < DP_FS_CAP) sts(r.fs + 4u * at++, c1);
                if (c2 && at < DP_FS_CAP) sts(r.fs + 4u * at++, c2);
                s.n_free = min(s.n_free + tot, DP_FS_CAP);
            }
        }
        __syncwarp();
        // what is complete now: the events whose last micro-op (the one that carries the record entry) was in this round
        const u32 om = __ballot_sync(BB_FULL, own != 0u);
        if (om) {
            const u32 ev_done = __shfl_sync(BB_FULL, v.w, 31u - (u32)__clz(om));
            bk_publish(r, s, lane, ev_done);
        }
        return n_round;
    }
}

// ---- the replay warp: rounds while micro-ops are published; parks when the chain warp asks for it ---------------------------------
__device__ __forceinline__ void bk_replay_warp(const BkReg& r, u32 lane, u32 n_tr0) {
    BkSt s;
    s.err = 0u;
    s.ret_room = 0u;  // (first use reads the retire warp's counter)
#ifdef DP_PROF
    s.pf_rounds = s.pf_mops = 0u;
#endif
    u32 head = 0u, lane_err = 0u, parked = 0u, ok_final = 1u;
    (void)n_tr0;
    for (;;) {
        u32 tail = 0u, drain = 0u, fin = 0u, ok = 1u;
        if (lane == 0u) {
            ok = dp_wait(r.ctl, [&] {
                fin = ld_acq(r.ctl + CT_FIN_L);   // read before the tail: set after the last publication
                drain = ld_acq(r.ctl + CT_DRAIN);  // (likewise)
                tail = ld_acq(r.ctl + CT_MOP_TAIL);
                return tail != head || fin != 0u || ((drain & 1u) && drain != parked);
            }, 7) ? 1u : 0u;
        }
        ok = __shfl_sync(BB_FULL, ok, 0);
        tail = __shfl_sync(BB_FULL, tail, 0);
        drain = __shfl_sync(BB_FULL, drain, 0);
        fin = __shfl_sync(BB_FULL, fin, 0);
        if (!ok) { ok_final = 0u; break; }
        if (tail != head) {
            s.bump = lds(r.ctl + RS_BUMP);
            s.n_free = lds(r.ctl + RS_NFREE);
            s.n_tr = lds(r.ctl + RS_NTR);
            s.ret_tail = s.ret_pub = lds(r.ctl + RS_RET_TAIL);
            if (s.ret_room < s.ret_tail) s.ret_room = s.ret_tail;
            while (tail != head) {
                const u32 n = bk_replay_round(r, s, lane, head, min(32u, tail - head), lane_err);
                if (n == 0u) { ok = 0u; break; }
                head += n;
                if (lane == 0u) st_rel(r.ctl + CT_MOP_DONE, head);
            }
            __syncwarp();
            if (lane == 0u) {
                if (s.ret_pub != s.ret_tail) st_rel(r.ctl + CT_RET_TAIL, s.ret_tail);
                sts(r.ctl + RS_BUMP, s.bump);
                sts(r.ctl + RS_NFREE, s.n_free);
                sts(r.ctl + RS_NTR, s.n_tr);
                sts(r.ctl + RS_RET_TAIL, s.ret_tail);
            }
            s.ret_pub = s.ret_tail;
            if (!ok) { ok_final = 0u; break; }
            continue;
        }
        if ((drain & 1u) && drain != parked) {  // everything published is done: the chain warp may borrow the queues
            parked = drain;
            if (lane == 0u) st_rel(r.ctl + CT_PARKED, parked);
            continue;
        }
        if (fin) break;
    }
    lane_err = __reduce_or_sync(BB_FULL, lane_err | s.err);
    if (lane == 0u) {
        sts(r.ctl + RS_ERR, lane_err);
        if (!ok_final) st_rel(r.ctl + CT_ABORT, 1u);
    }
#ifdef DP_PROF
    if (lane == 0u && blockIdx.x == 0) printf("k_deepw replay warp: rounds %u, micro-ops %u\n", s.pf_rounds, s.pf_mops);
#endif
}

// ---- chain warp: the replay warp finishes what is published and parks; its scalars come over (complex events, market-data
// records and the end of the launch work on the queues from the chain warp) -----------------------------------------------------------
__device__ __forceinline__ bool bk_borrow(const BkReg& r, BkSt& s, u32 lane) {
    s.drain_seq += 1;  // odd
    const u32 seq = s.drain_seq;
    __syncwarp();
    if (lane == 0u) st_rel(r.ctl + CT_DRAIN, seq);
    if (!bk_wait(r, lane, [&] { return ld_acq(r.ctl + CT_PARKED) == seq; }, 5)) return false;
    s.bump = lds(r.ctl + RS_BUMP);
    s.n_free = lds(r.ctl + RS_NFREE);
    s.n_tr = lds(r.ctl + RS_NTR);
    s.ret_tail = s.ret_pub = lds(r.ctl + RS_RET_TAIL);
    s.ret_room = s.ret_tail;  // (re-read the retire warp's counter on first use)
    s.done_seen = s.n_emit;
    return true;
}
__device__ __forceinline__ void bk_give_back(const BkReg& r, BkSt& s, u32 lane) {
    __syncwarp();
    if (lane == 0u) {
        if (s.ret_pub != s.ret_tail) st_rel(r.ctl + CT_RET_TAIL, s.ret_tail);
        sts(r.ctl + RS_BUMP, s.bump);
        sts(r.ctl + RS_NFREE, s.n_free);
        sts(r.ctl + RS_NTR, s.n_tr);
        sts(r.ctl + RS_RET_TAIL, s.ret_tail);
    }
    s.ret_pub = s.ret_tail;
    s.drain_seq += 1;  // even: run
    __syncwarp();
    if (lane == 0u) st_rel(r.ctl + CT_DRAIN, s.drain_seq);
}


// The placement half of an event on the chain (lane 0 alone): match_bid / match_ask (orderbook.rs:429-487) level by level —
// how much each crossed level gives — then rest or finish (orderbook.rs:495-531, 699-722).  SIDE is the order's side, a
// compile-time constant so that "the other side's touch" is a register, not a select.  Returns true when the output list is
// full in the middle of a sweep (the caller flushes and calls again: rem and the ladder carry the state).
template <u32 SIDE_T>
__device__ __forceinline__ bool bk_chain_place(const BkReg& r, BkSt& s, u32 co, u32& n_out, u32 ea, u32 f, u32 e, u32 mark, u32& rem, u32& last_t,
                                               u32& last_a) {
    // SIDE_T 0 / 1: the side as a compile-time constant; 2: one generic copy — the compact kernel (several books per SM) is bound by
    // instruction-cache refills and wins with the smaller hot loop, the roomy one with the shorter chain (profiles/r02_summary.md)
    const u32 SIDE = SIDE_T < 2u ? SIDE_T : ((f & EF_PSIDE) ? 1u : 0u);
    const u32 OPP = SIDE ^ 1u;
    const u32 HAS_OPP = FL_HAS_ASK << OPP, HAS_OWN = FL_HAS_ASK << SIDE;
    const u32 price = lds(ea + 32u);
    const u32 ebits = e << 18;
    while (rem > 0u && (s.flags & HAS_OPP)) {
        const u32 bq = SIDE ? s.bq_ask : s.bq_bid;
        const u32 bprice = r.win_lo + bq;
        if (SIDE ? (price < bprice) : (price > bprice)) break;
        if (n_out + 2u > DW_COUT) return true;  // (a sweep through more levels than the list holds)
        const u32 la = r.lvol + 4u * bq;
        const u32 lv = lds(la);
        const u32 take = min(rem, lv), nv = lv - take;
        rem -= take;
        sts(la, nv);
        last_t = n_out;
        sts(r.swept + 4u * (bq & r.swept_mask), mark);
        sts128(co + 16u * n_out++, make_uint4(bq | (MK_T << 13) | (rem > 0u ? 1u << 16 : 0u) | (OPP << 17) | ebits, take, 0u, 0u));
        if (nv == 0u) bk_level_gone<true>(r, s, 0u, OPP, bq);
    }
    const u32 ekind = (f & EF_REPLACE) ? RK_REPLACE : RK_NEW;
    if (rem == 0u || (f & EF_MARKET)) {
        const u32 status = rem == 0u ? ST_FILLED : ST_CANCELLED;  // (trading is enabled on this path)
        const u32 own = ekind | (SIDE << 8) | (status << 12);
        const u32 aux = ekind == RK_REPLACE ? price : rem;
        if (last_t != 0xFFFFFFFFu) {  // the entry rides on the event's last take
            sts64(co + 16u * last_t + 8u, ((u64)own << 32) | aux);
        } else {  // a market order that found no other side
            sts128(co + 16u * n_out++, make_uint4((MK_N << 13) | ebits, 0u, aux, own));
        }
    } else {  // insert_order (side.rs:54-66), the ladder half
        const u32 q = price - r.win_lo;
        const u32 ba = (SIDE ? r.bmb : r.bma) + 4u * (q >> 5), bit = 1u << (q & 31u);
        const u32 la = r.lvol + 4u * q;
        const u32 bw = lds(ba);
        if (!(bw & bit)) {
            if (lds((SIDE ? r.bma : r.bmb) + 4u * (q >> 5)) & bit) {  // (cannot happen while trading is enabled and volumes are > 0)
                s.err |= ERR_LOCKED;
            } else {
                sts(la, rem);
                sts(ba, bw | bit);
                if (bw == 0u) {
                    const u32 sa = (SIDE ? r.smb : r.sma) + 4u * (q >> 10);
                    sts(sa, lds(sa) | (1u << ((q >> 5) & 31u)));
                }
                if (!(s.flags & HAS_OWN) || (SIDE ? q > s.bq_bid : q < s.bq_ask)) {
                    if (SIDE) s.bq_bid = q; else s.bq_ask = q;
                    s.flags |= HAS_OWN;
                }
            }
        } else {
            sts(la, lds(la) + rem);
        }
        last_a = e;
        sts128(co + 16u * n_out++, make_uint4(q | (MK_A << 13) | (SIDE << 17) | ebits, rem, 0u, ekind | (SIDE << 8) | (ST_ACTIVE << 12)));
    }
    return false;
}

#define CXR_EMIT 0
#define CXR_STATE 1
#define CXR_BIG 2
#define CXR_DOUBT 3
#define CXR_SAMEID 4
#define CXR_TIME 5
#define CXR_ZERO 6
#define CXR_OTHER 7

// The events of one batch still to do (`pending`: a contiguous run of lanes; lane i holds event i: x, y pre-decoded
// instruction, a, c prefetched record).  `ev0`: events complete before this batch.  Comes back early (obs_lane < 32) after an
// event that asks for a market-data record.  Returns false when a bounded wait ran out.
// ENV (bb_step_device): every id the step's rows created is below s.n_orders from the start, so a cancel / modify is checked
// against that count alone and a NEW does not add to it.
template <bool COMPACT, bool ENV = false>
__device__ __forceinline__ bool bk_batch(const BkReg& r, BkSt& s, u32 lane, u32& pending, uint4 x, uint4 y, uint4 a, uint4 c, u32 ev0, u32 rf,
                                         u32 fast, u32& lane_err, u32& obs_lane) {
    constexpr bool compact = COMPACT;
    const u32 lt = (1u << lane) - 1u;
    const u32 op = x.z & BB_OP_MASK;
    const u32 t_lo = x.x, t_hi = x.y;
    const u64 t = ((u64)t_hi << 32) | t_lo;
    u32 rfl = rf;  // per lane: events whose record writes were in HBM when THIS lane's record (a, c) was read
    obs_lane = 32u;
    while (pending) {
        const u32 first = (u32)__ffs(pending) - 1u;
        const bool valid = (pending >> lane) & 1u;
        // events whose fills are all in the touched-order filter (sampled BEFORE the filter is read below)
        u32 qev = 0u;
        if (lane == 0u) qev = ld_acq(r.ctl + CT_Q_EV);
        qev = __shfl_sync(BB_FULL, qev, 0);
        // ---- decode: everything that does not depend on the book -------------------------------------------------------
        bool cx = false;
        u32 why = CXR_OTHER;
        u32 ef = 0u, q1 = 0u, v1 = 0u, pos1 = 0u, red_vol = 0u, pprice = 0u, pvol = 0u;
        const u32 id = x.w;
        const bool is_new = valid && op == BB_OP_NEW, is_cm = valid && (op == BB_OP_CANCEL || op == BB_OP_MODIFY);
        const u32 newm = __ballot_sync(BB_FULL, is_new);
        if (valid) {
            if (!fast || s.zv || !(s.flags & FL_TRADING)) { cx = true; why = CXR_STATE; }
            if (x.z & BB_F_EMIT) { cx = true; why = CXR_EMIT; }
            if (is_new) {
                if (x.z & DPF_CAP_ORDERS) cx = true;
                ef = EF_PLACE | EF_INSTR | EF_NEW | (((x.z >> 8) & 1u) ? EF_PSIDE : 0u) | ((x.z & DPF_MARKET) ? EF_MARKET : 0u);
                pprice = y.x;
                pvol = y.y;
            } else if (is_cm) {
                ef = EF_INSTR;
                if (id >= s.n_orders + (ENV ? 0u : __popc(newm & lt)) || id >= r.max_orders) {
                    cx = true;  // unknown id
                } else {
                    if (lds(r.dirty + 4u * (id & r.dirty_mask)) > rfl) { cx = true; why = CXR_DOUBT; }
                    const bool has_p = (x.z & BB_F_HAS_PRICE) != 0u, has_v = (x.z & BB_F_HAS_VOL) != 0u;
                    q1 = a.x - r.win_lo;
                    if ((c.z & META_STATUS_MASK) != ST_ACTIVE || (op == BB_OP_MODIFY && !has_p && !has_v) || q1 >= r.W) {
                        // nothing to do (cancel / modify of an order that is not on the book are no-ops)
                    } else {
                        const u32 oside = (c.z & META_BID) ? 1u : 0u;
                        ef |= oside ? EF_OSIDE : 0u;
                        v1 = a.y;
                        pos1 = a.z;
                        if (op == BB_OP_MODIFY && !has_p && has_v && y.y < a.y) {
                            ef |= EF_RED;
                            red_vol = y.y;
                        } else {
                            ef |= EF_REM;
                            if (op == BB_OP_MODIFY) {  // replace_order: never a market order (N4)
                                ef |= EF_PLACE | EF_REPLACE | (oside ? EF_PSIDE : 0u);
                                pprice = has_p ? y.x : a.x;
                                pvol = has_v ? y.y : a.y;
                            }
                        }
                    }
                }
            } else {
                cx = true;  // SET_TRADING, RESTORE, no-ops: the serial path knows
            }
            if ((ef & EF_RED) && red_vol == 0u) { cx = true; why = CXR_ZERO; }
            if (ef & EF_PLACE) {
                if (pvol == 0u) { cx = true; why = CXR_ZERO; }
                if (pvol > DW_FILLS) { cx = true; why = CXR_BIG; }
                // a limit price outside the window can only be handled where it never rests; leave it to the serial path
                if (!(ef & EF_MARKET) && pprice - r.win_lo >= r.W) cx = true;
            }
        }
        {   // time moves strictly forward through the batch and past every resting order's key
            const u32 pl = __shfl_up_sync(BB_FULL, t_lo, 1), ph = __shfl_up_sync(BB_FULL, t_hi, 1);
            const u64 tp = lane == first ? s.max_key_time : (((u64)ph << 32) | pl);
            if (valid && t <= tp) { cx = true; why = CXR_TIME; }
        }
        {   // two events of the batch naming one order: the later one cannot trust its prefetched record
            const u32 key = (is_new || is_cm) ? id : (0xFFFFFF00u | lane);
            const u32 mg = __match_any_sync(BB_FULL, key);
            if ((is_new || is_cm) && (mg & lt)) { cx = true; why = CXR_SAMEID; }
        }
        const u32 cm = __ballot_sync(BB_FULL, cx && valid);
        const u32 kcut = cm ? (u32)__ffs(cm) - 1u : 32u;
        const u32 clean = cm ? (pending & ((1u << kcut) - 1u)) : pending;
        if (clean) {
            // the decoded events go to shared memory: the chain reads them one after the other (broadcast loads)
            if ((clean >> lane) & 1u) {
                const u32 ea = r.scr + SC_EVD + 48u * lane;
                sts128(ea, make_uint4(ef, id, t_lo, t_hi));
                sts128(ea + 16u, make_uint4(q1, v1, pos1, red_vol));
                sts128(ea + 32u, make_uint4(pprice, pvol, 0u, 0u));
            }
            __syncwarp();
            const u32 e_end = 32u - (u32)__clz(clean);
            // ---- chain: the ladder, in event order, on LANE 0 ALONE (plain loads and stores, no warp synchronisation inside).  It
            // reads the decoded events and writes one 16-byte record per micro-op {level | kind << 13 | exhaust << 16 |
            // passive side << 17 | event << 18, volume, aux, record entry}; everything that is not part of the recurrence
            // (counters, side totals, the full micro-op with its ids and times) is worked out by all lanes afterwards.
            // It stops where its output list (or the volume one flush may take) is full — possibly in the middle of an
            // aggressive order's sweep — and goes on after the flush below.
            // A cancel / modify trusts the order record the fetch warp prefetched; the decode step above has checked it against
            // every fill the replay warp had made by then (`qev`), but not against takes that are still on their way through
            // the ring: an event that names an order on a level taken from since then stops the run (`late`), waits for the
            // replay warp to get there and is decoded again.
            u32 e = first, rem = 0u, last_t = 0xFFFFFFFFu;  // (rem, last_t, in_place: lane 0's)
            bool in_place = false, late = false;
            for (;;) {
                u32 n_out = 0u, last_a = 32u, stop = 0u;  // stop: the mark to wait for (late)
                if (lane == 0u) {
                    const u32 co = r.scr + SC_COUT;
                    last_t = 0xFFFFFFFFu;  // (the list is empty again; a sweep under way continues with its next take)
                    if (in_place) {  // the sweep the last run had to leave
                        const u32 ea = r.scr + SC_EVD + 48u * e;
                        const u32 f = lds(ea);
                        in_place = compact              ? bk_chain_place<2u>(r, s, co, n_out, ea, f, e, ev0 + e + 1u, rem, last_t, last_a)
                                   : (f & EF_PSIDE) ? bk_chain_place<1u>(r, s, co, n_out, ea, f, e, ev0 + e + 1u, rem, last_t, last_a)
                                                    : bk_chain_place<0u>(r, s, co, n_out, ea, f, e, ev0 + e + 1u, rem, last_t, last_a);
                        if (!in_place) ++e;
                    }
                    while (!in_place && e < e_end) {
                        const u32 ea = r.scr + SC_EVD + 48u * e;
                        const u32 f = lds(ea);
                        if (n_out + 4u > DW_COUT) break;
                        if (f & (EF_REM | EF_RED)) {
                            const uint4 d1 = lds128(ea + 16u);
                            const u32 sw = lds(r.swept + 4u * (d1.x & r.swept_mask));
                            if (sw > qev) {
                                stop = sw;
                                break;
                            }
                            const u32 oside = (f & EF_OSIDE) ? 1u : 0u;
                            const u32 la = r.lvol + 4u * d1.x;
                            const u32 lv = lds(la);
                            if (f & EF_RED) {  // reduce in place: priority kept (orderbook.rs:755-757)
                                sts(la, lv - (d1.y - d1.w));
                                sts128(co + 16u * n_out++, make_uint4(d1.x | (MK_D << 13) | (oside << 17) | (e << 18), d1.y - d1.w, 0u, RK_REDUCE));
                            } else {  // cancel_order (orderbook.rs:622-644), or the remove half of replace_order (:679-723)
                                const u32 nv = lv - d1.y;
                                sts(la, nv);
                                sts128(co + 16u * n_out++, make_uint4(d1.x | (MK_R << 13) | (oside << 17) | (e << 18), d1.y, 0u,
                                                                      (f & EF_PLACE) ? 0u : (RK_CANCEL | (oside << 8))));
                                if (nv == 0u) bk_level_gone<true>(r, s, 0u, oside, d1.x);
                            }
                        }
                        if (f & EF_PLACE) {
                            rem = lds(ea + 36u);
                            last_t = 0xFFFFFFFFu;
                            in_place = compact              ? bk_chain_place<2u>(r, s, co, n_out, ea, f, e, ev0 + e + 1u, rem, last_t, last_a)
                                       : (f & EF_PSIDE) ? bk_chain_place<1u>(r, s, co, n_out, ea, f, e, ev0 + e + 1u, rem, last_t, last_a)
                                                        : bk_chain_place<0u>(r, s, co, n_out, ea, f, e, ev0 + e + 1u, rem, last_t, last_a);
                            if (in_place) break;
                        }
                        ++e;
                    }
                }
                __syncwarp();
                // ---- back to 32 lanes: lane 0's view of the ladder, then everything that was left off the chain -----------------
                e = __shfl_sync(BB_FULL, e, 0);
                n_out = __shfl_sync(BB_FULL, n_out, 0);
                last_a = __shfl_sync(BB_FULL, last_a, 0);
                stop = __shfl_sync(BB_FULL, stop, 0);
                late = stop != 0u;
                s.bq_ask = __shfl_sync(BB_FULL, s.bq_ask, 0);
                s.bq_bid = __shfl_sync(BB_FULL, s.bq_bid, 0);
                s.flags = __shfl_sync(BB_FULL, s.flags, 0);
                s.err = __shfl_sync(BB_FULL, s.err, 0);
                // the micro-ops in full — ids, times, positions and marks come from the decoded events — go into the ring
                if (s.n_emit + n_out - s.done_seen > DW_MOPS) {
                    u32 done = 0u;
                    const u32 need = s.n_emit + n_out - DW_MOPS;
                    if (!bk_wait(r, lane, [&] {
                            done = ld_acq(r.ctl + CT_MOP_DONE);
                            return (int)(done - need) >= 0;
                        }, 4))
                        return false;
                    s.done_seen = __shfl_sync(BB_FULL, done, 0);
                }
                int d_ask = 0, d_bid = 0;
                u32 tv = 0u;
                for (u32 m0 = 0; m0 < n_out; m0 += 32u) {
                    const u32 m = m0 + lane;
                    if (m < n_out) {
                        const uint4 cr = lds128(r.scr + SC_COUT + 16u * m);
                        const u32 ce = (cr.x >> 18) & 31u, kind = (cr.x >> 13) & 7u, sd = (cr.x >> 17) & 1u;
                        const u32 ea = r.scr + SC_EVD + 48u * ce;
                        const uint4 d0 = lds128(ea);
                        u32 a2 = cr.y, a3 = cr.z;
                        int dv = 0;
                        if (kind == MK_T) {
                            dv = -(int)cr.y;
                            tv += cr.y;
                        } else if (kind == MK_A) {
                            dv = (int)cr.y;
                        } else if (kind == MK_R) {
                            dv = -(int)cr.y;
                            a2 = lds(ea + 24u);
                        } else if (kind == MK_D) {
                            dv = -(int)cr.y;
                            a2 = lds(ea + 24u);
                            a3 = lds(ea + 28u);
                        }
                        if (sd) d_bid += dv; else d_ask += dv;
                        const u32 ma = r.scr + SC_MOP + 32u * ((s.n_emit + m) & (DW_MOPS - 1u));
                        const u32 mark = ev0 + ce + 1u;
                        sts128(ma, make_uint4(cr.x & 0x3FFFFu, d0.y, a2, a3));
                        sts128(ma + 16u, make_uint4(d0.z, d0.w, cr.w, mark));
                        // the order this event names is in flight from now on: its prefetched record is not to be trusted
                        if (cr.w) reds_max(r.dirty + 4u * (d0.y & r.dirty_mask), mark);
                    }
                }
                s.n_emit += n_out;
                __syncwarp();
                if (lane == 0u && n_out) st_rel(r.ctl + CT_MOP_TAIL, s.n_emit);
#ifdef DP_PROF
                s.pf_flush += 1;
#endif
                s.vol_ask += (u32)__reduce_add_sync(BB_FULL, d_ask);
                s.vol_bid += (u32)__reduce_add_sync(BB_FULL, d_bid);
                s.trade_vol += __reduce_add_sync(BB_FULL, tv);
                if (last_a < 32u) s.max_key_time = ((u64)lds(r.scr + SC_EVD + 48u * last_a + 12u) << 32) | lds(r.scr + SC_EVD + 48u * last_a + 8u);
                if (late) {  // the replay warp has to get past the take that may have filled the order this event names
                    const u32 need = stop;
                    if (!bk_wait(r, lane, [&] { return ld_acq(r.ctl + CT_Q_EV) >= need; }, 14)) return false;
                }
                if (e >= e_end || late) break;
            }
            {   // the counters of the events done (a cancel / modify of an order that is not on the book counts as an instruction only)
                const bool mine = ((clean >> lane) & 1u) && lane < e;
                s.d_instr += __popc(__ballot_sync(BB_FULL, mine && (ef & EF_INSTR)));
                s.d_applied += __popc(__ballot_sync(BB_FULL, mine && (ef & (EF_PLACE | EF_REM | EF_RED))));
                if (!ENV) s.n_orders += __popc(__ballot_sync(BB_FULL, mine && (ef & EF_NEW)));
                if (e > first) s.t = ((u64)__shfl_sync(BB_FULL, t_hi, e - 1u) << 32) | __shfl_sync(BB_FULL, t_lo, e - 1u);
            }
            pending &= ~(clean & (e >= 32u ? BB_FULL : ((1u << e) - 1u)));
            if (late) continue;  // (decode the rest again: the fills made meanwhile are in the filter now)
        }
        if (cm) {
#ifdef DP_PROF
            s.pf_ser += 1;
            s.pf_reason[__shfl_sync(BB_FULL, why, kcut) & 7u] += 1;
#endif
            const u32 k = kcut;
            if (__shfl_sync(BB_FULL, why, k) == CXR_DOUBT) {
                // A doubtful record is no reason for the serial path: everything that is on its way drains (the micro-ops are all
                // published), the record is read again, and the event is decoded again — with a record it can trust now.
                const u32 need = __shfl_sync(BB_FULL, lds(r.dirty + 4u * (id & r.dirty_mask)), k);
                u32 seen = 0u;
                if (!bk_wait(r, lane, [&] {
                        seen = ld_acq(r.ctl + CT_EV_RETIRED);
                        return seen >= need;
                    }, 13))
                    return false;
                seen = __shfl_sync(BB_FULL, seen, 0);
                if (lane == k) {
                    a = ldg128_cg(r.oh + (u64)id * ORD_STRIDE);
                    c = ldg128_cg(r.oh + (u64)id * ORD_STRIDE + 16u);
                    rfl = seen;
                }
                continue;
            }
            uint4 kx, ky, ka, kc;
            kx.x = __shfl_sync(BB_FULL, x.x, k); kx.y = __shfl_sync(BB_FULL, x.y, k); kx.z = __shfl_sync(BB_FULL, x.z, k); kx.w = __shfl_sync(BB_FULL, x.w, k);
            ky.x = __shfl_sync(BB_FULL, y.x, k); ky.y = __shfl_sync(BB_FULL, y.y, k); ky.z = __shfl_sync(BB_FULL, y.z, k); ky.w = __shfl_sync(BB_FULL, y.w, k);
            ka.x = __shfl_sync(BB_FULL, a.x, k); ka.y = __shfl_sync(BB_FULL, a.y, k); ka.z = __shfl_sync(BB_FULL, a.z, k); ka.w = __shfl_sync(BB_FULL, a.w, k);
            kc.x = __shfl_sync(BB_FULL, c.x, k); kc.y = __shfl_sync(BB_FULL, c.y, k); kc.z = __shfl_sync(BB_FULL, c.z, k); kc.w = __shfl_sync(BB_FULL, c.w, k);
            // the replay warp parks; the whole reference algorithm for this event runs here, on the queues as they are
            if (!bk_borrow(r, s, lane)) return false;
            const bool sok = bk_serial<ENV>(r, s, lane, kx, ky, ka, kc, ev0 + k + 1u, rf, lane_err);
            pending &= ~(1u << k);
            if (sok && (kx.z & BB_F_EMIT)) {  // the caller writes the market-data record, gives the queues back and returns for the rest
                obs_lane = k;
                return true;
            }
            bk_give_back(r, s, lane);
            if (!sok) return false;
        }
        (void)why;
    }
    return true;
}

}  // namespace bb
