// Dense-window engine: the shallow-book specialisation of the device order book (included by book.cuh).
//
// Same reference semantics as the paged engine in book.cuh (side.rs:36-143, orderbook.rs:429-772), different
// data structure — the one BASELINE.json's north_star describes: the price ladder is a DENSE tick-indexed array
// in shared memory with one non-empty-level bitmap per side, and every resting order lives in a shared-memory
// slot, so matching, cancelling and modifying never read HBM.  The order table in HBM is written through (it is
// the reference's `orders: Vec<OrderEntry>` log and what agents gather statuses from) but never read back on the
// matching path.
//
// Book image in shared memory; every offset is a compile-time constant of the engine variant (DenseLayout):
//   0       BookHdr (128 B)
//   OFF_ID  slot_id[LP]   u32   order id resting in the slot, BB_NIL when free (searched lane-parallel by id)
//   OFF_SV  slot_vol[LP]  u32   remaining volume
//   OFF_SL  slot_link[LP] u32   next u8 | prev u8 | (level index | side << 15) u16; a head's prev and a tail's next
//                               are don't-care (queue ends are identified by the level record)
//   OFF_FS  free[LP]      u8    stack of free slot indices, Book::free_top entries
//   OFF_BM  bitmap[ask][NWMAX], bitmap[bid][NWMAX]      bit q set <=> level q of that side has a queue
//   OFF_LV  level[W][2]   8 B each (ask, bid interleaved): vol u32 | cnt u16 | head u8 | tail u8
// W = Geo::d_levels <= 32 * NWMAX price levels, L = Geo::d_live <= min(LP, 254) slots (0xFF is the null link).
// Two variants are compiled: ENG_DENSE (LP 128, W <= 256) and ENG_DENSE_L (LP 256, W <= 1024).
//
// Preconditions (violations set a sticky per-env error bit, they never change results silently):
//   * resting prices inside [d_win_lo, d_win_lo + W)                      else ERR_CAP_PAGES
//   * at most L resting orders per book                                     else ERR_CAP_LIVE
//   * per price level, resting orders arrive in strictly increasing time    else ERR_TIME_ORDER
//     (no equal-(price,time) key collisions, SURVEY.md N1: those need the paged engine's sorted queues)
// After an error the book of that env is no longer meaningful, but every access stays inside its own image.
#pragma once

namespace bb {

#define D_NIL 0xFFu

template <u32 LP_, u32 NWMAX_> struct DenseLayout {
    static constexpr u32 LP = LP_, NWMAX = NWMAX_;
    static constexpr u32 OFF_ID = 128u, OFF_SV = OFF_ID + 4u * LP, OFF_SL = OFF_SV + 4u * LP, OFF_FS = OFF_SL + 4u * LP;
    static constexpr u32 OFF_BM = OFF_FS + LP, OFF_LV = OFF_BM + 8u * NWMAX;
    static constexpr u32 image_bytes(u32 W) { return OFF_LV + 16u * W; }
};
typedef DenseLayout<128u, 8u> DenseSmall;
typedef DenseLayout<256u, 32u> DenseLarge;

// write-once streams (the trade log) are stored with the evict-first policy so they do not displace order records in L2
__device__ __forceinline__ void stg128_cs(u64 a, u32 x, u32 y, u32 z, u32 w) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void stg64v(u64 a, u32 x, u32 y) { asm volatile("st.global.v2.u32 [%0], {%1,%2};" ::"l"(a), "r"(x), "r"(y) : "memory"); }

template <class G> __device__ __forceinline__ u32 d_lv(const Book& b, u32 side, u32 q) { return b.sb + G::DL::OFF_LV + 16u * q + 8u * side; }
template <class G> __device__ __forceinline__ u32 d_bm(const Book& b, u32 side, u32 w) {
    return b.sb + G::DL::OFF_BM + 4u * (side ? G::DL::NWMAX : 0u) + 4u * w;
}

// The touch level q of `side` just lost its queue; `m` is its bitmap word with bit q already cleared.  q was the
// best level, so every other non-empty level is on the far side of it: scan words outwards from q's word (words
// beyond the configured window are always zero).
template <class G> __device__ __forceinline__ void d_next_best(Book& b, u32 side, u32 q, u32 m) {
    u32 w = q >> 5;
    if (side == 0u) {
        while (m == 0u) {
            if (++w >= G::DL::NWMAX) {
                b.flags &= ~FL_HAS_ASK;
                return;
            }
            m = lds(d_bm<G>(b, 0u, w));
        }
        b.bq_ask = (w << 5) + (u32)__ffs(m) - 1u;
    } else {
        while (m == 0u) {
            if (w == 0u) {
                b.flags &= ~FL_HAS_BID;
                return;
            }
            --w;
            m = lds(d_bm<G>(b, 1u, w));
        }
        b.bq_bid = (w << 5) + 31u - (u32)__clz(m);
    }
}

template <class G> __device__ __forceinline__ void d_log_trade(const G& g, Book& b, u64 t, u32 passive_bid, u32 price, u32 vol,
                                                               u32 active, u32 passive) {
    if (b.n_trades < g.max_trades) {
        stg128_cs(b.tr_ptr, (u32)t, (u32)(t >> 32), price, vol);
        stg128_cs(b.tr_ptr + 16u, active, passive, passive_bid, 0u);
        b.tr_ptr += 32u;
    } else if (g.max_trades) {
        b.err |= ERR_CAP_TRADES;
    }
    b.n_trades += 1;
}

template <class G> __device__ __forceinline__ void d_free_slot(Book& b, u32 slot) {
    sts(b.sb + 4u * slot + G::DL::OFF_ID, BB_NIL);
    sts8(b.sb + G::DL::OFF_FS + b.free_top, slot);
    b.free_top += 1;
}

// match_bid / match_ask (orderbook.rs:429-487) + match_orders (:843-870) against shared-memory slots.
// Returns the aggressor's remaining volume; the caller derives Status::Filled as (vol > 0 && remaining == 0):
// the loop body only runs while volume is left, so that is exactly "some fill brought the volume to zero".
// STEPPED (k_sim): the per-launch transition / volume counters are settled once per env-step by the caller (from the
// trade count and the step's trade_vol) instead of once per fill.
// JRN: each fill leaves one trade-journal entry instead of its trade record, passive-record stores and counter updates
// (see d_flush); the loop stops early, with volume left, when the journal is full.
template <bool STEPPED, bool JRN, class G> __device__ __forceinline__ u32 d_match(const G& g, Book& b, u32 side, u32 price, u32 vol, u32 id, u64 t) {
    const u32 o = side ^ 1u;
    while (vol > 0u && has_best(b, o)) {
        const u32 bq = best_q(b, o);
        const u32 bprice = g.d_win_lo + bq;
        if (side ? (price < bprice) : (price > bprice)) break;
        if (JRN && b.jp == b.jend) break;
        const u32 la = d_lv<G>(b, o, bq);
        const u64 lv = lds64(la);
        const u32 lvol = (u32)lv, hi = (u32)(lv >> 32);
        const u32 head = (hi >> 16) & 0xFFu;
        const u32 sa = b.sb + 4u * head;
        const u32 pid = lds(sa + G::DL::OFF_ID), pvol = lds(sa + G::DL::OFF_SV);
        const u32 tv = min(vol, pvol);
        vol -= tv;
        if (JRN) {
            sts128(b.jp, make_uint4(b.ev | (bq << 20), pid, tv, pvol - tv));
            b.jp += 16u;
        } else {
            d_log_trade(g, b, t, o, bprice, tv, id, pid);
            b.trade_vol += tv;
        }
        if (!STEPPED) {
            b.d_volume += tv;
            b.d_trans += 1;
        }
        add_side_vol(b, o, 0u - tv);
        const u64 pa = b.oh + (u64)pid * ORD_STRIDE;
        if (pvol == tv) {  // passive order Filled: leaves its slot and the head of its level
            if (!JRN) {
                stg32(pa + OH_VOL, 0u);
                stg32(pa + OH_META, ST_FILLED | (o ? META_BID : 0u));
                stg64(pa + OC_END, t);
            }
            const u32 nxt = lds8(sa + G::DL::OFF_SL);
            d_free_slot<G>(b, head);
            if ((hi & 0xFFFFu) == 1u) {  // last order of the level (its `next` byte is stale by design)
                const u32 ba = d_bm<G>(b, o, bq >> 5);
                const u32 m = lds(ba) & ~(1u << (bq & 31u));
                sts(ba, m);
                d_next_best<G>(b, o, bq, m);
            } else {
                sts64(la, ((u64)((hi & 0xFF00FFFFu) - 1u + (nxt << 16)) << 32) | (u64)(lvol - tv));
            }
        } else {
            sts(sa + G::DL::OFF_SV, pvol - tv);
            if (!JRN) stg32(pa + OH_VOL, pvol - tv);
            sts(la, lvol - tv);  // side.remove_vol(price, tv)
        }
    }
    return vol;
}

// insert_order (side.rs:54-66) for an order that rests: append to its level's queue.  Capacity violations are
// recorded and leave the image consistent: a price outside the window is clamped to level 0, an order that finds no
// free slot is dropped.
// CHECK_TIME: the caller cannot guarantee that time moves strictly forward between resting inserts (replay mode).
// CHECK_SLOTS: false when the caller has already made sure that a free slot exists (k_sim validates a whole env-step's
// new orders against the free-slot count up front, so the event loop carries no per-insert test).
// JRN: max_key_time is settled by d_flush.
template <bool CHECK_TIME, bool CHECK_SLOTS, bool JRN, class G>
__device__ __forceinline__ u32 d_insert(const G& g, Book& b, u32 side, u32 price, u64 t, u32 id, u32 vol) {
    u32 q = price - g.d_win_lo;
    if (q >= g.d_levels) {
        b.err |= ERR_CAP_PAGES;
        q = 0u;
    }
    if (CHECK_SLOTS && b.free_top == 0u) {  // no free slot: the order is NOT put on the book (flagged; the image stays
        b.err |= ERR_CAP_LIVE;              // consistent — a reused live slot would hand d_match a stale order id and send
        return 0u;                          // its record write out of bounds)
    }
    b.free_top -= 1;
    const u32 slot = lds8(b.sb + G::DL::OFF_FS + b.free_top);
    const u32 la = d_lv<G>(b, side, q);
    const u32 ba = d_bm<G>(b, side, q >> 5);
    const u32 bit = 1u << (q & 31u);
    const u32 bw = lds(ba);
    const u32 sa = b.sb + 4u * slot;
    u32 prev = D_NIL;
    if (bw & bit) {
        const u64 lv = lds64(la);
        const u32 hi = (u32)(lv >> 32);
        prev = hi >> 24;
        if (CHECK_TIME && t <= b.max_key_time) {  // rare: valid only while still strictly after this level's current tail
            const u32 tid = lds(b.sb + 4u * prev + G::DL::OFF_ID);
            if (t <= ldg64(b.oh + (u64)tid * ORD_STRIDE + OH_KEYT)) b.err |= ERR_TIME_ORDER;
        }
        sts64(la, ((u64)(((hi & 0x00FFFFFFu) + 1u) | (slot << 24)) << 32) | (u64)((u32)lv + vol));
        sts8(b.sb + 4u * prev + G::DL::OFF_SL, slot);  // old tail's next
    } else {
        sts64(la, ((u64)(1u | (slot << 16) | (slot << 24)) << 32) | (u64)vol);
        sts(ba, bw | bit);
        const bool better = !has_best(b, side) || (side ? q > b.bq_bid : q < b.bq_ask);
        if (better) set_best(b, side, q);
    }
    sts(sa + G::DL::OFF_ID, id);
    sts(sa + G::DL::OFF_SV, vol);
    sts(sa + G::DL::OFF_SL, D_NIL | (prev << 8) | ((q | (side << 15)) << 16));
    add_side_vol(b, side, vol);
    if (CHECK_TIME) {
        if (t > b.max_key_time) b.max_key_time = t;
    } else if (!JRN) {
        b.max_key_time = t;  // time is strictly increasing by construction
    }
    return slot;
}

// slot holding order `id`, or D_NIL when the order is not resting: every lane compares four slot ids
template <class G> __device__ __forceinline__ u32 d_find(const Book& b, u32 id) {
#pragma unroll
    for (u32 base = 0; base < G::DL::LP; base += 128u) {
        const uint4 v = lds128(b.sb + G::DL::OFF_ID + 4u * base + 16u * b.lane);
        const u32 hit = v.x == id ? 0u : v.y == id ? 1u : v.z == id ? 2u : v.w == id ? 3u : 4u;
        const u32 m = __ballot_sync(BB_FULL, hit != 4u);
        if (m) {
            const u32 src = (u32)__ffs(m) - 1u;
            return base + 4u * src + __shfl_sync(BB_FULL, hit, src);
        }
    }
    return D_NIL;
}

// remove_order (side.rs:75-84): unlink the slot from its level and free it
template <class G> __device__ __forceinline__ void d_remove(Book& b, u32 slot, u32 side, u32 q, u32 next, u32 prev, u32 svol) {
    const u32 la = d_lv<G>(b, side, q);
    const u64 lv = lds64(la);
    const u32 hi = (u32)(lv >> 32);
    if ((hi & 0xFFFFu) == 1u) {
        const u32 ba = d_bm<G>(b, side, q >> 5);
        const u32 m = lds(ba) & ~(1u << (q & 31u));
        sts(ba, m);
        if (best_q(b, side) == q) d_next_best<G>(b, side, q, m);
    } else {
        // head / tail are recognised by the level record, never by null links: the `prev` of a head and the `next`
        // of a tail may be stale, which saves the link fix-ups when a queue advances
        const u32 head = (hi >> 16) & 0xFFu, tail = hi >> 24;
        const bool is_head = head == slot, is_tail = tail == slot;
        const u32 nh = is_head ? next : head, nt = is_tail ? prev : tail;
        if (!is_head) sts8(b.sb + 4u * prev + G::DL::OFF_SL, next);
        if (!is_tail) sts8(b.sb + 4u * next + G::DL::OFF_SL + 1u, prev);
        sts64(la, ((u64)(((hi & 0xFFFFu) - 1u) | (nh << 16) | (nt << 24)) << 32) | (u64)((u32)lv - svol));
    }
    d_free_slot<G>(b, slot);
    add_side_vol(b, side, 0u - svol);
}

// process_event (orderbook.rs:782-792) on the dense book; same contract as book_apply in book.cuh.
// HINT (k_sim's in-kernel agents): 0 = none; 1 = every event carries a hint; 2 = hint present iff non-zero.
//   NEW    hint = 1 + index of the issuing agent in the launch's agent-slot table (Book::ags): the slot the order
//          rests in is recorded there, so the agent's next "is my order still live" test is one shared-memory compare
//   CANCEL hint = 1 + the slot the order was resting in when the agent looked: a mismatch of the slot's id means
//          the order has left the book since (filled earlier in this step) and the cancel is a no-op
// With HINT != 0 ids are trusted (generated in-kernel, capacity validated once per step by the caller).
// JRN (k_sim with RandomAgents only; HINT == 1, NEW and CANCEL only): no order record, trade record or trade counter is
// written here.  The event leaves its outcome in its own queue entry at shared address Book::ev (NEW: the remaining
// volume in the id word; CANCEL: 2 | side in the last word when it took effect, which the agents leave 0) and one
// trade-journal entry per fill; d_flush turns them into the HBM writes.  `t` is unused.  Returns 0, or, when a fill
// found the journal full, the NEW order's remaining volume: the event is then suspended before it rests, and the
// caller flushes and runs it again with that volume.
template <bool IS_NEW, bool CHECK_TIME, int HINT, bool JRN = false, class G>
__device__ __forceinline__ u32 d_apply(const G& g, Book& b, u32 kind, u32 id, u32 side, u32 price, u32 vol, u32 trader, bool has_p,
                                       bool has_v, u64 t, u32 hint) {
    static_assert(!JRN || HINT == 1, "the journal derives order ids from the agents' hints");
    const u64 ra = b.oh + (u64)id * ORD_STRIDE;
    if (IS_NEW) {
        if (HINT == 0 && id >= g.max_orders) {
            b.err |= ERR_CAP_ORDERS;
            return 0u;
        }
        const bool trading = (b.flags & FL_TRADING) != 0u;
        u32 rem = vol;
        if (trading) rem = d_match<HINT != 0, JRN>(g, b, side, price, vol, id, t);
        if (JRN && rem != 0u && b.jp == b.jend) return rem;
        const bool filled = vol != 0u && rem == 0u;
        const bool market = side ? (price == 0xFFFFFFFFu) : (price == 0u);  // N3
        const bool ended = filled || market;
        // Filled, or an unfilled market order: Cancelled when trading, Rejected otherwise (orderbook.rs:517-531)
        const u32 status = filled ? ST_FILLED : market ? (trading ? ST_CANCELLED : ST_REJECTED) : ST_ACTIVE;
        if (!ended) {
            const u32 slot = d_insert<CHECK_TIME, HINT == 0, JRN>(g, b, side, price, t, id, rem);
            if (HINT == 1 || (HINT == 2 && hint)) sts8(b.ags + hint, slot);
        }
        if (JRN) {
            sts(b.ev + 4u, rem);
            return 0u;
        }
        // order record; the queue links of the HBM record are not used by this engine
        const u64 kt = ended ? 0ULL : t, end_time = ended ? t : ~0ULL;
        // 52 of the record's 64 bytes are written (the link and padding words are not): L2 therefore reads the two
        // partially written sectors back from DRAM when it evicts them (10 GB per C3 pass).  Writing both sectors
        // in full removes those reads but was measured 4.6 % SLOWER end to end, twice: with zero-filled words
        // (profiles/r01_s5_summary.md) and with the don't-care words taken from live registers (38.74 vs 37.03 ms,
        // profiles/r02_summary.md) — the cost is in the store path, not in register pressure — and DRAM is at 11 % of
        // its bandwidth either way.
        stg64v(ra + OH_PRICE, price, rem);
        stg128(ra + OH_KEYT, (u32)kt, (u32)(kt >> 32), status | (side ? META_BID : 0u), vol);
        stg128(ra + OC_ARR, (u32)t, (u32)(t >> 32), (u32)end_time, (u32)(end_time >> 32));
        stg32(ra + OC_TRADER, trader);
        if (HINT == 0) b.d_trans += 1;
        return 0u;
    }
    if (HINT == 0 && (id >= b.n_orders || id >= g.max_orders)) {
        b.err |= ERR_BAD_ID;  // the reference panics (orderbook.rs:642, :749)
        return 0u;
    }
    u32 slot;
    if (HINT == 1 || (HINT == 2 && hint)) {
        slot = hint - 1u;
        if (lds(b.sb + 4u * slot + G::DL::OFF_ID) != id) return 0u;
    } else {
        slot = d_find<G>(b, id);
        if (slot == D_NIL) return 0u;  // not Active: cancel / modify are no-ops
    }
    const u32 sa = b.sb + 4u * slot;
    const u32 link = lds(sa + G::DL::OFF_SL), svol = lds(sa + G::DL::OFF_SV);
    const u32 next = link & 0xFFu, prev = (link >> 8) & 0xFFu, q = (link >> 16) & 0x7FFFu;
    side = link >> 31;
    if (kind == EV_MODIFY) {
        if (!has_p && !has_v) return 0u;
        if (!has_p && vol < svol) {  // reduce in place: priority kept (orderbook.rs:755-757)
            const u32 la = d_lv<G>(b, side, q);
            sts(sa + G::DL::OFF_SV, vol);
            sts(la, lds(la) - (svol - vol));
            add_side_vol(b, side, vol - svol);
            stg32(ra + OH_VOL, vol);
            b.d_trans += 1;
            return 0u;
        }
        if (!has_p) price = g.d_win_lo + q;
        if (!has_v) vol = svol;
    }
    d_remove<G>(b, slot, side, q, next, prev, svol);
    const u32 side_bit = side ? META_BID : 0u;
    if (JRN || kind == EV_CANCEL) {
        if (JRN) {
            sts(b.ev + 12u, 2u | side);
        } else {
            stg32(ra + OH_META, ST_CANCELLED | side_bit);
            stg64(ra + OC_END, t);
        }
        b.d_trans += 1;
        return 0u;
    }
    // replace_order (orderbook.rs:679-723): re-match, re-rest under key time t; never a market order (N4)
    u32 rem = vol;
    if (b.flags & FL_TRADING) rem = d_match<HINT != 0, false>(g, b, side, price, vol, id, t);
    const bool filled = vol != 0u && rem == 0u;
    if (!filled) d_insert<CHECK_TIME, HINT == 0, false>(g, b, side, price, t, id, rem);
    stg64v(ra + OH_PRICE, price, rem);
    stg32(ra + OH_META, (filled ? ST_FILLED : ST_ACTIVE) | side_bit);
    stg64(ra + (filled ? OC_END : OH_KEYT), t);
    b.d_trans += 1;
    return 0u;
}

// Write-out of a journaled (JRN) stretch of an env-step, all lanes: the events at queue positions [e_lo, e_hi) — complete,
// outcomes in place — and the `nj` trade-journal entries at `jb` (16 B each: queue-entry address | level << 20, passive
// id, traded volume, passive volume left).  The stores, and the bytes they leave in the order table and the trade log,
// are those of the write-through path: the write-out only moves them off lane 0's chain, where each record cost several
// dependent instructions, to one store per lane.  Every record is written by at most one lane per instruction, and in
// event order across instructions (a passive order's volume word keeps the value of its last fill); the __syncwarp
// calls order the stores of different lanes to one record.  Settles the counters the event loop no longer keeps:
// n_trades, trade_vol and max_key_time.  `agh`: the agents' held ids (a NEW event's id, by its hint).
template <class G>
__device__ __forceinline__ void d_flush(const G& g, Book& b, u32 qs, u32 agh, u64 start, u32 e_lo, u32 e_hi, u32 jb, u32 nj) {
    const bool trading = (b.flags & FL_TRADING) != 0u;
    u32 last_rest = 0;  // 1 + queue position of the last order that rested
    for (u32 i = e_lo + b.lane; i < e_hi; i += 32u) {
        const uint4 ev = lds128(qs + 16u * i);
        const u64 t = start + i;
        const u32 side_bit = (ev.x & 2u) ? META_BID : 0u;
        if (ev.x & 1u) {
            const u32 id = lds(agh + 4u * ((ev.x >> 2) & 0x7FFu) - 4u);
            const u32 price = ev.z, vol = ev.w, rem = ev.y;
            const bool filled = vol != 0u && rem == 0u;
            const bool market = side_bit ? (price == 0xFFFFFFFFu) : (price == 0u);
            const bool ended = filled || market;
            const u32 status = filled ? ST_FILLED : market ? (trading ? ST_CANCELLED : ST_REJECTED) : ST_ACTIVE;
            if (!ended) last_rest = i + 1u;
            // 52 of the record's 64 bytes, as on the write-through path (see d_apply)
            const u64 ra = b.oh + (u64)id * ORD_STRIDE;
            const u64 kt = ended ? 0ULL : t, end_time = ended ? t : ~0ULL;
            stg64v(ra + OH_PRICE, price, rem);
            stg128(ra + OH_KEYT, (u32)kt, (u32)(kt >> 32), status | side_bit, vol);
            stg128(ra + OC_ARR, (u32)t, (u32)(t >> 32), (u32)end_time, (u32)(end_time >> 32));
            stg32(ra + OC_TRADER, ev.x >> 13);
        } else if (ev.w) {
            const u64 ra = b.oh + (u64)ev.y * ORD_STRIDE;
            stg32(ra + OH_META, ST_CANCELLED | ((ev.w & 1u) ? META_BID : 0u));
            stg64(ra + OC_END, t);
        }
    }
    last_rest = __reduce_max_sync(BB_FULL, last_rest);
    if (last_rest) b.max_key_time = start + (last_rest - 1u);
    __syncwarp();
    u32 err = 0, tv_sum = 0;
    const u64 tr_env = g.tr_base + (u64)b.env * g.max_trades * 32u;
    for (u32 k0 = 0; k0 < nj; k0 += 32u) {
        const u32 k = k0 + b.lane;
        const bool valid = k < nj;
        const uint4 je = valid ? lds128(jb + 16u * k) : make_uint4(0u, BB_NIL, 0u, 0u);
        const u32 same = __match_any_sync(BB_FULL, je.y);  // lanes of this chunk that fill the same passive order
        if (valid) {
            const u32 ea = je.x & 0xFFFFFu, pid = je.y, tv = je.z, left = je.w;
            const u32 ax = lds(ea);  // the aggressor's queue entry
            const u32 active = lds(agh + 4u * ((ax >> 2) & 0x7FFu) - 4u);
            const u32 o = ((ax >> 1) & 1u) ^ 1u;
            const u64 t = start + ((ea - qs) >> 4);
            const u32 idx = b.n_trades + k;
            if (idx < g.max_trades) {
                const u64 ta = tr_env + (u64)idx * 32u;
                stg128_cs(ta, (u32)t, (u32)(t >> 32), g.d_win_lo + (je.x >> 20), tv);
                stg128_cs(ta + 16u, active, pid, o, 0u);
            } else if (g.max_trades) {
                err |= ERR_CAP_TRADES;
            }
            if ((same >> b.lane) == 1u) {  // the chunk's last fill of this passive order
                const u64 pa = b.oh + (u64)pid * ORD_STRIDE;
                stg32(pa + OH_VOL, left);
                if (left == 0u) {
                    stg32(pa + OH_META, ST_FILLED | (o ? META_BID : 0u));
                    stg64(pa + OC_END, t);
                }
            }
            tv_sum += tv;
        }
        __syncwarp();
    }
    b.trade_vol += __reduce_add_sync(BB_FULL, tv_sum);
    b.n_trades += nj;
    b.err |= __reduce_or_sync(BB_FULL, err);
}

// bb_load_book: put an Active order read from its HBM record back on its side (orderbook.rs:898-905)
template <class G> __device__ __forceinline__ void d_restore(const G& g, Book& b, u32 order_id) {
    const u64 ra = b.oh + (u64)order_id * ORD_STRIDE;
    const uint4 a = ldg128(ra), c = ldg128(ra + 16u);
    if (order_id + 1u > b.n_orders) b.n_orders = order_id + 1u;
    if ((c.z & META_STATUS_MASK) == ST_ACTIVE)
        d_insert<true, true, false>(g, b, (c.z & META_BID) ? 1u : 0u, a.x, ((u64)c.y << 32) | c.x, order_id, a.y);
}

// (vol, count) at an arbitrary price; per-lane (prices may differ between lanes)
template <class G> __device__ __forceinline__ void d_level_at(const G& g, const Book& b, u32 side, u32 price, u32* vol, u32* cnt) {
    *vol = 0;
    *cnt = 0;
    const u32 q = price - g.d_win_lo;
    if (q >= g.d_levels) return;
    if (!((lds(d_bm<G>(b, side, q >> 5)) >> (q & 31u)) & 1u)) return;
    const u64 lv = lds64(d_lv<G>(b, side, q));
    *vol = (u32)lv;
    *cnt = (u32)(lv >> 32) & 0xFFFFu;
}

}  // namespace bb
