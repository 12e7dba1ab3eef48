// Device-side limit order book: one warp owns one book.
//
// Replaces, for the batched path, the reference's per-book data structures and matching engine:
//   crates/order_book/src/side.rs:36-143      OrderBookSide{vol, volumes: BTreeMap, orders: BTreeMap}
//   crates/order_book/src/orderbook.rs:429-772 match_bid/ask, place_*, cancel, reduce, replace, modify
//   crates/order_book/src/orderbook.rs:229-324 bid_ask, *_levels, level_1_data, level_2_data
//
// B200-first layout instead of two B-trees per side:
//   * price ladder = dense 32-level "pages" (vol[32], cnt[32], head[32], tail[32] = 512 B) tagged
//     (price / granule) >> 5 | side.  A page exists only while it holds a level, so any u32 price
//     is representable; the first `p_smem` pages of a book live in shared memory, the rest in HBM.
//   * one lane per page tag: find-page is one __ballot_sync, best bid/ask is one
//     __reduce_min/max_sync over (page key * 32 + __ffs/__clz of the page's 32-bit non-empty bitmap).
//   * two bitmaps per page mirror the reference's two maps: `vmap` <=> key present in `volumes`
//     (count > 0), `qmap` <=> some key of that price present in `orders` (queue non-empty).  They
//     differ only under the reference's equal-(price,time) key collisions (SURVEY.md N1).
//   * price-time queue per level = intrusive doubly linked list through the 32-byte hot order
//     records in HBM, kept sorted by key time; the common case (time moved forward) appends without
//     reading the tail record.
//   * the book header (time, counters, side totals, cached touch) lives in REGISTERS for the whole
//     launch; shared memory and global memory are addressed with explicit ld/st.shared / ld/st.global
//     so no generic-address or stack traffic is generated (profiles/r01_v1_summary.md).
// All book code is warp-uniform: every lane executes it with identical values (loads broadcast, stores
// coalesce to one transaction); lanes diverge only in the explicitly lane-parallel helpers.
#pragma once
#include <cstdint>

namespace bb {

typedef uint32_t u32;
typedef uint64_t u64;

#define BB_NIL 0xFFFFFFFFu
#define BB_TAG_FREE 0xFFFFFFFFu
#define BB_FULL 0xFFFFFFFFu

enum { ST_NEW = 0, ST_ACTIVE = 1, ST_FILLED = 2, ST_CANCELLED = 3, ST_REJECTED = 4 };  // types.rs:51-75
#define META_STATUS_MASK 7u
#define META_BID 8u     // side bit (types.rs:26-47: true <-> Bid)
#define META_GHOST 16u  // Active but no longer owning a queue key (N1)

// device error bits == BB_ERR_* of include/bourse_b200.h
#define ERR_CAP_ORDERS 0x01u
#define ERR_CAP_TRADES 0x02u
#define ERR_CAP_PAGES 0x04u
#define ERR_CAP_QUEUE 0x08u
#define ERR_BAD_ID 0x10u
#define ERR_GRANULE 0x20u
#define ERR_CAP_STEPS 0x40u
#define ERR_CAP_LIVE 0x80u
#define ERR_TIME_ORDER 0x100u
#define ERR_PRICE 0x200u  // bb_step_device: a NEW row's limit price was off the tick grid (row dropped)
#define ERR_ROW_OP 0x400u  // bb_run_agents_with_rows: a row the in-kernel queue cannot carry (MODIFY, trader id >= 2^19)

// Order record (types.rs:79-101 `Order` + orderbook.rs:36-44 key), 64 bytes = two 32-byte sectors split
// by access pattern: the first sector is what matching / cancel / modify read and update, the second
// holds the write-only timestamps and the trader id.
struct __align__(16) OrderRec {
    u32 price, vol, next, prev;
    u64 key_time;  // time component of the queue key (arrival, or the last replace)
    u32 meta, start_vol;
    u64 arr_time, end_time;
    u32 trader, pad0, pad1, pad2;
};
#define ORD_STRIDE 64u
struct __align__(16) TradeRec {  // types.rs:105-118
    u64 t;
    u32 price, vol, active, passive, side_bid, pad;
};

struct __align__(16) BookHdr {  // 128 bytes, head of every book blob
    u64 t, max_key_time, rng_s0, rng_s1;
    u32 n_orders, n_trades, trade_vol, trading;
    u32 side_vol[2];  // [0] ask, [1] bid
    u32 best_q[2];    // best level index (price / granule) by queue, valid iff has_best
    u32 has_best[2];
    u32 err, n_steps;
    u32 step_counter, free_top;  // free_top: dense engine's free-slot stack height
    u64 n_instr, n_transitions, traded_volume, n_trades_total, n_created;
};
static_assert(sizeof(BookHdr) == 128, "BookHdr must stay 128 bytes");
static_assert(sizeof(OrderRec) == 64 && sizeof(TradeRec) == 32, "record sizes");

// ---- address-space-explicit memory operations ---------------------------------------------------------
__device__ __forceinline__ u32 lds(u32 a) {
    u32 v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts(u32 a, u32 v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u64 lds64(u32 a) {
    u64 v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts64(u32 a, u64 v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ u32 lds8(u32 a) {
    u32 v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts8(u32 a, u32 v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u32 lds16(u32 a) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts16(u32 a, u32 v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ uint4 lds128(u32 a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128(u32 a, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ u32 ldg32(u64 a) {
    u32 v;
    asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(a));
    return v;
}
__device__ __forceinline__ u64 ldg64(u64 a) {
    u64 v;
    asm volatile("ld.global.u64 %0, [%1];" : "=l"(v) : "l"(a));
    return v;
}
__device__ __forceinline__ uint4 ldg128(u64 a) {
    uint4 v;
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(a));
    return v;
}
__device__ __forceinline__ void stg32(u64 a, u32 v) { asm volatile("st.global.u32 [%0], %1;" ::"l"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void stg64(u64 a, u64 v) { asm volatile("st.global.u64 [%0], %1;" ::"l"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void stg128(u64 a, u32 x, u32 y, u32 z, u32 w) {
    asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

// fire-and-forget pull of one 32-byte sector towards L2 (deep books: order records are DRAM-cold when first touched)
__device__ __forceinline__ void prefetch_l2(u64 a) { asm volatile("prefetch.global.L2 [%0];" ::"l"(a)); }
__device__ __forceinline__ void prefetch_l1(u64 a) { asm volatile("prefetch.global.L1 [%0];" ::"l"(a)); }

// byte offsets inside records
#define OH_PRICE 0u
#define OH_VOL 4u
#define OH_NEXT 8u
#define OH_PREV 12u
#define OH_KEYT 16u
#define OH_META 24u
#define OH_SVOL 28u
#define OC_ARR 32u
#define OC_END 40u
#define OC_TRADER 48u
// byte offsets inside a 512-byte page: level l has (vol, cnt) at PG_VC + 8l and (head, tail) at PG_HT + 8l
#define PG_VC 0u
#define PG_HT 256u
#define PG_VOL(l) (8u * (l))
#define PG_CNT(l) (8u * (l) + 4u)
#define PG_HEAD(l) (256u + 8u * (l))
#define PG_TAIL(l) (260u + 8u * (l))

#define FL_TRADING 1u
#define FL_HAS_ASK 2u  // FL_HAS_ASK << side
#define FL_HAS_BID 4u

// Launch-invariant geometry (lives in the constant bank through the kernel parameter block).
struct Geo {
    u32 p_total, p_smem, granule;
    u32 pc_off;       // paged engine: offset (from the warp's shared-memory base) of the 128-entry page lookup cache
    u32 max_orders, max_trades;
    u64 tr_base;      // trade slabs  [n_envs][max_trades] x 32 B
    u64 blobs_base;   // book blobs   [n_envs] x blob_stride
    u64 blob_stride;
    // tick size of each env's book [n_envs] (bb_set_tick_sizes).  Read where it is used — once per level-2 record, row
    // batch or agent update (k_deepw: once per launch, into a control word), never per event — so that it holds no
    // register across the event loop.
    const u32* ticks;
    // dense-window engine (dense.cuh): first price of the window, number of levels, number of order slots
    u32 d_win_lo, d_levels, d_live;
};
template <u32 LP_, u32 NWMAX_> struct DenseLayout;
// Compile-time engine selection.
//   ENG_PAGED  any granule, any number of pages, HBM-resident pages
//   ENG_FAST   granule == 1 && p_total == 32, every page resident: no price division, directory loops become one ballot
//   ENG_DENSE* dense tick-indexed window + shared-memory order slots (dense.cuh), two size classes
#define ENG_PAGED 0
#define ENG_FAST 1
#define ENG_DENSE 2    // <= 128 order slots, window <= 256 levels
#define ENG_DENSE_L 3  // <= 254 order slots, window <= 1024 levels
// the generic geometry with EVERY page resident in shared memory (deep books at one or two books per CTA): the HBM-page
// variants of every page access drop out of the instruction stream.  Only k_apply is instantiated for it.
#define ENG_PAGED_RES 4
// deep-book engine (deep.cuh): its own kernel (k_deep, one CTA per book); never a GeoT<> instantiation
#define ENG_DEEP 5
template <int ENG_> struct GeoT : Geo {
    static constexpr bool FAST = ENG_ == ENG_FAST;
    static constexpr bool RES = ENG_ == ENG_FAST || ENG_ == ENG_PAGED_RES;  // no page lives in HBM
    static constexpr bool DENSE = ENG_ == ENG_DENSE || ENG_ == ENG_DENSE_L;
    typedef DenseLayout<(ENG_ == ENG_DENSE_L ? 256u : 128u), (ENG_ == ENG_DENSE_L ? 32u : 8u)> DL;
};
template <class G> __device__ __forceinline__ u32 ptot(const G& g) { return G::FAST ? 32u : g.p_total; }
template <class G> __device__ __forceinline__ u32 gran(const G& g) { return G::FAST ? 1u : g.granule; }

// Register-resident state of the warp's book.
struct Book {
    u64 t, max_key_time;
    u32 n_orders, n_trades, trade_vol;  // n_trades counts every trade, logged or not
    u32 vol_ask, vol_bid;  // side totals (side.rs:38)
    u32 bq_ask, bq_bid;    // cached touch level index by queue
    u32 flags, err;
    u32 d_instr, d_trans, d_volume;  // per-launch deltas of the u64 header counters
    u32 sb;                // shared-space address of the blob image
    u32 tag_lane;          // shared-space address of this lane's page tag: sb + 128 + 4 * lane
    u64 oh;                // global address of this env's order slab
    u32 env;               // env index inside the handle (cold addresses are rebuilt from it)
    u64 blob;              // global address of this env's book blob (HBM-resident pages of the generic geometry)
    u32 lane;
    u32 free_top;          // dense engine: entries on the free-slot stack
    u32 ags;               // dense engine, k_sim: shared-space address of the agent -> slot table (u8, entry 0 unused)
    u64 tr_ptr;            // dense engine: address of the next trade record
    u32 ev, jp, jend;      // dense k_sim, journaled (d_apply JRN): the event's queue entry, next / end of the trade journal
};

__device__ __forceinline__ u32 tag_addr(const Book& b, u32 i) { return b.sb + 128u + 4u * i; }
template <class G> __device__ __forceinline__ u32 vmap_addr(const G& g, const Book& b, u32 i) { return b.sb + 128u + 4u * (ptot(g) + i); }
template <class G> __device__ __forceinline__ u32 qmap_addr(const G& g, const Book& b, u32 i) { return b.sb + 128u + 4u * (2u * ptot(g) + i); }

// A page lives in shared memory when its slot is resident (slot < p_smem), else in the env's HBM page
// array.  The two cases are distinct TYPES so that every accessor compiles to exactly one ld/st; the
// choice is made once per operation by the callers (see the `*_at` implementation templates).
// Page layout: 32 x (vol, cnt) pairs, then 32 x (head, tail) pairs.
struct PageS {
    u32 a;  // shared-space byte address of the page
};
struct PageG {
    u64 a;  // global address of the page
};
__device__ __forceinline__ u32 pld(PageS p, u32 off) { return lds(p.a + off); }
__device__ __forceinline__ u32 pld(PageG p, u32 off) { return ldg32(p.a + off); }
__device__ __forceinline__ void pst(PageS p, u32 off, u32 v) { sts(p.a + off, v); }
__device__ __forceinline__ void pst(PageG p, u32 off, u32 v) { stg32(p.a + off, v); }
__device__ __forceinline__ uint2 pld2(PageS p, u32 off) {
    const u64 v = lds64(p.a + off);
    return make_uint2((u32)v, (u32)(v >> 32));
}
__device__ __forceinline__ uint2 pld2(PageG p, u32 off) {
    const u64 v = ldg64(p.a + off);
    return make_uint2((u32)v, (u32)(v >> 32));
}
__device__ __forceinline__ void pst2(PageS p, u32 off, u32 x, u32 y) { sts64(p.a + off, ((u64)y << 32) | x); }
__device__ __forceinline__ void pst2(PageG p, u32 off, u32 x, u32 y) { stg64(p.a + off, ((u64)y << 32) | x); }

template <class G> __device__ __forceinline__ u32 page_off(const G& g, u32 slot) { return 128u + 12u * ptot(g) + slot * 512u; }
template <class G> __device__ __forceinline__ PageS page_s(const G& g, const Book& b, u32 slot) {
    return PageS{b.sb + page_off(g, slot)};
}
template <class G> __device__ __forceinline__ PageG page_g(const G& g, const Book& b, u32 slot) {
    return PageG{b.blob + page_off(g, slot)};
}
// (vol, cnt) of a level of any page; for the cold observation paths where the slot may differ per lane
template <class G> __device__ __forceinline__ uint2 level_pair_any(const G& g, const Book& b, u32 slot, u32 l) {
    return (G::RES || slot < g.p_smem) ? pld2(page_s(g, b, slot), PG_VC + 8u * l) : pld2(page_g(g, b, slot), PG_VC + 8u * l);
}

__device__ __forceinline__ bool has_best(const Book& b, u32 side) { return (b.flags >> (1u + side)) & 1u; }
__device__ __forceinline__ u32 best_q(const Book& b, u32 side) { return side ? b.bq_bid : b.bq_ask; }
__device__ __forceinline__ void set_best(Book& b, u32 side, u32 q) {
    if (side) b.bq_bid = q; else b.bq_ask = q;
    b.flags |= FL_HAS_ASK << side;
}
__device__ __forceinline__ void add_side_vol(Book& b, u32 side, u32 dv) {
    if (side) b.vol_bid += dv; else b.vol_ask += dv;
}

// price -> level index; false when the price is not a multiple of the ladder granule
template <class G> __device__ __forceinline__ bool to_level(const G& g, u32 price, u32* q) {
    if (G::FAST || gran(g) == 1u) {
        *q = price;
        return true;
    }
    const u32 x = price / gran(g);
    *q = x;
    return x * gran(g) == price;
}

// ---- page directory -----------------------------------------------------------------------------
// The generic geometry (hundreds of pages per book) keeps a 128-entry direct-mapped lookup cache in front of the
// associative directory search: entry (tag & 127) holds the slot that tag was last found in.  The tag array stays
// authoritative (a cached slot is used only if its tag still matches), so stale entries are harmless and the cache
// is never persisted.  A deep book's live pages are consecutive page keys, which map to distinct entries.
#define PCACHE_ENTRIES 128u
template <class G> __device__ __forceinline__ u32 find_page(const G& g, const Book& b, u32 side, u32 pkey) {
    const u32 want = (pkey << 1) | side;
    u32 ca = 0;
    if constexpr (!G::FAST) {
        ca = b.sb + g.pc_off + (want & (PCACHE_ENTRIES - 1u));
        const u32 s = lds8(ca);
        if (lds(tag_addr(b, s)) == want) return s;
    }
    for (u32 base = 0; base < ptot(g); base += 32) {
        const u32 m = __ballot_sync(BB_FULL, lds(b.tag_lane + 4u * base) == want);
        if (m) {
            const u32 slot = base + __ffs(m) - 1;
            if constexpr (!G::FAST) sts8(ca, slot);
            return slot;
        }
    }
    return BB_NIL;
}

template <class G> __device__ __forceinline__ u32 alloc_page(const G& g, Book& b, u32 side, u32 pkey) {
    for (u32 base = 0; base < ptot(g); base += 32) {
        // in the all-resident geometries only the slots [0, p_smem) exist
        const bool usable = !G::RES || (base + b.lane) < g.p_smem;
        const u32 m = __ballot_sync(BB_FULL, usable && lds(b.tag_lane + 4u * base) == BB_TAG_FREE);
        if (m) {
            const u32 slot = base + __ffs(m) - 1;
            sts(tag_addr(b, slot), (pkey << 1) | side);
            if constexpr (!G::FAST) sts8(b.sb + g.pc_off + (((pkey << 1) | side) & (PCACHE_ENTRIES - 1u)), slot);
            sts(vmap_addr(g, b, slot), 0);
            sts(qmap_addr(g, b, slot), 0);
            return slot;
        }
    }
    b.err |= ERR_CAP_PAGES;
    return BB_NIL;
}

// best level by the given bitmap family (qmap: first key of `orders`, side.rs:99-104; vmap: first key
// of `volumes`, side.rs:107-120).  Returns false when the side is empty.
template <class G> __device__ __forceinline__ bool scan_best(const G& g, const Book& b, u32 side, bool by_queue, u32* out_q) {
    u32 best = side ? 0u : 0xFFFFFFFFu;
    u32 any = 0;
    for (u32 base = 0; base < ptot(g); base += 32) {
        const u32 tg = lds(tag_addr(b, base + b.lane));
        const u32 bm = lds(by_queue ? qmap_addr(g, b, base + b.lane) : vmap_addr(g, b, base + b.lane));
        const bool ok = (tg != BB_TAG_FREE) && ((tg & 1u) == side) && (bm != 0);
        any |= __ballot_sync(BB_FULL, ok);
        if (side) {
            const u32 v = ok ? (((tg >> 1) << 5) + (31u - __clz(bm))) : 0u;
            best = max(best, __reduce_max_sync(BB_FULL, v));
        } else {
            const u32 v = ok ? (((tg >> 1) << 5) + (__ffs(bm) - 1u)) : 0xFFFFFFFFu;
            best = min(best, __reduce_min_sync(BB_FULL, v));
        }
    }
    *out_q = best;
    return any != 0;
}

template <class G> __device__ __forceinline__ void recompute_best(const G& g, Book& b, u32 side) {
    u32 q;
    if (scan_best(g, b, side, true, &q)) set_best(b, side, q);
    else b.flags &= ~(FL_HAS_ASK << side);
}

// The touch level (page `slot`, page key `pkey`) just lost its last queued order and `qm` is that page's
// remaining queue bitmap.  Pages of one side never overlap in price, so when the page that held the best
// level still has a queued level, the new best is in the same page: one bit scan instead of a directory scan.
template <class G> __device__ __forceinline__ void next_best_after(const G& g, Book& b, u32 side, u32 pkey, u32 qm) {
    if (qm) {
        const u32 l = side ? (31u - __clz(qm)) : (__ffs(qm) - 1u);
        set_best(b, side, (pkey << 5) + l);
    } else {
        recompute_best(g, b, side);
    }
}

// side.rs:99-104 + 194-196: empty ask => u32::MAX, empty bid => 0
template <class G> __device__ __forceinline__ u32 best_price(const G& g, const Book& b, u32 side) {
    if (!has_best(b, side)) return side ? 0u : 0xFFFFFFFFu;
    if constexpr (G::DENSE) return g.d_win_lo + best_q(b, side);
    return best_q(b, side) * gran(g);
}

// side.rs:138-143 through the bid/ask wrappers: (vol, count) at an arbitrary price; warp-cooperative
template <class G> __device__ __forceinline__ void level_at(const G& g, const Book& b, u32 side, u32 price, u32* vol, u32* cnt);
template <class G> __device__ __forceinline__ void d_level_at(const G& g, const Book& b, u32 side, u32 price, u32* vol, u32* cnt);
template <class G> __device__ __forceinline__ void level_at(const G& g, const Book& b, u32 side, u32 price, u32* vol, u32* cnt) {
    if constexpr (G::DENSE) {
        d_level_at(g, b, side, price, vol, cnt);
        return;
    }
    *vol = 0;
    *cnt = 0;
    u32 q;
    if (!to_level(g, price, &q)) return;
    const u32 slot = find_page(g, b, side, q >> 5);
    if (slot == BB_NIL) return;
    if (!((lds(vmap_addr(g, b, slot)) >> (q & 31u)) & 1u)) return;
    const uint2 vc = level_pair_any(g, b, slot, q & 31u);
    *vol = vc.x;
    *cnt = vc.y;
}

// same lookup done independently by each lane (divergent prices) — used by the level-2 emitter
template <class G> __device__ __forceinline__ void level_at_lane(const G& g, const Book& b, u32 side, u32 price, u32* vol, u32* cnt) {
    if constexpr (G::DENSE) {
        d_level_at(g, b, side, price, vol, cnt);
        return;
    }
    *vol = 0;
    *cnt = 0;
    u32 q;
    if (!to_level(g, price, &q)) return;
    const u32 want = ((q >> 5) << 1) | side;
    u32 slot = BB_NIL;
    const u32 n_tags = G::RES ? g.p_smem : g.p_total;  // the all-resident geometries only have the slots [0, p_smem)
    for (u32 j = 0; j < n_tags; ++j)
        if (lds(tag_addr(b, j)) == want) slot = j;
    if (slot == BB_NIL) return;
    if (!((lds(vmap_addr(g, b, slot)) >> (q & 31u)) & 1u)) return;
    const uint2 vc = level_pair_any(g, b, slot, q & 31u);
    *vol = vc.x;
    *cnt = vc.y;
}

// first level of the reference's `volumes` map (side.rs:107-120)
template <class G> __device__ __forceinline__ void best_by_volumes(const G& g, const Book& b, u32 side, u32* vol, u32* cnt) {
    if constexpr (G::DENSE) {  // no key collisions in the dense engine: the two maps of side.rs always agree
        d_level_at(g, b, side, best_price(g, b, side), vol, cnt);
        return;
    }
    *vol = 0;
    *cnt = 0;
    u32 q;
    if (!scan_best(g, b, side, false, &q)) return;
    const u32 slot = find_page(g, b, side, q >> 5);
    const uint2 vc = level_pair_any(g, b, slot, q & 31u);
    *vol = vc.x;
    *cnt = vc.y;
}

// ---- volumes-map half of insert_order / remove_order / remove_vol (side.rs:54-96) ------------------
template <class G, class P> __device__ __forceinline__ void level_add(const G& g, Book& b, u32 side, u32 slot, P pr, u32 l, u32 vol) {
    const u32 bit = 1u << l;
    const u32 vm = lds(vmap_addr(g, b, slot));
    if (vm & bit) {
        const uint2 vc = pld2(pr, PG_VC + 8u * l);
        pst2(pr, PG_VC + 8u * l, vc.x + vol, vc.y + 1u);
    } else {
        pst2(pr, PG_VC + 8u * l, vol, 1u);
        sts(vmap_addr(g, b, slot), vm | bit);
    }
    add_side_vol(b, side, vol);
}

// returns true when the page was released
template <class G, class P> __device__ __forceinline__ bool level_remove(const G& g, Book& b, u32 side, u32 slot, P pr, u32 l, u32 vol) {
    const u32 bit = 1u << l;
    const uint2 vc = pld2(pr, PG_VC + 8u * l);
    const u32 cnt = vc.y - 1u;
    pst2(pr, PG_VC + 8u * l, vc.x - vol, cnt);
    add_side_vol(b, side, 0u - vol);
    if (cnt == 0) {
        const u32 vm = lds(vmap_addr(g, b, slot)) & ~bit;
        sts(vmap_addr(g, b, slot), vm);
        if (vm == 0 && lds(qmap_addr(g, b, slot)) == 0) {
            sts(tag_addr(b, slot), BB_TAG_FREE);
            return true;
        }
    }
    return false;
}

// ---- orders-map half: the price-time queue ----------------------------------------------------------
// unlink a record with links (prev,next) from level (slot,l); maintains qmap and the cached touch
template <class G, class P> __device__ __forceinline__ void queue_unlink(const G& g, Book& b, u32 side, u32 slot, P pr, u32 l, u32 q,
                                                                        u32 prev, u32 next) {
    if (prev == BB_NIL) pst(pr, PG_HEAD(l), next); else stg32(b.oh + (u64)prev * ORD_STRIDE + OH_NEXT, next);
    if (next == BB_NIL) pst(pr, PG_TAIL(l), prev); else stg32(b.oh + (u64)next * ORD_STRIDE + OH_PREV, prev);
    if (prev == BB_NIL && next == BB_NIL) {
        const u32 qm = lds(qmap_addr(g, b, slot)) & ~(1u << l);
        sts(qmap_addr(g, b, slot), qm);
        if (has_best(b, side) && best_q(b, side) == q) next_best_after(g, b, side, q >> 5, qm);
    }
}

// orders.remove(&(price', key_time)) for an order that does NOT own its key any more (N1 ghost):
// whoever owns that key now loses it and becomes a ghost itself.
template <class G, class P> __device__ __forceinline__ void queue_remove_key_slow(const G& g, Book& b, u32 side, u32 slot, P pr,
                                                                                 u32 l, u32 q, u64 key_time) {
    if (!((lds(qmap_addr(g, b, slot)) >> l) & 1u)) return;
    u32 cur = pld(pr, PG_HEAD(l));
    while (cur != BB_NIL) {
        const u64 ra = b.oh + (u64)cur * ORD_STRIDE;
        const uint4 a = ldg128(ra);
        const u64 kt = ldg64(ra + OH_KEYT);
        if (kt == key_time) {
            stg32(ra + OH_META, ldg32(ra + OH_META) | META_GHOST);
            queue_unlink(g, b, side, slot, pr, l, q, a.w, a.z);
            return;
        }
        if (kt > key_time) return;
        cur = a.z;
    }
}

// orders.insert((price', t), id) when time did not move strictly forward: sorted position, or take
// over an existing equal key.  Returns the (prev,next) links the new record must carry.
template <class P> __device__ __forceinline__ void queue_insert_slow(const Book& b, P pr, u32 l, u32 id, u64 t, u32* out_prev,
                                                                     u32* out_next) {
    u32 cur = pld(pr, PG_TAIL(l));  // walk back from the tail
    u32 after = BB_NIL;             // node that will follow the new one
    while (cur != BB_NIL) {
        const u64 ra = b.oh + (u64)cur * ORD_STRIDE;
        const uint4 a = ldg128(ra);
        const u64 kt = ldg64(ra + OH_KEYT);
        if (kt < t) break;
        if (kt == t) {
            // BTreeMap::insert on an existing key: value replaced, position kept (side.rs:55)
            stg32(ra + OH_META, ldg32(ra + OH_META) | META_GHOST);
            if (a.w == BB_NIL) pst(pr, PG_HEAD(l), id); else stg32(b.oh + (u64)a.w * ORD_STRIDE + OH_NEXT, id);
            if (a.z == BB_NIL) pst(pr, PG_TAIL(l), id); else stg32(b.oh + (u64)a.z * ORD_STRIDE + OH_PREV, id);
            *out_prev = a.w;
            *out_next = a.z;
            return;
        }
        after = cur;
        cur = a.w;
    }
    // insert between cur (may be NIL => new head) and after (may be NIL => new tail)
    if (cur == BB_NIL) pst(pr, PG_HEAD(l), id); else stg32(b.oh + (u64)cur * ORD_STRIDE + OH_NEXT, id);
    if (after == BB_NIL) pst(pr, PG_TAIL(l), id); else stg32(b.oh + (u64)after * ORD_STRIDE + OH_PREV, id);
    *out_prev = cur;
    *out_next = after;
}

template <class G, class P> __device__ __forceinline__ void book_insert_at(const G& g, Book& b, u32 side, u32 q, u32 slot, P pr, u64 t,
                                                                          u32 id, u32 vol, u32* out_prev, u32* out_next) {
    const u32 l = q & 31u;
    level_add(g, b, side, slot, pr, l, vol);
    const u32 bit = 1u << l;
    const u32 qm = lds(qmap_addr(g, b, slot));
    if (!(qm & bit)) {
        pst2(pr, PG_HT + 8u * l, id, id);
        sts(qmap_addr(g, b, slot), qm | bit);
        const bool better = !has_best(b, side) || (side ? q > b.bq_bid : q < b.bq_ask);
        if (better) set_best(b, side, q);
    } else if (t > b.max_key_time) {
        const u32 tail = pld(pr, PG_TAIL(l));
        stg32(b.oh + (u64)tail * ORD_STRIDE + OH_NEXT, id);
        pst(pr, PG_TAIL(l), id);
        *out_prev = tail;
    } else {
        queue_insert_slow(b, pr, l, id, t, out_prev, out_next);
    }
}

// side.rs:54-66 insert_order for a resting order.  Returns false when the order could not rest.
template <class G> __device__ __forceinline__ bool book_insert(const G& g, Book& b, u32 side, u32 price, u64 t, u32 id, u32 vol,
                                                               u32* out_prev, u32* out_next) {
    *out_prev = BB_NIL;
    *out_next = BB_NIL;
    u32 q;
    if (!to_level(g, price, &q)) {
        b.err |= ERR_GRANULE;
        return false;
    }
    u32 slot = find_page(g, b, side, q >> 5);
    if (slot == BB_NIL) {
        slot = alloc_page(g, b, side, q >> 5);
        if (slot == BB_NIL) return false;
    }
    if (G::RES || slot < g.p_smem) book_insert_at(g, b, side, q, slot, page_s(g, b, slot), t, id, vol, out_prev, out_next);
    else book_insert_at(g, b, side, q, slot, page_g(g, b, slot), t, id, vol, out_prev, out_next);
    if (t > b.max_key_time) b.max_key_time = t;
    return true;
}

template <class G, class P> __device__ __forceinline__ void book_remove_at(const G& g, Book& b, u32 side, u32 q, u32 slot, P pr, u32 prev,
                                                                          u32 next, u64 key_time, bool ghost, u32 vol) {
    const u32 l = q & 31u;
    if (ghost) queue_remove_key_slow(g, b, side, slot, pr, l, q, key_time);
    else queue_unlink(g, b, side, slot, pr, l, q, prev, next);
    level_remove(g, b, side, slot, pr, l, vol);
}

// side.rs:75-84 remove_order(key, vol) for an order with the given record fields
template <class G> __device__ __forceinline__ void book_remove(const G& g, Book& b, u32 side, u32 price, u32 prev, u32 next,
                                                               u64 key_time, bool ghost, u32 vol) {
    u32 q;
    to_level(g, price, &q);
    const u32 slot = find_page(g, b, side, q >> 5);
    if (slot == BB_NIL) return;  // unreachable for Active orders
    if (G::RES || slot < g.p_smem) book_remove_at(g, b, side, q, slot, page_s(g, b, slot), prev, next, key_time, ghost, vol);
    else book_remove_at(g, b, side, q, slot, page_g(g, b, slot), prev, next, key_time, ghost, vol);
}

// remove_vol(price, dv) (side.rs:93-96) for the in-place volume reduction of modify_order
template <class G> __device__ __forceinline__ void book_reduce(const G& g, Book& b, u32 side, u32 price, u32 dv) {
    u32 q;
    to_level(g, price, &q);
    const u32 slot = find_page(g, b, side, q >> 5);
    if (slot == BB_NIL) return;
    if (G::RES || slot < g.p_smem) {
        const PageS pr = page_s(g, b, slot);
        pst(pr, PG_VOL(q & 31u), pld(pr, PG_VOL(q & 31u)) - dv);
    } else {
        const PageG pr = page_g(g, b, slot);
        pst(pr, PG_VOL(q & 31u), pld(pr, PG_VOL(q & 31u)) - dv);
    }
    add_side_vol(b, side, 0u - dv);
}

template <class G> __device__ __forceinline__ void log_trade(const G& g, Book& b, u64 t, u32 passive_bid, u32 price, u32 vol, u32 active,
                                                             u32 passive) {
    const u32 n = b.n_trades;
    if (n < g.max_trades) {
        const u64 a = g.tr_base + ((u64)b.env * g.max_trades + n) * 32u;
        stg128(a, (u32)t, (u32)(t >> 32), price, vol);
        stg128(a + 16u, active, passive, passive_bid, 0u);
    } else if (g.max_trades) {
        b.err |= ERR_CAP_TRADES;
    }
    b.n_trades = n + 1;
}

// One fill of the aggressor against the head of the touch level (slot, l) of side `o`
// (match_orders, orderbook.rs:843-870, plus the side bookkeeping of :443-447).  Returns false when the
// book turned out to be inconsistent.  *released is set when the page was freed.
template <class G, class P> __device__ __forceinline__ bool fill_one(const G& g, Book& b, u32 o, u32 bq, u32 slot, P pr, u32 id, u64 t,
                                                                    u32* vol, bool* filled, bool* released) {
    const u32 l = bq & 31u;
    const u32 hid = pld(pr, PG_HEAD(l));
    if (hid >= g.max_orders) {
        b.err |= ERR_BAD_ID;
        return false;
    }
    const u64 ha = b.oh + (u64)hid * ORD_STRIDE;
    const uint4 ph = ldg128(ha);  // price, vol, next, prev
    const u32 tv = min(*vol, ph.y);
    *vol -= tv;
    const u32 pvol = ph.y - tv;
    log_trade(g, b, t, o, ph.x, tv, id, hid);
    b.trade_vol += tv;
    b.d_volume += tv;
    b.d_trans += 1;
    if (pvol == 0) {
        stg32(ha + OH_VOL, 0u);
        stg32(ha + OH_META, ST_FILLED | (o ? META_BID : 0u));
        stg64(ha + OC_END, t);
        // side.remove_order(match.key, tv): the head always owns its key
        const u32 nxt = ph.z;
        bool emptied = false;
        u32 qm = 0;
        if (nxt == BB_NIL) {
            pst2(pr, PG_HT + 8u * l, BB_NIL, BB_NIL);
            qm = lds(qmap_addr(g, b, slot)) & ~(1u << l);
            sts(qmap_addr(g, b, slot), qm);
            emptied = true;
        } else {
            pst(pr, PG_HEAD(l), nxt);
            if constexpr (!G::FAST) prefetch_l2(b.oh + (u64)nxt * ORD_STRIDE);  // the new head is what the next fill reads
            stg32(b.oh + (u64)nxt * ORD_STRIDE + OH_PREV, BB_NIL);
        }
        *released = level_remove(g, b, o, slot, pr, l, tv);
        if (emptied) next_best_after(g, b, o, bq >> 5, qm);
    } else {
        stg32(ha + OH_VOL, pvol);
        pst(pr, PG_VOL(l), pld(pr, PG_VOL(l)) - tv);  // side.remove_vol(price, tv)
        add_side_vol(b, o, 0u - tv);
    }
    if (*vol == 0) *filled = true;
    return true;
}

// orderbook.rs:429-487 match_bid / match_ask.  Sweeps the opposite side in price-time order; returns the
// aggressor's remaining volume, *filled as the reference's Status::Filled.
template <class G> __device__ __forceinline__ u32 book_match(const G& g, Book& b, u32 side, u32 price, u32 vol, u32 id, u64 t,
                                                             bool* filled) {
    const u32 o = side ^ 1u;
    *filled = false;
    u32 slot = BB_NIL, slot_key = BB_NIL;
    while (vol > 0 && has_best(b, o)) {
        const u32 bq = best_q(b, o);
        const u32 bprice = bq * gran(g);
        if (side ? (price < bprice) : (price > bprice)) break;
        if (slot_key != (bq >> 5)) {
            slot = find_page(g, b, o, bq >> 5);
            slot_key = bq >> 5;
            if (slot == BB_NIL) {  // only reachable after a capacity error left the book inconsistent
                b.err |= ERR_CAP_PAGES;
                break;
            }
        }
        bool released = false, ok;
        if (G::RES || slot < g.p_smem) ok = fill_one(g, b, o, bq, slot, page_s(g, b, slot), id, t, &vol, filled, &released);
        else ok = fill_one(g, b, o, bq, slot, page_g(g, b, slot), id, t, &vol, filled, &released);
        if (!ok) break;
        if (released) slot_key = BB_NIL;
    }
    return vol;
}

__device__ __forceinline__ void write_order(const Book& b, u32 id, u32 price, u32 vol, u32 next, u32 prev, u64 key_time, u32 meta,
                                            u32 start_vol) {
    const u64 a = b.oh + (u64)id * ORD_STRIDE;
    stg128(a, price, vol, next, prev);
    stg128(a + 16u, (u32)key_time, (u32)(key_time >> 32), meta, start_vol);
}

// One event against the book: process_event (orderbook.rs:782-792) with place_order (:583-611),
// cancel_order (:622-644) and modify_order (:743-772; reduce_order_vol :656-667, replace_order :679-723)
// folded into one pipeline so that the remove / match / insert code exists once in the instruction stream:
//
//     NEW ------------------------------.
//     CANCEL --> load record --> remove --+--> done (cancel)
//     MODIFY --> load record --> reduce in place --> done
//                           `--> remove ---------.
//                                                  v
//                                   match (if trading) --> rest or finish --> write record
//
// For NEW the caller supplies every field (create_order :356-396 happened at submission).
#define EV_NEW 1u
#define EV_CANCEL 2u
#define EV_MODIFY 3u
}  // namespace bb
#include "dense.cuh"
namespace bb {
// IS_NEW is the compile-time specialisation for the dominant event kind (no record load, no replace state).
// CHECK_TIME (dense engine only): the caller cannot guarantee strictly increasing time between resting inserts.
template <bool IS_NEW, bool CHECK_TIME, class G, int HINT = 0>
__device__ __forceinline__ void book_apply(const G& g, Book& b, u32 kind, u32 id, u32 side, u32 price, u32 vol, u32 trader, bool has_p,
                                           bool has_v, u64 t, u32 hint = 0u) {
    if constexpr (G::DENSE) {
        d_apply<IS_NEW, CHECK_TIME, HINT>(g, b, kind, id, side, price, vol, trader, has_p, has_v, t, hint);
        return;
    }
    u32 start_vol = vol, meta_keep = 0;
    u64 old_kt = 0;
    const u64 ra = b.oh + (u64)id * ORD_STRIDE;
    if (IS_NEW) {
        if (id >= g.max_orders) {
            b.err |= ERR_CAP_ORDERS;
            return;
        }
    } else {
        if (id >= b.n_orders || id >= g.max_orders) {
            b.err |= ERR_BAD_ID;  // the reference panics (orderbook.rs:642, :749)
            return;
        }
        const uint4 a = ldg128(ra);        // price, vol, next, prev
        const uint4 c = ldg128(ra + 16u);  // key_time lo, hi, meta, start_vol
        if ((c.z & META_STATUS_MASK) != ST_ACTIVE) return;
        side = (c.z & META_BID) ? 1u : 0u;
        if (kind == EV_MODIFY) {
            if (!has_p && !has_v) return;
            if (!has_p && vol < a.y) {  // reduce in place: priority kept (orderbook.rs:755-757)
                stg32(ra + OH_VOL, vol);
                book_reduce(g, b, side, a.x, a.y - vol);
                b.d_trans += 1;
                return;
            }
            if (!has_p) price = a.x;
            if (!has_v) vol = a.y;
        }
        old_kt = ((u64)c.y << 32) | c.x;
        book_remove(g, b, side, a.x, a.w, a.z, old_kt, (c.z & META_GHOST) != 0, a.y);
        if (kind == EV_CANCEL) {
            stg32(ra + OH_META, ST_CANCELLED | (c.z & META_BID));
            stg64(ra + OC_END, t);
            b.d_trans += 1;
            return;
        }
        start_vol = c.w;
        meta_keep = c.z & META_BID;
    }
    // placement: a replaced order never takes the market-order path (N4), a new one does by price value (N3)
    const bool market = IS_NEW && (side ? (price == 0xFFFFFFFFu) : (price == 0u));
    u32 rem = vol, status = ST_ACTIVE, prev = BB_NIL, next = BB_NIL;
    bool filled = false, ended = false;
    if (b.flags & FL_TRADING) rem = book_match(g, b, side, price, vol, id, t, &filled);
    if (filled) {
        status = ST_FILLED;
        ended = true;
    } else if (market) {
        status = (b.flags & FL_TRADING) ? ST_CANCELLED : ST_REJECTED;  // orderbook.rs:517-531
        ended = true;
    } else {
        book_insert(g, b, side, price, t, id, rem, &prev, &next);  // orderbook.rs:499-504 / :699-722
    }
    if (!IS_NEW) {
        write_order(b, id, price, rem, next, prev, filled ? old_kt : t, status | meta_keep, start_vol);
        if (ended) stg64(ra + OC_END, t);
    } else {
        // the key's time component is only stamped when the order rests (orderbook.rs:499-504); 0 otherwise
        write_order(b, id, price, rem, next, prev, ended ? 0ULL : t, status | (side ? META_BID : 0u), start_vol);
        const u64 end_time = ended ? t : ~0ULL;
        stg128(ra + OC_ARR, (u32)t, (u32)(t >> 32), (u32)end_time, (u32)(end_time >> 32));
        stg128(ra + OC_ARR + 16u, trader, 0u, 0u, 0u);
    }
    b.d_trans += 1;
}

// ---- observation emission ------------------------------------------------------------------------
// Level-1 / level-2 record in the array layout of rust/src/step_sim_numpy.rs:300-368:
// [trade_vol, bid_price, ask_price, ask_vol, bid_vol, then per level i: bid_vol_i, n_bid_i, ask_vol_i, n_ask_i]
// Levels sit at FIXED offsets of the env's tick from the touch with wrapping arithmetic (orderbook.rs:229-264).
// Each lane returns the word(s) it owns: word index = lane (and lane + 32 for the 45-word record).
template <class G> __device__ __forceinline__ void book_obs(const G& g, const Book& b, u32 n_words, u32* w0, u32* w1) {
    // the tick is issued first so that its load overlaps the touch lookups (45-word records only)
    const u32 tick = n_words > 9u ? __ldg(g.ticks + b.env) : 0u;
    const u32 bid = best_price(g, b, 1), ask = best_price(g, b, 0);
    u32 x = 0, y = 0;
    if (n_words <= 9u) {
        u32 bv, bc, av, ac;
        level_at(g, b, 1, bid, &bv, &bc);
        level_at(g, b, 0, ask, &av, &ac);
        const u32 l = b.lane;
        x = l == 0 ? b.trade_vol : l == 1 ? bid : l == 2 ? ask : l == 3 ? b.vol_ask : l == 4 ? b.vol_bid
          : l == 5 ? bv : l == 6 ? bc : l == 7 ? av : l == 8 ? ac : 0u;
    } else {
        // words 5..44: level i = (w-5)/4, field f = (w-5)%4 -> f<2 bid (vol,cnt), else ask (vol,cnt)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const u32 w = b.lane + 32u * half;
            u32 val = 0;
            if (w >= 5u && w < 45u) {
                const u32 i = (w - 5u) >> 2, f = (w - 5u) & 3u;
                u32 v, n;
                if (f < 2u) level_at_lane(g, b, 1, bid - i * tick, &v, &n);
                else level_at_lane(g, b, 0, ask + i * tick, &v, &n);
                val = (f & 1u) ? n : v;
            } else if (w < 5u) {
                val = w == 0 ? b.trade_vol : w == 1 ? bid : w == 2 ? ask : w == 3 ? b.vol_ask : b.vol_bid;
            }
            if (half == 0) x = val; else y = val;
        }
    }
    *w0 = x;
    *w1 = y;
}

// ---- header <-> registers ---------------------------------------------------------------------------
// n_steps, step_counter and the xoroshiro state stay in the shared-memory header (touched once per step).
#define HDR_T 0u
#define HDR_MAXKT 8u
#define HDR_RNG0 16u
#define HDR_RNG1 24u
#define HDR_NORDERS 32u
#define HDR_NTRADES 36u
#define HDR_TRADEVOL 40u
#define HDR_TRADING 44u
#define HDR_SIDEVOL 48u
#define HDR_BESTQ 56u
#define HDR_HASBEST 64u
#define HDR_ERR 72u
#define HDR_NSTEPS 76u
#define HDR_STEPCTR 80u
#define HDR_FREETOP 84u
#define HDR_NINSTR 88u
#define HDR_NTRANS 96u
#define HDR_VOLUME 104u
#define HDR_NTRADES_TOTAL 112u
#define HDR_NCREATED 120u

template <class G> __device__ __forceinline__ void book_from_header(const G& g, Book& b) {
    if constexpr (G::DENSE) {
        b.free_top = lds(b.sb + HDR_FREETOP);
        b.tr_ptr = g.tr_base + ((u64)b.env * g.max_trades + min((u32)lds64(b.sb + HDR_NTRADES_TOTAL), g.max_trades)) * 32u;
    }
    b.t = lds64(b.sb + HDR_T);
    b.max_key_time = lds64(b.sb + HDR_MAXKT);
    b.n_orders = lds(b.sb + HDR_NORDERS);
    b.n_trades = (u32)lds64(b.sb + HDR_NTRADES_TOTAL);
    b.trade_vol = lds(b.sb + HDR_TRADEVOL);
    b.vol_ask = lds(b.sb + HDR_SIDEVOL);
    b.vol_bid = lds(b.sb + HDR_SIDEVOL + 4u);
    b.bq_ask = lds(b.sb + HDR_BESTQ);
    b.bq_bid = lds(b.sb + HDR_BESTQ + 4u);
    b.flags = (lds(b.sb + HDR_TRADING) ? FL_TRADING : 0u) | (lds(b.sb + HDR_HASBEST) ? FL_HAS_ASK : 0u) |
              (lds(b.sb + HDR_HASBEST + 4u) ? FL_HAS_BID : 0u);
    // Book::err collects the errors raised DURING THIS LAUNCH only (they are what the launch reports through err_flag);
    // the header word they are OR-ed into at write-back is the env's sticky record (bb_env_errors / bb_clear_errors)
    b.err = 0u;
    b.d_instr = b.d_trans = b.d_volume = 0;
}

// One lane writes (every lane holds the same values): the read-modify-write counters must not be applied per lane.
template <class G> __device__ __forceinline__ void book_to_header(const G& g, const Book& b) {
    __syncwarp();
    if (b.lane != 0u) {
        __syncwarp();
        return;
    }
    if constexpr (G::DENSE) sts(b.sb + HDR_FREETOP, b.free_top);
    sts64(b.sb + HDR_T, b.t);
    sts64(b.sb + HDR_MAXKT, b.max_key_time);
    sts64(b.sb + HDR_NCREATED, lds64(b.sb + HDR_NCREATED) + (b.n_orders - lds(b.sb + HDR_NORDERS)));
    sts(b.sb + HDR_NORDERS, b.n_orders);
    sts(b.sb + HDR_TRADEVOL, b.trade_vol);
    sts(b.sb + HDR_SIDEVOL, b.vol_ask);
    sts(b.sb + HDR_SIDEVOL + 4u, b.vol_bid);
    sts(b.sb + HDR_BESTQ, b.bq_ask);
    sts(b.sb + HDR_BESTQ + 4u, b.bq_bid);
    sts(b.sb + HDR_TRADING, (b.flags & FL_TRADING) ? 1u : 0u);
    sts(b.sb + HDR_HASBEST, (b.flags & FL_HAS_ASK) ? 1u : 0u);
    sts(b.sb + HDR_HASBEST + 4u, (b.flags & FL_HAS_BID) ? 1u : 0u);
    sts(b.sb + HDR_ERR, lds(b.sb + HDR_ERR) | b.err);
    sts64(b.sb + HDR_NINSTR, lds64(b.sb + HDR_NINSTR) + b.d_instr);
    sts64(b.sb + HDR_NTRANS, lds64(b.sb + HDR_NTRANS) + b.d_trans);
    sts64(b.sb + HDR_VOLUME, lds64(b.sb + HDR_VOLUME) + b.d_volume);
    const u64 tt = lds64(b.sb + HDR_NTRADES_TOTAL);
    sts64(b.sb + HDR_NTRADES_TOTAL, tt + (u32)(b.n_trades - (u32)tt));
    sts(b.sb + HDR_NTRADES, min(b.n_trades, g.max_trades));  // records actually present in the trade log
    __syncwarp();
}

}  // namespace bb
