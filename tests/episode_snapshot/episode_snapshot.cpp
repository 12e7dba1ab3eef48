// Test infrastructure: the snapshot restore of bb_restore_device restated on the oracle's own objects (oracle/env.hpp) — a
// Sim / MarketSim (env, agent groups with their state, Philox step counter) and its Xoroshiro128** shuffle stream copied
// from another handle with C++ value semantics.  The copy's per-step records are cleared (a restored book's history starts
// empty), and its stream is optionally re-seeded (Xoroshiro128StarStar::seed_from_u64(seed)) with the step counter kept.
//
// The oracle's C API is compiled in (for its SimHandle / MarketHandle); every symbol of this library is hidden except the
// ess_* calls, so the copies of the orc_* functions never meet liboracle's.  It operates on handles liboracle created
// (oracle.StepEnv._h, oracle.MarketEnv._h): both libraries are built from the same headers with the same flags.
#include "../../oracle/oracle_capi.cpp"

#define ESS_API extern "C" __attribute__((visibility("default")))

ESS_API void ess_sim_copy(void* dst, const void* src, int reseed, uint64_t seed) {
    SimHandle* d = (SimHandle*)dst;
    const SimHandle* s = (const SimHandle*)src;
    if (d != s) {
        d->sim = s->sim;
        d->rng = s->rng;
    }
    d->sim.env.records = Level2DataRecords{};
    d->sim.env.trade_vols.clear();
    if (reseed) d->rng = Xoroshiro128StarStar::seed_from_u64(seed);
}

ESS_API void ess_market_copy(void* dst, const void* src, int reseed, uint64_t seed) {
    MarketHandle* d = (MarketHandle*)dst;
    const MarketHandle* s = (const MarketHandle*)src;
    if (d != s) {
        d->sim = s->sim;  // (d->env refers to d->sim.env, which is assigned in place)
        d->rng = s->rng;
    }
    for (auto& r : d->env.records) r = Level2DataRecords{};
    for (auto& v : d->env.trade_vols) v.clear();
    if (reseed) d->rng = Xoroshiro128StarStar::seed_from_u64(seed);
}
