// Test infrastructure: the per-env reset of bb_reset_device restated on the oracle's own objects (oracle/env.hpp) — an
// Env / MarketEnv rebuilt from its construction parameters with its agent groups' state cleared, and the env's random
// streams either kept (shuffle generator and the step counter of the agents' Philox draws) or re-seeded
// (Xoroshiro128StarStar::seed_from_u64(seed), step counter 0), as a freshly constructed StepEnvNumpy(seed, ...) /
// MarketEnv has them.
//
// The oracle's C API is compiled in (for its SimHandle / MarketHandle); every symbol of this library is hidden except the
// ers_* calls, so the copies of the orc_* functions never meet liboracle's.  It operates on handles liboracle created
// (oracle.StepEnv._h, oracle.MarketEnv._h): both libraries are built from the same headers with the same flags.
#include "../../oracle/oracle_capi.cpp"

#define ERS_API extern "C" __attribute__((visibility("default")))

namespace {
// the groups of `from`, in declaration order, with the state a freshly added group has
template <class S> void add_groups_like(S& to, const S& from) {
    for (const auto& g : from.order) {
        if constexpr (std::is_same<S, Sim>::value) {
            if (g.first == GROUP_RANDOM) to.add_random(from.randoms[g.second].p);
            else if (g.first == GROUP_MOMENTUM) to.add_momentum(from.momentums[g.second].p);
            else to.add_noise(from.noises[g.second].p);
        } else {
            if (g.kind == GROUP_RANDOM) to.add_random(g.asset, from.randoms[g.idx].p);
            else if (g.kind == GROUP_MOMENTUM) to.add_momentum(g.asset, from.momentums[g.idx].p);
            else to.add_noise(g.asset, from.noises[g.idx].p);
        }
    }
}
}  // namespace

ERS_API void ers_sim_reset(void* s, uint64_t start_time, int trading, int reseed, uint64_t seed) {
    SimHandle* h = (SimHandle*)s;
    Sim fresh(start_time, h->sim.env.book.tick_size, h->sim.env.step_size, trading != 0);
    add_groups_like(fresh, h->sim);
    fresh.env.keep_records = h->sim.env.keep_records;
    fresh.step_counter = reseed ? 0u : h->sim.step_counter;
    fresh.n_instructions = h->sim.n_instructions;
    h->sim = std::move(fresh);
    if (reseed) h->rng = Xoroshiro128StarStar::seed_from_u64(seed);
}

ERS_API void ers_market_reset(void* m, uint64_t start_time, int trading, int reseed, uint64_t seed) {
    MarketHandle* h = (MarketHandle*)m;
    std::vector<Price> ticks;
    for (const auto& b : h->env.books) ticks.push_back(b.tick_size);
    MarketSim fresh(start_time, ticks, h->env.step_size, trading != 0);
    add_groups_like(fresh, h->sim);
    fresh.step_counter = reseed ? 0u : h->sim.step_counter;
    fresh.n_instructions = h->sim.n_instructions;
    h->sim = std::move(fresh);  // (h->env refers to h->sim.env, which is assigned in place)
    if (reseed) h->rng = Xoroshiro128StarStar::seed_from_u64(seed);
}
