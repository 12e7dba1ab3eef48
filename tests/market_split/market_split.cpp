// Test infrastructure: the two halves of one keyed market step of the oracle's MarketSim (oracle/env.hpp), separately
// callable so that a test can queue its own instructions between them — `agents.update(env)`, `env.place_order(..)` /
// `env.cancel_order(..)`, `env.step()`, what bb_run_agents_with_rows_market does per market (runner.rs:107-131 with the
// caller's calls in between).  The halves restate MarketSim::run_keyed step for step on the oracle's own objects;
// tests/test_oracle_market_split_step.py checks that, with nothing queued between them, they are exactly run_keyed.
//
// The oracle's C API is compiled in (for its MarketHandle); every symbol of this library is hidden except the mks_* calls,
// so the copies of the orc_* functions never meet liboracle's.  It operates on handles liboracle created
// (oracle.MarketEnv._h): both libraries are built from the same headers with the same flags.
#include "../../oracle/oracle_capi.cpp"

#define MKS_API extern "C" __attribute__((visibility("default")))

namespace {
void agents_update_keyed(MarketSim& sim, uint64_t seed, uint32_t market_id) {  // the first half of MarketSim::run_keyed
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t step = sim.step_counter;
    uint32_t slot_base = 0, gi = 0;
    for (auto& g : sim.order) {
        AssetEnv ae(sim.env, g.asset);
        if (g.kind == GROUP_RANDOM) {
            sim.randoms[g.idx].update_keyed(ae, market_id, step, slot_base, k0, k1);
            slot_base += sim.randoms[g.idx].p.n_agents;
        } else if (g.kind == GROUP_MOMENTUM) {
            sim.momentums[g.idx].update_keyed(ae, market_id, step, gi, slot_base, k0, k1);
            slot_base += sim.momentums[g.idx].p.n_agents;
        } else {
            sim.noises[g.idx].update_keyed(ae, market_id, step, gi, slot_base, k0, k1);
            slot_base += sim.noises[g.idx].p.n_agents;
        }
        ++gi;
    }
}
void step_keyed(MarketSim& sim, uint64_t seed, uint32_t market_id) {  // the second half
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t step = sim.step_counter;
    sim.n_instructions += sim.env.transactions.size();
    sim.env.step_with([&](std::vector<MarketEnv::MarketEvent>& tx) {
        for (size_t i = tx.size(); i > 1; --i) {  // Fisher-Yates from the back, one Philox word per position
            const uint32_t idx = (uint32_t)(i - 1);
            const Philox4 r = philox4x32_10(market_id, step, PHILOX_SLOT_SHUFFLE, idx >> 2, k0, k1);
            std::swap(tx[i - 1], tx[mulhi_range(r.v[idx & 3], (uint32_t)i)]);
        }
    });
    ++sim.step_counter;
}
}  // namespace

MKS_API const char* mks_last_error(void) { return last_error.c_str(); }
// 0, or -1 when an agent's limit price was off its book's tick (the reference agents panic; as orc_market_run)
MKS_API int mks_agents_update(void* m, uint64_t seed, uint32_t market_id) {
    try {
        agents_update_keyed(((MarketHandle*)m)->sim, seed, market_id);
    } catch (const PriceError& e) {
        last_error = e.what();
        return -1;
    }
    return 0;
}
// 0, or -2 when an event names an order id the book never issued (as orc_market_step)
MKS_API int mks_step_keyed(void* m, uint64_t seed, uint32_t market_id) {
    try {
        step_keyed(((MarketHandle*)m)->sim, seed, market_id);
    } catch (const std::out_of_range&) {
        return -2;
    }
    return 0;
}
