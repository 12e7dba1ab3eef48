// Test infrastructure: bb_set_agent_params_device restated on the oracle's own objects (oracle/env.hpp) — the parameters of
// agent group gi of an Env / MarketEnv overwritten in place, from a bb_agent_group record converted as the oracle's C API
// converts it at set_groups.  The agents' state (held orders, MomentumAgent momentum and last price, live-order lists) is
// left as it is, as on the device, where the parameters are configuration read at every step.
//
// The oracle's C API is compiled in (for its SimHandle / MarketHandle and orc_group); every symbol of this library is hidden
// except the aps_* calls.  It operates on handles liboracle created (oracle.StepEnv._h, oracle.MarketEnv._h): both libraries
// are built from the same headers with the same flags.
#include "../../oracle/oracle_capi.cpp"

#define APS_API extern "C" __attribute__((visibility("default")))

namespace {
// the group's parameters replaced; 0, or -1 when gi names no group or the record's kind is not the group's
template <class S> int set_group(S& sim, GroupKind kind, size_t idx, const orc_group& g) {
    if ((uint32_t)kind != g.kind) return -1;
    if (kind == GROUP_RANDOM)
        sim.randoms[idx].p = RandomAgentsParams{g.n_agents, g.tick_lo, g.tick_hi, g.vol_lo, g.vol_hi, g.tick_size, g.rate};
    else if (kind == GROUP_MOMENTUM)
        sim.momentums[idx].p = MomentumParams{g.tick_lo, g.n_agents, g.tick_size, g.rate, g.vol_lo, g.decay, g.demand, g.scale,
                                              g.order_ratio, g.mu, g.sigma};
    else  // NoiseAgent: p_limit / p_market travel in the decay / demand slots
        sim.noises[idx].p = NoiseParams{g.tick_lo, g.n_agents, g.tick_size, (float)g.decay, (float)g.demand, g.rate, g.vol_lo, g.mu, g.sigma};
    return 0;
}
}  // namespace

APS_API int aps_sim_set_group(void* s, uint32_t gi, const orc_group* g) {
    Sim& sim = ((SimHandle*)s)->sim;
    if (gi >= sim.order.size()) return -1;
    return set_group(sim, sim.order[gi].first, sim.order[gi].second, *g);
}

APS_API int aps_market_set_group(void* m, uint32_t gi, const orc_group* g) {
    MarketSim& sim = ((MarketHandle*)m)->sim;
    if (gi >= sim.order.size()) return -1;
    return set_group(sim, sim.order[gi].kind, sim.order[gi].idx, *g);
}
