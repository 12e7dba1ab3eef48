"""Episodes that start from a warm book: device-resident snapshots (`snapshots`, `save`, `restore`).  4096 envs with the C3
population (50 + 50 background RandomAgents each) warm up for a few hundred steps; a handful of their states are saved into
a device store.  The loop then runs per-env episodes of random length against a (random) torch policy, and the envs whose
episode ended are restored from slot `env % n_slots` with fresh seeds, so every episode starts with resting liquidity, a
spread and a price instead of the empty book `reset(mask)` gives, and each env's shuffles differ from its slot's source.
For comparison the same loop then runs with `reset(done)`.  Nothing crosses PCIe inside either loop.

    python examples/vector_env_warm_start_torch.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bourse_b200 import abi, gym, workloads  # noqa: E402

N_ENVS, ROWS, WARMUP, STEPS, MAX_STEPS, N_SLOTS = 4096, 4, 300, 200, 64, 8
env = gym.VectorEnv(N_ENVS, ROWS, seed=0, start_time=0, tick_size=1, step_size=1_000_000, max_queue=128, max_orders=16384,
                    max_trades=16384, max_steps=MAX_STEPS, agents=workloads.c3_groups(), agent_seed=7)
stream = torch.cuda.Stream()   # the env's launches and the torch code below share one stream
torch.cuda.set_stream(stream)
env.env.set_stream(stream.cuda_stream)
gen = torch.Generator(device="cuda").manual_seed(0)
actions = torch.zeros((N_ENVS, ROWS, 8), dtype=torch.int32, device="cuda")
idle = torch.zeros((N_ENVS, ROWS, 8), dtype=torch.int32, device="cuda")   # OP_NOOP rows: the agents alone


def depth(obs):
    """Resting volume on both sides of each book (level-2 words 3 and 4: ask and bid volume)."""
    return obs[:, 3].long() + obs[:, 4].long()


def policy(obs):
    mid = ((obs[:, 1].long() + obs[:, 2].long()) // 2).clamp(40, 160)   # quote around the mid price (bid, ask = words 1, 2)
    side = torch.randint(0, 2, (N_ENVS, ROWS), device="cuda", generator=gen)
    off = torch.randint(0, 6, (N_ENVS, ROWS), device="cuda", generator=gen)
    actions[:, :, 2] = (abi.OP_NEW | torch.where(side == 1, abi.F_BID, 0)).int()
    actions[:, :, 4] = ((mid[:, None] + torch.where(side == 1, -off, off)) // 2 * 2).int()   # on the agents' tick grid
    actions[:, :, 5] = 5
    actions[:, :, 6] = 1000
    return actions


env.reset()
for _ in range(WARMUP):
    env.step(idle)
store = env.snapshots(N_SLOTS)
env.save(store, torch.arange(N_SLOTS, dtype=torch.int32, device="cuda") * (N_ENVS // N_SLOTS))   # a handful of warm states
env_ids = torch.arange(N_ENVS, device="cuda")


def run(warm: bool):
    """Per-env episodes; returns (episodes completed, mean resting depth of the books episodes started from)."""
    obs = torch.as_tensor(env.restore(store, (env_ids % N_SLOTS).int()) if warm else env.reset(), device="cuda")
    horizon = torch.randint(8, MAX_STEPS + 1, (N_ENVS,), device="cuda", generator=gen)
    t = torch.zeros(N_ENVS, dtype=torch.int64, device="cuda")
    episodes = torch.zeros((), dtype=torch.int64, device="cuda")
    start_depth = depth(obs).sum()
    starts = torch.full((), N_ENVS, dtype=torch.int64, device="cuda")
    for step in range(STEPS):
        env.step(policy(obs))
        t += 1
        done = t >= horizon
        episodes += done.sum()
        t.masked_fill_(done, 0)
        horizon = torch.where(done, torch.randint(8, MAX_STEPS + 1, (N_ENVS,), device="cuda", generator=gen), horizon)
        if warm:   # one launch per call: the ended episodes restart from a warm state with fresh seeds, the rest are untouched
            seeds = torch.randint(0, 2**62, (N_ENVS,), device="cuda", generator=gen)
            env.restore(store, torch.where(done, env_ids % N_SLOTS, gym.NO_SLOT).int(), seeds)
        else:
            env.reset(done)
        start_depth += torch.where(done, depth(obs), 0).sum()   # the rows restore / reset just wrote for the new episodes
        starts += done.sum()
    stream.synchronize()
    return int(episodes), int(start_depth) / int(starts)


n_warm, d_warm = run(True)
n_cold, d_cold = run(False)
env.check_errors()
print(f"warm start: {n_warm} episodes over {STEPS} steps of {N_ENVS} envs, mean resting depth at episode start {d_warm:.1f}")
print(f"empty-book reset: {n_cold} episodes, mean resting depth at episode start {d_cold:.1f}")
print(f"store: {N_SLOTS} slots, {store.nbytes / 2**20:.1f} MiB on the device")
print(f"error_envs: {env.env.stats()['error_envs']}")
env.close()
