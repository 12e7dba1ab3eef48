"""Episodes of different lengths in one batch: gymnasium-style per-env autoreset on the device.  A (random) torch policy
trades against 100 background RandomAgents in each of 4096 envs; every env ends its episode at its own horizon (drawn per
episode), and `reset(mask=done)` after every step restarts exactly the envs whose episodes ended, each with a fresh book,
a fresh history and its order table and trade log back at slot 0, while the others keep running.  The episode return here
is the traded volume the learner's env saw; it is read from the last observation before the reset overwrites it.  Nothing
crosses PCIe inside the loop.

    python examples/vector_env_episodes_torch.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bourse_b200 import abi, core, gym  # noqa: E402

N_ENVS, ROWS, STEPS, MAX_STEPS = 4096, 4, 400, 64
env = gym.VectorEnv(N_ENVS, ROWS, seed=0, start_time=0, tick_size=1, step_size=1_000_000, max_queue=128, max_orders=8192,
                    max_trades=8192, max_steps=MAX_STEPS,
                    agents=[core.random_group(50, (40, 60), (10, 20), 2, 0.8), core.random_group(50, (10, 90), (50, 70), 2, 0.2)],
                    agent_seed=7)
stream = torch.cuda.Stream()   # the env's launches and the torch code below share one stream
torch.cuda.set_stream(stream)
env.env.set_stream(stream.cuda_stream)
obs = torch.as_tensor(env.reset(), device="cuda")
actions = torch.zeros((N_ENVS, ROWS, 8), dtype=torch.int32, device="cuda")
gen = torch.Generator(device="cuda").manual_seed(0)
horizon = torch.randint(8, MAX_STEPS + 1, (N_ENVS,), device="cuda", generator=gen)   # each env's episode length
t = torch.zeros(N_ENVS, dtype=torch.int64, device="cuda")
ret = torch.zeros(N_ENVS, dtype=torch.int64, device="cuda")          # running return of each env's current episode
episodes = torch.zeros((), dtype=torch.int64, device="cuda")
returns = torch.zeros((), dtype=torch.int64, device="cuda")          # summed over completed episodes

for step in range(STEPS):
    mid = ((obs[:, 1].long() + obs[:, 2].long()) // 2).clamp(40, 160)   # quote around the mid price (bid, ask = words 1, 2)
    side = torch.randint(0, 2, (N_ENVS, ROWS), device="cuda", generator=gen)
    off = torch.randint(0, 6, (N_ENVS, ROWS), device="cuda", generator=gen)
    actions[:, :, 2] = (abi.OP_NEW | torch.where(side == 1, abi.F_BID, 0)).int()
    actions[:, :, 4] = ((mid[:, None] + torch.where(side == 1, -off, off)) // 2 * 2).int()   # on the agents' tick grid
    actions[:, :, 5] = 5
    actions[:, :, 6] = 1000
    env.step(actions)                                  # one launch: agents + these rows + Env::step
    ret += obs[:, 0].long()                            # this step's traded volume (word 0), read before the reset below
    t += 1
    done = t >= horizon
    episodes += done.sum()
    returns += torch.where(done, ret, 0).sum()
    ret.masked_fill_(done, 0)
    t.masked_fill_(done, 0)
    horizon = torch.where(done, torch.randint(8, MAX_STEPS + 1, (N_ENVS,), device="cuda", generator=gen), horizon)
    env.reset(done)                                    # one launch: the ended episodes restart, the rest are untouched
stream.synchronize()
env.check_errors()
n_ep = int(episodes)
print(f"episodes completed: {n_ep} over {STEPS} steps of {N_ENVS} envs, mean return (traded volume): {int(returns) / max(n_ep, 1):.1f}")
print("longest history of any env:", max(env.env.n_steps(e) for e in range(0, N_ENVS, 97)), f"(<= max_steps = {MAX_STEPS})")
print(f"error_envs: {env.env.stats()['error_envs']}")
