"""The loop of vector_env_torch.py, plus what a learner needs for a reward: the fills of its own orders.  A (random) torch
policy trades against 100 background RandomAgents in each of 4096 envs; after every step `trades(cap)` hands over the
trades each env logged during the step, `orders(...)` on their order ids tells which side of each trade was the learner's
(its trader id) and whether it bought or sold, and the learner's inventory and cash per env are kept in torch.  Nothing
crosses PCIe inside the loop.  At the end the totals of a sample of envs are checked against the host reads
(`get_trades` / `get_orders`).

    python examples/vector_env_fills_torch.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bourse_b200 import abi, core, gym  # noqa: E402

N_ENVS, ROWS, CAP, LEARNER = 4096, 4, 64, 1000
env = gym.VectorEnv(N_ENVS, ROWS, seed=0, start_time=0, tick_size=1, step_size=1_000_000, max_queue=128, max_orders=16384,
                    max_trades=16384, max_steps=256,
                    agents=[core.random_group(50, (40, 60), (10, 20), 2, 0.8), core.random_group(50, (10, 90), (50, 70), 2, 0.2)],
                    agent_seed=101)
stream = torch.cuda.Stream()   # the env's launches and the torch code below share one stream
torch.cuda.set_stream(stream)
env.env.set_stream(stream.cuda_stream)
obs = torch.as_tensor(env.reset(), device="cuda")
actions = torch.zeros((N_ENVS, ROWS, 8), dtype=torch.int32, device="cuda")
inventory = torch.zeros(N_ENVS, dtype=torch.int64, device="cuda")   # units bought - units sold
cash = torch.zeros(N_ENVS, dtype=torch.int64, device="cuda")        # price x volume received - paid


def book_fills():
    """Fold the trades logged since the last call into the learner's inventory and cash; returns the per-env counts."""
    cols, count = env.trades(CAP)
    t = {k: torch.as_tensor(v, device="cuda") for k, v in cols.items()}
    # both sides of every trade in one query block: [N_ENVS, 2 * CAP].  Unused slots hold NO_ID, which reads as "no order"
    # (trader 0), so they drop out below.
    ids = torch.cat([t["active_id"].view(torch.int64), t["passive_id"].view(torch.int64)], dim=1)
    o = env.orders(ids)
    trader = torch.as_tensor(o["trader"], device="cuda").view(torch.int32)
    bid = torch.as_tensor(o["side_is_bid"], device="cuda").bool()
    vol = t["vol"].view(torch.int32).long().repeat(1, 2)
    price = t["price"].view(torch.int32).long().repeat(1, 2)
    signed = torch.where(bid, vol, -vol) * (trader == LEARNER)
    inventory.add_(signed.sum(1))
    cash.sub_((signed * price).sum(1))
    return torch.as_tensor(count, device="cuda").view(torch.int32)


gen = torch.Generator(device="cuda").manual_seed(0)
for step in range(100):
    mid = ((obs[:, 1].long() + obs[:, 2].long()) // 2).clamp(40, 160)        # quote around the mid price (bid, ask = words 1, 2)
    side = torch.randint(0, 2, (N_ENVS, ROWS), device="cuda", generator=gen)
    off = torch.randint(0, 6, (N_ENVS, ROWS), device="cuda", generator=gen)
    price = ((mid[:, None] + torch.where(side == 1, -off, off)) // 2 * 2)    # on the agents' tick grid
    actions[:, :, 2] = (abi.OP_NEW | torch.where(side == 1, abi.F_BID, 0)).int()
    actions[:, :, 4] = price.int()
    actions[:, :, 5] = 5
    actions[:, :, 6] = LEARNER
    env.step(actions)                                                        # one launch: agents + these rows + Env::step
    book_fills()                                                             # two launches: trades, then orders
while (book_fills() > CAP).any():   # a step that logged more than CAP trades left the rest for later calls
    pass
stream.synchronize()
env.check_errors()

# the same totals from the host reads of a sample of envs
for e in range(0, N_ENVS, N_ENVS // 16):
    orders = env.env.get_orders(e)
    inv = csh = 0
    for (_, _, price, vol, active, passive) in env.env.get_trades(e):
        for oid in (active, passive):
            if orders[oid][7] == LEARNER:
                signed = vol if orders[oid][0] else -vol
                inv, csh = inv + signed, csh - signed * price
    assert (inv, csh) == (int(inventory[e]), int(cash[e])), (e, inv, csh, int(inventory[e]), int(cash[e]))
print("learner inventory (mean |units|):", inventory.abs().float().mean().item(), "| cash of env 0:", int(cash[0]),
      "| inventory of env 0:", int(inventory[0]))
print("device fills match the host reads of 16 sampled envs")
print(env.env.stats())
