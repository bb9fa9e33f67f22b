"""The PPO loop of train_ppo_puzzle8.py, trained on rank 0 from the episodes of every GPU: each rank collects its shard of
the 4096 * W episodes on its own GPU and rank 0 receives all of them (`dist.ShardedCollector`, one NCCL gather) as torch
CUDA tensors; the other ranks only serve.  Not part of the product path.

    torchrun --nproc-per-node W examples/train_ppo_sharded.py [iterations]
"""
import os
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import twisterl_b200 as tw
from twisterl_b200 import dist as twd
from train_ppo_puzzle8 import TorchPolicy


def main(iters=60):
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.manual_seed(0)
    # one engine per process, shared by the collect and (on rank 0) the evaluation
    tw.configure(device=local, precision="f16x2", seed=1, rank=rank, world=world)
    comm = twd.Comm(tw.default_engine())
    env = tw.env.Puzzle(3, 3, 1, 2, 256)
    collector = tw.collector.PPOCollector(num_episodes=4096 * world, gamma=0.995, num_cores=32, **{"lambda": 0.995})
    sharded = twd.ShardedCollector(collector, comm)
    if rank != 0:
        rs = TorchPolicy().to_engine()             # its weights are replaced by rank 0's every iteration
        n = sharded.serve(env, rs)
        print(f"rank {rank}: served {n} iterations", flush=True)
        comm.close()
        return None
    dev = torch.device("cuda", local)
    policy = TorchPolicy().to(dev)
    opt = torch.optim.Adam(policy.parameters(), lr=1.5e-4)
    rs = policy.to_engine()
    t0 = time.time()
    try:
        for it in range(iters):
            rs.update_from_torch(policy)
            succ, rew = tw.collector.evaluate(env, rs, 256, False, 1, 0, 0, 1.41, 1, 32)
            data = sharded.collect_torch(env, rs)          # every rank's episodes, on this GPU
            obs, logits, acts, rets, advs = data["obs"], data["logits"], data["actions"], data["rets"], data["advs"]
            advs = (advs - advs.mean()) / (advs.std() + 1e-8)
            old_lp = torch.distributions.Categorical(logits=logits).log_prob(acts)
            illegal = logits <= -1e9
            for _ in range(10):
                pl, pv = policy(obs)
                dist = torch.distributions.Categorical(logits=pl.masked_fill(illegal, -1e10))
                ratio = torch.exp(dist.log_prob(acts) - old_lp)
                loss = (-torch.min(ratio * advs, torch.clamp(ratio, 0.9, 1.1) * advs).mean()
                        + 0.8 * torch.nn.functional.mse_loss(pv.squeeze(1), rets) - 0.01 * dist.entropy().mean())
                opt.zero_grad(); loss.backward(); opt.step()
            print(f"it {it:3d} difficulty {env.difficulty:2d} success {succ:.2f} reward {rew:+.3f} episodes "
                  f"{data['stats']['episodes']} records {len(acts)} loss {loss.item():+.4f} ({time.time() - t0:.1f}s)", flush=True)
            if succ >= 0.85 and env.difficulty < 32:
                env.difficulty = env.difficulty + 1
    finally:
        sharded.close()                                    # the other ranks leave serve()
    comm.close()
    return env.difficulty


if __name__ == "__main__":
    d = main(int(sys.argv[1]) if len(sys.argv) > 1 else 60)
    if d is not None:
        print("final difficulty", d)
