"""2+ ranks: the peer-memory gradient exchange against NCCL all-reduce on identical rollouts: parameters after a few
minibatch updates must be equal (bitwise at 2 ranks: a + b in either order).
    torchrun --nproc-per-node 2 tools/ppo_peer_check.py [--terrain]
--terrain: the networks of the terrain env with the height scan (terrain measure_heights, 674 observation columns)."""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, '.')
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = f"cuda:{local}"
dist.init_process_group("nccl", device_id=torch.device(dev))
from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
terrain = "--terrain" in sys.argv[1:]
res = {}
for mode in ("nccl", "peer", "peer2"):
    cfg = default_cfg(256)
    if terrain:
        cfg["env"]["terrain"] = {"measure_heights": True, "seed": 2}
    env = DyrosDynamicWalk(cfg, dev, rank=rank, use_cuda_graph=False)
    tr = PPOTrainer(env, PPOConfig(horizon_length=8, minibatch_size=512, grad_sync=mode, use_cuda_graph=(mode != "nccl"),
                                   num_obs=env.num_obs), rank=rank, world=world)
    g = torch.Generator(device=dev); g.manual_seed(100 + rank)       # different data per rank, same in both modes
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    N, H = tr.N, tr.H
    tr.x_roll.copy_(r(N * H, tr.packed.K0).to(torch.bfloat16)); tr.x_roll[:, env.num_obs:] = 0
    b = tr.buf
    b["mus"].copy_(0.3 * r(N, H, 13)); b["actions"].copy_(b["mus"] + 0.12 * r(N, H, 13))
    b["neglogp"].copy_(13 * 0.9189385 + tr.net.logstd.sum() + 0.5 * (((b["actions"] - b["mus"]) / tr.net.logstd.exp()) ** 2).sum(-1) + 0.3 * r(N, H))
    b["values"].copy_(r(N, H)); b["returns"].copy_(b["values"] + r(N, H)); b["advantages"].copy_(b["returns"] - b["values"])
    tr.net.flat.copy_(tr.net.flat * 30); tr.packed.pack()
    dist.broadcast(tr.net.flat, 0); tr.packed.pack()
    tr.update()                                                       # mini_epochs x minibatches optimiser steps
    torch.cuda.synchronize()
    res[mode] = tr.net.flat.clone()
    all_p = [torch.empty_like(tr.net.flat) for _ in range(world)]
    dist.all_gather(all_p, tr.net.flat)
    same_across = all(torch.equal(all_p[0], p) for p in all_p)
    print(f"{rank} {mode} steps {int(tr.opt_step.item())} identical across ranks {same_across}\n", end="", flush=True)
    dist.barrier()
    if tr.peers is not None:
        tr.peers.close()
    env.close()
for mode in ("peer", "peer2"):
    d = (res[mode] - res["nccl"]).abs().max().item()
    print(f"{rank} {mode} vs nccl max |diff| {d} rel {d / res['nccl'].abs().max().item()}\n", end="", flush=True)
dist.barrier(); torch.cuda.synchronize()
os._exit(0)
