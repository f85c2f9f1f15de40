"""On-device PPO for a few hundred epochs on one GPU (4096 envs x 128 steps per epoch, the reference's hyper-parameters):
episode statistics every 20 epochs, plus a finite-state check of the env.

    python tools/ppo_learning_curve.py [epochs] [--terrain] [--critic-states]

--terrain trains on the generated sub-terrain grid with its curriculum and the height scan (terrain measure_heights:
674 observation columns, PPOConfig(num_obs=674)) and adds the mean terrain level to the table. With --critic-states the
heights go into the critic's state row only (criticStates): a blind 487-input actor and a privileged 705-input critic,
PPOConfig(num_states=705)."""
import argparse, sys, time, torch
sys.path.insert(0, '.')
from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
ap = argparse.ArgumentParser()
ap.add_argument("epochs", nargs="?", type=int, default=400)
ap.add_argument("--terrain", action="store_true", help="generated terrain, curriculum and measure_heights")
ap.add_argument("--critic-states", action="store_true", help="blind actor, privileged critic (criticStates)")
args = ap.parse_args()
E = args.epochs
cfg = default_cfg(4096)
if args.terrain:
    cfg["env"]["terrain"] = {"curriculum": True, "measure_heights": True, "seed": 2}
if args.critic_states:
    cfg["env"]["criticStates"] = True
env = DyrosDynamicWalk(cfg, "cuda:0", use_cuda_graph=False)
tr = PPOTrainer(env, PPOConfig(num_obs=env.num_obs, num_states=env.num_states if args.critic_states else 0))
where = "curriculum terrain with the height scan" if args.terrain else "the plane"
if args.critic_states:
    where += f", critic states ({env.num_states} columns, blind actor)"
print(f"# On-device PPO, one B200, 4096 envs x 128 steps per epoch on {where}, {env.num_obs} observation columns "
      "(DyrosDynamicWalkPPO.yaml hyper-parameters, self-collision on)\n")
lvl = args.terrain
print("| epoch | frames | mean episode reward | mean episode length | episodes ended |" + (" terrain level |" if lvl else "")
      + " actor loss | critic loss | kl | lr |")
print("|---|---|---|---|---|" + ("---|" if lvl else "") + "---|---|---|---|")
t0 = time.time()
for ep in range(1, E + 1):
    out = tr.train_epoch()
    if ep % 20 == 0 or ep == 1:
        print(f"| {ep} | {ep * 4096 * 128:,} | {out['mean_reward']:.1f} | {out['mean_length']:.1f} | {int(out['episodes'])} | "
              + (f"{out['terrain_level']:.2f} | " if lvl else "")
              + f"{out['a_loss']:.4f} | {out['c_loss']:.3f} | {out['kl']:.5f} | {out['lr']:.2e} |", flush=True)
torch.cuda.synchronize()
dt = time.time() - t0
finite = bool(torch.isfinite(env.core.sim_t["root_states"]).all() and torch.isfinite(env.core.sim_t["dof_state"]).all() and torch.isfinite(env.obs_buf).all())
print(f"\n{E} epochs = {E * 4096 * 128:,} env-steps in {dt:.1f} s wall ({E * 4096 * 128 / dt / 1e6:.2f} M env-steps/s including the host loop); "
      f"all env state finite at the end: {finite}.")
