"""Epoch time of the on-device PPO on the plane (487 observation columns) and on curriculum terrain with the height scan
(terrain measure_heights, 674 columns), in one process, alternating, split into rollout and update; then the library
kernels of the first-layer GEMMs of both widths under torch.profiler (source of profiles/ppo_terrain.md).

With --critic-states the two trainers are instead the 674-wide perceptive one (actor and critic read the observation row
with the heights) and the blind-actor one (criticStates: a 487-input actor, a 705-input critic on the state rows,
PPOConfig(num_states=705)), both on curriculum terrain.

    python tools/ppo_terrain_time.py [--epochs 10] [--trace-dir DIR] [--critic-states]"""
import argparse, subprocess, sys, time
import torch
sys.path.insert(0, '.')
from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer

ap = argparse.ArgumentParser()
ap.add_argument("--epochs", type=int, default=10, help="timed epochs per env, alternating")
ap.add_argument("--trace-dir", default=None, help="also write the torch.profiler traces there")
ap.add_argument("--critic-states", action="store_true", help="perceptive (674) against blind actor + critic states (487 / 705)")
args = ap.parse_args()
N = 4096
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else 'n/a'}")


def make(terrain: bool, states: bool = False):
    cfg = default_cfg(N)
    if terrain:
        cfg["env"]["terrain"] = {"curriculum": True, "measure_heights": True, "seed": 2}
    if states:
        cfg["env"]["criticStates"] = True
    env = DyrosDynamicWalk(cfg, "cuda:0", use_cuda_graph=False)
    return env, PPOTrainer(env, PPOConfig(num_obs=env.num_obs, num_states=env.num_states if states else 0))


runs = ({"perceptive": make(True), "blind+states": make(True, True)} if args.critic_states
        else {"plane": make(False), "terrain": make(True)})


# ---- the first-layer GEMMs (eager: the same shapes and library calls the CUDA graphs capture)
def gemm_kernels(tr):
    """{(role, kernel name): [us per call]} of the bmm calls whose operands are K0 wide."""
    K0 = tr.packed.K0
    for _ in range(2):                                      # warm-up: library heuristics and workspaces
        tr._rollout_step(); tr._minibatch(0)
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts, record_shapes=True) as prof:
        for _ in range(3):
            tr._rollout_step(); tr._minibatch(0)
        torch.cuda.synchronize()
    if args.trace_dir:
        prof.export_chrome_trace(f"{args.trace_dir}/ppo_gemms_K0_{K0}.pt.trace.json")

    def kernels(e):
        out = list(e.kernels)
        for c in e.cpu_children:
            out += kernels(c)
        return out
    table = prof.key_averages().table(sort_by="self_device_time_total", row_limit=12)
    print("\n".join(l for l in table.splitlines() if l.strip()))
    res = {}
    for e in prof.events():
        if e.name != "aten::bmm" or not e.input_shapes or len(e.input_shapes[0]) != 3:
            continue
        a, b = e.input_shapes[0], e.input_shapes[1]
        if a[-1] == K0:                                     # (the rollout's N and the minibatch are both 4096 rows here)
            role = f"forward x W0^T ({a[1]} x {K0} . {K0} x 256, x2)"
        elif b[-1] == K0:
            role = f"update backward dW0 = d0^T x (256 x {a[-1]} . {a[-1]} x {K0}, x2)"
        else:
            continue
        for k in kernels(e):
            res.setdefault((role, k.name), []).append(k.duration)
    return res


for name, (env, tr) in runs.items():
    print(f"\n## first-layer GEMMs, {name}: W = {env.num_obs}, K0 = {tr.packed.K0}")
    for (role, kname), d in sorted(gemm_kernels(tr).items()):
        print(f"- {role}: `{kname}` {sum(d) / len(d):.1f} us per call ({len(d)} calls)")


# ---- epoch time, alternating (CUDA graphs on: PPOTrainer's default)
def timed_epoch(tr):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    r, u = tr.rollout, tr.update
    tr.rollout = lambda: (ev[0].record(), r(), ev[1].record())
    tr.update = lambda: (u(), ev[2].record())
    t0 = time.perf_counter()
    out = tr.train_epoch()                                  # ends in its one device->host read
    wall = time.perf_counter() - t0
    del tr.rollout, tr.update
    return wall * 1e3, ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), out


for name, (env, tr) in runs.items():                        # graph capture + warm-up
    for _ in range(2):
        timed_epoch(tr)
times = {k: [] for k in runs}
for i in range(args.epochs):
    for name, (env, tr) in runs.items():
        times[name].append(timed_epoch(tr))
print(f"\n## epoch time, {N} envs x 128 steps, 5 mini-epochs x 128 minibatches of 4096 rows, {args.epochs} epochs each, alternating")
print("| env | W | K0 | epoch wall ms (median, min-max) | rollout ms (median) | update ms (median) | M env-steps/s |")
print("|---|---|---|---|---|---|---|")
for name, (env, tr) in runs.items():
    t = times[name]
    med = lambda xs: sorted(xs)[len(xs) // 2]
    w = [x[0] for x in t]
    print(f"| {name} | {env.num_obs} | {tr.packed.K0} | {med(w):.1f} ({min(w):.1f}-{max(w):.1f}) | {med([x[1] for x in t]):.1f} | "
          f"{med([x[2] for x in t]):.1f} | {N * 128 / med(w) / 1e3:.2f} |")
print("\nlast epoch outputs:", {k: {kk: round(v, 4) for kk, v in times[k][-1][3].items()} for k in runs})
for env, tr in runs.values():
    env.close()
