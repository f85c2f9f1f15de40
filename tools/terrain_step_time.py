"""What a heightfield ground costs: the fused DyrosDynamicWalk step at 4096 envs (default task, CUDA graph) on six
grounds, and what the height scan adds on the generated terrain, timed alternately in one process with the L2 flushed between timed steps (dyros_flush_l2, as bench.py does):
  plane      the plane z = 0 (the default build path)
  flat       a heightfield of zeros (same contacts as the plane, heightfield code path)
  rough      uniform heights in [-5 cm, +5 cm] at 0.1 m spacing
  stairs     5 cm steps every 0.3 m along x (0.05 m spacing)
  generated  the terrain generator's default grid (isaacgymdyros_b200/terrain.py: 10 levels x 20 types of 8 m, 0.1 m
             spacing), envs fixed on their sub-terrains (terrain curriculum: False)
  curriculum the same field with the terrain curriculum: levels move on every reset
  scan       the curriculum row with measure_heights (legged_gym's 187-point height scan appended to the observation)
The first four fields cover the default env grid (T:709-718); the envs stand on them at their origins. Also prints the per-phase
clock64() breakdown of the physics kernel (CTA 0, per role; marks of physics_roles.cuh, as tools/trace_physics.py)
and the card's name and power limit, and times the fused post-physics launch alone (dyros_task_post_step, L2 flushed
before each) for the curriculum and scan rows: the kernel the scan runs in. TOCABI's roles: 0 torso + left arm, 1 head + right arm + base, 2 left leg,
3 right leg (only the two legs have contact phases).
With --critic-states it times instead, alternating, with the L2 flushed before each timed step and back to back, the
fused step and the post-physics launch alone of
  plane         the plane, no critic states
  plane+states  the plane with criticStates (state rows of 518 floats)
  scan          the curriculum with the height scan in the observation (rows of 674 floats), no critic states
  scan+states   the same with criticStates: a blind 487-float observation and state rows of 705 floats
Usage: python tools/terrain_step_time.py [--envs 4096] [--steps 60] [--rounds 5] [--critic-states] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg  # noqa: E402
from isaacgymdyros_b200.core import env_origins  # noqa: E402

# phases of one sub-step of a role (mark ids of physics_roles.cuh): name, from, to
PHASES = [("pass 1", 0, 1), ("pass 2", 2, 4), ("feet part 1 + plane candidates", 4, 5), ("pass 3", 5, 6),
          ("contact rows (+ heightfield candidates)", 6, 7), ("sweeps", 7, 8), ("impulse, down pass, integration", 8, 12)]


def field(kind, N, spacing=5.0):
    o = env_origins(N, spacing)
    x0, y0 = o[:, 0].min() - 3.0, o[:, 1].min() - 3.0
    size = max(o[:, 0].max() - x0, o[:, 1].max() - y0) + 3.0
    dx = 0.05 if kind == "stairs" else 0.1
    n = int(np.ceil(size / dx)) + 1
    vs = 0.005
    if kind == "flat":
        s = np.zeros((n, n), np.int16)
    elif kind == "rough":
        s = np.random.default_rng(0).integers(-10, 11, (n, n)).astype(np.int16)  # +-5 cm
    else:
        x = x0 + dx * np.arange(n)
        s = np.repeat((np.floor((x - x0) / 0.3) * 10).astype(np.int16)[:, None], n, 1)  # 5 cm per 0.3 m
    return {"samples": s, "row_scale": dx, "column_scale": dx, "vertical_scale": vs, "origin": (float(x0), float(y0), 0.0)}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "unknown"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--out", default=None)
    ap.add_argument("--critic-states", action="store_true", help="time the critic state rows (DESIGN.md section 4)")
    a = ap.parse_args()
    N = a.envs
    name, power = card()
    print(f"card: {name}; power limit, max SM clock: {power}", flush=True)
    if a.critic_states:
        return critic_states(a, name, power)
    kinds = ["plane", "flat", "rough", "stairs", "generated", "curriculum", "scan"]
    envs = {}
    for k in kinds:
        cfg = default_cfg(N)
        if k in ("generated", "curriculum", "scan"):
            cfg["env"]["terrain"] = {"curriculum": k != "generated", "measure_heights": k == "scan"}
        elif k != "plane":
            cfg["env"]["heightfield"] = field(k, N)
        envs[k] = DyrosDynamicWalk(cfg, "cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator(device="cuda:0")
    g.manual_seed(1)
    acts = [torch.rand(N, 13, device="cuda:0", generator=g) * 2 - 1 for _ in range(8)]
    for k in kinds:
        for i in range(a.warmup):
            envs[k].step(acts[i % 8])
    torch.cuda.synchronize()
    times = {k: [] for k in kinds}
    for r in range(a.rounds):
        for k in kinds:  # alternating: the grounds see the same machine state
            env = envs[k]
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
            for i in range(a.steps):
                env.core.flush_l2(flush, i)
                ev[i][0].record()
                env.step(acts[i % 8])
                ev[i][1].record()
            torch.cuda.synchronize()
            times[k] += [e0.elapsed_time(e1) for e0, e1 in ev]
    # the post-physics launch alone (after the step timings: it advances the envs without physics)
    post = {k: [] for k in ("curriculum", "scan")}
    for r in range(a.rounds):
        for k in post:
            core = envs[k].core
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
            for i in range(a.steps):
                core.flush_l2(flush, i)
                ev[i][0].record()
                core.post_step()
                ev[i][1].record()
            torch.cuda.synchronize()
            post[k] += [e0.elapsed_time(e1) for e0, e1 in ev]
    # phase breakdown: clock64() marks of the physics launch of CTA 0 (a separate, traced launch)
    phases = {}
    for k in kinds:
        core = envs[k].core
        acc = np.zeros((len(PHASES), 4))
        reps = 20
        for _ in range(reps):
            core.flush_l2(flush, 0)
            tr = core.task_physics_trace().cpu().numpy().astype(np.float64)  # (skipframe, roles, 32)
            for p, (_n, m0, m1) in enumerate(PHASES):
                # (a role without a foot never writes marks 7 and 8: its contact phases stay empty)
                d = np.where((tr[:, :, m0] > 0) & (tr[:, :, m1] > 0), tr[:, :, m1] - tr[:, :, m0], np.nan)
                acc[p] += d.mean(0)
        phases[k] = {n: [None if np.isnan(c) else round(float(c), 0) for c in acc[p] / reps]
                     for p, (n, _m0, _m1) in enumerate(PHASES)}
    res = {"card": name, "power_limit_and_max_sm_clock": power, "envs": N, "steps_per_round": a.steps, "rounds": a.rounds,
           "l2": "flushed between timed steps (dyros_flush_l2, 256 MiB)",
           "launch_info": {k: envs[k].core.launch_info() for k in kinds}, "step_ms": {}, "phase_cycles_per_substep_by_role": phases}
    for k in kinds:
        t = np.array(times[k])
        res["step_ms"][k] = {"median": round(float(np.median(t)), 4), "p10": round(float(np.percentile(t, 10)), 4),
                             "p90": round(float(np.percentile(t, 90)), 4),
                             "round_medians": [round(float(np.median(t[i * a.steps:(i + 1) * a.steps])), 4) for i in range(a.rounds)],
                             "Menv_steps_per_s": round(N / np.median(t) / 1e3, 2)}
    res["post_step_ms"] = {k: {"median": round(float(np.median(v)), 4), "p10": round(float(np.percentile(v, 10)), 4),
                               "p90": round(float(np.percentile(v, 90)), 4)} for k, v in post.items()}
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


def critic_states(a, name, power):
    N = a.envs
    kinds = {"plane": (None, None), "plane+states": (None, True),
             "scan": ({"curriculum": True, "measure_heights": True}, None),
             "scan+states": ({"curriculum": True, "measure_heights": True}, True)}
    envs = {}
    for k, (terrain, cs) in kinds.items():
        cfg = default_cfg(N)
        if terrain is not None:
            cfg["env"]["terrain"] = dict(terrain)
        if cs is not None:
            cfg["env"]["criticStates"] = cs
        envs[k] = DyrosDynamicWalk(cfg, "cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator(device="cuda:0")
    g.manual_seed(1)
    acts = [torch.rand(N, 13, device="cuda:0", generator=g) * 2 - 1 for _ in range(8)]
    for k in kinds:
        for i in range(a.warmup):
            envs[k].step(acts[i % 8])
    torch.cuda.synchronize()
    modes = [(what, flushed) for what in ("step", "post") for flushed in (True, False)]
    times = {(k, w, f): [] for k in kinds for w, f in modes}
    for r in range(a.rounds):
        for w, f in modes:
            for k in kinds:  # alternating
                env = envs[k]
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
                for i in range(a.steps):
                    if f:
                        env.core.flush_l2(flush, i)
                    ev[i][0].record()
                    env.step(acts[i % 8]) if w == "step" else env.core.post_step()
                    ev[i][1].record()
                torch.cuda.synchronize()
                times[(k, w, f)] += [e0.elapsed_time(e1) for e0, e1 in ev]
    res = {"card": name, "power_limit_and_max_sm_clock": power, "envs": N, "steps_per_round": a.steps, "rounds": a.rounds,
           "widths": {k: {"obs": envs[k].num_obs, "states": envs[k].num_states} for k in kinds}, "ms": {}}
    print(f"\n| env | obs | states | L2 | step ms (median, p10-p90) | post-physics launch ms (median, p10-p90) |")
    print("|---|---|---|---|---|---|")
    for f in (True, False):
        for k in kinds:
            row = {}
            for w in ("step", "post"):
                t = np.array(times[(k, w, f)])
                row[w] = {"median": round(float(np.median(t)), 4), "p10": round(float(np.percentile(t, 10)), 4),
                          "p90": round(float(np.percentile(t, 90)), 4)}
            res["ms"][f"{k}, {'flushed' if f else 'back to back'}"] = row
            fmt = lambda d: f"{d['median']:.4f} ({d['p10']:.4f}-{d['p90']:.4f})"
            print(f"| {k} | {envs[k].num_obs} | {envs[k].num_states} | {'flushed' if f else 'back to back'} | "
                  f"{fmt(row['step'])} | {fmt(row['post'])} |")
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    for e in envs.values():
        e.close()


if __name__ == "__main__":
    main()
