"""What a triangle-mesh ground costs: the fused DyrosDynamicWalk step at 4096 envs (default task, CUDA graph) on the same
grounds as a heightfield and as legged_gym's trimesh of that heightfield (terrain.convert_heightfield_to_trimesh with
slope_treshold 0.75), timed alternately in one process, with the L2 flushed between timed steps (dyros_flush_l2, as
bench.py does) and back to back:
  plane                   the plane z = 0
  field/mesh flat         zeros at 0.1 m spacing
  field/mesh rough        uniform heights in [-5 cm, +5 cm] at 0.1 m spacing
  field/mesh stairs       5 cm steps every 0.3 m along x at 0.05 m spacing (the mesh's risers are vertical walls)
  field/mesh curriculum   the generator's default terrain (10 x 20 sub-terrains of 8 m, 1300 x 2100 samples) with the
                          terrain curriculum; the mesh arm is cfg["env"]["terrainMesh"]
For every mesh it also records the registration (dyros_sim_set_triangle_mesh: copy, grid build, upload; host wall clock,
re-registered on the live sim) and dyros_sim_triangle_mesh_info (device bytes, triangles kept and dropped, buckets), and
the card's name and power limit.
Usage: python tools/trimesh_step_time.py [--envs 4096] [--steps 60] [--rounds 5] [--out FILE.json]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg, native, terrain  # noqa: E402
from isaacgymdyros_b200.core import HeightField  # noqa: E402
from isaacgymdyros_b200.tasks import dyros_dynamic_walk as task  # noqa: E402
from tools.terrain_step_time import card, field  # noqa: E402


def make_env(cfg, mesh):
    """The task with cfg's heightfield, or (mesh) with that heightfield's trimesh as the ground."""
    if not mesh or "heightfield" not in cfg["env"]:
        return DyrosDynamicWalk(cfg, "cuda:0")
    base = task.core_config_from_cfg

    def to_mesh(cfg_, generator=None):
        c = base(cfg_, generator)
        hf = c.heightfield
        tm = terrain.trimesh_from_field(HeightField(hf.samples, hf.row_scale, hf.column_scale, hf.vertical_scale,
                                                    hf.origin, hf.friction), 0.75)
        c.heightfield, c.triangle_mesh = None, tm
        return c
    task.core_config_from_cfg = to_mesh
    try:
        return DyrosDynamicWalk(cfg, "cuda:0")
    finally:
        task.core_config_from_cfg = base


def reregister(core):
    """Host wall clock of dyros_sim_set_triangle_mesh on the live sim (the same mesh again)."""
    tm = core.cfg.triangle_mesh
    v = np.ascontiguousarray(tm.vertices, np.float32)
    t = np.ascontiguousarray(tm.triangles, np.uint32)
    d = native.DyrosTriangleMesh()
    d.vertices, d.triangles, d.num_vertices, d.num_triangles = v.ctypes.data, t.ctypes.data, len(v), len(t)
    d.origin = (C.c_float * 3)(*tm.origin)
    d.dynamic_friction = core.cfg.friction
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    native.check(core.lib.dyros_sim_set_triangle_mesh(core.sim_handle, C.byref(d)), "dyros_sim_set_triangle_mesh")
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    N = a.envs
    name, power = card()
    print(f"card: {name}; power limit, max SM clock: {power}", flush=True)
    arms = ["plane"] + [f"{g} {k}" for k in ("flat", "rough", "stairs", "curriculum") for g in ("field", "mesh")]
    envs, reg = {}, {}
    for arm in arms:
        cfg = default_cfg(N)
        kind = arm.split()[-1]
        if kind == "curriculum":
            cfg["env"]["terrain"] = {"curriculum": True}
            cfg["env"]["terrainMesh"] = arm.startswith("mesh")
        elif kind != "plane":
            cfg["env"]["heightfield"] = field(kind, N)
        t0 = time.perf_counter()
        envs[arm] = make_env(cfg, arm.startswith("mesh"))
        built = time.perf_counter() - t0
        core = envs[arm].core
        if core.mesh_info is not None:
            reg[arm] = dict(core.mesh_info, env_build_s=round(built, 2), register_s=round(reregister(core), 3))
            print(arm, reg[arm], flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.Generator(device="cuda:0")
    g.manual_seed(1)
    acts = [torch.rand(N, 13, device="cuda:0", generator=g) * 2 - 1 for _ in range(8)]
    for arm in arms:
        for i in range(a.warmup):
            envs[arm].step(acts[i % 8])
    torch.cuda.synchronize()
    times = {(arm, l2): [] for arm in arms for l2 in ("flushed", "warm")}
    for r in range(a.rounds):
        for l2 in ("flushed", "warm"):
            for arm in arms:  # alternating: the grounds see the same machine state
                env = envs[arm]
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
                for i in range(a.steps):
                    if l2 == "flushed":
                        env.core.flush_l2(flush, i)
                    ev[i][0].record()
                    env.step(acts[i % 8])
                    ev[i][1].record()
                torch.cuda.synchronize()
                times[(arm, l2)] += [e0.elapsed_time(e1) for e0, e1 in ev]
    res = {"card": name, "power_limit_and_max_sm_clock": power, "envs": N, "steps_per_round": a.steps, "rounds": a.rounds,
           "registration": reg, "step_ms": {}}
    for arm in arms:
        res["step_ms"][arm] = {}
        for l2 in ("flushed", "warm"):
            t = np.array(times[(arm, l2)])
            res["step_ms"][arm][l2] = {"median": round(float(np.median(t)), 4), "p10": round(float(np.percentile(t, 10)), 4),
                                       "p90": round(float(np.percentile(t, 90)), 4)}
        ro = envs[arm].core.sim_t["root_states"]
        res["step_ms"][arm]["finite"] = bool(torch.isfinite(ro).all())
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
