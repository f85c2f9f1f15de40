#!/usr/bin/env python
"""bench.py -- env-steps/s of the DyrosDynamicWalk hot path (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs 4096] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one VecTask.step of every env of the shard: PD/delay + 2 physics sub-steps + sensor noise +
termination + reward + reset + observations (SURVEY 8d). Envs shard across ranks with no data-path collective
(weak scaling: 4096 envs per GPU); NCCL is used for the barrier, the max-over-ranks timing and the episode statistics.

Prints ONE JSON line (rank 0). `value` is device-resident throughput with the L2 flushed between timed steps;
`e2e` goes through DyrosDynamicWalk.step_async / step_wait with pinned HOST buffers (actions read from pinned host memory
by the step's first kernel; obs / reward / reset / time_outs packed and moved device->host every step on a copy stream,
overlapping the next step's kernels); `e2e_sync` is DyrosDynamicWalk.step + copies on one stream, nothing overlapped.
`--impl reference` times the CPU oracle port (oracle/env_oracle.py) on the host cores: the reference's own physics
is closed-source PhysX whose binaries are absent from the checkout (SURVEY fact 2), so the "reference arm" is the port.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/s at 4096 envs/GPU"
UNIT = "env-steps/s"
WORKLOAD = "DyrosDynamicWalk 4096 envs/GPU, random actions, physics + PD + obs/reward/reset kernels (BASELINE configs[1])"
K1_BYTES_PER_ENV_STEP = 2 * 1648 + 2 * 1296   # per policy step: 2 x K1 sub-step (SURVEY 8d: 412 words) + 2 x (torque/delay ring + sensor noise: 324 words), DESIGN.md section 6
ENV_STEP_BYTES = 7044                # SURVEY 8d canonical bytes per env-step


def k1_profile():
    """Executed FP32 FLOP and DRAM bytes of ONE k_step_physics launch of the CURRENT build, per env: read from
    profiles/current.json, which tools/ncu_summary.py --json writes from the ncu --set full capture of this build
    (ffma*2 + fadd + fmul; dram__bytes_read + write with the caches flushed by ncu before the launch, as in the timed
    launches here). Returns (flop_per_env, dram_bytes_per_env, source) or (None, None, why)."""
    path = os.path.join(ROOT, "profiles", "current.json")
    try:
        d = json.load(open(path))["k_step_physics"]
        return d["flop"] / d["envs"], d["dram_bytes"] / d["envs"], f"profiles/{d['source']} ({d['envs']} envs, one launch)"
    except Exception as exc:  # noqa: BLE001
        return None, None, f"profiles/current.json unreadable: {exc}"



def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--envs", type=int, default=4096, help="envs per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--force-perturb", action="store_true", help="pushes forced on (BASELINE configs[3]; T:491)")
    ap.add_argument("--dr-extra", action="store_true",
                    help="also randomise friction x[0.7,1.3] and the PD gains x[0.9,1.1] per env (BASELINE configs[3])")
    ap.add_argument("--physics-program", default="roles", choices=["roles", "lanes"],
                    help="roles: one lane per env (default); lanes: 8 lanes per env (DESIGN.md section 4, the measured negative result)")
    ap.add_argument("--no-self-collision", action="store_true",
                    help="drop k_self_collision (the reference always has it: create_actor filter 0, T:354)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--workload", default="env", choices=["env", "ppo"],
                    help="env: the env-step hot path (BASELINE configs[1], the default and the driver's line); ppo: end-to-end "
                         "on-device PPO training (BASELINE configs[4]): --steps / --warmup count EPOCHS of 128 env steps + 640 updates")
    ap.add_argument("--horizon", type=int, default=128)
    ap.add_argument("--ppo-dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--grad-sync", default="peer", choices=["peer", "peer2", "nccl"],
                    help="PPO gradient exchange at N > 1: sum over peer-mapped buffers inside the optimiser's kernels, or one NCCL all-reduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed env step returned to rank 0 (obs, rew, reset, "
                         "time_outs, stacked_rewards) as DIR/<name>.npy, float32 / float64; beyond 64 MiB a fixed, seeded "
                         "sample of envs (DIR/env_index.npy). The inputs are the same on every run with the same arguments.")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.workload != "env"):
        ap.error("--dump-outputs writes the outputs of the env-step path (--impl ours --workload env)")
    return a


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML from a thread every 5 ms (nvidia_ml_py), so
    that even a 30 ms region gets samples; `nvidia-smi -lms` as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.stop = index, [], None, False

    def _nvml_loop(self):
        import pynvml as nv
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        bits = [(0x8, 3), (0x40, 4), (0x20, 5), (0x4, 6)]  # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap (NVML reason bits)
        while not self.stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:  # noqa: BLE001  (older bindings)
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = [str(sm), str(mx), "", "", "", "", ""]
                for bit, col in bits:
                    row[col] = "Active" if rs & bit else "Not Active"
                self.rows.append(row)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.005)

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return self
        except Exception:  # noqa: BLE001
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        self.stop = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:  # noqa: BLE001
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ outputs
DUMP_BYTES = 64 << 20


def step_outputs(out, seed=0):
    """What DyrosDynamicWalk.step returned, as host arrays (float32; integer buffers as float64, exactly). The env's own
    buffers, overwritten by the next step: call this before that. If the arrays exceed DUMP_BYTES, the rows of a fixed,
    seeded sample of envs; `env_index` lists which."""
    import numpy as np
    obs, rew, reset, extras = out
    arrays = {"obs": obs["obs"], "rew": rew, "reset": reset, "time_outs": extras["time_outs"],
              "stacked_rewards": extras["stacked_rewards"]}
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v.astype(np.float64 if v.dtype.kind in "biu" else np.float32) for k, v in arrays.items()}
    n = len(arrays["rew"])
    row_bytes = 8 + sum(v.nbytes for v in arrays.values()) // n
    keep = np.arange(n)
    if n * row_bytes > DUMP_BYTES - (1 << 16):  # (room for the .npy headers)
        keep = np.sort(np.random.default_rng(seed).choice(n, (DUMP_BYTES - (1 << 16)) // row_bytes, replace=False))
    arrays = {k: v[keep] for k, v in arrays.items()}
    arrays["env_index"] = keep.astype(np.float64)
    return arrays


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), v)


# ------------------------------------------------------------------------------------------------ CPU oracle port
def make_cpu_env(n_envs, seed):
    import numpy as np
    from oracle.env_oracle import EnvOracle
    from oracle import task_oracle as O
    from isaacgymdyros_b200.model.tables import ModelTables
    assets = os.path.join(ROOT, "isaacgymdyros_b200", "assets")
    tables = ModelTables.load(os.path.join(assets, "tocabi_tables.npz"))
    mocap, obs_norm = np.load(os.path.join(assets, "mocap_walk.npy")), np.load(os.path.join(assets, "obs_norm.npy"))
    rng = np.random.default_rng(seed)
    env = EnvOracle(n_envs, tables, mocap, obs_norm, rng=rng)
    return env, rng, O


def cpu_worker(args):
    """Steps a 64-env shard of the workload with the oracle port for up to `steps` steps or `seconds` seconds."""
    n_envs, steps, warmup, seconds, seed = args
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=1)
    except Exception:  # noqa: BLE001
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        env, rng, O = make_cpu_env(n_envs, seed)
        import numpy as np
        act = lambda: rng.uniform(-1, 1, (n_envs, 13)).astype(np.float32)
        for _ in range(warmup):
            env.step(act(), O.draw_noise(n_envs, 2, rng))
        done, t0 = 0, time.perf_counter()
        while done < steps and (time.perf_counter() - t0) < seconds:
            env.step(act(), O.draw_noise(n_envs, 2, rng))
            done += 1
        return done, time.perf_counter() - t0


def cpu_baseline(seconds):
    done, el = cpu_worker((64, 10 ** 9, 1, seconds, 42))
    return {"value": 64 * done / el, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{done} steps of a 64-env shard (BASELINE configs[0] size) with oracle/env_oracle.py "
                      f"(numpy task restatement + dense fp64 physics), 1 thread, {el:.1f} s; not PhysX"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    workers = max(1, min(os.cpu_count() or 1, 32))
    budget = 150.0
    per_step_guess = 0.2
    steps = max(1, min(a.steps, int(budget / per_step_guess)))
    warm = max(a.warmup, 3) if a.warmup <= 5 else 5  # >= 3 as in our arm; capped: a port step costs ~0.1 s
    with mp.get_context("spawn").Pool(workers) as pool:
        res = pool.map(cpu_worker, [(64, steps, warm, budget, 42 + i) for i in range(workers)])
    total = sum(64 * d for d, _ in res)
    el = max(e for _, e in res)
    value = total / el
    steps_done = min(d for d, _ in res)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": steps_done,
            "warmup": warm, "ms_per_step": 1e3 * el / max(steps_done, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": a.envs,
                       "sample": f"bounded: {workers} host processes x 64-env shards = {workers * 64} envs per step (not "
                                 f"{a.envs}: a 4096-env port step takes minutes); throughput is per env-step, so comparable"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port",
                             "sample": f"{workers} processes x 64-env shards x {steps_done} steps of the oracle port "
                                       f"(reference PhysX binaries absent: SURVEY fact 2), {el:.1f} s"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(a):
    import torch
    import torch.distributed as dist
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    from isaacgymdyros_b200.core import measure_fp32_peak

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = f"cuda:{local}"
    torch.cuda.set_device(dev)
    N, K, W = a.envs, a.steps, max(a.warmup, 3)
    extra = dict(friction_range=(0.7, 1.3), pd_gain_range=(0.9, 1.1)) if a.dr_extra else {}
    cfg = default_cfg(N, **extra)
    cfg["env"]["physicsProgram"] = a.physics_program
    cfg["env"]["selfCollision"] = not a.no_self_collision
    # tickets in flight for step_async: 3 hides the host's reaction time when the PCIe link of ONE GPU is the limit
    # (155 vs 172 us per step); with more ranks the host's memory system is the limit (8 ranks: ~112 GB/s of device->host
    # writes in total) and fewer, cache-resident host blocks do better (8 ranks: 56.9 M with 2, 51.4 M with 3;
    # profiles/r1j_step_async.txt)
    depth = 3 if world <= 2 else 2
    cfg["async_depth"] = depth
    env = DyrosDynamicWalk(cfg, dev, rank=rank)
    if a.force_perturb:
        env.core.task_t["perturb_start"].fill_(1)
    g = torch.Generator(device=dev)
    g.manual_seed(42 + rank)  # reference default seed, cfg/config.yaml:11
    pool = [torch.rand(N, 13, device=dev, generator=g) * 2 - 1 for _ in range(16)]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def device_step(i):
        # the public call; the action tensors are resident in HBM and the step's first kernel reads them in place (one
        # CUDA graph per action tensor, captured the second time `step` sees it)
        return env.step(pool[i % len(pool)])

    for i in range(2 * len(pool)):  # every pool entry seen twice: all graphs captured before the warm-up
        device_step(i)
    for i in range(W):
        device_step(i)
    barrier()
    # ---- (1) device-resident, L2 flushed between timed steps: `value`
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    with ClockSampler(local) as clk:
        barrier()
        t_wall0 = time.perf_counter()
        for i in range(K):
            env.core.flush_l2(flush, i)
            ev[i][0].record()
            out = device_step(W + i)
            ev[i][1].record()
        barrier()
        t_wall_flush = time.perf_counter() - t_wall0
        cold_ms = sum(s.elapsed_time(e) for s, e in ev)
        last_outputs = step_outputs(out) if a.dump_outputs and rank == 0 else None
        # ---- (2) back to back (state L2-resident, as in the real rollout loop)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        s0.record()
        for i in range(K):
            device_step(W + K + i)
        s1.record()
        barrier()
        warm_ms = s0.elapsed_time(s1)
        # ---- (3) end to end through the public API with host buffers
        h_act = [p.cpu().pin_memory() for p in pool]
        h_obs = torch.empty(N, 487).pin_memory()
        h_rew = torch.empty(N).pin_memory()
        h_rst = torch.empty(N, dtype=torch.int64).pin_memory()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(K):
            # the pinned host tensor goes to the public API as it is: the first kernel of the step reads it over PCIe
            obs, rew, rst, _ = env.step(h_act[i % len(h_act)])
            h_obs.copy_(obs["obs"], non_blocking=True)
            h_rew.copy_(rew, non_blocking=True)
            h_rst.copy_(rst, non_blocking=True)
        e1.record()
        barrier()
        e2e_sync_ms = e0.elapsed_time(e1)
        # ---- (3b) the same through step_async / step_wait: results packed into one block by dyros_task_pack_results,
        #           ONE device->host transfer per step on a copy stream, `depth` steps in flight, the host consumes (waits
        #           for) the results of step i-depth+1 right after submitting step i
        # every ticket slot captures its CUDA graph on first use: use each slot (twice) BEFORE the timed region, so that
        # no capture (a device synchronisation + graph instantiation) lands inside it
        for j in range(2 * depth):
            env.step_wait(env.step_async(h_act[j % len(h_act)]))
        cs = env._pipe.copy_stream
        barrier()
        e0.record()
        ticks = []
        for i in range(K):
            ticks.append(env.step_async(h_act[i % len(h_act)]))
            if len(ticks) == depth:  # `depth` steps in flight: consume the oldest
                env.step_wait(ticks.pop(0))
        for tick in ticks:
            env.step_wait(tick)
        torch.cuda.current_stream().wait_stream(cs)
        e1.record()
        barrier()
        e2e_ms = e0.elapsed_time(e1)
        # ---- (3c) what the host link gives at this rank count, same run: the same packed block (obs | rew | reset |
        #           time_outs) copied device -> pinned host back to back on the copy stream, nothing else running, all
        #           ranks at once. e2e cannot beat it; the fraction says how well the pipelined step hides its kernels.
        pipe = env._pipe
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(cs):
            c0.record(cs)
            for i in range(K):
                pipe.host[i % depth].copy_(pipe.dev[i % depth], non_blocking=True)
            c1.record(cs)
        c1.synchronize()
        barrier()
        d2h_ms = c0.elapsed_time(c1)
    clocks = clk.summary()
    h2d, d2h = N * 13 * 4, env.core.result_bytes()
    # ---- (4) the dominant kernel alone (k_step_physics = 2 x (torque, physics sub-step, noise) in one launch), inside
    #          real staged steps, L2 flushed before each launch
    KS = min(K, 50)
    kev, scev = [], []
    core = env.core
    for i in range(KS):
        core.prologue(pool[i % len(pool)])
        core.flush_l2(flush, i)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        core.task_physics_kernel()
        a1.record()
        kev.append((a0, a1))
        if core.step_launches() == 3:
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            core.self_collision()
            b1.record()
            scev.append((b0, b1))
        env.post_physics_step()
    torch.cuda.synchronize()
    k1_ms = statistics.mean(s.elapsed_time(e) for s, e in kev)
    sc_ms = statistics.mean(s.elapsed_time(e) for s, e in scev) if scev else 0.0
    reset_rate = float(env.reset_buf.float().mean().item())
    # ---- (5) as (1), with the env state pinned in the persisting part of L2 (dyros_sim_set_l2_persistence): the same
    #          256 MiB fill between the steps no longer evicts it. Reported beside `value`, not as `value`.
    persist_ms, set_aside = float("nan"), 0
    try:
        set_aside = env.set_l2_persistence(True)
        for i in range(len(pool) + W):
            device_step(i)
        barrier()
        pev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for i in range(K):
            env.core.flush_l2(flush, i)
            pev[i][0].record()
            device_step(W + i)
            pev[i][1].record()
        barrier()
        persist_ms = sum(s.elapsed_time(e) for s, e in pev)
        env.set_l2_persistence(False)
    except Exception as exc:  # noqa: BLE001  (an informational extra must not cost the run its JSON line)
        print(f"l2 persistence measurement skipped: {exc}", file=sys.stderr)

    from isaacgymdyros_b200.sharding import max_over_ranks, reduce_episode_stats
    cold_ms, warm_ms, e2e_ms, e2e_sync_ms, k1_ms, persist_ms, d2h_ms = (max_over_ranks(x, dev) for x in (cold_ms, warm_ms, e2e_ms, e2e_sync_ms, k1_ms, persist_ms, d2h_ms))
    # episode statistics across ranks (the only data the env path ever reduces; SURVEY 8e)
    stats = reduce_episode_stats({"epi_len_log": env.epi_len_log, "contact_reward_mean": env.contact_reward_mean})
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        fp32_peak = measure_fp32_peak(local)
        k1_flop_env, k1_dram_env, k1_src = k1_profile()
        total_envs = N * world
        value = total_envs * K / (cold_ms * 1e-3)
        k1_bytes = K1_BYTES_PER_ENV_STEP * N
        achieved = k1_bytes / (k1_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": cold_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": N, "actions": "torch.rand(N,13)*2-1, seed 42",
                       "domain_randomisation": "mass, damping, armature, friction, PD gains" if a.dr_extra else "mass, damping, armature (CFG:81-115)",
                       "perturbation": "forced on (T:491)" if a.force_perturb else "gated as in the reference (T:489)",
                       "self_collision": not a.no_self_collision, "physics_program": a.physics_program,
                       "l2": "flushed between timed steps (256 MiB fill outside the timed intervals, by a kernel with the step kernels' L1 / shared-memory split: dyros_flush_l2)",
                       "timing": "CUDA events per step on the launch stream, summed; max over ranks",
                       "launch_geometry": dict(core.launch_info(), threads_per_cta_fused_step=256), "reset_rate_last_step": reset_rate},
            "clocks": clocks,
            "e2e": {"value": total_envs * K / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K,
                    "api": "DyrosDynamicWalk.step_async / step_wait: pinned host actions in, one packed pinned host block "
                           "(obs, rew, reset, time_outs) out per step; the transfer of step k overlaps the kernels of step k+1",
                    "tickets_in_flight": depth,
                    "d2h_ceiling": {"value": total_envs * K / (d2h_ms * 1e-3), "unit": UNIT, "ms_per_step": d2h_ms / K,
                                    "gb_per_s_per_rank": d2h / (d2h_ms / K * 1e-3) / 1e9,
                                    "what": "the same result block copied device -> pinned host back to back, all ranks at once, no kernels"},
                    "frac_of_d2h_ceiling": d2h_ms / e2e_ms},
            "e2e_sync": {"value": total_envs * K / (e2e_sync_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_sync_ms / K,
                         "d2h_bytes_per_step": N * 487 * 4 + N * 4 + N * 8,
                         "api": "DyrosDynamicWalk.step + three device->host copies on the same stream, nothing overlapped"},
            "gpu_launches": K * core.step_launches(),
            "value_warm_l2": total_envs * K / (warm_ms * 1e-3), "ms_per_step_warm_l2": warm_ms / K,
            "l2_persisting_state": None if persist_ms != persist_ms else {
                                    "value": total_envs * K / (persist_ms * 1e-3), "unit": UNIT, "ms_per_step": persist_ms / K,
                                    "set_aside_bytes": set_aside, "state_bytes": int(core.state_arena.numel()),
                                    "note": "same flushed-L2 loop as `value`, env state pinned in the persisting part of L2 "
                                            "(DyrosDynamicWalk.set_l2_persistence): an opt-in of the product, not the headline; "
                                            "it buys ~2 us of the ~24 us a flushed L2 costs: the rest is not env state"},
            "roofline": {"bound": "hbm", "kernel": "k_step_physics (2 x (PD/delay torque, physics sub-step, sensor noise) of all envs, one launch)",
                         "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                         "traffic": None if k1_dram_env is None else k1_dram_env * N,
                         "traffic_source": k1_src + "; ncu --set full, cold caches as in the timed launches; scaled per env",
                         "launch_ms": k1_ms, "algorithmic_bytes_per_launch": k1_bytes,
                         "note": "K1 is FP32-latency bound, not HBM bound (SURVEY 8d): see fp32"},
            "fp32": None if k1_flop_env is None else {
                     "achieved": k1_flop_env * N / (k1_ms * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": k1_flop_env * N / (k1_ms * 1e-3) / 1e12 / fp32_peak,
                     "flop_per_launch": k1_flop_env * N, "flop_source": k1_src + ": executed ffma*2 + fadd + fmul",
                     "peak_source": "dyros_measure_fp32_peak (FFMA saturation, this run)"},
            "step_kernels": {"k_step_physics_ms": k1_ms, "k_self_collision_ms": sc_ms,
                             "note": "CUDA events around each launch inside staged steps, L2 flushed before the physics launch "
                                     "(k_self_collision then finds the link poses in L2, as in the fused step); the rest of "
                                     "ms_per_step is k_post_fused and launch gaps"},
            "whole_step_hbm": {"achieved": ENV_STEP_BYTES * N / (cold_ms / K * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s"},
            "episode_stats": stats,
            "wall_s_flush_loop": t_wall_flush,
        }
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(a.cpu_seconds)
        if last_outputs is not None:
            write_outputs(a.dump_outputs, last_outputs)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ PPO (configs[4])
def run_ppo(a):
    """End-to-end PPO training on the device (isaacgymdyros_b200/ppo.py): per epoch horizon x envs env-steps (policy
    forward on the GPU reading obs_buf in place) + mini_epochs x minibatches updates, each with one NCCL all-reduce of
    the flat 1.54 MB gradient bucket when world > 1. Times K epochs after W warm-up epochs (graph captures land there)."""
    import torch
    import torch.distributed as dist
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = f"cuda:{local}"
    torch.cuda.set_device(dev)
    N, K, W = a.envs, a.steps, max(a.warmup, 1)
    env = DyrosDynamicWalk(default_cfg(N), dev, rank=rank, use_cuda_graph=False)
    cfg = PPOConfig(horizon_length=a.horizon, mixed_precision=a.ppo_dtype, grad_sync=a.grad_sync)
    tr = PPOTrainer(env, cfg, rank=rank, world=world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        out = tr.train_epoch()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    t_roll = t_upd = 0.0
    with ClockSampler(local) as clk:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            tr.epoch += 1
            tr.net.update_action_noise((cfg.max_epochs - tr.epoch) / cfg.max_epochs)
            tr.buf["ep_stats"].zero_()
            ev[0].record(); tr.rollout(); ev[1].record(); tr.update(); ev[2].record()
            ev[2].synchronize()
            t_roll += ev[0].elapsed_time(ev[1]); t_upd += ev[1].elapsed_time(ev[2])
        e1.record()
        barrier()
        total_ms = e0.elapsed_time(e1)
        # the collective alone: the same flat bucket, all-reduced back to back
        ar_ms = 0.0
        if world > 1:
            reps = 200
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(reps):
                dist.all_reduce(tr.net.grad)
            a1.record()
            barrier()
            ar_ms = a0.elapsed_time(a1) / reps
    from isaacgymdyros_b200.sharding import max_over_ranks
    total_ms, t_roll, t_upd, ar_ms = (max_over_ranks(x, dev) for x in (total_ms, t_roll, t_upd, ar_ms))
    out = tr.train_epoch()
    if rank == 0:
        frames = N * a.horizon * world * K
        updates = cfg.mini_epochs * tr.num_minibatches
        line = {"metric": "env-steps/s, end-to-end on-device PPO training (BASELINE configs[4])", "value": frames / (total_ms * 1e-3),
                "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": a.ppo_dtype, "data": "synthetic",
                "config": {"workload": "DyrosDynamicWalk PPO (DyrosDynamicWalkPPO.yaml): per epoch horizon x envs env-steps with the "
                                       "policy on the GPU + mini_epochs x minibatches updates; one step = one epoch",
                           "envs_per_gpu": N, "horizon_length": a.horizon, "minibatch_size": cfg.minibatch_size,
                           "mini_epochs": cfg.mini_epochs, "updates_per_epoch": updates, "parameters": tr.net.n,
                           "gradient_bucket_bytes": tr.net.n * 4,
                           "networks": "packed bf16 (batch-2 GEMMs)" if tr.packed is not None else "fp32 autograd",
                           "grad_sync": (("peer memory, two-phase (reduce-scatter + all-gather)" if cfg.grad_sync == "peer2" else "peer memory (dyros_ppo_reduce_peers)")
                                         if tr.peers is not None else "nccl all_reduce") if world > 1 else "none"},
                "clocks": clk.summary(),
                "breakdown_ms_per_epoch": {"rollout_and_gae": t_roll / K, "update": t_upd / K,
                                           "update_per_minibatch": t_upd / K / updates,
                                           "allreduce_alone_per_call": ar_ms, "allreduce_alone_per_epoch": ar_ms * updates},
                # this library's kernels per epoch (the cuBLAS GEMMs between them are not counted): per rollout step
                # cast_obs, 2 x bias_relu, act, the env step's launches, reward, advance; GAE; per update 2 x bias_relu,
                # loss_grad, 2 x relu_bwd, unpack (+ reduce_peers at N > 1), adam_pack, adam_finish
                "gpu_launches": (K * (tr.H * (6 + env.core.step_launches()) + 1 + tr.cfg.mini_epochs * tr.num_minibatches * (8 + (world > 1)))
                                 if tr.packed is not None else None),
                "last_epoch": out}
        emit(line)
    if world > 1:
        # the CUDA graphs hold captured NCCL work: drop them before the communicator goes, and do not wait on a
        # destroy_process_group that was seen to hang behind them (the JSON line is out; nothing is left to flush)
        tr._g_update.clear()
        tr._g_rollout = None
        dist.barrier()
        torch.cuda.synchronize()
        sys.stderr.flush()
        os._exit(0)


_JSON_FD = None


def emit(line: dict):
    """The ONE JSON line, on the process's original stdout."""
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


def main():
    global _JSON_FD
    a = parse()
    # stdout carries the JSON line and nothing else: whatever libraries print there from C (NCCL prints its version to
    # stdout when the box sets NCCL_DEBUG) goes to stderr instead
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "ppo":
        run_ppo(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
