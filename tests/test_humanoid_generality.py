"""BASELINE configs[2]: the stock IsaacGymEnvs Humanoid (assets/mjcf/nv_humanoid.xml: 16 bodies, 21 hinges with 2-3 hinges
on one body and anchored joints, capsule / sphere geoms, joint stiffness, masses from geometry, legs branching at the
pelvis) through the SAME loader, C ABI and physics kernel as TOCABI. Parity: kernel (float32, O(n)) vs the dense fp64
oracle on identical states, Humanoid.yaml sim parameters (dt 1/60, 2 sub-steps, contact_offset 0.02, 4+0 iterations)."""
import os

import numpy as np
import pytest

from isaacgymdyros_b200.core import ASSETS, CoreConfig, stable_penalty
from isaacgymdyros_b200.model.tables import ModelTables, role_programs
from oracle.physics_oracle import PhysicsOracle
from tests.physics_util import emulate_substep, emulate_substep_lanes, oracle_params
from tests.test_physics_emulation import compare

HUMANOID_CFG = dict(dt=0.0166, substeps=1, contact_offset=0.02, num_position_iterations=4, num_velocity_iterations=0,
                    dof_vel_limit=1.0e3, max_angular_velocity=64.0, solver_bodies=("right_foot", "left_foot"))
STAND_Z = 1.2855  # torso height at which the soles touch the plane in the zero pose


def humanoid():
    return ModelTables.load(os.path.join(ASSETS, "humanoid_tables.npz"))


def humanoid_states(N, rng, t, kind):
    root = np.zeros((N, 13))
    root[:, 6] = 1.0
    q = np.zeros((N, 21))
    qd = np.zeros((N, 21))
    for n in range(N):
        mode = {"air": 0, "stand": 1}.get(kind, rng.integers(0, 3))
        if mode == 0:
            root[n, 2] = 2.5
            quat = rng.normal(0, 1, 4)
            root[n, 3:7] = quat / np.linalg.norm(quat)
            root[n, 7:13] = rng.normal(0, 0.5, 6)
            q[n] = rng.normal(0, 0.2, 21)
            qd[n] = rng.normal(0, 1.0, 21)
        elif mode == 1:
            root[n, 2] = STAND_Z + rng.uniform(-0.01, 0.01)
            quat = np.array([0, 0, 0, 1.0]) + np.append(rng.normal(0, 0.01, 3), 0)
            root[n, 3:7] = quat / np.linalg.norm(quat)
            root[n, 7:13] = rng.normal(0, 0.05, 6)
            q[n] = rng.normal(0, 0.01, 21)
            qd[n] = rng.normal(0, 0.1, 21)
        else:
            root[n, 2] = rng.uniform(0.2, 0.9)
            quat = np.array([0, 0, 0, 1.0]) + np.append(rng.normal(0, 0.5, 3), 0)
            root[n, 3:7] = quat / np.linalg.norm(quat)
            root[n, 7:13] = rng.normal(0, 0.3, 6)
            q[n] = rng.normal(0, 0.3, 21)
            qd[n] = rng.normal(0, 0.5, 21)
    q = np.clip(q, t.dof_lower + 0.02, t.dof_upper - 0.02)
    f = lambda a: a.astype(np.float32).astype(np.float64)
    tau = rng.normal(0, 10, (N, 21))
    return dict(root=f(root), q=f(q), qd=f(qd), tau=f(tau), damping=f(np.tile(t.dof_damping, (N, 1))),
                armature=f(np.tile(t.dof_armature, (N, 1))), mass_scale=f(rng.uniform(0.9, 1.1, (N, 16))))


def test_humanoid_tables_known_answers():
    t = humanoid()
    assert (t.num_bodies, t.num_links, t.num_dofs) == (16, 22, 21)
    assert abs(t.total_mass() - 40.844) < 0.01  # MuJoCo humanoid at density 1000
    assert t.body_names[0] == "torso" and t.body_link[1] == 0  # head is welded to the torso
    # lower_waist carries two hinges: one massless link, the body rides on the second
    assert list(t.body_link).count(1) == 0 and t.body_link[2] == 2
    assert t.dof_stiffness.max() == 20.0 and t.dof_armature.max() == pytest.approx(0.02)
    assert np.allclose(np.linalg.norm(t.link_axis[1:], axis=1), 1.0)
    prog = role_programs(t.link_parent, [9, 15])
    links = sorted(int(l) for l in prog.flatten() if l > 0)
    assert links == list(range(1, 22))


@pytest.mark.parametrize("program", ["roles", "lanes"])
@pytest.mark.parametrize("kind,seed", [("air", 0), ("stand", 1), ("mixed", 2)])
def test_humanoid_lane_program_matches_dense_oracle(kind, seed, program):
    """`roles`: the single-lane statement of the algorithm; `lanes`: the 8-lanes-per-env program the CUDA kernels run."""
    t = humanoid()
    cfg = CoreConfig(**HUMANOID_CFG)
    o = PhysicsOracle(t, oracle_params(cfg), solver_bodies=cfg.solver_bodies)
    st = humanoid_states(8, np.random.default_rng(seed), t, kind)
    want = o.substep(st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"], st["mass_scale"])
    got = (emulate_substep if program == "roles" else emulate_substep_lanes)(t, cfg, st)
    compare(st, got, want, ctx=f"humanoid {kind}: ")
    if kind == "stand":
        feet = [t.body_names.index("right_foot"), t.body_names.index("left_foot")]
        assert (want[3][:, feet, 2] > 0).any()


def test_role_program_does_not_depend_on_role_timing():
    """The roles exchange results through the env's scratch block, ordered by stage flags only. Holding any one role back
    at any stage marker of physics_roles.cuh lets the others run ahead as far as the flags allow; the result must stay
    bit for bit the same. (The Humanoid's arms hang off the base while its feet hang off the pelvis: no foot waits for
    an arm's pass 3, so an arm may run its pass 3 after the base response has overwritten the base's velocity.)"""
    import ctypes as C
    from tests.golden_util import load_assets
    from tests.physics_util import hostemu, random_states
    t, tocabi = humanoid(), load_assets()[0]
    cases = [(t, CoreConfig(**HUMANOID_CFG), humanoid_states(2, np.random.default_rng(0), t, "air")),
             (t, CoreConfig(**HUMANOID_CFG), humanoid_states(2, np.random.default_rng(1), t, "stand")),
             (tocabi, CoreConfig(), random_states(2, np.random.default_rng(2), tocabi, "mixed"))]
    hold = hostemu().dyros_hostemu_hold_role
    try:
        for tab, cfg, st in cases:
            free = emulate_substep(tab, cfg, st)
            for role in range(8):
                for mark in (0, 16, 17, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12):
                    hold(role, mark, 2000)
                    held = emulate_substep(tab, cfg, st)
                    hold(-1, -1, 0)
                    for a, b in zip(held, free):
                        assert np.array_equal(a, b), f"{tab.num_links} links: role {role} held at mark {mark} changes the result"
    finally:
        hold(-1, -1, 0)


def test_humanoid_stands_on_the_oracle():
    """Zero pose on the ground, zero torques: joint springs (stiffness 2..20) and damping hold the pose for a while and
    the ground reaction approaches the weight (40.8 kg)."""
    t = humanoid()
    cfg = CoreConfig(**{**HUMANOID_CFG, "dt": 0.0166 / 2})
    o = PhysicsOracle(t, oracle_params(cfg), solver_bodies=cfg.solver_bodies)
    root = np.zeros((1, 13)); root[:, 6] = 1; root[:, 2] = STAND_Z
    q, qd = np.zeros((1, 21)), np.zeros((1, 21))
    damp, arm, ms = t.dof_damping[None], t.dof_armature[None], np.ones((1, 16))
    fz = []
    for s in range(30):
        root, q, qd, cf, _ = o.substep(root, q, qd, np.zeros((1, 21)), damp, arm, ms)
        fz.append(cf[0, :, 2].sum())
    assert np.isfinite(root).all() and abs(np.mean(fz[10:]) - 40.844 * 9.81) < 0.25 * 40.844 * 9.81
    assert root[0, 2] > 1.2


@pytest.mark.gpu
def test_humanoid_cuda_simulate_matches_oracle_and_runs_4096():
    import torch
    from isaacgymdyros_b200.core import DyrosCore
    t = humanoid()
    cfg = CoreConfig(**HUMANOID_CFG, self_collision=False)   # (PhysicsOracle.substep has no self-collision pass; its own
    o = PhysicsOracle(t, oracle_params(cfg), solver_bodies=cfg.solver_bodies)   # test: tests/test_self_collision.py)
    N = 40
    st = humanoid_states(N, np.random.default_rng(5), t, "mixed")
    want = o.substep(st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"], st["mass_scale"])
    core = DyrosCore(N, "cuda:0", cfg, tables=t, with_task=False)
    T = lambda a: torch.tensor(np.ascontiguousarray(a, dtype=np.float32), device="cuda:0")
    core.sim_t["root_states"].copy_(T(st["root"]))
    ds = core.sim_t["dof_state"].view(N, 21, 2)
    ds[:, :, 0], ds[:, :, 1] = T(st["q"]), T(st["qd"])
    core.sim_t["dof_actuation_force"].copy_(T(st["tau"]).reshape(-1))
    core.sim_t["body_mass_scale"].copy_(T(st["mass_scale"]))
    core.simulate()
    torch.cuda.synchronize()
    f = lambda x: x.cpu().numpy().astype(np.float64)
    got = (f(core.sim_t["root_states"]), f(ds[:, :, 0]), f(ds[:, :, 1]), f(core.sim_t["net_contact_force"].view(N, 16, 3)))
    compare(st, got, want, ctx="humanoid cuda: ")
    core.close()
    # BASELINE configs[2] size: 4096 humanoids, Humanoid.yaml stepping (dt 1/60 in 2 sub-steps), held upright by a
    # weak joint-space PD with random torque noise for a quarter of a second (a humanoid without a balance controller
    # buckles after ~0.5 s, in MuJoCo and PhysX too). (Only the soles are constraint-solved; other bodies get
    # the soft, explicitly integrated penalty contact that TOCABI uses to flag a fall, so a rollout of *fallen*
    # humanoids is out of scope here: DESIGN.md section 8.)
    N = 4096
    k_pen, c_pen = stable_penalty(0.0166 / 2)
    cfg2 = CoreConfig(**{**HUMANOID_CFG, "substeps": 2, "penalty_stiffness": k_pen, "penalty_damping": c_pen})
    core = DyrosCore(N, "cuda:0", cfg2, tables=t, with_task=False)
    core.sim_t["root_states"][:, 2] = STAND_Z
    g = torch.Generator(device="cuda:0"); g.manual_seed(0)
    gear = torch.tensor(t.dof_effort, dtype=torch.float32, device="cuda:0")
    ds = core.sim_t["dof_state"].view(N, 21, 2)
    for _ in range(15):
        noise = (torch.rand(N, 21, device="cuda:0", generator=g) * 2 - 1) * 0.05 * gear
        core.sim_t["dof_actuation_force"].copy_((-20.0 * ds[:, :, 0] - 1.0 * ds[:, :, 1] + noise).reshape(-1))
        core.simulate()
    torch.cuda.synchronize()
    assert torch.isfinite(core.sim_t["root_states"]).all() and torch.isfinite(core.sim_t["dof_state"]).all()
    z = core.sim_t["root_states"][:, 2]
    assert z.min().item() > 1.2 and z.max().item() < 1.4  # everybody is still on their feet
    cf = core.sim_t["net_contact_force"].view(N, 16, 3)
    feet = [t.body_names.index("right_foot"), t.body_names.index("left_foot")]
    others = [b for b in range(16) if b not in feet]
    assert cf[:, others].abs().max().item() == 0.0
    w = 40.844 * 9.81
    assert (cf[:, feet, 2].sum(1) - w).abs().mean().item() < 0.15 * w  # the soles carry the weight
    core.close()
