"""Triangle-mesh ground on the B200: the CUDA role program with Ground = MeshGround against the plane and the
heightfield it must reproduce, weight on the feet, the CTA size, the C ABI's refusals and the terrainMesh task."""
import ctypes as C

import numpy as np
import pytest
import torch

from isaacgymdyros_b200 import native, terrain
from isaacgymdyros_b200.core import CoreConfig, INIT_DOF_POS, KP, KV
from tests.golden_util import load_assets
from tests.physics_util import random_states
from tests.terrain_util import flat_field, ramp_field
from tests.test_physics_emulation import compare
from tests.test_physics_parity_gpu import load_sim_state, read_sim_state
from tests.test_terrain_gpu import core_field, run_simulate

pytestmark = pytest.mark.gpu
W = 104.48712 * 9.81  # TOCABI's weight (N)


def mesh_of(field):
    return terrain.trimesh_from_field(core_field(field), None)


def run_simulate_mesh(N, mesh, st):
    from isaacgymdyros_b200.core import DyrosCore
    core = DyrosCore(N, "cuda:0", CoreConfig(self_collision=False, triangle_mesh=mesh), with_task=False)
    load_sim_state(core, st)
    core.simulate()
    torch.cuda.synchronize()
    out = read_sim_state(core)
    info = core.mesh_info
    core.close()
    return out, info


def _states(seed):
    """Standing and airborne envs: sole contacts and none. (The 'mixed' states also bury tilted links deeper than the
    mesh's depth allowance D = 0.1 m, where a mesh point loses its ground by design and the plane's does not.)"""
    tables = load_assets()[0]
    a = random_states(150, np.random.default_rng(seed), tables, "stand")
    b = random_states(150, np.random.default_rng(seed + 1), tables, "air")
    return {k: np.concatenate([a[k], b[k]]) for k in a}


def test_cuda_flat_mesh_matches_plane():
    st = _states(2)
    plane = run_simulate(300, None, st)
    flat, info = run_simulate_mesh(300, mesh_of(flat_field()), st)
    assert info["bytes"] > 0 and info["dropped"] == 0
    compare(st, flat, plane, ctx="flat mesh vs plane: ")


def test_cuda_ramp_mesh_matches_heightfield():
    field = ramp_field()
    st = _states(5)
    hf = run_simulate(300, field, st)
    mesh, _ = run_simulate_mesh(300, mesh_of(field), st)
    compare(st, mesh, hf, ctx="ramp mesh vs heightfield: ")


def test_cuda_standing_on_flat_mesh_carries_weight_on_feet_only():
    from isaacgymdyros_b200.core import DyrosCore
    N = 512
    field = flat_field(z=0.3, size=(200.0, 200.0), origin_xy=(-5.0, -5.0))
    core = DyrosCore(N, "cuda:0", CoreConfig(triangle_mesh=mesh_of(field), self_collision=False))
    dev = core.device
    origins = core.task_t["env_origins"].clone()
    assert (origins[:, 2] - 0.3).abs().max().item() < 1e-5, "default origins sit on the mesh"
    kp, kv = torch.tensor(KP, device=dev), torch.tensor(KV, device=dev)
    q0 = torch.tensor(INIT_DOF_POS, device=dev)
    ds = core.sim_t["dof_state"].view(N, 33, 2)
    ds[:, :, 0] = q0
    for s in range(400):
        core.sim_t["dof_actuation_force"].copy_((kp * (q0 - ds[:, :, 0]) - kv * ds[:, :, 1]).reshape(-1))
        core.simulate()
    torch.cuda.synchronize()
    cf = core.sim_t["net_contact_force"].view(N, 38, 3)
    assert torch.isfinite(core.sim_t["root_states"]).all()
    fz = cf[:, :, 2].sum(1)
    assert (fz - W).abs().max().item() < 0.05 * W, (fz.min().item(), fz.max().item())
    others = [b for b in range(38) if b not in (8, 16)]
    assert cf[:, others].abs().max().item() == 0.0
    core.close()


def test_mesh_cta_holds_28_envs_on_the_gpu():
    from isaacgymdyros_b200.core import DyrosCore
    core = DyrosCore(4096, "cuda:0", CoreConfig(self_collision=False, triangle_mesh=mesh_of(flat_field())), with_task=False)
    info = core.launch_info()
    assert info["envs_per_cta"] == 28 and info["ctas"] == 147, info
    core.close()


def _desc(v, t):
    d = native.DyrosTriangleMesh()
    d.vertices, d.triangles, d.num_vertices, d.num_triangles = v.ctypes.data, t.ctypes.data, len(v), len(t)
    d.dynamic_friction = 1.0
    return d


def test_c_abi_refusals():
    from isaacgymdyros_b200.core import DyrosCore
    m = mesh_of(flat_field())
    v, t = np.ascontiguousarray(m.vertices), np.ascontiguousarray(m.triangles)
    lanes = DyrosCore(8, "cuda:0", CoreConfig(self_collision=False, physics_program="lanes"), with_task=False)
    assert lanes.lib.dyros_sim_set_triangle_mesh(lanes.sim_handle, C.byref(_desc(v, t))) != 0
    assert b"lanes" in lanes.lib.dyros_last_error()
    lanes.close()
    with pytest.raises(native.DyrosError, match="lanes"):
        DyrosCore(8, "cuda:0", CoreConfig(self_collision=False, physics_program="lanes", triangle_mesh=m), with_task=False)
    core = DyrosCore(8, "cuda:0", CoreConfig(self_collision=False), with_task=False)
    lib, h = core.lib, core.sim_handle
    bad = t.copy()
    bad[3, 1] = len(v)
    assert lib.dyros_sim_set_triangle_mesh(h, C.byref(_desc(v, bad))) != 0 and b"vertex index" in lib.dyros_last_error()
    vn = v.copy()
    vn[2, 0] = np.inf
    assert lib.dyros_sim_set_triangle_mesh(h, C.byref(_desc(vn, t))) != 0 and b"not finite" in lib.dyros_last_error()
    assert lib.dyros_sim_set_triangle_mesh(h, C.byref(_desc(v, t))) == 0
    out = (C.c_int64 * 4)()
    assert lib.dyros_sim_triangle_mesh_info(h, C.byref(out)) == 0 and out[0] > 0 and out[2] == len(t)
    s = torch.zeros(4, 4, dtype=torch.int16, device=core.device)
    d = native.DyrosHeightField()
    d.samples = s.data_ptr()
    d.num_rows = d.num_columns = 4
    d.row_scale = d.column_scale = d.vertical_scale = 0.1
    assert lib.dyros_sim_set_heightfield(h, C.byref(d)) != 0 and b"one ground" in lib.dyros_last_error()
    assert lib.dyros_sim_set_triangle_mesh(h, None) == 0
    assert lib.dyros_sim_triangle_mesh_info(h, C.byref(out)) == 0 and out[0] == 0
    assert lib.dyros_sim_set_heightfield(h, C.byref(d)) == 0
    assert lib.dyros_sim_set_triangle_mesh(h, C.byref(_desc(v, t))) != 0 and b"one ground" in lib.dyros_last_error()
    core.close()


def _walk(N, mesh, seed=3):
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import DyrosDynamicWalk, default_cfg
    cfg = default_cfg(N)
    cfg["env"]["terrain"] = dict(num_rows=4, num_cols=5, terrain_length=4.0, terrain_width=4.0, border_size=2.0,
                                 measure_heights=True, seed=seed)
    if mesh:
        cfg["env"]["terrainMesh"] = True
    return DyrosDynamicWalk(cfg, "cuda:0")


def test_terrain_mesh_task_steps_and_scan_equals_heightfield():
    N = 4096
    envm = _walk(N, True)
    envh = _walk(N, False)
    om, oh = envm.reset(), envh.reset()
    om = om["obs"] if isinstance(om, dict) else om
    oh = oh["obs"] if isinstance(oh, dict) else oh
    # same roots (same seed, same origins) -> the height-scan columns are the field's samples on both grounds
    assert torch.equal(om[:, 487:], oh[:, 487:])
    g = torch.Generator(device="cuda:0").manual_seed(0)
    for _ in range(300):
        a = torch.rand((N, 13), device="cuda:0", generator=g) * 2 - 1
        obs, rew, done, extras = envm.step(a)
    o = obs["obs"] if isinstance(obs, dict) else obs
    assert torch.isfinite(o).all() and torch.isfinite(rew).all()
    assert "terrain_level" in envm.extras.get("episode", {})
    envm.close() if hasattr(envm, "close") else None
    envh.close() if hasattr(envh, "close") else None


# ---------------------------------------------------------------- against the fp64 oracle, risers, fused/staged, facade

from tests.mesh_util import mesh_from, stair_mesh_field  # noqa: E402
from tests.terrain_util import rough_field  # noqa: E402
from tests.test_terrain import terrain_states  # noqa: E402
from tests.test_trimesh_program import MESHES, mesh_case, mesh_oracle  # noqa: E402


@pytest.mark.parametrize("name", list(MESHES))
def test_cuda_simulate_on_mesh_matches_oracle_ragged_n(name):
    """k_simulate<MeshGround> at N = 2 waves of 148 CTAs plus a partial CTA: the envs are 16 distinct states tiled, so
    the fp64 oracle checks all of them, the last (partial) CTA's included."""
    field, mesh = mesh_case(name)
    base = terrain_states(field, "mixed", seed=17, N=8)
    stand = terrain_states(field, "stand", seed=18, N=8)
    base = {k: np.concatenate([base[k], stand[k]]) for k in base}
    N = 28 * 148 * 2 + 13
    reps = -(-N // 16)
    st = {k: np.tile(v, (reps,) + (1,) * (v.ndim - 1))[:N] for k, v in base.items()}
    got, _ = run_simulate_mesh(N, mesh, st)
    want = mesh_oracle(mesh).substep(base["root"], base["q"], base["qd"], base["tau"], base["damping"], base["armature"],
                                     base["mass_scale"])[:4]
    for part, idx in (("first", np.arange(16)), ("last", np.arange(N - 16, N))):
        order = idx % 16
        sub = {k: v[order] for k, v in base.items()}
        compare(sub, tuple(g[idx] for g in got), tuple(w[order] for w in want), ctx=f"{name} {part}: ")


def _riser_states(axis, sign, n=24):
    """Standing TOCABIs on the lower tread of a 0.1 m riser at 0.3 m (ascending, sign +1, wall facing -axis) or at 0
    (descending, sign -1, wall facing +axis), swept along `axis` so that some feet overlap the wall."""
    tables = load_assets()[0]
    st = random_states(n, np.random.default_rng(4), tables, "stand")
    st["root"][:, 7:13] = 0.0
    st["qd"][:] = 0.0
    if axis == 0:  # (feet side by side: both reach the wall with their toes, or their heels)
        sweep = np.linspace(0.1, 0.3, n) if sign > 0 else np.linspace(0.0, 0.2, n)
    else:  # (the left foot at about +0.1 m reaches the ascending wall, the right one at -0.1 m the descending one)
        sweep = np.linspace(0.1, 0.3, n) if sign > 0 else np.linspace(-0.05, 0.1, n)
    st["root"][:, axis] = sweep
    st["root"][:, 1 - axis] = 0.0
    st["root"] = st["root"].astype(np.float32).astype(np.float64)
    return st


@pytest.mark.parametrize("axis", [0, 1])
@pytest.mark.parametrize("sign", [1, -1])
def test_cuda_riser_pushes_the_foot_back_horizontally(axis, sign):
    """A foot that overlaps a vertical riser of legged_gym's trimesh gets a horizontal net_contact_force away from the
    wall: -x / -y in front of an ascending riser, +x / +y behind a descending one (the wall facing +-y is the tangent
    fallback case). A heightfield has no such force: its riser is a ramp."""
    from isaacgymdyros_b200.core import DyrosCore
    field = stair_mesh_field(step=0.1 * sign, size=(4.0, 4.0), origin_xy=(-2.0, -2.0), axis=axis)
    mesh = mesh_from(field, 0.75)
    st = _riser_states(axis, sign)
    N = len(st["root"])
    core = DyrosCore(N, "cuda:0", CoreConfig(self_collision=False, triangle_mesh=mesh), with_task=False)
    load_sim_state(core, st)
    core.simulate()
    torch.cuda.synchronize()
    cf = core.sim_t["net_contact_force"].view(N, 38, 3)[:, [8, 16]].cpu().numpy()
    core.close()
    f = -sign * cf[..., axis].ravel()  # > 0: away from the wall
    assert f.max() > 0.1 * W and f.sum() > 0 and f.min() > -0.5 * f.max(), (f.min(), f.max())
    want = mesh_oracle(mesh).substep(st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"],
                                     st["mass_scale"])[3][:, [8, 16]]
    w = -sign * want[..., axis].ravel()
    assert np.abs(w - f).max() < 0.02 * np.abs(w).max(), np.abs(w - f).max()


def test_cuda_standing_on_a_stair_tread_carries_weight_on_feet_only():
    from isaacgymdyros_b200.core import DyrosCore, env_origins
    N = 64
    field = stair_mesh_field(step=0.1, tread=0.6, size=(45.0, 45.0), origin_xy=(-5.0, -5.0))
    mesh = mesh_from(field, 0.75)
    o = env_origins(N, 5.0).astype(np.float64)
    o[:, 0] = np.floor(o[:, 0] / 0.6) * 0.6 + 0.3  # tread centres
    o[:, 2] = mesh.height_at(o[:, 0], o[:, 1])[0]
    mesh.env_origins = o
    core = DyrosCore(N, "cuda:0", CoreConfig(triangle_mesh=mesh, self_collision=False))
    dev = core.device
    assert np.abs(core.task_t["env_origins"].cpu().numpy()[:, 2] - np.floor(o[:, 0] / 0.6) * 0.1).max() < 1e-4
    kp, kv = torch.tensor(KP, device=dev), torch.tensor(KV, device=dev)
    q0 = torch.tensor(INIT_DOF_POS, device=dev)
    ds = core.sim_t["dof_state"].view(N, 33, 2)
    ds[:, :, 0] = q0
    for s in range(400):
        core.sim_t["dof_actuation_force"].copy_((kp * (q0 - ds[:, :, 0]) - kv * ds[:, :, 1]).reshape(-1))
        core.simulate()
    torch.cuda.synchronize()
    cf = core.sim_t["net_contact_force"].view(N, 38, 3)
    fz = cf[:, :, 2].sum(1)
    assert (fz - W).abs().max().item() < 0.05 * W, (fz.min().item(), fz.max().item())
    others = [b for b in range(38) if b not in (8, 16)]
    assert cf[:, others].abs().max().item() == 0.0
    core.close()


def test_fused_step_equals_staged_sequence_on_mesh():
    from isaacgymdyros_b200.core import DyrosCore
    from oracle import task_oracle as O
    from tests.test_task_parity_gpu import inject_noise, load_state, read_state
    N = 257
    field = rough_field(size=(100.0, 100.0), origin_xy=(-5.0, -5.0), spacing=0.25)
    cfg = CoreConfig(with_rb_force_tensors=True, triangle_mesh=mesh_from(field, 0.75))
    a, b = DyrosCore(N, "cuda:0", cfg), DyrosCore(N, "cuda:0", cfg)
    rng = np.random.default_rng(3)
    tables, mocap, obs_norm = load_assets()
    s, _c = O.new_state(N, mocap, obs_norm, np.full(N, np.float32(tables.total_mass())), tables.dof_lower,
                        tables.dof_upper, O.Params(), rng=rng)
    load_state(a, s)
    load_state(b, s)
    for c in (a, b):
        c.sim_t["root_states"][:, 0:3] = c.task_t["env_origins"] + torch.tensor([0.0, 0.0, 0.93], device=c.device)
    touched = 0.0
    for t in range(4):
        noise = O.draw_noise(N, 2, rng)
        actions = torch.tensor(rng.uniform(-1, 1, (N, 13)).astype(np.float32), device=a.device)
        inject_noise(a, noise)
        inject_noise(b, noise)
        a.step(actions)
        b.prologue(actions)
        for k in range(2):
            b.substep_torque()
            if k == 0:
                b.sim_t["rb_force"].zero_()
                b.sim_t["rb_force"].view(N, 38, 3)[:, 0, :] = b.task_t["push_force"]
                b.simulate(apply_wrench=True)
            else:
                b.simulate()
            b.sensor_noise(k)
        b.epilogue(); b.check_termination(); b.compute_reward(); b.compact_resets(); b.reset_idx(None)
        b.compute_observations(); b.late_update(); b.end_step()
        a.compact_resets()
        torch.cuda.synchronize()
        ga, gb = read_state(a), read_state(b)
        touched = max(touched, float(np.abs(ga["contact_forces_pre"]).max()))
        for g in (ga, gb):
            g["contact_forces_pre"] = g["contact_forces_pre"].reshape(N, 38, 3)[:, [8, 16]]
        for k in ga:
            assert np.array_equal(ga[k], gb[k], equal_nan=True), f"step {t}: {k} differs between fused and staged"
    assert touched > 100.0, "the robots should stand on the mesh"
    a.close(); b.close()


def test_terrain_mesh_resets_land_on_the_terrain_and_levels_move():
    N = 1024
    env = _walk(N, True)
    core = env.core
    levels0 = core.task_t["terrain_levels"].clone()
    core.sim_t["root_states"].fill_(7.0)
    core.reset_idx(torch.arange(N, device=core.device))
    torch.cuda.synchronize()
    r = core.sim_t["root_states"].cpu().numpy()
    o = core.task_t["env_origins"].cpu().numpy()
    assert np.abs(r[:, 0:2] - o[:, 0:2]).max() < 1e-6
    assert np.abs(r[:, 2] - (o[:, 2] + np.float32(0.93))).max() < 1e-6
    # origins of the sub-terrains lie on the mesh surface
    z, ok = core.cfg.triangle_mesh.height_at(o[:, 0].astype(np.float64), o[:, 1].astype(np.float64))
    assert ok.all() and np.abs(z - o[:, 2]).max() < 1e-3
    g = torch.Generator(device="cuda:0").manual_seed(1)
    for _ in range(200):
        env.step(torch.rand((N, 13), device="cuda:0", generator=g) * 2 - 1)
    torch.cuda.synchronize()
    moved = (core.task_t["terrain_levels"] != levels0).sum().item()
    assert moved > 0, "the curriculum moved no env"
    lvl = float(env.extras["episode"]["terrain_level"])
    assert abs(lvl - core.task_t["terrain_levels"].float().mean().item()) < 1e-4
    env.close()


def test_gym_facade_loop_on_triangle_mesh():
    from isaacgymdyros_b200 import gymapi, gymtorch
    N = 4
    gym = gymapi.acquire_gym()
    sp = gymapi.SimParams()
    sp.dt, sp.substeps, sp.up_axis = 0.002, 1, gymapi.UP_AXIS_Z
    sp.gravity = gymapi.Vec3(0.0, 0.0, -9.81)
    sp.physx.contact_offset, sp.physx.max_depenetration_velocity = 0.002, 10.0
    sim = gym.create_sim(0, -1, gymapi.SIM_PHYSX, sp)
    field = flat_field(z=0.3, size=(24.0, 6.0), origin_xy=(-3.0, -3.0))
    vertices, triangles = terrain.convert_heightfield_to_trimesh(field.samples, field.row_scale, field.vertical_scale, 0.75)
    tp = gymapi.TriangleMeshParams()
    tp.nb_vertices, tp.nb_triangles = vertices.shape[0], triangles.shape[0]
    tp.transform.p.x, tp.transform.p.y, tp.transform.p.z = field.origin
    tp.static_friction = tp.dynamic_friction = 1.0
    gym.add_triangle_mesh(sim, vertices.flatten(order="C"), triangles.flatten(order="C"), tp)
    ao = gymapi.AssetOptions()
    ao.angular_damping, ao.max_angular_velocity = 0.0, 100.0
    asset = gym.load_asset(sim, "../assets", "mjcf/dyros_tocabi/xml/dyros_tocabi.xml", ao)
    for i in range(N):
        env = gym.create_env(sim, gymapi.Vec3(0, 0, 0), gymapi.Vec3(0, 0, 0), 4)
        h = gym.create_actor(env, asset, gymapi.Transform(gymapi.Vec3(5.0 * i, 0.0, 0.3 + 0.93), gymapi.Quat(0, 0, 0, 1)),
                             "humanoid", i, 0, 0)
        props = gym.get_actor_dof_properties(env, h)
        props["damping"], props["velocity"], props["armature"] = 0.1, 4.03, 0.5
        gym.set_actor_dof_properties(env, h, props)
    assert gym.prepare_sim(sim)
    dof = gymtorch.wrap_tensor(gym.acquire_dof_state_tensor(sim))
    contact = gymtorch.wrap_tensor(gym.acquire_net_contact_force_tensor(sim))
    root = gymtorch.wrap_tensor(gym.acquire_actor_root_state_tensor(sim))
    dof.view(N, 33, 2)[:, :, 0] = torch.tensor(INIT_DOF_POS, device=dof.device)
    gym.set_dof_state_tensor(sim, gymtorch.unwrap_tensor(dof))
    q0 = dof.view(N, 33, 2)[:, :, 0].clone()
    for _ in range(150):
        tau = (2000.0 * (q0 - dof.view(N, 33, 2)[:, :, 0]) - 30.0 * dof.view(N, 33, 2)[:, :, 1]).reshape(-1).contiguous()
        gym.set_dof_actuation_force_tensor(sim, gymtorch.unwrap_tensor(tau))
        gym.simulate(sim)
        gym.refresh_dof_state_tensor(sim)
    gym.fetch_results(sim, True)
    gym.refresh_net_contact_force_tensor(sim)
    fz = contact.view(N, 38, 3)[:, :, 2].sum(1)
    assert ((fz - W).abs() < 0.08 * W).all(), fz
    assert ((root[:, 2] - 1.23).abs() < 0.03).all(), root[:, 2]
    gym.destroy_sim(sim)
