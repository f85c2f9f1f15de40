"""Heightfield ground on the B200: the CUDA role program (Ground = FieldGround) against the fp64 oracle on each kind of
field, flat field against plane, weight on the feet on raised and sloped ground, fused step against the staged
sequence, resets onto the terrain, a ragged multi-wave N, the lanes program's refusal and the gym facade."""
import numpy as np
import pytest
import torch

from isaacgymdyros_b200 import native
from isaacgymdyros_b200.core import CoreConfig, HeightField, INIT_DOF_POS, KP, KV
from oracle.physics_oracle import PhysicsOracle
from tests.golden_util import load_assets
from tests.physics_util import oracle_params, random_states
from tests.terrain_oracle import TerrainOracle
from tests.terrain_util import flat_field, ramp_field, rough_field, stairs_field
from tests.test_physics_emulation import compare
from tests.test_physics_parity_gpu import load_sim_state, read_sim_state
from tests.test_terrain import FIELDS, terrain_states

pytestmark = pytest.mark.gpu
W = 104.48712 * 9.81  # TOCABI's weight (N)


def core_field(f):
    """tests' oracle HeightField -> the product's (DyrosCore) HeightField."""
    return HeightField(np.asarray(f.samples, np.int16), f.row_scale, f.column_scale, f.vertical_scale, tuple(f.origin))


def sim_core(N, field, **kw):
    from isaacgymdyros_b200.core import DyrosCore
    cfg = CoreConfig(self_collision=False, heightfield=core_field(field) if field is not None else None, **kw)
    return DyrosCore(N, "cuda:0", cfg, with_task=False), cfg


def run_simulate(N, field, st):
    core, _ = sim_core(N, field)
    load_sim_state(core, st)
    core.simulate()
    torch.cuda.synchronize()
    out = read_sim_state(core)
    core.close()
    return out


def oracle(field, st, cfg=None):
    o = TerrainOracle(load_assets()[0], oracle_params(cfg or CoreConfig()), ground=field)
    return o.substep(st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"], st["mass_scale"])


@pytest.mark.parametrize("kind", ["stand", "mixed"])
@pytest.mark.parametrize("name", list(FIELDS))
def test_cuda_simulate_on_field_matches_oracle(name, kind):
    field = FIELDS[name]()
    st = terrain_states(field, kind, seed=5, N=96)
    # On the field raised by 0.25 m the base stands above z = 1 m, where float32 positions are spaced twice as widely as
    # below it: the same batch in the host emulation has 1.7 x the joint-velocity error it has on the plane
    # (4.0e-4 against 2.4e-4; the same at z = -0.25 as at z = 0), so the raised stance gets 1.5 x the tolerance.
    slack = 1.5 if name == "raised" else 1.0
    compare(st, run_simulate(96, field, st), oracle(field, st), ctx=f"{name} {kind}: ", slack=slack)


def test_cuda_flat_field_matches_plane():
    """A flat field at z = 0 against the plane kernel, at the oracle's tolerance (the two are different instantiations
    of the role program, compiled separately)."""
    tables = load_assets()[0]
    st = random_states(300, np.random.default_rng(2), tables, "mixed")
    plane = run_simulate(300, None, st)
    flat = run_simulate(300, flat_field(), st)
    want = PhysicsOracle(tables, oracle_params(CoreConfig())).substep(
        st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"], st["mass_scale"])
    compare(st, plane, want, ctx="plane: ")
    compare(st, flat, want, ctx="flat field: ")
    compare(st, flat, plane, ctx="flat field vs plane: ")


def grid_field(kind, N, spacing=5.0):
    """A field under the default env grid (T:709-718) of N envs: 'raised' flat at 0.3 m, 'slope' rising 2 % along x."""
    n = int(np.ceil(np.sqrt(N))) + 1
    size = spacing * n
    if kind == "raised":
        return flat_field(z=0.3, size=(size, size), origin_xy=(-2.0, -2.0), spacing=0.5)
    return ramp_field(slope=0.02, size=(size, size), origin_xy=(-2.0, -2.0), spacing=0.25, vscale=0.005)


@pytest.mark.parametrize("kind", ["raised", "slope"])
def test_cuda_standing_on_terrain_carries_weight_on_feet_only(kind):
    from isaacgymdyros_b200.core import DyrosCore
    N = 1024
    field = grid_field(kind, N)
    core = DyrosCore(N, "cuda:0", CoreConfig(heightfield=core_field(field), self_collision=False))
    dev = core.device
    origins = core.task_t["env_origins"].clone()
    h = torch.tensor(field.query(origins[:, 0].cpu().numpy(), origins[:, 1].cpu().numpy())[0], dtype=torch.float32, device=dev)
    assert (origins[:, 2] - h).abs().max().item() < 1e-4, "default origins sit on the terrain"
    assert (core.sim_t["root_states"][:, 2] - origins[:, 2] - 0.93).abs().max().item() < 1e-5
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
    assert (core.sim_t["root_states"][:, 2] - origins[:, 2] - 0.93).abs().max().item() < 0.02
    core.close()


def test_fused_step_equals_staged_sequence_on_terrain():
    from isaacgymdyros_b200.core import DyrosCore
    from oracle import task_oracle as O
    from tests.test_task_parity_gpu import inject_noise, load_state, read_state
    N = 257
    field = rough_field(size=(100.0, 100.0), origin_xy=(-5.0, -5.0), spacing=0.25)
    cfg = CoreConfig(with_rb_force_tensors=True, heightfield=core_field(field))
    a, b = DyrosCore(N, "cuda:0", cfg), DyrosCore(N, "cuda:0", cfg)
    rng = np.random.default_rng(3)
    tables, mocap, obs_norm = load_assets()
    s, _c = O.new_state(N, mocap, obs_norm, np.full(N, np.float32(tables.total_mass())), tables.dof_lower,
                        tables.dof_upper, O.Params(), rng=rng)
    load_state(a, s)
    load_state(b, s)
    for c in (a, b):  # on the terrain: every env starts at its origin
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
    assert touched > 100.0, "the robots should stand on the field"
    a.close(); b.close()


def test_reset_puts_root_on_the_terrain():
    from isaacgymdyros_b200.core import DyrosCore
    N = 64
    field = rough_field(size=(50.0, 50.0), origin_xy=(-5.0, -5.0), spacing=0.25, amp=0.2)
    origins = np.random.default_rng(0).uniform(-4.0, 40.0, (N, 3))
    origins[:, 2] = field.query(origins[:, 0], origins[:, 1])[0]
    hf = core_field(field)
    hf.env_origins = origins
    core = DyrosCore(N, "cuda:0", CoreConfig(heightfield=hf))
    core.sim_t["root_states"].fill_(7.0)
    core.reset_idx(torch.arange(N, device=core.device))
    torch.cuda.synchronize()
    r = core.sim_t["root_states"].cpu().numpy()
    o = origins.astype(np.float32)
    assert np.abs(r[:, 0:2] - o[:, 0:2]).max() < 1e-6
    assert np.abs(r[:, 2] - (o[:, 2] + np.float32(0.93))).max() < 1e-6
    core.close()


def test_ragged_multi_wave_n_matches_oracle():
    """N = 2 waves of 148 CTAs plus a partial CTA; the oracle checks a sample of envs that includes the last ones."""
    N = 28 * 148 * 2 + 13
    field = stairs_field(size=(8.0, 8.0), origin_xy=(-4.0, -4.0))
    st = terrain_states(field, "mixed", seed=9, N=N)
    got = run_simulate(N, field, st)
    idx = np.r_[np.random.default_rng(1).choice(N - 40, 60, replace=False), np.arange(N - 40, N)]
    sub = {k: v[idx] for k, v in st.items()}
    compare(sub, tuple(g[idx] for g in got), oracle(field, sub), ctx="ragged: ")


def test_terrain_cta_holds_28_envs_on_the_gpu():
    core, _ = sim_core(4096, flat_field())
    info = core.launch_info()
    assert info["envs_per_cta"] == 28 and info["ctas"] == 147, info
    core.close()


def test_lanes_program_refuses_a_heightfield():
    import ctypes as C
    with pytest.raises(native.DyrosError, match="lanes"):
        sim_core(8, flat_field(), physics_program="lanes")
    core, _ = sim_core(8, None, physics_program="lanes")
    s = torch.zeros(4, 4, dtype=torch.int16, device=core.device)
    d = native.DyrosHeightField()
    d.samples = s.data_ptr()
    d.num_rows = d.num_columns = 4
    d.row_scale = d.column_scale = d.vertical_scale = 0.1
    rc = core.lib.dyros_sim_set_heightfield(core.sim_handle, C.byref(d))
    assert rc != 0 and b"lanes" in core.lib.dyros_last_error()
    core.close()


def test_origin_outside_the_field_is_an_error():
    from isaacgymdyros_b200.core import DyrosCore
    with pytest.raises(native.DyrosError, match="outside the field"):
        DyrosCore(64, "cuda:0", CoreConfig(heightfield=core_field(flat_field())))


def test_gym_facade_loop_on_heightfield():
    from isaacgymdyros_b200 import gymapi, gymtorch
    N = 4
    gym = gymapi.acquire_gym()
    sp = gymapi.SimParams()
    sp.dt, sp.substeps, sp.up_axis = 0.002, 1, gymapi.UP_AXIS_Z
    sp.gravity = gymapi.Vec3(0.0, 0.0, -9.81)
    sp.physx.contact_offset, sp.physx.max_depenetration_velocity = 0.002, 10.0
    sim = gym.create_sim(0, -1, gymapi.SIM_PHYSX, sp)
    field = flat_field(z=0.3, size=(24.0, 6.0), origin_xy=(-3.0, -3.0))
    hp = gymapi.HeightFieldParams()
    hp.nbRows, hp.nbColumns = field.samples.shape
    hp.row_scale, hp.column_scale, hp.vertical_scale = field.row_scale, field.column_scale, field.vertical_scale
    hp.transform.p = gymapi.Vec3(*field.origin)
    gym.add_heightfield(sim, field.samples.reshape(-1), hp)
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
