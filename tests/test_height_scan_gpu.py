"""Height scan on the B200: the observation kernels against tests/height_scan_oracle.py (staged and fused, generated
field, random poses, far-off roots, the plane, ragged N), fused against staged steps bit for bit, an env with the scan
against the same env without it, the post-reset root of a reset env, and DyrosDynamicWalk with measure_heights."""
import dataclasses

import numpy as np
import pytest
import torch

from isaacgymdyros_b200.core import CoreConfig, DyrosCore, TerrainCurriculum
from isaacgymdyros_b200.terrain import TerrainConfig, generate, height_points
from oracle import task_oracle as O
from tests import height_scan_oracle as H
from tests.golden_util import load_assets
from tests.test_task_parity_gpu import inject_noise, load_state, read_state

pytestmark = pytest.mark.gpu
f32 = np.float32
POINTS = height_points(TerrainConfig(measure_heights=True))  # legged_gym's 17 x 11 grid


@pytest.fixture(scope="module")
def terrain():
    return generate(TerrainConfig(seed=11))


def field_extent(hf):
    nr, nc = hf.samples.shape
    return (hf.origin[0], hf.origin[0] + (nr - 1) * hf.row_scale), (hf.origin[1], hf.origin[1] + (nc - 1) * hf.column_scale)


def scan_core(N, hf, points=POINTS, origins=None, **kw):
    if hf is not None:
        if origins is None:
            (x0, x1), (y0, y1) = field_extent(hf)
            origins = np.zeros((N, 3))
            origins[:, 0] = np.linspace(x0 + 1, x1 - 1, N)
            origins[:, 1] = np.linspace(y0 + 1, y1 - 1, N)[::-1]
        hf = dataclasses.replace(hf, env_origins=origins)
    kw.setdefault("self_collision", False)
    return DyrosCore(N, "cuda:0", CoreConfig(heightfield=hf, height_scan=points, **kw))


def random_roots(N, hf, rng, far=False):
    """Root poses: x-y over the field (or +-1e6 m), a random yaw plus a tilt, z in [-2, 3] m."""
    r = np.zeros((N, 13), f32)
    if far:
        r[:, 0:2] = rng.choice([-1e6, 1e6], (N, 2)) + rng.uniform(-1, 1, (N, 2))
    else:
        (x0, x1), (y0, y1) = field_extent(hf)
        r[:, 0], r[:, 1] = rng.uniform(x0 - 2, x1 + 2, N), rng.uniform(y0 - 2, y1 + 2, N)
    r[:, 2] = rng.uniform(-2, 3, N)
    yaw, tilt, ax = rng.uniform(-np.pi, np.pi, N), rng.uniform(0, 0.6, N), rng.uniform(0, 2 * np.pi, N)
    qy = np.stack([np.zeros(N), np.zeros(N), np.sin(yaw / 2), np.cos(yaw / 2)], 1)
    qt = np.stack([np.cos(ax) * np.sin(tilt / 2), np.sin(ax) * np.sin(tilt / 2), np.zeros(N), np.cos(tilt / 2)], 1)
    x1, y1, z1, w1 = qy.T
    x2, y2, z2, w2 = qt.T
    q = np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                  w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], 1)
    r[:, 3:7] = q
    r[:, 7:13] = rng.normal(0, 0.3, (N, 6))
    return r


def assert_scan_matches_oracle(core, hf, points=POINTS):
    """measured_heights and the obs columns of the root now in root_states: exact, except that a point within 1e-5 grid
    units of a cell boundary may take either neighbour's cell."""
    torch.cuda.synchronize()
    r = core.sim_t["root_states"].cpu().numpy()
    got_h = core.task_t["measured_heights"].cpu().numpy()
    obs = core.task_t["obs_buf"].cpu().numpy()
    assert obs.shape == (core.N, 487 + len(points))
    want = H.heights(r, points, hf)
    bad = got_h != want
    if bad.any():
        wx, wy = H.world_points(r, points)
        u = (wx.astype(np.float64) - hf.origin[0]) / hf.row_scale
        v = (wy.astype(np.float64) - hf.origin[1]) / hf.column_scale
        near = (np.abs(u - np.rint(u)) < 1e-5) | (np.abs(v - np.rint(v)) < 1e-5)
        assert near[bad].all(), f"{int((bad & ~near).sum())} heights differ away from cell boundaries"
        ix, iy = H.cell_index(wx, wy, hf)
        nr, nc = hf.samples.shape
        ok = np.zeros_like(bad)
        for di in (-1, 0, 1):
            for dj in (-1, 0, 1):
                ok |= got_h == H.heights_at(np.clip(ix + di, 0, nr - 2), np.clip(iy + dj, 0, nc - 2), hf)
        assert ok[bad].all()
    np.testing.assert_array_equal(obs[:, 487:], H.obs_columns(r, got_h))
    return r, got_h


@pytest.mark.parametrize("path", ["staged", "fused"])
def test_kernel_matches_oracle_on_the_generated_field(terrain, path):
    hf, _ = terrain
    N = 1000
    rng = np.random.default_rng(1 if path == "staged" else 2)
    core = scan_core(N, hf)
    core.sim_t["root_states"].copy_(torch.tensor(random_roots(N, hf, rng), device=core.device))
    if path == "staged":
        core.compute_observations()
    else:
        core.post_step()  # (tilted envs terminate and reset: their heights are those of the post-reset root)
    r, h = assert_scan_matches_oracle(core, hf)
    assert np.ptp(h) > 0.5 and len(np.unique(h)) > 100
    core.close()


def test_far_off_roots_take_the_edge_samples(terrain):
    hf, _ = terrain
    N = 256
    core = scan_core(N, hf)
    core.sim_t["root_states"].copy_(torch.tensor(random_roots(N, hf, np.random.default_rng(3), far=True), device=core.device))
    core.compute_observations()
    r, h = assert_scan_matches_oracle(core, hf)
    s = hf.samples
    edge = np.concatenate([s[:2].ravel(), s[-2:].ravel(), s[:, :2].ravel(), s[:, -2:].ravel()])
    assert np.isin(np.rint((h - hf.origin[2]) / f32(hf.vertical_scale)), edge).all()
    core.close()


def test_plane_heights_are_zero():
    N = 100
    core = scan_core(N, None)
    rng = np.random.default_rng(4)
    r = random_roots(N, None, rng, far=True)
    r[:50, 0:2] = rng.uniform(-50, 50, (50, 2))
    core.sim_t["root_states"].copy_(torch.tensor(r, device=core.device))
    core.compute_observations()
    torch.cuda.synchronize()
    h = core.task_t["measured_heights"].cpu().numpy()
    assert h.shape == (N, 187) and not h.any()
    np.testing.assert_array_equal(core.task_t["obs_buf"].cpu().numpy()[:, 487:], H.obs_columns(r, h))
    core.close()


@pytest.mark.parametrize("N", [1, 33, 1025])
def test_ragged_n(terrain, N):
    hf, _ = terrain
    for path in ("staged", "fused"):
        core = scan_core(N, hf)
        core.sim_t["root_states"].copy_(torch.tensor(random_roots(N, hf, np.random.default_rng(N)), device=core.device))
        core.compute_observations() if path == "staged" else core.post_step()
        assert_scan_matches_oracle(core, hf)
        core.close()


def oracle_state(N, rng):
    tables, mocap, obs_norm = load_assets()
    return O.new_state(N, mocap, obs_norm, np.full(N, f32(tables.total_mass())), tables.dof_lower, tables.dof_upper,
                       O.Params(), rng=rng)


def load_wide(core, s):
    """load_state for a core whose obs_buf rows are wider than the oracle's 487 columns."""
    full = core.task_t["obs_buf"]
    core.task_t["obs_buf"] = full[:, :487]
    try:
        load_state(core, s)
    finally:
        core.task_t["obs_buf"] = full


def curriculum_cores(N, terrain, rng, scans):
    hf, origins = terrain
    L, T = origins.shape[:2]
    levels, types = rng.integers(0, L, N).astype(np.int32), np.floor(np.arange(N) / (N / T)).astype(np.int32)
    cores = [DyrosCore(N, "cuda:0", CoreConfig(heightfield=hf, with_rb_force_tensors=True, height_scan=p,
                                               terrain_curriculum=TerrainCurriculum(origins, types, levels, 4.0, 16.0)))
             for p in scans]
    s, _c = oracle_state(N, rng)
    s["progress_buf"][::3] = 7999  # time-outs at the first step
    jump = torch.tensor(rng.uniform(-3, 3, (N, 2)).astype(f32), device=cores[0].device)
    for core in cores:
        load_wide(core, s)
        core.sim_t["root_states"][:, 0:3] = core.task_t["env_origins"] + torch.tensor([0.0, 0.0, 0.93], device=core.device)
        core.sim_t["root_states"][:, 0:2] += jump
    return cores


def staged(b, actions):
    N = b.N
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


def test_fused_step_equals_staged_with_scan(terrain):
    N = 257
    rng = np.random.default_rng(5)
    a, b = curriculum_cores(N, terrain, rng, [POINTS, POINTS])
    for t in range(5):
        noise = O.draw_noise(N, 2, rng)
        actions = torch.tensor(rng.uniform(-1, 1, (N, 13)).astype(f32), device=a.device)
        inject_noise(a, noise)
        inject_noise(b, noise)
        a.step(actions)
        staged(b, actions)
        a.compact_resets()
        torch.cuda.synchronize()
        ga, gb = read_state(a), read_state(b)
        for g in (ga, gb):
            g["contact_forces_pre"] = g["contact_forces_pre"].reshape(N, 38, 3)[:, [8, 16]]
        assert ga["obs_buf"].shape == (N, 674) and "measured_heights" in ga
        for k in ga:
            assert np.array_equal(ga[k], gb[k], equal_nan=True), f"step {t}: {k} differs between fused and staged"
        assert_scan_matches_oracle(a, terrain[0])
    a.close(); b.close()


def test_scan_changes_nothing_else(terrain):
    N = 512
    rng = np.random.default_rng(6)
    on, off = curriculum_cores(N, terrain, rng, [POINTS, None])
    g = torch.Generator(device="cuda:0").manual_seed(1)
    resets = 0
    for t in range(40):
        actions = torch.rand(N, 13, device="cuda:0", generator=g) * 2 - 1
        on.step(actions)
        off.step(actions)
        torch.cuda.synchronize()
        resets += int(off.task_t["reset_buf"].sum())
        ga, gb = read_state(on), read_state(off)
        assert np.array_equal(ga.pop("obs_buf")[:, :487], gb.pop("obs_buf"))
        ga.pop("measured_heights"), ga.pop("height_points")
        assert ga.keys() == gb.keys()
        for k in gb:
            assert np.array_equal(ga[k], gb[k], equal_nan=True), f"step {t}: {k} differs with the scan on"
    assert resets > 0
    on.close(); off.close()


def test_reset_env_sees_its_post_reset_root(terrain):
    N = 256
    rng = np.random.default_rng(7)
    hf, _ = terrain
    core = scan_core(N, hf, with_rb_force_tensors=True)
    s, _c = oracle_state(N, rng)
    load_wide(core, s)
    r = random_roots(N, hf, rng)
    r[:, 3:7] = (0, 0, 0, 1)
    core.sim_t["root_states"].copy_(torch.tensor(r, device=core.device))
    forced = np.zeros(N, bool)
    forced[::2] = True
    core.task_t["progress_buf"][torch.tensor(forced, device=core.device)] = 7999  # time-out now: reset in this step
    core.post_step()
    torch.cuda.synchronize()
    assert core.task_t["reset_buf"].cpu().numpy()[forced].all()
    after = core.sim_t["root_states"].cpu().numpy()
    org = core.task_t["env_origins"].cpu().numpy()
    np.testing.assert_array_equal(after[forced, 0:2], org[forced, 0:2])  # the reset moved them home ...
    _r, h = assert_scan_matches_oracle(core, hf)                         # ... and the heights are measured there
    moved = np.abs(r[forced, 0:2] - org[forced, 0:2]).max(1) > 1.0
    assert moved.sum() > 50
    assert not np.array_equal(h[forced][moved], H.heights(r[forced][moved], POINTS, hf))
    core.close()


def walk_env(N, **terrain):
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    cfg = default_cfg(N)
    cfg["env"]["terrain"] = {"seed": 2, **terrain}
    return DyrosDynamicWalk(cfg, "cuda:0")


def test_dynamic_walk_with_measure_heights():
    N = 4096
    env = walk_env(N, measure_heights=True)
    pipe = walk_env(N, measure_heights=True)
    assert env.num_obs == 674 and env.observation_space.shape == (674,) and env.num_height_points == 187
    assert env.measured_heights.shape == (N, 187) and env.terrain_level_mean is not None
    g = torch.Generator(device="cuda:0").manual_seed(0)
    resets = 0
    for i in range(60):
        act = torch.rand(N, 13, device="cuda:0", generator=g) * 2 - 1
        obs, _rew, reset, _extras = env.step(act)
        obs = obs["obs"].clone()
        o2, rew2, reset2, ex2 = pipe.step_wait(pipe.step_async(act))
        resets += int(reset.sum())
        assert obs.shape == (N, 674) and torch.isfinite(obs).all()
        hc = obs[:, 487:]
        assert hc.min() >= -5 and hc.max() <= 5
        assert torch.equal(o2["obs"], obs.cpu()), f"step {i}: step_async / step_wait obs differ from step"
        assert torch.equal(rew2, env.rew_buf.cpu()) and torch.equal(reset2, reset.cpu())
        assert torch.equal(ex2["time_outs"], env.timeout_buf.cpu())
    assert resets > 0
    assert env.core.step_launches() == 3
    from isaacgymdyros_b200.ppo import PPOTrainer
    with pytest.raises(ValueError, match="height scan"):
        PPOTrainer(env)
    env.close(); pipe.close()
