"""Terrain curriculum on the B200: the level update of the reset stage against tests/curriculum_oracle.py, fused step
against the staged sequence bit for bit (levels and the mean level included), the production draw of an env that
climbed past the top level, and DyrosDynamicWalk on the generated terrain."""
import numpy as np
import pytest
import torch

from isaacgymdyros_b200.core import CoreConfig, DyrosCore, TerrainCurriculum
from isaacgymdyros_b200.terrain import TerrainConfig, generate
from oracle import task_oracle as O
from tests import curriculum_oracle as CO
from tests.golden_util import load_assets
from tests.test_task_parity_gpu import inject_noise, load_state, read_state

pytestmark = pytest.mark.gpu
f32 = np.float32
UP, DOWN = 4.0, 16.0  # terrain_length / 2, episodeLength * 0.5


@pytest.fixture(scope="module")
def terrain():
    return generate(TerrainConfig(seed=11))


def curriculum_core(N, terrain, levels, types, **kw):
    hf, origins = terrain
    tc = TerrainCurriculum(origins, types.astype(np.int32), levels.astype(np.int32), UP, DOWN)
    return DyrosCore(N, "cuda:0", CoreConfig(heightfield=hf, terrain_curriculum=tc, **kw))


def oracle_state(N, rng):
    tables, mocap, obs_norm = load_assets()
    return O.new_state(N, mocap, obs_norm, np.full(N, f32(tables.total_mass())), tables.dof_lower, tables.dof_upper,
                       O.Params(), rng=rng)


def displaced_roots(origin_xy, tv, rng):
    """Root x-y of each env so that every branch of the update is taken, at least 1e-4 m from both thresholds, plus
    roots exactly at a threshold as float32 forms it (the oracle forms the same float32 distance)."""
    N = len(origin_xy)
    down_thr = np.sqrt(tv[:, 0] * tv[:, 0] + tv[:, 1] * tv[:, 1]) * f32(DOWN)
    kind = rng.integers(0, 5, N)
    d = np.where(kind == 0, rng.uniform(UP + 1e-4, 12.0, N),                                          # up
        np.where(kind == 1, rng.uniform(0.0, np.maximum(np.minimum(down_thr, UP) - 1e-4, 0.0)),     # down (or stay if tv = 0)
        np.where(kind == 2, rng.uniform(np.minimum(down_thr + 1e-4, UP - 2e-4), UP - 1e-4), UP)))  # stay / exactly UP
    d = np.where(kind == 4, down_thr, d)                                                           # exactly the down threshold
    ang = rng.uniform(0, 2 * np.pi, N)
    xy = np.stack([origin_xy[:, 0] + d * np.cos(ang), origin_xy[:, 1] + d * np.sin(ang)], 1)
    xy[kind >= 3, 1] = origin_xy[kind >= 3, 1]  # threshold cases along x only
    xy[kind >= 3, 0] = (origin_xy[kind >= 3, 0].astype(np.float64) + d[kind >= 3]).astype(f32)
    return xy.astype(f32), kind


def test_kernel_level_update_matches_oracle(terrain):
    N = 1000
    rng = np.random.default_rng(5)
    hf, origins = terrain
    L, T = origins.shape[:2]
    levels = rng.integers(0, L, N)
    levels[:100] = L - 1  # many envs at the top level: the overflow draw
    types = rng.integers(0, T, N)
    core = curriculum_core(N, terrain, levels, types, self_collision=False)
    s, c = oracle_state(N, rng)
    s["env_origins"] = core.task_t["env_origins"].cpu().numpy()
    np.testing.assert_array_equal(s["env_origins"], origins.astype(f32)[levels, types])
    s["target_vel"] = np.stack([rng.uniform(0, 0.8, N), rng.uniform(-0.1, 0.1, N)], 1).astype(f32)
    s["target_vel"][::7] = 0.0
    xy, kind = displaced_roots(s["env_origins"][:, 0:2], s["target_vel"], rng)
    s["root_states"][:, 0:2] = xy
    load_state(core, s)
    noise = O.draw_noise(N, 2, rng)
    inject_noise(core, noise)
    cur = {"origins": origins.astype(f32), "types": types.astype(np.int32), "levels": levels.astype(np.int32),
           "move_up_distance": UP, "move_down_scale": DOWN}
    before = levels.copy()
    CO.reset_idx(s, c, np.arange(N), noise, cur)
    core.reset_idx(torch.arange(N, device=core.device))
    torch.cuda.synchronize()
    got_levels = core.task_t["terrain_levels"].cpu().numpy()
    np.testing.assert_array_equal(got_levels, cur["levels"])
    np.testing.assert_array_equal(core.task_t["env_origins"].cpu().numpy(), s["env_origins"])
    r = core.sim_t["root_states"].cpu().numpy()
    assert np.abs(r - s["root_states"]).max() < 1e-6
    # every branch was taken
    moved = got_levels.astype(int) - before
    assert (moved == 1).sum() > 50 and (moved == -1).sum() > 50 and (moved == 0).sum() > 50
    assert ((before == L - 1) & (got_levels < L - 1) & (kind == 0)).sum() > 5, "overflow redraws"
    assert (kind >= 3).sum() > 100
    core.close()


def test_fused_step_equals_staged_with_curriculum(terrain):
    N = 257
    rng = np.random.default_rng(3)
    hf, origins = terrain
    L, T = origins.shape[:2]
    levels, types = rng.integers(0, L, N), np.floor(np.arange(N) / (N / T)).astype(np.int32)
    a = curriculum_core(N, terrain, levels, types, with_rb_force_tensors=True)
    b = curriculum_core(N, terrain, levels, types, with_rb_force_tensors=True)
    s, _c = oracle_state(N, rng)
    s["progress_buf"][::3] = 7999  # time-outs at the first step: resets with the curriculum
    load_state(a, s)
    load_state(b, s)
    jump = torch.tensor(rng.uniform(-7, 7, (N, 2)).astype(f32), device=a.device)
    for core in (a, b):
        core.sim_t["root_states"][:, 0:3] = core.task_t["env_origins"] + torch.tensor([0.0, 0.0, 0.93], device=core.device)
        core.sim_t["root_states"][:, 0:2] += jump
    level_moves = 0
    for t in range(5):
        noise = O.draw_noise(N, 2, rng)
        actions = torch.tensor(rng.uniform(-1, 1, (N, 13)).astype(np.float32), device=a.device)
        inject_noise(a, noise)
        inject_noise(b, noise)
        lv0 = a.task_t["terrain_levels"].clone()
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
        level_moves += int((a.task_t["terrain_levels"] != lv0).sum())
        ga, gb = read_state(a), read_state(b)
        for g in (ga, gb):
            g["contact_forces_pre"] = g["contact_forces_pre"].reshape(N, 38, 3)[:, [8, 16]]
        assert "terrain_levels" in ga and "terrain_level_mean" in ga
        for k in ga:
            assert np.array_equal(ga[k], gb[k], equal_nan=True), f"step {t}: {k} differs between fused and staged"
        lv = ga["terrain_levels"]
        assert ga["terrain_level_mean"] == np.float32(lv.astype(np.float64).mean())
    assert level_moves > 50, level_moves
    a.close(); b.close()


def test_production_draw_past_the_top_is_uniform(terrain):
    N = 8192
    hf, origins = terrain
    L, T = origins.shape[:2]
    core = curriculum_core(N, terrain, np.full(N, L - 1), np.arange(N) % T, self_collision=False)
    core.sim_t["root_states"][:, 0:2] = core.task_t["env_origins"][:, 0:2] + torch.tensor([6.0, 0.0], device=core.device)
    core.reset_idx(torch.arange(N, device=core.device))
    torch.cuda.synchronize()
    lv = core.task_t["terrain_levels"].cpu().numpy()
    counts = np.bincount(lv, minlength=L)
    assert len(counts) == L
    chi2 = ((counts - N / L) ** 2 / (N / L)).sum()
    assert chi2 < 27.88, (chi2, counts)  # 9 degrees of freedom, p = 0.001
    types = core.task_t["terrain_types"].cpu().numpy()
    np.testing.assert_array_equal(core.task_t["env_origins"].cpu().numpy(), origins.astype(f32)[lv, types])
    core.close()


def walk_env(N, curriculum):
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    cfg = default_cfg(N)
    cfg["env"]["terrain"] = {"curriculum": curriculum, "seed": 2}
    return DyrosDynamicWalk(cfg, "cuda:0")


@pytest.mark.parametrize("curriculum", [True, False])
def test_dynamic_walk_loop_on_generated_terrain(curriculum):
    N, steps = 4096, 300 if curriculum else 120
    env = walk_env(N, curriculum)
    rows = 10
    lv0 = env.terrain_levels.clone()
    assert int(lv0.max()) <= (5 if curriculum else rows - 1)
    torch.testing.assert_close(env.core.task_t["env_origins"], env.terrain_origins[lv0.long(), env.terrain_types.long()],
                               rtol=0, atol=0)
    g = torch.Generator(device="cuda:0").manual_seed(0)
    resets = 0
    for i in range(steps):
        act = torch.rand(N, 13, device="cuda:0", generator=g) * 2 - 1
        _obs, _rew, reset, extras = env.step(act)
        done = reset.bool()
        resets += int(done.sum())
        o = env.core.task_t["env_origins"]
        r = env.root_states
        assert (r[done, 0:2] - o[done, 0:2]).abs().max().item() < 1e-6 if done.any() else True
        assert (r[done, 2] - (o[done, 2] + 0.93)).abs().max().item() < 1e-6 if done.any() else True
        if curriculum:
            assert extras["episode"]["terrain_level"].dim() == 0
            assert extras["episode"]["terrain_level"].item() == env.terrain_levels.float().mean().item()
        if i % 50 == 0 or i == steps - 1:
            assert torch.isfinite(env.root_states).all() and torch.isfinite(env.obs_buf).all()
            assert int(env.terrain_levels.min()) >= 0 and int(env.terrain_levels.max()) < rows
            torch.testing.assert_close(o, env.terrain_origins[env.terrain_levels.long(), env.terrain_types.long()],
                                       rtol=0, atol=0)
    assert resets > 100, resets
    if curriculum:
        assert "terrain_level" in extras["episode"]
        assert int((env.terrain_levels != lv0).sum()) > min(resets // 4, N // 10)
    else:
        assert "episode" not in extras
        assert torch.equal(env.terrain_levels, lv0)
    assert env.core.step_launches() == 3
    env.close()
