"""Terrain curriculum on the CPU: the generator (isaacgymdyros_b200/terrain.py) against known answers, the oracle of the
level update (tests/curriculum_oracle.py) on hand-built cases, the cfg["env"]["terrain"] plumbing of the task, and the
C ABI's new entry point."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

from isaacgymdyros_b200 import native
from isaacgymdyros_b200.terrain import TerrainConfig, generate
from tests.curriculum_oracle import f32, reset_idx, update_levels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def default_terrain():
    cfg = TerrainConfig(seed=3)
    return cfg, *generate(cfg)


def sub(cfg, samples, i, j):
    """Samples of sub-terrain (i, j)."""
    b = int(cfg.border_size / cfg.horizontal_scale)
    lx, ly = int(cfg.terrain_length / cfg.horizontal_scale), int(cfg.terrain_width / cfg.horizontal_scale)
    return samples[b + i * lx:b + (i + 1) * lx, b + j * ly:b + (j + 1) * ly].astype(np.int64)


def kind_columns(cfg):
    """Columns of each kind under the curriculum (choice j / num_cols + 0.001)."""
    cum = np.cumsum(cfg.terrain_proportions)
    ch = np.arange(cfg.num_cols) / cfg.num_cols + 0.001
    return {"slope_down": np.flatnonzero(ch < cum[0] / 2), "slope_up": np.flatnonzero((ch >= cum[0] / 2) & (ch < cum[0])),
            "rough": np.flatnonzero((ch >= cum[0]) & (ch < cum[1])),
            "stairs": np.flatnonzero((ch >= cum[1]) & (ch < cum[3])), "obstacles": np.flatnonzero(ch >= cum[3])}


# ------------------------------------------------------------------ generator
def test_field_shape_border_and_transform(default_terrain):
    cfg, hf, origins = default_terrain
    b = 2 * cfg.border_size / cfg.horizontal_scale
    assert hf.samples.shape == (round(b + cfg.num_rows * cfg.terrain_length / cfg.horizontal_scale),
                                round(b + cfg.num_cols * cfg.terrain_width / cfg.horizontal_scale)) == (1300, 2100)
    assert hf.samples.dtype == np.int16
    assert hf.origin == (-cfg.border_size, -cfg.border_size, 0.0)
    assert hf.row_scale == hf.column_scale == cfg.horizontal_scale and hf.vertical_scale == cfg.vertical_scale
    nb = int(cfg.border_size / cfg.horizontal_scale)
    s = hf.samples
    assert not s[:nb].any() and not s[-nb:].any() and not s[:, :nb].any() and not s[:, -nb:].any(), "flat border"
    assert origins.shape == (cfg.num_rows, cfg.num_cols, 3)


def test_row_0_slopes_are_flat_and_slopes_grow_down_the_rows(default_terrain):
    cfg, hf, _ = default_terrain
    cols = kind_columns(cfg)
    for j in np.r_[cols["slope_down"], cols["slope_up"]]:
        assert not sub(cfg, hf.samples, 0, j).any(), f"column {j}: difficulty 0 is flat"
        tops = [np.abs(sub(cfg, hf.samples, i, j)).max() for i in range(cfg.num_rows)]
        assert all(a <= b for a, b in zip(tops, tops[1:])) and tops[-1] > tops[1] > 0, tops
    for j in cols["slope_up"]:
        assert sub(cfg, hf.samples, 5, j).min() >= 0
    for j in cols["slope_down"]:
        assert sub(cfg, hf.samples, 5, j).max() <= 0


def test_stair_risers(default_terrain):
    cfg, hf, _ = default_terrain
    cols = kind_columns(cfg)
    cum = np.cumsum(cfg.terrain_proportions)
    for j in cols["stairs"]:
        sign = -1 if j / cfg.num_cols + 0.001 < cum[2] else 1
        for i in range(cfg.num_rows):
            riser = int((0.05 + 0.18 * i / cfg.num_rows) / cfg.vertical_scale)  # truncated as terrain_utils does
            h = sub(cfg, hf.samples, i, j)
            line = h[:, h.shape[1] // 2]  # along x through the centre: 0, then one riser per 0.31 m step
            steps = np.diff(line[:len(line) // 2])
            steps = steps[steps != 0]
            assert len(steps) >= 3 and np.all(steps == sign * riser), (i, j, riser, steps)


def test_origins_lie_on_the_field_at_the_central_patch_maximum(default_terrain):
    cfg, hf, origins = default_terrain
    hs, vs = cfg.horizontal_scale, cfg.vertical_scale
    inside = hf.height_at(origins[..., 0], origins[..., 1])[1]
    assert inside.all()
    x1, x2 = int((cfg.terrain_length / 2 - 1) / hs), int((cfg.terrain_length / 2 + 1) / hs)
    y1, y2 = int((cfg.terrain_width / 2 - 1) / hs), int((cfg.terrain_width / 2 + 1) / hs)
    for i in range(cfg.num_rows):
        for j in range(cfg.num_cols):
            np.testing.assert_allclose(origins[i, j, :2], [(i + 0.5) * cfg.terrain_length, (j + 0.5) * cfg.terrain_width])
            assert origins[i, j, 2] == sub(cfg, hf.samples, i, j)[x1:x2, y1:y2].max() * vs
    # the root of an env placed there stands on the terrain, not inside it
    h = hf.height_at(origins[..., 0], origins[..., 1])[0]
    assert np.all(origins[..., 2] >= h - 1e-9)


def test_same_seed_same_field():
    small = dict(num_rows=3, num_cols=5, terrain_length=4.0, terrain_width=4.0, border_size=2.0)
    for cur in (True, False):
        a, b = generate(TerrainConfig(curriculum=cur, seed=7, **small)), generate(TerrainConfig(curriculum=cur, seed=7, **small))
        assert np.array_equal(a[0].samples, b[0].samples) and np.array_equal(a[1], b[1])
    c = generate(TerrainConfig(curriculum=False, seed=8, **small))
    assert not np.array_equal(a[0].samples, c[0].samples)


@pytest.mark.parametrize("kw, match", [
    (dict(terrain_proportions=[0.1, 0.1, 0.3, 0.2, 0.2, 0.1]), "at most 5"),
    (dict(terrain_proportions=[0.1, 0.1, 0.35, 0.25, 0.1]), "sum to 1"),
    (dict(vertical_scale=1e-5), "overflow int16"),
    (dict(mesh_type="trimesh"), "heightfield"),
    (dict(static_friction=1.0, dynamic_friction=0.5), "friction"),
])
def test_refused_configurations(kw, match):
    with pytest.raises(native.DyrosError, match=match):
        generate(TerrainConfig(num_rows=2, num_cols=5, **kw))


# ------------------------------------------------------------------ oracle of the update rule
def one(root_x, level, tv=0.0, u=0.5, num_levels=10, up=4.0, down_scale=16.0, origin_x=0.0):
    return int(update_levels([[root_x, 0.0]], [[origin_x, 0.0]], [[tv, 0.0]], [level], [u], num_levels, up, down_scale)[0])


def test_update_up_threshold_exact_and_just_past():
    assert one(4.0, 3) == 3, "exactly terrain_length / 2: not up"
    assert one(float(np.nextafter(f32(4.0), f32(5.0))), 3) == 4, "one ulp past: up"
    assert one(3.0, 3, origin_x=-1.0) == 3
    assert one(5.0, 3, origin_x=1.0000001) == 3  # d = 3.9999998 in float32


def test_update_down_and_up_over_down():
    assert one(1.0, 3, tv=0.5) == 2, "walked 1 m of the 8 m asked: down"
    assert one(5.0, 3, tv=0.5) == 4, "farther than the up distance: up, even though it is less than asked"
    assert one(8.0, 3, tv=0.5) == 4
    assert one(1.0, 3, tv=0.0) == 3, "standing target: never down"
    assert one(8.0, 3, tv=0.25) == 4
    # exactly at the down threshold: not down
    assert one(float(f32(0.25) * f32(16.0)) - 1e-6, 3, tv=0.25, up=10.0) == 2
    assert one(float(f32(0.25) * f32(16.0)), 3, tv=0.25, up=10.0) == 3


def test_update_clip_at_level_0_and_overflow_through_u():
    assert one(0.0, 0, tv=0.5) == 0
    assert one(5.0, 9, u=0.73) == 7, "past the top: int(u * num_levels)"
    assert one(5.0, 9, u=0.0) == 0
    assert one(5.0, 9, u=float(np.nextafter(f32(1.0), f32(0.0)))) == 9
    assert one(5.0, 8, u=0.0) == 9, "reaching the top level itself is no overflow"
    assert one(5.0, 0, u=0.3, num_levels=1) == 0


def test_oracle_reset_moves_env_to_its_new_origin():
    from oracle import task_oracle as O
    from tests.golden_util import load_assets
    N = 6
    tables, mocap, obs_norm = load_assets()
    rng = np.random.default_rng(0)
    s, c = O.new_state(N, mocap, obs_norm, np.full(N, f32(tables.total_mass())), tables.dof_lower, tables.dof_upper,
                       O.Params(), rng=rng)
    origins = rng.uniform(0, 50, (3, 2, 3)).astype(f32)
    cur = {"origins": origins, "types": np.array([0, 1, 0, 1, 0, 1], np.int32), "levels": np.array([0, 1, 2, 2, 1, 0], np.int32),
           "move_up_distance": 4.0, "move_down_scale": 16.0}
    s["env_origins"][:] = origins[cur["levels"], cur["types"]]
    s["root_states"][:, 0:2] = s["env_origins"][:, 0:2] + np.array([[5, 0], [0, 1], [0, 0], [3, 4.5], [0.5, 0], [0, 0]], f32)
    s["target_vel"][:] = np.array([0.5, 0], f32)
    noise = O.draw_noise(N, 2, rng)
    noise["reset_f"][:, 30] = 0.5
    reset_idx(s, c, np.arange(N), noise, cur)
    assert cur["levels"].tolist() == [1, 0, 1, 1, 0, 0]
    np.testing.assert_array_equal(s["env_origins"], origins[cur["levels"], cur["types"]])
    np.testing.assert_array_equal(s["root_states"][:, 0:2], s["env_origins"][:, 0:2])
    np.testing.assert_array_equal(s["root_states"][:, 2], s["env_origins"][:, 2] + f32(0.93))


# ------------------------------------------------------------------ task plumbing and ABI
def walk_cfg(N=64, **terrain):
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import default_cfg
    cfg = default_cfg(N)
    cfg["env"]["terrain"] = dict(num_rows=4, num_cols=5, terrain_length=4.0, terrain_width=4.0, border_size=2.0, **terrain)
    return cfg


def test_core_config_from_cfg_terrain():
    import torch
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import core_config_from_cfg
    N = 64
    c = core_config_from_cfg(walk_cfg(N, max_init_terrain_level=2, seed=4), torch.Generator().manual_seed(1))
    hf, tc = c.heightfield, c.terrain_curriculum
    assert hf.samples.shape == (4 * 40 + 40, 5 * 40 + 40) and hf.origin == (-2.0, -2.0, 0.0)
    assert np.array_equal(hf.samples, generate(TerrainConfig(num_rows=4, num_cols=5, terrain_length=4.0, terrain_width=4.0,
                                                             border_size=2.0, seed=4))[0].samples)
    assert tc.curriculum and tc.origins.shape == (4, 5, 3)
    assert tc.move_up_distance == 2.0 and tc.move_down_scale == 32 * 0.5
    assert np.array_equal(tc.types, np.floor(np.arange(N) / (N / 5)).astype(np.int32))
    assert tc.levels.min() >= 0 and tc.levels.max() <= 2 and len(set(tc.levels.tolist())) == 3
    tc.validate(N)
    # without the curriculum: initial levels over every row, no updates
    c = core_config_from_cfg(walk_cfg(N, curriculum=False), torch.Generator().manual_seed(1))
    assert not c.terrain_curriculum.curriculum and c.terrain_curriculum.levels.max() == 3
    # the plane, and the two grounds together
    cfg = walk_cfg(N, mesh_type="plane")
    assert core_config_from_cfg(cfg).heightfield is None and core_config_from_cfg(cfg).terrain_curriculum is None
    cfg = walk_cfg(N)
    cfg["env"]["heightfield"] = {"samples": np.zeros((4, 4), np.int16), "row_scale": 1.0, "column_scale": 1.0,
                                 "vertical_scale": 0.01}
    with pytest.raises(native.DyrosError, match="not both"):
        core_config_from_cfg(cfg)
    with pytest.raises(native.DyrosError, match="unknown keys"):
        core_config_from_cfg(walk_cfg(N, terrain_lenght=3.0))
    with pytest.raises(native.DyrosError, match="heightfield"):
        core_config_from_cfg(walk_cfg(N, mesh_type="trimesh"))


def test_set_terrain_curriculum_exported_and_mirrored():
    lib = native.load()
    assert hasattr(lib, "dyros_task_set_terrain_curriculum")
    assert "dyros_task_set_terrain_curriculum" in native.header_symbols()
    assert lib.dyros_task_set_terrain_curriculum(None, None) != 0 and b"task is NULL" in lib.dyros_last_error()
    src = '#include <stdio.h>\n#include "dyros_b200.h"\nint main(void){printf("%zu\\n", sizeof(DyrosTerrainCurriculum)); return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        assert int(subprocess.check_output([os.path.join(d, "s")])) == ctypes.sizeof(native.DyrosTerrainCurriculum)
