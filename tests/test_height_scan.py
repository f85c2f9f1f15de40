"""Height scan on the CPU: the oracle (tests/height_scan_oracle.py) against known answers on a hand-built 4 x 4 field,
the cfg["env"]["terrain"] plumbing of measure_heights, the layout of a pack_results block with the wider rows, the C
ABI's new entry point and the PPO trainer's refusal of the wider observation."""
import ctypes
import os
import subprocess
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from isaacgymdyros_b200 import native
from isaacgymdyros_b200.core import DyrosCore, HeightField
from isaacgymdyros_b200.terrain import TerrainConfig, height_points
from tests import height_scan_oracle as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
# samples s[i, j] = 10 i + j (rows along x, columns along y), 1 m cells, 0.1 m per unit, vertex (0, 0) at (10, 20, 1)
FIELD = HeightField((10 * np.arange(4)[:, None] + np.arange(4)[None, :]).astype(np.int16), 1.0, 1.0, 0.1,
                    origin=(10.0, 20.0, 1.0))


def root(x, y, z, q=(0.0, 0.0, 0.0, 1.0)):
    r = np.zeros((1, 13), f32)
    r[0, 0:3], r[0, 3:7] = (x, y, z), q
    return r


def yaw_quat(a):
    return (0.0, 0.0, np.sin(a / 2), np.cos(a / 2))


def h_expected(i, j):
    """Lowest of the three samples legged_gym reads in cell (i, j) of FIELD, in m."""
    s = FIELD.samples.astype(np.float64)
    return 1.0 + 0.1 * min(s[i, j], s[i + 1, j], s[i, j + 1])


def test_yaw_zero():
    pts = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [0.3, 0.3]], f32)
    r = root(11.5, 21.2, 2.5)
    h = H.heights(r, pts, FIELD)
    np.testing.assert_allclose(h[0], [h_expected(1, 1), h_expected(2, 1), h_expected(1, 2), h_expected(1, 1)], atol=1e-6)
    obs = H.obs_columns(r, h)
    np.testing.assert_allclose(obs[0], np.clip(2.5 - 0.5 - h[0], -1, 1) * 5, atol=1e-5)


def test_yaw_90_degrees():
    # +90 deg about z: the yaw frame's +x is the world's +y, its +y the world's -x
    pts = np.array([[1.0, 0.0], [0.0, 1.0]], f32)
    r = root(11.5, 21.5, 2.0, yaw_quat(np.pi / 2))
    wx, wy = H.world_points(r, pts)
    np.testing.assert_allclose(np.stack([wx[0], wy[0]], 1), [[11.5, 22.5], [10.5, 21.5]], atol=1e-6)
    np.testing.assert_allclose(H.heights(r, pts, FIELD)[0], [h_expected(1, 2), h_expected(0, 1)], atol=1e-6)


@pytest.mark.parametrize("axis", [0, 1])
def test_tilted_base_only_yaw_matters(axis):
    """A base yawed by a and then rolled (axis 0) or pitched (axis 1) by 0.4 rad: q's (z, w) is cos(0.2) times the yaw
    quaternion's, so the points land where the yaw alone puts them (legged_gym's quat_apply_yaw drops x and y)."""
    rng = np.random.default_rng(0)
    pts = rng.uniform(-0.8, 0.8, (50, 2)).astype(f32)
    a, t = 0.7, 0.4
    qy = np.array(yaw_quat(a))
    qt = np.zeros(4)
    qt[axis], qt[3] = np.sin(t / 2), np.cos(t / 2)
    ax, ay, az, aw = qy
    bx, by, bz, bw = qt
    q = np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by - ax * bz + ay * bw + az * bx,
                  aw * bz + ax * by - ay * bx + az * bw, aw * bw - ax * bx - ay * by - az * bz])  # qy (x) qt, xyzw
    assert np.hypot(q[0], q[1]) > 0.15
    wt = H.world_points(root(11.6, 21.4, 1.0, q), pts)
    wy = H.world_points(root(11.6, 21.4, 1.0, qy), pts)
    np.testing.assert_allclose(wt[0], wy[0], atol=5e-6)
    np.testing.assert_allclose(wt[1], wy[1], atol=5e-6)
    # away from cell edges: the same samples, the same heights
    u, v = (wy[0] - 10.0) % 1.0, (wy[1] - 20.0) % 1.0
    ok = (np.minimum(u, 1 - u) > 1e-4) & (np.minimum(v, 1 - v) > 1e-4)
    assert ok.sum() > 40
    np.testing.assert_array_equal(H.heights(root(11.6, 21.4, 1.0, q), pts, FIELD)[ok],
                                  H.heights(root(11.6, 21.4, 1.0, qy), pts, FIELD)[ok])


def test_min_of_three_ignores_the_far_corner():
    s = np.full((4, 4), 50, np.int16)
    s[1, 1], s[2, 1], s[1, 2], s[2, 2] = 30, 40, 20, -100  # (2, 2) is the lowest vertex but not one of the three
    f = HeightField(s, 1.0, 1.0, 0.01)
    h = H.heights(root(1.5, 1.5, 1.0), np.zeros((1, 2), f32), f)
    np.testing.assert_allclose(h[0], [0.2], atol=1e-7)
    s[1, 2] = 60
    np.testing.assert_allclose(H.heights(root(1.5, 1.5, 1.0), np.zeros((1, 2), f32), f)[0], [0.3], atol=1e-7)


@pytest.mark.parametrize("x, y, cell", [(-50.0, 21.5, (0, 1)), (99.0, 21.5, (2, 1)), (11.5, -70.0, (1, 0)),
                                        (11.5, 1e6, (1, 2)), (-1e6, -1e6, (0, 0)), (1e6, 1e6, (2, 2))])
def test_points_off_the_field_take_the_edge_cell(x, y, cell):
    h = H.heights(root(x, y, 1.0), np.zeros((1, 2), f32), FIELD)
    np.testing.assert_allclose(h[0], [h_expected(*cell)], atol=1e-6)


def test_plane_gives_zero_heights():
    rng = np.random.default_rng(1)
    r = np.zeros((5, 13), f32)
    r[:, 0:3] = rng.uniform(-100, 100, (5, 3))
    r[:, 6] = 1
    h = H.heights(r, rng.uniform(-1, 1, (7, 2)).astype(f32), None)
    assert h.shape == (5, 7) and not h.any()
    np.testing.assert_array_equal(H.obs_columns(r, h), np.repeat(np.clip(r[:, 2:3] - f32(0.5), -1, 1) * f32(5), 7, 1))


def test_obs_clip_and_scale():
    r = root(11.5, 21.5, 0.0)
    h = np.array([[-2.0, 0.0, -0.7, 3.0]], f32)
    r[0, 2] = 0.5
    np.testing.assert_allclose(H.obs_columns(r, h)[0], [5.0, 0.0, 3.5, -5.0], atol=1e-6)


def test_point_order_is_torch_meshgrid_ij():
    cfg = TerrainConfig(measure_heights=True)
    p = height_points(cfg)
    x = torch.tensor(cfg.measured_points_x)
    y = torch.tensor(cfg.measured_points_y)
    gx, gy = torch.meshgrid(x, y, indexing="ij")
    ref = torch.stack([gx.flatten(), gy.flatten()], 1).numpy()
    assert p.shape == (187, 2) and p.dtype == np.float32
    np.testing.assert_array_equal(p, ref)
    assert p[1].tolist() == [f32(-0.8), f32(-0.4)] and p[11].tolist() == [f32(-0.7), f32(-0.5)]


def walk_cfg(**terrain):
    from isaacgymdyros_b200 import default_cfg
    cfg = default_cfg(64)
    cfg["env"]["terrain"] = dict(num_rows=2, num_cols=2, terrain_length=4.0, terrain_width=4.0, border_size=2.0, **terrain)
    return cfg


def test_cfg_plumbing():
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import core_config_from_cfg, num_observations
    cfg = walk_cfg(measure_heights=True)
    c = core_config_from_cfg(cfg, torch.Generator().manual_seed(0))
    assert c.height_scan.shape == (187, 2) and c.heightfield is not None
    assert num_observations(cfg) == 674
    # off by default, and off when asked
    for cfg in (walk_cfg(), walk_cfg(measure_heights=False)):
        assert core_config_from_cfg(cfg, torch.Generator().manual_seed(0)).height_scan is None
        assert num_observations(cfg) == 487
    from isaacgymdyros_b200 import default_cfg
    assert num_observations(default_cfg(8)) == 487
    # on the plane too
    cfg = walk_cfg(mesh_type="plane", measure_heights=True, measured_points_x=[0.0, 0.5], measured_points_y=[-0.2, 0.0, 0.2])
    c = core_config_from_cfg(cfg)
    assert c.heightfield is None and c.height_scan.shape == (6, 2) and num_observations(cfg) == 493
    # bad point lists
    for bad in ({"measured_points_x": []}, {"measured_points_y": [0.0, float("nan")]},
                {"measured_points_x": [[0.0, 1.0]]}, {"measured_points_x": list(range(33)), "measured_points_y": list(range(32))}):
        with pytest.raises(native.DyrosError, match="measured_points|1024"):
            core_config_from_cfg(walk_cfg(measure_heights=True, **bad))
    # (a bad list with the scan off is not looked at)
    assert core_config_from_cfg(walk_cfg(measured_points_x=[]), torch.Generator()).height_scan is None
    with pytest.raises(native.DyrosError, match="heightfield"):
        core_config_from_cfg(walk_cfg(mesh_type="trimesh", measure_heights=True))


def test_pack_results_offsets_for_odd_n_and_wide_rows():
    c = DyrosCore.__new__(DyrosCore)
    c.N, c.obs_width = 5, 674
    rew, rst, tmo, end = c.result_offsets()
    assert rew == 5 * 674 * 4 and rst == 5 * 675 * 4 + 4 and rst % 8 == 0  # 13500 bytes: 4 bytes of padding
    assert tmo == rst + 40 and end == rst + 80 and c.result_bytes() == end
    c.N, c.obs_width = 5, 487  # without a scan: the layout of before, N * (487 * 4 + 4 + 8 + 8) bytes
    assert c.result_offsets() == (5 * 487 * 4, 5 * 488 * 4, 5 * 488 * 4 + 40, 5 * (487 * 4 + 20))
    c.N, c.obs_width = 6, 674
    assert c.result_offsets()[1] == 6 * 675 * 4


def test_set_height_scan_exported_and_mirrored():
    lib = native.load()
    assert "dyros_task_set_height_scan" in native.header_symbols()
    assert lib.dyros_task_set_height_scan(None, None) != 0 and b"task is NULL" in lib.dyros_last_error()
    src = '#include <stdio.h>\n#include "dyros_b200.h"\nint main(void){printf("%zu\\n", sizeof(DyrosHeightScan)); return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        assert int(subprocess.check_output([os.path.join(d, "s")])) == ctypes.sizeof(native.DyrosHeightScan)


def test_ppo_refuses_the_wider_observation():
    from isaacgymdyros_b200.ppo import PPOTrainer
    with pytest.raises(ValueError, match="height scan"):
        PPOTrainer(SimpleNamespace(num_obs=674, num_envs=8, device="cpu"))
