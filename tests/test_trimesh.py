"""Triangle-mesh ground, host side: legged_gym's convert_heightfield_to_trimesh, the grid and narrow phase of the
kernel (host-compiled from its source) against the fp64 brute force of tests/mesh_oracle.py, the refusals of every
layer and the C ABI layout."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from isaacgymdyros_b200 import gymapi, native, terrain
from isaacgymdyros_b200.core import CoreConfig, HeightField, TriangleMesh
from tests.mesh_oracle import MeshOracle
from tests import mesh_util
from tests.physics_util import HERE

ROOT = os.path.dirname(HERE)
MARGIN = 0.15


def kernel_query(v, t, c, r, origin=(0.0, 0.0, 0.0), margin=MARGIN, contact_offset=1e30):
    return mesh_util.kernel_query(v, t, c, r, origin, margin, contact_offset)


# ---------------------------------------------------------------- convert_heightfield_to_trimesh

def _step_field():
    """3 x 3 samples: a step of 40 units between rows 0 and 1 (along x) and one of 40 between columns 1 and 2 (along y)."""
    return np.array([[0, 0, 40], [40, 40, 80], [40, 40, 80]], np.int16)


def test_convert_moves_hand_computed():
    hs, vs = 0.1, 0.005  # threshold 0.75 * hs / vs = 15 sample units
    v, t = terrain.convert_heightfield_to_trimesh(_step_field(), hs, vs, 0.75)
    xy = v[:, :2].reshape(3, 3, 2)
    # (0, 0): row 1 higher -> +x; column 1 level, but (1, 1) higher diagonally and move_y = 0 -> +y
    assert np.allclose(xy[0, 0], [0.1, 0.1])
    # (0, 1): row 1 higher -> +x, column 2 higher -> +y
    assert np.allclose(xy[0, 1], [0.1, 0.2])
    # (1, 0): no higher neighbour (row 0 is lower; a lower neighbour moves nothing)
    assert np.allclose(xy[1, 0], [0.1, 0.0])
    # (1, 1): column 2 higher -> +y; move_x = 0 and (2, 2) higher diagonally -> +x
    assert np.allclose(xy[1, 1], [0.2, 0.2])
    assert np.allclose(xy[2, 2], [0.2, 0.2]) and np.allclose(xy[0, 2], [0.1, 0.2])
    assert np.allclose(v[:, 2], _step_field().ravel() * vs)
    v0, _ = terrain.convert_heightfield_to_trimesh(_step_field(), hs, vs, None)
    gy, gx = np.meshgrid(np.arange(3) * hs, np.arange(3) * hs)
    assert np.allclose(v0[:, 0], gx.ravel()) and np.allclose(v0[:, 1], gy.ravel())  # None: no moves


def test_convert_triangle_order_and_winding():
    hf = np.zeros((3, 4), np.int16)
    v, t = terrain.convert_heightfield_to_trimesh(hf, 0.1, 0.005, None)
    nc = 4
    assert t.dtype == np.uint32 and t.shape == (2 * 2 * 3, 3)
    for i in range(2):
        for j in range(3):
            k = 2 * (i * 3 + j)
            a = i * nc + j
            assert list(t[k]) == [a, a + nc + 1, a + 1]
            assert list(t[k + 1]) == [a, a + nc, a + nc + 1]
    P = v[t.astype(np.int64)].astype(np.float64)
    n = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
    assert np.all(n[:, 2] > 0)  # every face up


def test_unmoved_mesh_surface_equals_heightfield():
    rng = np.random.default_rng(3)
    s = rng.integers(-60, 60, (9, 7)).astype(np.int16)
    hf = HeightField(s, 0.1, 0.1, 0.005, origin=(-0.3, 0.2, 0.05))
    tm = terrain.trimesh_from_field(hf, None)
    x = rng.uniform(-0.3, -0.3 + 0.8, 200)
    y = rng.uniform(0.2, 0.2 + 0.6, 200)
    zm, ok = tm.height_at(x, y)
    zf, inside = hf.height_at(x, y)
    assert ok.all() and inside.all()
    assert np.allclose(zm, zf, atol=1e-6)


# ---------------------------------------------------------------- kernel query against the fp64 brute force

def _meshes():
    rng = np.random.default_rng(0)
    out = {}
    out["flat"] = terrain.convert_heightfield_to_trimesh(np.zeros((8, 8), np.int16), 0.1, 0.005, None)
    ramp = (np.arange(8)[:, None] * 10 + np.zeros((1, 8))).astype(np.int16)
    out["ramp"] = terrain.convert_heightfield_to_trimesh(ramp, 0.1, 0.005, None)
    st = np.zeros((12, 12), np.int16)
    st[4:, :] += 30   # riser facing -x
    st[:, 7:] += 30   # riser facing -y
    st[9:, :] -= 50   # riser facing +x (a step down)
    out["stairs"] = terrain.convert_heightfield_to_trimesh(st, 0.1, 0.005, 0.75)
    out["rough"] = terrain.convert_heightfield_to_trimesh(rng.integers(-10, 10, (10, 10)).astype(np.int16), 0.1, 0.005, 0.75)
    return out


@pytest.mark.parametrize("name", ["flat", "ramp", "stairs", "rough"])
def test_mesh_query_matches_brute_force(name):
    v, t = _meshes()[name]
    origin = (100.0, -150.0, 0.3)  # coordinates far from 0, as on the generated terrain
    orc = MeshOracle(v, t, origin, MARGIN)
    rng = np.random.default_rng(7)
    n = 600
    lo = v.min(0) + origin - 0.3
    hi = v.max(0) + origin + np.array([0.3, 0.3, 0.3])
    c = rng.uniform(lo, hi, (n, 3))
    r = rng.choice([0.0, 0.02, 0.05], n)
    s, nrm, hit, info = kernel_query(v, t, c, r, origin)
    assert info[0] + info[1] == len(t)
    checked = 0
    for k in range(n):
        q = orc.query(c[k])
        if q is None:
            assert not hit[k] or abs(s[k]) > MARGIN - 1e-4, f"point {k}: ground where the oracle has none"
            continue
        if abs(q["s"]) > MARGIN - 1e-4:
            continue  # (at the margin the float32 distance may fall either side)
        assert hit[k], f"point {k}: the grid missed a triangle within the margin ({q['s']})"
        assert abs(abs(s[k]) - abs(q["s"])) < 2e-5, (k, s[k], q["s"])
        if q["tie_gap"] > 1e-4:  # (at a tie the faces of a shared edge or vertex may disagree on the side)
            assert abs(s[k] - q["s"]) < 2e-5, (k, s[k], q["s"])
            assert np.abs(nrm[k] - q["n"]).max() < 2e-3 * max(1.0, 1e-3 / max(abs(q["s"]), 1e-6)), (k, nrm[k], q["n"])
            cp_k = c[k] - (r[k]) * nrm[k]
            cp_o = c[k] - r[k] * q["n"]
            assert np.abs(cp_k - cp_o).max() < 1e-4
        checked += 1
    assert checked > n // 8


def test_zero_area_triangles_dropped():
    v, t = terrain.convert_heightfield_to_trimesh(np.array([[0, 0, 40], [0, 40, 40], [40, 40, 40]], np.int16),
                                                  0.1, 0.005, 0.75)
    orc = MeshOracle(v, t)
    s, nrm, hit, info = kernel_query(v, t, np.array([[0.1, 0.1, 0.5]]), np.array([0.0]))
    assert info[1] == orc.dropped and info[0] == len(t) - info[1]
    bad = np.vstack([t, [[0, 0, 1]]]).astype(np.uint32)  # an explicit degenerate triangle is dropped, not refused
    assert kernel_query(v, bad, np.zeros((1, 3)), np.zeros(1))[3][1] == info[1] + 1


def test_off_mesh_and_far_points_have_no_ground():
    v, t = _meshes()["flat"]
    c = np.array([[-1.0, 0.3, 0.0], [0.3, 2.0, 0.0], [0.3, 0.3, 0.5], [0.3, 0.3, -0.5], [0.3, 0.3, 0.1]])
    s, nrm, hit, _ = kernel_query(v, t, c, np.zeros(len(c)))
    assert list(hit) == [False, False, False, False, True]
    assert abs(s[4] - 0.1) < 1e-6 and np.allclose(nrm[4], [0, 0, 1])


def test_bucket_cull_never_drops_a_contact():
    for name, (v, t) in _meshes().items():
        rng = np.random.default_rng(11)
        # (inside the mesh's x-y extent: past an open edge a point can lie behind the edge's face, where the side is
        #  not meaningful; DESIGN.md section 4)
        c = rng.uniform(v.min(0) + [0.05, 0.05, -0.1], v.max(0) + [-0.05, -0.05, 0.2], (800, 3))
        r = rng.choice([0.0, 0.03], len(c))
        co = 0.002
        s0, n0, h0, _ = kernel_query(v, t, c, r)                      # no cull
        s1, n1, h1, _ = kernel_query(v, t, c, r, contact_offset=co)   # the cull of the kernels
        touch = h0 & (s0 - r < co)
        assert np.all(h1[touch]), name
        assert np.array_equal(s0[touch], s1[touch]) and np.array_equal(n0[touch], n1[touch])


def test_grid_refusals():
    v, t = _meshes()["flat"]
    with pytest.raises(native.DyrosError, match="vertex index"):
        kernel_query(v, np.array([[0, 1, len(v)]]), np.zeros((1, 3)), np.zeros(1))
    vv = v.copy()
    vv[3, 2] = np.nan
    with pytest.raises(native.DyrosError, match="not finite"):
        kernel_query(vv, t, np.zeros((1, 3)), np.zeros(1))
    with pytest.raises(native.DyrosError, match="zero area"):
        kernel_query(v, np.array([[0, 0, 1]]), np.zeros((1, 3)), np.zeros(1))
    big = np.array([[0, 0, 0], [1e5, 0, 0], [0, 1e5, 0]], np.float32)
    with pytest.raises(native.DyrosError, match="buckets"):
        kernel_query(big, np.array([[0, 1, 2]]), np.zeros((1, 3)), np.zeros(1))
    dense = np.zeros((3 * 1100, 3), np.float32)
    dense[1::3, 0] = 0.01
    dense[2::3, 1] = 0.01
    with pytest.raises(native.DyrosError, match="more than 1024 triangles"):
        kernel_query(dense, np.arange(3 * 1100).reshape(-1, 3), np.zeros((1, 3)), np.zeros(1))


# ---------------------------------------------------------------- refusals of the Python layers

def _params(nv, nt):
    p = gymapi.TriangleMeshParams()
    p.nb_vertices, p.nb_triangles = nv, nt
    return p


def test_gym_add_triangle_mesh_validation():
    gym = gymapi.acquire_gym()
    sim = gymapi.Sim(0, gymapi.SimParams())
    v, t = _meshes()["flat"]
    p = _params(len(v), len(t))
    p.transform.r = gymapi.Quat(0.0, 0.0, 0.38268343, 0.92387953)
    with pytest.raises(native.DyrosError, match="transform.r"):
        gym.add_triangle_mesh(sim, v.ravel(), t.ravel(), p)
    p = _params(len(v), len(t))
    with pytest.raises(native.DyrosError, match="float32"):
        gym.add_triangle_mesh(sim, v.ravel().astype(np.float64), t.ravel(), p)
    with pytest.raises(native.DyrosError, match="uint32"):
        gym.add_triangle_mesh(sim, v.ravel(), t.ravel().astype(np.int32), p)
    with pytest.raises(native.DyrosError, match="nb_vertices"):
        gym.add_triangle_mesh(sim, v.ravel()[:-3], t.ravel(), p)
    p.transform.p = gymapi.Vec3(1.0, 2.0, 3.0)
    p.dynamic_friction = 0.6
    gym.add_triangle_mesh(sim, v.ravel(), t.ravel(), p)
    assert sim.triangle_mesh.vertices.shape == v.shape and sim.triangle_mesh.origin == (1.0, 2.0, 3.0)
    assert sim.triangle_mesh.friction == 0.6
    with pytest.raises(native.DyrosError, match="one ground"):
        gym.add_triangle_mesh(sim, v.ravel(), t.ravel(), p)
    with pytest.raises(native.DyrosError, match="one ground"):
        gym.add_ground(sim, gymapi.PlaneParams())
    hp = gymapi.HeightFieldParams()
    hp.nbRows, hp.nbColumns = 2, 2
    with pytest.raises(native.DyrosError, match="one ground"):
        gym.add_heightfield(sim, np.zeros(4, np.int16), hp)
    sim2 = gymapi.Sim(0, gymapi.SimParams())
    pp = gymapi.PlaneParams()
    pp.normal = gymapi.Vec3(0.0, 0.0, 1.0)
    gym.add_ground(sim2, pp)
    with pytest.raises(native.DyrosError, match="one ground"):
        gym.add_triangle_mesh(sim2, v.ravel(), t.ravel(), _params(len(v), len(t)))


def test_triangle_mesh_validation():
    v, t = _meshes()["flat"]
    for kw, msg in ((dict(vertices=v.astype(np.float64)), "float32"), (dict(triangles=t.astype(np.int64)), "uint32"),
                    (dict(triangles=t + np.uint32(1000)), "out of range"), (dict(origin=(0, np.inf, 0)), "origin"),
                    (dict(friction=-1.0), "friction")):
        args = dict(vertices=v, triangles=t)
        args.update(kw)
        with pytest.raises(native.DyrosError, match=msg):
            TriangleMesh(**args).validate()


@pytest.mark.parametrize("value", [-0.1, float("nan"), "0.75", True])
def test_slope_treshold_validation(value):
    with pytest.raises(native.DyrosError, match="slope_treshold"):
        terrain.validate(terrain.TerrainConfig(slope_treshold=value))
    terrain.validate(terrain.TerrainConfig(slope_treshold=None))


def _walk_cfg(**env):
    from tests.test_curriculum import walk_cfg
    cfg = walk_cfg(8)
    cfg["env"].update(env)
    return cfg


def test_terrain_mesh_key():
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import core_config_from_cfg
    c = core_config_from_cfg(_walk_cfg(terrainMesh=True))
    assert c.heightfield is None and c.triangle_mesh is not None and c.terrain_curriculum is not None
    tm = c.triangle_mesh
    assert tm.scan_field is not None and tm.origin == tm.scan_field.origin
    nr, nc = tm.scan_field.samples.shape
    assert tm.vertices.shape == (nr * nc, 3) and tm.triangles.shape == (2 * (nr - 1) * (nc - 1), 3)
    cfg = _walk_cfg(terrainMesh=True)
    del cfg["env"]["terrain"]
    with pytest.raises(native.DyrosError, match="needs a generated terrain"):
        core_config_from_cfg(cfg)
    cfg = _walk_cfg(terrainMesh=True)
    cfg["env"]["heightfield"] = dict(samples=np.zeros((4, 4), np.int16), row_scale=0.1, column_scale=0.1, vertical_scale=0.005)
    with pytest.raises(native.DyrosError, match="heightfield"):
        core_config_from_cfg(cfg)
    with pytest.raises(ValueError, match="terrainMesh"):
        core_config_from_cfg(_walk_cfg(terrainMesh="yes"))


# ---------------------------------------------------------------- C ABI layout

def test_abi_layout_and_symbols():
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "dyros_b200.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu\\n",'
           ' sizeof(DyrosTriangleMesh), offsetof(DyrosTriangleMesh, num_triangles), offsetof(DyrosTriangleMesh, origin),'
           ' offsetof(DyrosTriangleMesh, dynamic_friction), sizeof(DyrosHeightScan), offsetof(DyrosHeightScan, field));'
           ' return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "s.c"), "w") as f:
            f.write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "s"), os.path.join(d, "s.c")])
        got = [int(x) for x in subprocess.check_output([os.path.join(d, "s")]).split()]
    M, S = native.DyrosTriangleMesh, native.DyrosHeightScan
    assert got == [C.sizeof(M), M.num_triangles.offset, M.origin.offset, M.dynamic_friction.offset, C.sizeof(S),
                   S.field.offset]
    hdr = open(os.path.join(ROOT, "include", "dyros_b200.h")).read()
    so = os.path.join(ROOT, "isaacgymdyros_b200", "libdyros_b200.so")
    syms = subprocess.check_output(["nm", "-D", "--defined-only", so]).decode()
    for fn in ("dyros_sim_set_triangle_mesh", "dyros_sim_triangle_mesh_info"):
        assert f"int {fn}(" in hdr and fn in syms and fn in native.SIGNATURES
