"""Heightfield ground on the CPU: the height / normal query (kernel, oracle and host-side restatements) against hand-computed
values, the fp64 oracle against the plane oracle, and the kernel's heightfield role program (host emulation, float32)
against the oracle on flat, raised, sloped, rough and stair fields and off the field's edge."""
import dataclasses
import zlib

import numpy as np
import pytest

from isaacgymdyros_b200 import gymapi, native
from isaacgymdyros_b200.core import CoreConfig
from isaacgymdyros_b200.core import HeightField as CoreHeightField
from isaacgymdyros_b200.tasks.dyros_dynamic_walk import core_config_from_cfg, default_cfg
from oracle.physics_oracle import PhysicsOracle
from tests.golden_util import load_assets
from tests.physics_util import emulate_substep, oracle_params, random_states
from tests.terrain_oracle import HeightField, TerrainOracle
from tests.terrain_util import (emulate_substep_terrain, flat_field, query_kernel, ramp_field, rough_field,
                                stairs_field)
from tests.test_physics_emulation import SLIDING_SLACK, compare, sliding_states

# 3 x 3 field, 0.5 m spacing, 0.25 m per unit, vertex (0, 0) at (1, 2, 0.5): every value below is exact in float32
S3 = np.array([[0, 1, 2], [0, 2, 4], [1, 1, 1]], np.int16)
F3 = dict(row_scale=0.5, column_scale=0.5, vertical_scale=0.25, origin=(1.0, 2.0, 0.5))
r2, r15, r125, r425 = np.sqrt(2.0), np.sqrt(1.5), np.sqrt(1.25), np.sqrt(4.25)
CASES = [  # (x, y) -> inside, h, n
    ((1.0, 2.0), True, 0.5, (0.0, -1 / r2, 1 / r2)),                           # vertex (0, 0): cell (0, 0), lower triangle
    ((1.25, 2.125), True, 0.625, (0.0, -1 / r2, 1 / r2)),                      # inside the lower triangle (fu > fv)
    ((1.125, 2.25), True, 0.6875, (-0.5 / r15, -0.5 / r15, 1 / r15)),          # inside the upper triangle (fu < fv)
    ((1.25, 2.25), True, 0.75, (0.0, -1 / r2, 1 / r2)),                        # on the diagonal: the lower triangle
    ((1.5, 2.25), True, 0.75, (1 / 3, -2 / 3, 2 / 3)),                         # on a cell edge (u = 1): cell (1, 0), upper
    ((2.0, 3.0), True, 0.75, (0.5 / r125, 0.0, 1 / r125)),                     # far corner: last cell, lower triangle
    ((1.75, 3.0), True, 1.125, (1.5 / r425, -1 / r425, 1 / r425)),             # far edge v = 2: last cell column, upper
    ((0.99, 2.5), False, None, None), ((1.5, 3.01), False, None, None), ((2.01, 2.5), False, None, None),
    ((1.5, 1.99), False, None, None),
]


def _field3():
    return HeightField(S3, **F3)


def test_query_hand_computed_3x3():
    xy = np.array([c[0] for c in CASES])
    want_in = np.array([c[1] for c in CASES])
    h_o, n_o, in_o = _field3().query(xy[:, 0], xy[:, 1])
    h_k, n_k, in_k = query_kernel(_field3(), xy)
    hc, in_c = CoreHeightField(S3, **F3).height_at(xy[:, 0], xy[:, 1])
    for inside in (in_o, in_k, in_c):
        assert np.array_equal(inside, want_in)
    for k, (_xy, inside, h, n) in enumerate(CASES):
        if not inside:
            continue
        assert abs(h_o[k] - h) < 1e-12 and abs(hc[k] - h) < 1e-12, (k, h_o[k], hc[k], h)
        assert np.abs(n_o[k] - n).max() < 1e-12, (k, n_o[k], n)
        assert abs(h_k[k] - h) < 1e-6 and np.abs(n_k[k] - n).max() < 1e-6, (k, h_k[k], n_k[k])


def test_query_random_points_agree():
    """The kernel's per-triangle gradients and the oracle's vertex planes on a rough field, away from the cell edges
    (where a float32 rounding of u, v may pick the neighbouring triangle)."""
    f = rough_field(size=(2.0, 2.0), origin_xy=(-1.0, -1.0))
    rng = np.random.default_rng(0)
    xy = rng.uniform(-1.1, 1.1, (4000, 2))
    g = (xy - np.array([-1.0, -1.0])) / 0.1
    fu, fv = g[:, 0] - np.floor(g[:, 0]), g[:, 1] - np.floor(g[:, 1])
    xy = xy[(np.minimum(fu, 1 - fu) > 1e-3) & (np.minimum(fv, 1 - fv) > 1e-3) & (np.abs(fu - fv) > 1e-3)]
    h_o, n_o, in_o = f.query(xy[:, 0], xy[:, 1])
    h_k, n_k, in_k = query_kernel(f, xy)
    assert np.array_equal(in_o, in_k) and 0 < in_o.sum() < len(xy)
    assert np.abs(h_o - h_k)[in_o].max() < 1e-6 and np.abs(n_o - n_k)[in_o].max() < 1e-5


def _sub(o, st, **kw):
    return o.substep(st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"], st["mass_scale"], **kw)


def test_oracle_flat_field_equals_plane():
    tables = load_assets()[0]
    cfg = CoreConfig()
    rng = np.random.default_rng(2)
    st = random_states(12, rng, tables, "mixed")
    push = rng.normal(0, 300, (12, 3))
    want = _sub(PhysicsOracle(tables, oracle_params(cfg)), st, push=push)
    got = _sub(TerrainOracle(tables, oracle_params(cfg), ground=flat_field()), st, push=push)
    for a, b in zip(want[:4], got[:4]):
        assert np.abs(a - b).max() <= 1e-12
    assert np.abs(want[3]).max() > 100, "the batch should touch the ground"


def test_oracle_translation_invariance():
    """A field raised by c with the robot raised by c: the plane's result, shifted by c."""
    tables = load_assets()[0]
    cfg = CoreConfig()
    st = random_states(12, np.random.default_rng(4), tables, "mixed")
    c = 0.37
    up = dict(st, root=st["root"] + np.array([0, 0, c] + [0] * 10))
    want = _sub(PhysicsOracle(tables, oracle_params(cfg)), st)
    got = _sub(TerrainOracle(tables, oracle_params(cfg), ground=flat_field(z=c, vscale=0.01)), up)
    assert abs(got[0][:, 2] - want[0][:, 2] - c).max() < 1e-9
    assert np.abs(got[0][:, 3:] - want[0][:, 3:]).max() < 1e-9
    for a, b in zip(want[1:4], got[1:4]):
        assert np.abs(a - b).max() < 1e-6 * max(1.0, np.abs(a).max())


def _edge_field():
    """Flat at z = 0 for x >= 0 only: the soles straddle the field's edge."""
    return flat_field(size=(3.0, 6.0), origin_xy=(0.0, -3.0))


FIELDS = {"flat": flat_field, "raised": lambda: flat_field(z=0.25), "ramp": ramp_field, "rough": rough_field,
          "stairs": stairs_field, "edge": _edge_field}


def terrain_states(field, kind, seed, N=12):
    """random_states (or sliding_states) lifted onto the field: the base origin by the terrain height below it."""
    tables = load_assets()[0]
    rng = np.random.default_rng(seed)
    st = sliding_states(N, rng, tables, "mixed") if kind == "sliding" else random_states(N, rng, tables, kind)
    if kind == "stand":  # spread the stances over the field's features
        st["root"][:, 0:2] = rng.uniform(-0.4, 0.4, (N, 2))
    h, _n, inside = field.query(st["root"][:, 0], st["root"][:, 1])
    st["root"][:, 2] += np.where(inside, h, 0.0)
    st["root"] = st["root"].astype(np.float32).astype(np.float64)
    return st


@pytest.mark.parametrize("kind", ["stand", "mixed", "sliding"])
@pytest.mark.parametrize("name", list(FIELDS))
def test_terrain_program_matches_oracle(name, kind):
    tables = load_assets()[0]
    cfg = CoreConfig()
    field = FIELDS[name]()
    st = terrain_states(field, kind, seed=zlib.crc32(f"{name} {kind}".encode()) % 1000)
    want = _sub(TerrainOracle(tables, oracle_params(cfg), ground=field), st)
    got = emulate_substep_terrain(tables, cfg, st, field)
    compare(st, got, want, ctx=f"{name} {kind}: ", slack=SLIDING_SLACK if kind == "sliding" else 1.0)
    if kind == "stand":
        assert (np.abs(want[3][:, [8, 16]]).sum(-1) > 0).any(), "standing batch should load the soles"


def test_terrain_program_flat_field_equals_plane_program():
    """At z = 0 the heightfield program computes what the plane program computes (n = +z, t1 = x, t2 = y)."""
    tables = load_assets()[0]
    cfg = CoreConfig()
    st = random_states(12, np.random.default_rng(7), tables, "mixed")
    want = emulate_substep(tables, cfg, st)
    got = emulate_substep_terrain(tables, cfg, st, flat_field())
    for a, b in zip(want, got):
        assert np.array_equal(a, b)


def test_terrain_program_per_env_friction():
    tables = load_assets()[0]
    cfg = CoreConfig()
    field = ramp_field()
    st = terrain_states(field, "sliding", seed=21)
    mu = np.random.default_rng(3).uniform(0.2, 1.3, 12).astype(np.float32).astype(np.float64)
    want = _sub(TerrainOracle(tables, dataclasses.replace(oracle_params(cfg), mu=mu), ground=field), st)
    got = emulate_substep_terrain(tables, cfg, st, field, friction=mu)
    compare(st, got, want, slack=SLIDING_SLACK)


@pytest.mark.parametrize("name", ["rough", "stairs", "ramp"])
def test_reach_cull_never_drops_a_contact(name):
    """The per-link cull (pw.z < zmax + reach / min n_z) changes nothing: bit for bit the result without it, and every
    body the oracle finds in contact has a force."""
    tables = load_assets()[0]
    cfg = CoreConfig()
    field = FIELDS[name]()
    st = terrain_states(field, "mixed", seed=11, N=16)
    culled = emulate_substep_terrain(tables, cfg, st, field, cull=True)
    full = emulate_substep_terrain(tables, cfg, st, field, cull=False)
    for a, b in zip(culled, full):
        assert np.array_equal(a, b)
    want = _sub(TerrainOracle(tables, oracle_params(cfg), ground=field), st)[3]
    touching = np.abs(want).sum(-1) > 1e-3
    assert touching.sum() > 10
    assert (np.abs(culled[3]).sum(-1)[touching] > 0).all()


def test_humanoid_on_rough_field():
    from tests.test_humanoid_generality import HUMANOID_CFG, humanoid, humanoid_states
    t = humanoid()
    cfg = CoreConfig(**HUMANOID_CFG)
    field = rough_field(amp=0.03)
    st = humanoid_states(8, np.random.default_rng(5), t, "mixed")
    st["root"][:, 2] += field.query(st["root"][:, 0], st["root"][:, 1])[0]
    st["root"] = st["root"].astype(np.float32).astype(np.float64)
    want = _sub(TerrainOracle(t, oracle_params(cfg), solver_bodies=cfg.solver_bodies, ground=field), st)
    got = emulate_substep_terrain(t, cfg, st, field)
    compare(st, got, want, ctx="humanoid rough: ")
    assert np.abs(want[3]).sum() > 10


# ---- host-side validation
def _hf(**kw):
    base = dict(samples=np.zeros((4, 5), np.int16), row_scale=0.1, column_scale=0.1, vertical_scale=0.005)
    return CoreHeightField(**{**base, **kw})


@pytest.mark.parametrize("kw,msg", [
    (dict(samples=np.zeros((4, 5), np.float32)), "int16"), (dict(samples=np.zeros(20, np.int16)), "2-D"),
    (dict(samples=np.zeros((1, 5), np.int16)), "2 x 2"), (dict(row_scale=0.0), "row_scale"),
    (dict(column_scale=-1.0), "column_scale"), (dict(vertical_scale=float("nan")), "vertical_scale"),
    (dict(origin=(0.0, 0.0)), "origin"), (dict(friction=-0.5), "friction")])
def test_heightfield_validation(kw, msg):
    with pytest.raises(native.DyrosError, match=msg):
        _hf(**kw).validate()
    _hf().validate()


def test_task_cfg_heightfield_key():
    cfg = default_cfg(16)
    assert core_config_from_cfg(cfg).heightfield is None
    s = np.ones((30, 40), np.int16)
    cfg["env"]["heightfield"] = {"samples": s, "row_scale": 0.1, "column_scale": 0.2, "vertical_scale": 0.005,
                                 "origin": (-1.0, -2.0, 0.0), "friction": 0.8}
    hf = core_config_from_cfg(cfg).heightfield
    assert hf.samples is not None and hf.samples.shape == (30, 40) and hf.column_scale == 0.2 and hf.friction == 0.8
    assert hf.origin == (-1.0, -2.0, 0.0) and hf.env_origins is None


def test_gym_add_heightfield_validation():
    gym = gymapi.Gym()
    sim = gymapi.Sim(0, gymapi.SimParams())
    hp = gymapi.HeightFieldParams()
    hp.nbRows, hp.nbColumns = 4, 5
    hp.row_scale, hp.column_scale, hp.vertical_scale = 0.1, 0.1, 0.005
    hp.transform.r = gymapi.Quat(0.0, 0.0, 0.7071068, 0.7071068)
    with pytest.raises(native.DyrosError, match="identity"):
        gym.add_heightfield(sim, np.zeros(20, np.int16), hp)
    hp.transform.r = gymapi.Quat()
    with pytest.raises(native.DyrosError, match="int16"):
        gym.add_heightfield(sim, np.zeros(20, np.float32), hp)
    with pytest.raises(native.DyrosError, match="nbRows"):
        gym.add_heightfield(sim, np.zeros(21, np.int16), hp)
    hp.transform.p = gymapi.Vec3(1.0, 2.0, 3.0)
    hp.dynamic_friction = 0.7
    gym.add_heightfield(sim, np.arange(20, dtype=np.int16), hp)
    assert sim.heightfield.samples.shape == (4, 5) and sim.heightfield.samples[1, 0] == 5
    assert sim.heightfield.origin == (1.0, 2.0, 3.0) and sim.heightfield.friction == 0.7
    with pytest.raises(native.DyrosError, match="one ground"):
        gym.add_heightfield(sim, np.zeros(20, np.int16), hp)
    with pytest.raises(native.DyrosError, match="one ground"):
        gym.add_ground(sim, gymapi.PlaneParams())
    with pytest.raises(native.DyrosError, match="add_heightfield"):
        gym.add_triangle_mesh(sim, np.zeros((3, 3), np.float32), np.zeros((1, 3), np.uint32), gymapi.TriangleMeshParams())
