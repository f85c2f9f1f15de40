"""The role program with Ground = MeshGround, host-compiled from the kernel source (tests/native/hostemu_mesh.cu),
against the fp64 physics oracle on a mesh (tests/mesh_oracle.py: brute force over every triangle), against the plane
program on a flat mesh and the heightfield program on a planar ramp, and with its culls switched off."""
import zlib

import numpy as np
import pytest

from isaacgymdyros_b200.core import CoreConfig
from tests.golden_util import load_assets
from tests.mesh_oracle import MeshPhysicsOracle
from tests.mesh_util import emulate_substep_mesh, mesh_from, stair_mesh_field
from tests.physics_util import emulate_substep, oracle_params, random_states
from tests.terrain_util import emulate_substep_terrain, flat_field, ramp_field, rough_field
from tests.test_physics_emulation import compare
from tests.test_terrain import terrain_states


def _sub(o, st):
    return o.substep(st["root"], st["q"], st["qd"], st["tau"], st["damping"], st["armature"], st["mass_scale"])[:4]


# (field for the states' heights, mesh): 3 m x 3 m, so that the brute force stays small
MESHES = {
    "flat": lambda: (flat_field(size=(3.0, 3.0), origin_xy=(-1.5, -1.5)),) * 2,
    "ramp": lambda: (ramp_field(size=(3.0, 3.0), origin_xy=(-1.5, -1.5)),) * 2,
    "stairs": lambda: (stair_mesh_field(size=(3.0, 3.0), origin_xy=(-1.5, -1.5)),) * 2,
    "stairs_y": lambda: (stair_mesh_field(size=(3.0, 3.0), origin_xy=(-1.5, -1.5), axis=1),) * 2,
    "rough": lambda: (rough_field(size=(3.0, 3.0), origin_xy=(-1.5, -1.5)),) * 2,
}


def mesh_case(name):
    field, _ = MESHES[name]()
    # (rough: no vertex moves. With them, random +-5 cm heights make walls whose nearest points can sit at a near-tie
    #  between two triangles with different closest points, where float32 and float64 may pick different ones)
    return field, mesh_from(field, 0.75 if name.startswith("stairs") else None)


def mesh_oracle(mesh, cfg=None):
    cfg = cfg or CoreConfig()
    return MeshPhysicsOracle(load_assets()[0], oracle_params(cfg), mesh.vertices, mesh.triangles, mesh.origin)


@pytest.mark.parametrize("kind", ["stand", "mixed"])
@pytest.mark.parametrize("name", list(MESHES))
def test_mesh_program_matches_oracle(name, kind):
    tables = load_assets()[0]
    cfg = CoreConfig()
    field, mesh = mesh_case(name)
    st = terrain_states(field, kind, seed=zlib.crc32(f"mesh {name} {kind}".encode()) % 1000, N=8)
    want = _sub(mesh_oracle(mesh, cfg), st)
    got = emulate_substep_mesh(tables, cfg, st, mesh)
    compare(st, got, want, ctx=f"mesh {name} {kind}: ")
    if kind == "stand":
        assert (np.abs(want[3][:, [8, 16]]).sum(-1) > 0).any(), "standing batch should load the soles"


def test_flat_mesh_program_equals_plane_program():
    """Standing and airborne envs (no link deeper than the depth allowance): the mesh program computes what the plane
    program computes, to float32 rounding."""
    tables = load_assets()[0]
    cfg = CoreConfig()
    st = random_states(12, np.random.default_rng(7), tables, "stand")
    want = emulate_substep(tables, cfg, st)
    got = emulate_substep_mesh(tables, cfg, st, mesh_from(flat_field(size=(3.0, 3.0), origin_xy=(-1.5, -1.5))))
    compare(st, got, want, ctx="flat mesh vs plane program: ")


def test_ramp_mesh_program_equals_heightfield_program():
    tables = load_assets()[0]
    cfg = CoreConfig()
    field = ramp_field()
    st = terrain_states(field, "stand", seed=5)
    want = emulate_substep_terrain(tables, cfg, st, field)
    got = emulate_substep_mesh(tables, cfg, st, mesh_from(field))
    compare(st, got, want, ctx="ramp mesh vs heightfield program: ")


@pytest.mark.parametrize("name", ["stairs", "rough", "ramp"])
def test_mesh_culls_never_drop_a_contact(name):
    """The bucket and per-link height culls change nothing: bit for bit the result without them, and every body the
    oracle finds in contact has a force."""
    tables = load_assets()[0]
    cfg = CoreConfig()
    field, mesh = mesh_case(name)
    st = terrain_states(field, "mixed", seed=11, N=10)
    culled = emulate_substep_mesh(tables, cfg, st, mesh, cull=True)
    full = emulate_substep_mesh(tables, cfg, st, mesh, cull=False)
    for a, b in zip(culled, full):
        assert np.array_equal(a, b)
    want = _sub(mesh_oracle(mesh, cfg), st)[3]
    touching = np.abs(want).sum(-1) > 1e-3
    assert touching.sum() > 5
    assert (np.abs(culled[3]).sum(-1)[touching] > 0).all()
