"""Helpers of the triangle-mesh tests: the host build of the kernel's grid and narrow phase and of its role program
with Ground = MeshGround (tests/native/hostemu_mesh.cu), and the meshes of the tests."""
import ctypes as C
import os
import subprocess

import numpy as np

from isaacgymdyros_b200 import native, terrain
from isaacgymdyros_b200.core import HeightField, make_model_desc, make_sim_desc
from tests.physics_util import CSRC, HERE

_EMU = None


def hostemu_mesh():
    global _EMU
    if _EMU is None:
        so = os.path.join(HERE, "native", "libdyros_hostemu_mesh.so")
        src = os.path.join(HERE, "native", "hostemu_mesh.cu")
        deps = [src, os.path.join(HERE, "native", "hostemu.cu")] + [
            os.path.join(CSRC, f) for f in ("physics_roles.cuh", "phys_math.cuh", "host_model.h", "internal.h", "mesh_grid.h")]
        if not os.path.isfile(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["nvcc", "-O2", "-std=c++20", "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "20014",
                                   "-Wno-deprecated-gpu-targets", "-I", CSRC, "-o", so, src])
        _EMU = C.CDLL(so)
    return _EMU


def mesh_desc(v, t, origin=(0.0, 0.0, 0.0), friction=1.0):
    """(DyrosTriangleMesh, keep-alive arrays)."""
    v, t = np.ascontiguousarray(v, np.float32), np.ascontiguousarray(t, np.uint32)
    d = native.DyrosTriangleMesh()
    d.vertices, d.triangles, d.num_vertices, d.num_triangles = v.ctypes.data, t.ctypes.data, len(v), len(t)
    d.origin = (C.c_float * 3)(*origin)
    d.dynamic_friction = friction
    return d, (v, t)


def kernel_query(v, t, c, r, origin=(0.0, 0.0, 0.0), margin=0.15, contact_offset=1e30):
    """The kernel's grid + mesh_query (float32) -> s, n, hit, info; contact_offset=1e30 switches the sign cull off."""
    d, keep = mesh_desc(v, t, origin)
    c, r = np.ascontiguousarray(c, np.float32), np.ascontiguousarray(r, np.float32)
    n = len(c)
    s, nrm, hit = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.int32)
    info = (C.c_longlong * 4)()
    err = C.create_string_buffer(512)
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = hostemu_mesh().dyros_hostemu_mesh_query(C.byref(d), C.c_float(margin), C.c_float(contact_offset), P(c), P(r), n,
                                                 P(s), P(nrm), P(hit), info, err, 512)
    if rc:
        raise native.DyrosError(err.value.decode())
    return s.astype(np.float64), nrm.astype(np.float64), hit.astype(bool), list(info)


def emulate_substep_mesh(tables, cfg, st, mesh, friction=None, cull=True):
    """emulate_substep (tests/physics_util.py) on a triangle mesh (core.TriangleMesh): the kernel's role program with
    Ground = MeshGround on the CPU (float32), every cull included."""
    N = st["root"].shape[0]
    md, keep = make_model_desc(tables, cfg)
    sd = make_sim_desc(cfg, N)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    root = f32(st["root"])
    dof = f32(np.stack([st["q"], st["qd"]], -1))
    tau, damp, arm, ms = f32(st["tau"]), f32(st["damping"]), f32(st["armature"]), f32(st["mass_scale"])
    contact = np.zeros((N, tables.num_bodies, 3), np.float32)
    P = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    mu = f32(friction) if friction is not None else None
    d, keep2 = mesh_desc(mesh.vertices, mesh.triangles, mesh.origin, cfg.friction if mesh.friction is None else mesh.friction)
    err = C.create_string_buffer(512)
    rc = hostemu_mesh().dyros_hostemu_simulate_mesh(C.byref(sd), C.byref(md), C.byref(d), P(root), P(dof), P(tau), P(damp),
                                                    P(arm), P(ms), P(contact), None, P(mu), int(cull), err, 512)
    assert rc == 0, err.value
    return root.astype(np.float64), dof[:, :, 0].astype(np.float64), dof[:, :, 1].astype(np.float64), contact.astype(np.float64)


def mesh_from(field, slope_threshold=None):
    """tests' oracle HeightField -> core.TriangleMesh of legged_gym's converter (the field's origin, no friction)."""
    hf = HeightField(np.asarray(field.samples, np.int16), field.row_scale, field.column_scale, field.vertical_scale,
                     tuple(field.origin))
    return terrain.trimesh_from_field(hf, slope_threshold)


def stair_mesh_field(step=0.1, tread=0.3, size=(4.0, 4.0), origin_xy=(-2.0, -2.0), spacing=0.05, vscale=0.005, axis=0):
    """Steps of `step` every `tread` m along +x (axis 0) or +y (axis 1), z = 0 on the tread holding the origin; with
    slope_threshold 0.75 the mesh's risers are vertical walls facing -x (-y)."""
    from tests.terrain_oracle import HeightField as OHF
    nr, nc = int(round(size[0] / spacing)) + 1, int(round(size[1] / spacing)) + 1
    n = (nr, nc)[axis]
    x = (origin_xy[axis] + spacing * np.arange(n))
    k = (np.floor((x + 1e-9) / tread) * int(round(step / vscale))).astype(np.int16)
    s = np.repeat(k[:, None], nc, 1) if axis == 0 else np.repeat(k[None, :], nr, 0)
    return OHF(s.astype(np.int16), spacing, spacing, vscale, (origin_xy[0], origin_xy[1], 0.0))
