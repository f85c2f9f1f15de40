"""Helpers of the heightfield tests: field builders, the CPU emulation of the kernel's heightfield role program
(tests/native/hostemu_terrain.cu) and its height / normal query."""
import ctypes as C
import os
import subprocess

import numpy as np

from isaacgymdyros_b200.core import make_model_desc, make_sim_desc
from tests.physics_util import CSRC, HERE
from tests.terrain_oracle import HeightField

_EMU = None


def hostemu_terrain():
    global _EMU
    if _EMU is None:
        so = os.path.join(HERE, "native", "libdyros_hostemu_terrain.so")
        src = os.path.join(HERE, "native", "hostemu_terrain.cu")
        deps = [src, os.path.join(HERE, "native", "hostemu.cu")] + [
            os.path.join(CSRC, f) for f in ("physics_roles.cuh", "phys_math.cuh", "host_model.h", "internal.h")]
        if not os.path.isfile(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["nvcc", "-O2", "-std=c++20", "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "20014",
                                   "-Wno-deprecated-gpu-targets", "-I", CSRC, "-o", so, src])
        _EMU = C.CDLL(so)
        _EMU.dyros_hostemu_simulate_terrain.restype = C.c_int
    return _EMU


def _field_args(field: HeightField):
    s = np.ascontiguousarray(field.samples, dtype=np.int16)
    scale = np.array([field.row_scale, field.column_scale, field.vertical_scale], np.float32)
    origin = np.array(field.origin, np.float32)
    return s, scale, origin


def field_cull(field: HeightField):
    """(zmax, 1 / smallest n_z) as dyros_sim_set_heightfield derives them for the per-link reach cull."""
    s = np.asarray(field.samples, np.float64) * field.vertical_scale
    g = []
    for a, b, c, d in ((s[1:, :-1], s[:-1, :-1], s[1:, 1:], s[1:, :-1]), (s[1:, 1:], s[:-1, 1:], s[:-1, 1:], s[:-1, :-1])):
        g.append(((a - b) / field.row_scale) ** 2 + ((c - d) / field.column_scale) ** 2)
    return np.array([field.origin[2] + s.max() + 1e-4, np.sqrt(1 + max(x.max() for x in g)) * (1 + 1e-5)], np.float32)


def query_kernel(field: HeightField, xy):
    """The kernel's field_query (float32) at points xy (n, 2): h (n,), normal (n, 3), inside (n,) bool."""
    s, scale, origin = _field_args(field)
    xy = np.ascontiguousarray(xy, dtype=np.float32)
    n = xy.shape[0]
    h, nrm, inside = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.int32)
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    hostemu_terrain().dyros_hostemu_field_query(P(s), s.shape[0], s.shape[1], P(scale), P(origin), P(xy), n, P(h), P(nrm),
                                                P(inside))
    return h.astype(np.float64), nrm.astype(np.float64), inside.astype(bool)


def emulate_substep_terrain(tables, cfg, st, field: HeightField, push=None, friction=None, cull=True):
    """emulate_substep (tests/physics_util.py) on a heightfield: the kernel's role program with Ground = FieldGround on
    the CPU (float32). cull=True also runs the per-link reach cull with the bounds the library derives."""
    N = st["root"].shape[0]
    md, keep = make_model_desc(tables, cfg)
    sd = make_sim_desc(cfg, N)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    root = f32(st["root"])
    dof = f32(np.stack([st["q"], st["qd"]], -1))
    tau, damp, arm, ms = f32(st["tau"]), f32(st["damping"]), f32(st["armature"]), f32(st["mass_scale"])
    contact = np.zeros((N, tables.num_bodies, 3), np.float32)
    P = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    pf = f32(push) if push is not None else None
    mu = f32(friction) if friction is not None else None
    s, scale, origin = _field_args(field)
    cl = field_cull(field) if cull else None
    err = C.create_string_buffer(256)
    rc = hostemu_terrain().dyros_hostemu_simulate_terrain(C.byref(sd), C.byref(md), P(s), s.shape[0], s.shape[1], P(scale),
                                                          P(origin), P(cl), P(root), P(dof), P(tau), P(damp), P(arm), P(ms),
                                                          P(contact), P(pf), P(mu), err, 256)
    assert rc == 0, err.value
    return root.astype(np.float64), dof[:, :, 0].astype(np.float64), dof[:, :, 1].astype(np.float64), contact.astype(np.float64)


# ---- fields of the tests (all 0.1 m spacing unless stated; x along rows, y along columns)
def flat_field(z=0.0, size=(6.0, 6.0), origin_xy=(-3.0, -3.0), spacing=0.1, vscale=0.005):
    nr, nc = int(round(size[0] / spacing)) + 1, int(round(size[1] / spacing)) + 1
    k = int(round(z / vscale))
    return HeightField(np.full((nr, nc), k, np.int16), spacing, spacing, vscale, (origin_xy[0], origin_xy[1], z - k * vscale))


def ramp_field(slope=0.05, size=(6.0, 6.0), origin_xy=(-3.0, -3.0), spacing=0.125, vscale=0.0078125):
    """Linear ramp rising along +x: s[i, j] = i * steps; exactly representable (power-of-two scales) and planar, so
    every triangle has the same normal."""
    nr, nc = int(round(size[0] / spacing)) + 1, int(round(size[1] / spacing)) + 1
    steps = int(round(slope * spacing / vscale))
    s = (np.arange(nr)[:, None] * steps - (nr // 2) * steps + np.zeros(nc, int)[None, :]).astype(np.int16)
    return HeightField(s, spacing, spacing, vscale, (origin_xy[0], origin_xy[1], 0.0))


def rough_field(amp=0.05, size=(6.0, 6.0), origin_xy=(-3.0, -3.0), spacing=0.1, vscale=0.005, seed=0):
    """Uniform heights in [-amp, amp] at every vertex."""
    nr, nc = int(round(size[0] / spacing)) + 1, int(round(size[1] / spacing)) + 1
    k = int(round(amp / vscale))
    s = np.random.default_rng(seed).integers(-k, k + 1, (nr, nc)).astype(np.int16)
    return HeightField(s, spacing, spacing, vscale, (origin_xy[0], origin_xy[1], 0.0))


def stairs_field(step=0.05, tread=0.3, size=(6.0, 6.0), origin_xy=(-3.0, -3.0), spacing=0.05, vscale=0.005):
    """Steps of `step` height every `tread` metres along +x, centred on z = 0 at x = 0."""
    nr, nc = int(round(size[0] / spacing)) + 1, int(round(size[1] / spacing)) + 1
    x = origin_xy[0] + spacing * np.arange(nr)
    k = np.floor(x / tread) * int(round(step / vscale))
    s = np.repeat(k[:, None], nc, 1).astype(np.int16)
    return HeightField(s, spacing, spacing, vscale, (origin_xy[0], origin_xy[1], 0.0))
