"""Terrain generator of the curriculum (host, numpy): a grid of sub-terrains, num_rows difficulty levels by num_cols
terrain types, in one heightfield with a flat border, and the origin of each sub-terrain.

It follows legged_gym's Terrain (the layout of the reference's TerrainCfg) over isaacgym's terrain_utils, with the
kinds this project builds: pyramid slopes (smooth and rough), pyramid stairs (up and down) and discrete obstacles
(DESIGN.md section 4, "Curriculum"). It states that model; it does not reproduce the reference's samples one for one.
Randomness comes from numpy.random.default_rng(seed): the same seed gives the same field on every rank.
"""
from __future__ import annotations

from dataclasses import dataclass, field, fields
from typing import List, Optional

import numpy as np

from .core import HeightField, TriangleMesh
from .native import DyrosError


@dataclass
class TerrainConfig:
    """TerrainCfg's fields with legged_gym's defaults (mesh_type 'heightfield': the only kind built here), plus `seed`."""
    mesh_type: str = "heightfield"       # "plane" (no terrain) | "heightfield"; "trimesh" is refused
    horizontal_scale: float = 0.1        # m per sample
    vertical_scale: float = 0.005        # m per sample unit
    border_size: float = 25.0            # m of flat ground around the grid
    curriculum: bool = True
    static_friction: float = 1.0
    dynamic_friction: float = 1.0
    max_init_terrain_level: int = 5
    terrain_length: float = 8.0          # m along x of one sub-terrain
    terrain_width: float = 8.0           # m along y
    num_rows: int = 10                   # levels
    num_cols: int = 20                   # types
    # smooth slope, rough slope, stairs up, stairs down, discrete obstacles
    terrain_proportions: List[float] = field(default_factory=lambda: [0.1, 0.1, 0.35, 0.25, 0.2])
    # height scan (DESIGN.md section 4, "Height scan"), on any mesh_type. Off by default here (legged_gym: on), because it
    # widens the observation from 487 to 487 + len(x) * len(y) columns
    measure_heights: bool = False
    measured_points_x: List[float] = field(default_factory=lambda: [-0.8, -0.7, -0.6, -0.5, -0.4, -0.3, -0.2, -0.1, 0.,
                                                                    0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8])
    measured_points_y: List[float] = field(default_factory=lambda: [-0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3,
                                                                    0.4, 0.5])
    seed: int = 0
    # legged_gym's key (and spelling): convert_heightfield_to_trimesh moves vertices where neighbouring samples differ by
    # more than this slope, so that risers become vertical walls; None: no moves. Used only for a mesh ground
    # (cfg["env"]["terrainMesh"])
    slope_treshold: Optional[float] = 0.75

    @classmethod
    def from_dict(cls, d: dict) -> "TerrainConfig":
        known = {f.name for f in fields(cls)}
        unknown = sorted(set(d) - known)
        if unknown:
            raise DyrosError(f"terrain: unknown keys {unknown} (known: {sorted(known)})")
        return cls(**d)


def _pyramid_slope(h, slope, hs, vs, platform):
    """terrain_utils.pyramid_sloped_terrain."""
    w, l = h.shape
    cx, cy = w // 2, l // 2
    xx = ((cx - np.abs(cx - np.arange(w))) / cx).reshape(w, 1)
    yy = ((cy - np.abs(cy - np.arange(l))) / cy).reshape(1, l)
    top = int(slope * (hs / vs) * (w / 2))
    h += (top * xx * yy).astype(h.dtype)
    p = int(platform / hs / 2)
    x1, y1 = w // 2 - p, l // 2 - p
    lo, hi = min(h[x1, y1], 0), max(h[x1, y1], 0)
    np.clip(h, lo, hi, out=h)


def _random_uniform(h, rng, lo, hi, step, down, hs, vs):
    """terrain_utils.random_uniform_terrain: heights drawn on a grid `down` m apart, bilinear up to the samples, rounded."""
    w, l = h.shape
    lo, hi, step = int(lo / vs), int(hi / vs), int(step / vs)
    coarse = rng.choice(np.arange(lo, hi + step, step), (int(w * hs / down), int(l * hs / down))).astype(np.float64)
    xc, yc = np.linspace(0, w * hs, coarse.shape[0]), np.linspace(0, l * hs, coarse.shape[1])
    xf, yf = np.linspace(0, w * hs, w), np.linspace(0, l * hs, l)
    along_y = np.stack([np.interp(yf, yc, row) for row in coarse])                 # (coarse rows, l)
    fine = np.stack([np.interp(xf, xc, along_y[:, j]) for j in range(l)], axis=1)  # (w, l)
    h += np.rint(fine).astype(h.dtype)


def _pyramid_stairs(h, step_width, step_height, platform, hs, vs):
    """terrain_utils.pyramid_stairs_terrain (riser int(step_height / vs), truncated toward zero)."""
    step_width, step_height, platform = int(step_width / hs), int(step_height / vs), int(platform / hs)
    height, x0, x1, y0, y1 = 0, 0, h.shape[0], 0, h.shape[1]
    while (x1 - x0) > platform and (y1 - y0) > platform:
        x0, x1, y0, y1 = x0 + step_width, x1 - step_width, y0 + step_width, y1 - step_width
        height += step_height
        h[x0:x1, y0:y1] = height


def _discrete_obstacles(h, rng, max_height, min_size, max_size, num_rects, platform, hs, vs):
    """terrain_utils.discrete_obstacles_terrain."""
    max_height, min_size, max_size, platform = int(max_height / vs), int(min_size / hs), int(max_size / hs), int(platform / hs)
    ni, nj = h.shape
    heights = [-max_height, -max_height // 2, max_height // 2, max_height]
    sizes = range(min_size, max_size, 4)
    for _ in range(num_rects):
        wi, wj = rng.choice(sizes), rng.choice(sizes)
        si, sj = rng.choice(range(0, ni - wi, 4)), rng.choice(range(0, nj - wj, 4))
        h[si:si + wi, sj:sj + wj] = rng.choice(heights)
    x1, x2 = (ni - platform) // 2, (ni + platform) // 2
    y1, y2 = (nj - platform) // 2, (nj + platform) // 2
    h[x1:x2, y1:y2] = 0


def _sub_terrain(cfg: TerrainConfig, rng, choice: float, difficulty: float, shape):
    """legged_gym Terrain.make_terrain for the five kinds built here; heights in int64 sample units."""
    hs, vs = cfg.horizontal_scale, cfg.vertical_scale
    cum = np.cumsum(list(cfg.terrain_proportions) + [0.0] * (5 - len(cfg.terrain_proportions)))
    h = np.zeros(shape, np.int64)
    slope = difficulty * 0.4
    step_height = 0.05 + 0.18 * difficulty
    obstacle_height = 0.05 + difficulty * 0.2
    if choice < cum[0]:
        _pyramid_slope(h, -slope if choice < cum[0] / 2 else slope, hs, vs, 3.0)
    elif choice < cum[1]:
        _pyramid_slope(h, slope, hs, vs, 3.0)
        _random_uniform(h, rng, -0.05, 0.05, 0.005, 0.2, hs, vs)
    elif choice < cum[3]:
        _pyramid_stairs(h, 0.31, -step_height if choice < cum[2] else step_height, 3.0, hs, vs)
    else:  # choice < cum[4] = 1 (+ the 0.001 of the curriculum's last column: obstacles too)
        _discrete_obstacles(h, rng, obstacle_height, 1.0, 2.0, 20, 3.0, hs, vs)
    return h


def height_points(cfg: TerrainConfig) -> Optional[np.ndarray]:
    """legged_gym's _init_height_points: (P, 2) float32 points in the base's yaw frame, point k = (x[k // ny], y[k % ny])
    (torch.meshgrid(x, y) in "ij" order, flattened); None without measure_heights."""
    if not cfg.measure_heights:
        return None
    x = np.asarray(cfg.measured_points_x, np.float64)
    y = np.asarray(cfg.measured_points_y, np.float64)
    for k, v in (("measured_points_x", x), ("measured_points_y", y)):
        if v.ndim != 1 or len(v) < 1 or not np.all(np.isfinite(v)):
            raise DyrosError(f"terrain: {k} must be a non-empty list of finite numbers (got {getattr(cfg, k)!r})")
    if len(x) * len(y) > 1024:
        raise DyrosError(f"terrain: at most 1024 height points (got {len(x)} x {len(y)} = {len(x) * len(y)})")
    gx, gy = np.meshgrid(x.astype(np.float32), y.astype(np.float32), indexing="ij")
    return np.ascontiguousarray(np.stack([gx.ravel(), gy.ravel()], 1), np.float32)


def convert_heightfield_to_trimesh(height_field_raw, horizontal_scale, vertical_scale, slope_threshold=None):
    """isaacgym's terrain_utils.convert_heightfield_to_trimesh -> (vertices (R*C, 3) float32, triangles
    (2 (R-1)(C-1), 3) uint32). Vertex r*C + c sits at (r hs, c hs, vs h[r, c]); with slope_threshold, a vertex moves one
    horizontal step along x (y) toward a neighbour higher by more than slope_threshold * hs / vs sample units, and along
    the diagonal where it moved along neither, so that steep steps become vertical walls. Cell (i, j) gives the
    triangles (i,j),(i+1,j+1),(i,j+1) and (i,j),(i+1,j),(i+1,j+1), in that order: the heightfield's diagonal split,
    facing up."""
    hf = np.asarray(height_field_raw).astype(np.int64)
    nr, nc = hf.shape
    hs = float(horizontal_scale)
    yy, xx = np.meshgrid(np.linspace(0, (nc - 1) * hs, nc), np.linspace(0, (nr - 1) * hs, nr))
    if slope_threshold is not None:
        t = slope_threshold * hs / vertical_scale
        move_x, move_y, move_c = (np.zeros((nr, nc)) for _ in range(3))
        move_x[:nr - 1, :] += hf[1:, :] - hf[:nr - 1, :] > t
        move_x[1:, :] -= hf[:nr - 1, :] - hf[1:, :] > t
        move_y[:, :nc - 1] += hf[:, 1:] - hf[:, :nc - 1] > t
        move_y[:, 1:] -= hf[:, :nc - 1] - hf[:, 1:] > t
        move_c[:nr - 1, :nc - 1] += hf[1:, 1:] - hf[:nr - 1, :nc - 1] > t
        move_c[1:, 1:] -= hf[:nr - 1, :nc - 1] - hf[1:, 1:] > t
        xx = xx + (move_x + move_c * (move_x == 0)) * hs
        yy = yy + (move_y + move_c * (move_y == 0)) * hs
    vertices = np.zeros((nr * nc, 3), np.float32)
    vertices[:, 0] = xx.ravel()
    vertices[:, 1] = yy.ravel()
    vertices[:, 2] = hf.ravel() * vertical_scale
    i, j = np.meshgrid(np.arange(nr - 1), np.arange(nc - 1), indexing="ij")
    i0 = (i * nc + j).ravel()
    i1, i2 = i0 + 1, i0 + nc
    i3 = i2 + 1
    triangles = np.empty((2 * len(i0), 3), np.uint32)
    triangles[0::2] = np.stack([i0, i3, i1], 1)
    triangles[1::2] = np.stack([i0, i2, i3], 1)
    return vertices, triangles


def trimesh_from_field(hf: HeightField, slope_threshold) -> TriangleMesh:
    """legged_gym's trimesh terrain: the mesh of a generated field (equal row and column scales) at the field's origin,
    with the field's friction, and the field as the samples of the height scan."""
    if hf.row_scale != hf.column_scale:
        raise DyrosError(f"terrain: a trimesh needs equal row and column scales (legged_gym's horizontal_scale; got "
                         f"{hf.row_scale}, {hf.column_scale})")
    v, t = convert_heightfield_to_trimesh(hf.samples, hf.row_scale, hf.vertical_scale, slope_threshold)
    return TriangleMesh(v, t, origin=tuple(hf.origin), friction=hf.friction, scan_field=hf)


def validate(cfg: TerrainConfig):
    if cfg.mesh_type == "trimesh":
        raise DyrosError("terrain: mesh_type 'trimesh' is not accepted here; use mesh_type 'heightfield' (for legged_gym's "
                         "trimesh ground, set cfg[\"env\"][\"terrainMesh\"] = True beside it)")
    st = cfg.slope_treshold
    if st is not None and not (isinstance(st, (int, float)) and not isinstance(st, bool) and np.isfinite(st) and st >= 0):
        raise DyrosError(f"terrain: slope_treshold must be a number >= 0 or None (got {st!r})")
    if cfg.mesh_type != "heightfield":
        raise DyrosError(f"terrain: nothing to generate for mesh_type {cfg.mesh_type!r} (only 'heightfield')")
    p = np.asarray(cfg.terrain_proportions, np.float64)
    if p.ndim != 1 or len(p) < 1 or len(p) > 5:
        raise DyrosError(f"terrain: at most 5 terrain_proportions (smooth slope, rough slope, stairs up, stairs down, "
                         f"discrete obstacles); stepping stones, gaps and pits are not built (got {len(p)})")
    if np.any(p < 0) or abs(p.sum() - 1.0) > 1e-6:
        raise DyrosError(f"terrain: terrain_proportions must be >= 0 and sum to 1 (sum {p.sum()})")
    for k in ("horizontal_scale", "vertical_scale", "terrain_length", "terrain_width"):
        v = getattr(cfg, k)
        if not (np.isfinite(v) and v > 0):
            raise DyrosError(f"terrain: {k} must be positive (got {v})")
    if not (np.isfinite(cfg.border_size) and cfg.border_size >= 0):
        raise DyrosError(f"terrain: border_size must be >= 0 (got {cfg.border_size})")
    if cfg.num_rows < 1 or cfg.num_cols < 1:
        raise DyrosError(f"terrain: num_rows and num_cols must be >= 1 (got {cfg.num_rows}, {cfg.num_cols})")
    if cfg.static_friction != cfg.dynamic_friction:
        raise DyrosError("terrain: the contact model has one friction coefficient: static_friction and dynamic_friction "
                         f"must be equal (got {cfg.static_friction}, {cfg.dynamic_friction})")


def generate(cfg: TerrainConfig):
    """-> (HeightField, origins (num_rows, num_cols, 3) float64). Rows (levels) run along x, columns (types) along y;
    the field's vertex (0, 0) sits at (-border_size, -border_size, 0), so sub-terrain (i, j) covers
    [i terrain_length, (i + 1) terrain_length) x [j terrain_width, (j + 1) terrain_width)."""
    validate(cfg)
    rng = np.random.default_rng(cfg.seed)
    hs, vs = cfg.horizontal_scale, cfg.vertical_scale
    lx, ly = int(cfg.terrain_length / hs), int(cfg.terrain_width / hs)
    border = int(cfg.border_size / hs)
    raw = np.zeros((cfg.num_rows * lx + 2 * border, cfg.num_cols * ly + 2 * border), np.int64)
    origins = np.zeros((cfg.num_rows, cfg.num_cols, 3))
    cells = [(i, j) for j in range(cfg.num_cols) for i in range(cfg.num_rows)] if cfg.curriculum else \
        [(k // cfg.num_cols, k % cfg.num_cols) for k in range(cfg.num_rows * cfg.num_cols)]
    for i, j in cells:
        if cfg.curriculum:
            difficulty, choice = i / cfg.num_rows, j / cfg.num_cols + 0.001
        else:
            choice, difficulty = rng.uniform(0, 1), rng.choice([0.5, 0.75, 0.9])
        h = _sub_terrain(cfg, rng, choice, difficulty, (lx, ly))
        x0, y0 = border + i * lx, border + j * ly
        raw[x0:x0 + lx, y0:y0 + ly] = h
        # origin: the centre of the sub-terrain, on the highest sample of its central 2 m x 2 m
        x1, x2 = int((cfg.terrain_length / 2 - 1) / hs), int((cfg.terrain_length / 2 + 1) / hs)
        y1, y2 = int((cfg.terrain_width / 2 - 1) / hs), int((cfg.terrain_width / 2 + 1) / hs)
        origins[i, j] = ((i + 0.5) * cfg.terrain_length, (j + 0.5) * cfg.terrain_width, h[x1:x2, y1:y2].max() * vs)
    info = np.iinfo(np.int16)
    if raw.min() < info.min or raw.max() > info.max:
        raise DyrosError(f"terrain: heights [{raw.min()}, {raw.max()}] (units of vertical_scale {vs}) overflow int16; "
                         "raise vertical_scale")
    hf = HeightField(raw.astype(np.int16), hs, hs, vs, origin=(-cfg.border_size, -cfg.border_size, 0.0),
                     friction=cfg.static_friction)
    return hf, origins
