"""Height scan of the observation (DESIGN.md section 4, "Height scan") restated in numpy float32, operation for operation
in the order of stage_height_scan (task_kernels.cu): legged_gym's _get_heights, quat_apply_yaw and the height term of
compute_observations, with the field transform in place of border_size."""
import numpy as np

f32 = np.float32


def world_points(root, points):
    """(N, P) world x and y of the points (P, 2) of the base's yaw frame, for roots (N, 13) [pos, quat xyzw, ...]."""
    r = np.asarray(root, f32)
    qz, qw = r[:, 5:6], r[:, 6:7]
    n = np.maximum(np.sqrt(qz * qz + qw * qw), f32(1e-9))  # torch_utils normalize of (0, 0, qz, qw)
    z, w = qz / n, qw / n
    px, py = np.asarray(points, f32)[None, :, 0], np.asarray(points, f32)[None, :, 1]
    # quat_apply((0, 0, z, w), (px, py, 0)): t = cross(xyz, v) * 2; v + w t + cross(xyz, t) (zero terms left out)
    tx, ty = -(z * py) * f32(2), (z * px) * f32(2)
    wx = ((px + w * tx) - z * ty) + r[:, 0:1]
    wy = ((py + w * ty) + z * tx) + r[:, 1:2]
    return wx, wy


def cell_index(wx, wy, field):
    """legged_gym's px, py: trunc((w - origin) / scale), clamped to [0, n - 2]."""
    nr, nc = field.samples.shape
    ox, oy = f32(field.origin[0]), f32(field.origin[1])
    u = np.minimum(np.maximum((wx - ox) / f32(field.row_scale), f32(0)), f32(nr - 2))
    v = np.minimum(np.maximum((wy - oy) / f32(field.column_scale), f32(0)), f32(nc - 2))
    return u.astype(np.int64), v.astype(np.int64)


def heights_at(ix, iy, field):
    """origin.z + vertical_scale * min(s[px, py], s[px+1, py], s[px, py+1])."""
    s = field.samples
    m = np.minimum(np.minimum(s[ix, iy], s[ix + 1, iy]), s[ix, iy + 1])
    return f32(field.origin[2]) + f32(field.vertical_scale) * m.astype(f32)


def heights(root, points, field=None):
    """(N, P) measured heights in m; the plane (field None) gives 0."""
    wx, wy = world_points(root, points)
    if field is None:
        return np.zeros(wx.shape, f32)
    return heights_at(*cell_index(wx, wy, field), field)


def obs_columns(root, h, base_offset=0.5, scale=5.0):
    """obs[:, 487 + k] = clip(root_z - base_offset - h_k, -1, 1) * scale."""
    rz = np.asarray(root, f32)[:, 2:3]
    return np.minimum(np.maximum((rz - f32(base_offset)) - h, f32(-1)), f32(1)) * f32(scale)
