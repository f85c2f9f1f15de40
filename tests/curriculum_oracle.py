"""Oracle of the terrain curriculum (DESIGN.md section 4, "Curriculum"): legged_gym's _update_terrain_curriculum in
float32 numpy, operation for operation as the reset stage computes it, and T:598-669 with it (oracle/task_oracle.py's
reset_idx, which is left as it is, runs after the level update)."""
import numpy as np

from oracle import task_oracle as O

f32 = np.float32
U_COL = 30  # reset_f column of the draw that places an env that climbed past the top level


def update_levels(root_xy, origin_xy, target_vel, levels, u, num_levels, move_up_distance, move_down_scale):
    """New levels of resetting envs: up when the root walked farther than move_up_distance from its origin, else down
    when it walked less than |target_vel| * move_down_scale; past the top a uniform level int(u * num_levels)."""
    root_xy, origin_xy, target_vel = (np.asarray(a, f32) for a in (root_xy, origin_xy, target_vel))
    dx, dy = root_xy[:, 0] - origin_xy[:, 0], root_xy[:, 1] - origin_xy[:, 1]
    d = np.sqrt(dx * dx + dy * dy)
    tvx, tvy = target_vel[:, 0], target_vel[:, 1]
    up = d > f32(move_up_distance)
    down = ~up & (d < np.sqrt(tvx * tvx + tvy * tvy) * f32(move_down_scale))
    lvl = np.asarray(levels, np.int64) + up.astype(np.int64) - down.astype(np.int64)
    drawn = np.minimum((np.asarray(u, f32) * f32(num_levels)).astype(np.int64), num_levels - 1)
    return np.where(lvl >= num_levels, drawn, np.maximum(lvl, 0)).astype(np.int32)


def reset_idx(s, c, env_ids, noise, cur):
    """T:598-669 with the curriculum: `cur` holds origins (levels, types, 3) float32, types and levels (N,) int32 (updated
    in place), move_up_distance, move_down_scale."""
    e = np.asarray(env_ids, np.int64)
    if e.size:
        lvl = update_levels(s["root_states"][e, 0:2], s["env_origins"][e, 0:2], s["target_vel"][e], cur["levels"][e],
                            noise["reset_f"][e, U_COL], cur["origins"].shape[0], cur["move_up_distance"],
                            cur["move_down_scale"])
        cur["levels"][e] = lvl
        s["env_origins"][e] = cur["origins"][lvl, cur["types"][e]]
    O.reset_idx(s, c, env_ids, noise)
