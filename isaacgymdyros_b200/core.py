"""DyrosCore: owns every device buffer of one env shard (torch allocations) and the two native handles
(DyrosSim = what gym.create_sim returns, DyrosTask = the per-env state of DyrosDynamicWalk), and issues the
C-ABI calls on torch's current CUDA stream. The gym facade (gym.py) and the VecTask mirror
(tasks/dyros_dynamic_walk.py) are thin views over this object.

Reference: python/IsaacGymEnvs/isaacgymenvs/tasks/dyros_dynamic_walk.py (T) and tasks/base/vec_task.py (VT).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field, replace
from typing import Dict, Optional

import numpy as np
import torch

from . import native
from .model.tables import ModelTables, role_programs

ASSETS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets")
ND, NB, NA = 33, 38, 13
NOBS = 487  # columns of an observation row without a height scan
# height scan (legged_gym's measure_heights): obs = clip(root_z - BASE_OFFSET - h, -1, 1) * SCALE
HEIGHT_SCAN_BASE_OFFSET, HEIGHT_SCAN_SCALE = 0.5, 5.0  # _get_heights / compute_observations, obs_scales.height_measurements
MAX_HEIGHT_POINTS = 1024
NPRIV = 31  # privileged columns at the end of a critic state row (DESIGN.md section 4, "Critic states")

# T:58-70 (before the /9 and /3), T:296-301, T:95-100, T:366-371
KP = [2000.0, 5000.0, 4000.0, 3700.0, 3200.0, 3200.0, 2000.0, 5000.0, 4000.0, 3700.0, 3200.0, 3200.0,
      6000.0, 10000.0, 10000.0, 400.0, 1000.0, 400.0, 400.0, 400.0, 400.0, 100.0, 100.0, 100.0, 100.0,
      400.0, 1000.0, 400.0, 400.0, 400.0, 400.0, 100.0, 100.0]
KV = [15.0, 50.0, 20.0, 25.0, 24.0, 24.0, 15.0, 50.0, 20.0, 25.0, 24.0, 24.0, 200.0, 100.0, 100.0,
      10.0, 28.0, 10.0, 10.0, 10.0, 10.0, 3.0, 3.0, 2.0, 2.0, 10.0, 28.0, 10.0, 10.0, 10.0, 10.0, 3.0, 3.0]
ACTION_HIGH = [333, 232, 263, 289, 222, 166, 333, 232, 263, 289, 222, 166, 303, 303, 303, 64, 64, 64, 64,
               23, 23, 10, 10, 10, 10, 64, 64, 64, 64, 23, 23, 10, 10]
INIT_DOF_POS = [0.0, 0.0, -0.24, 0.6, -0.36, 0.0, 0.0, 0.0, -0.24, 0.6, -0.36, 0.0, 0.0, 0.0, 0.0,
                0.3, 0.3, 1.5, -1.27, -1.0, 0.0, -1.0, 0.0, 0.0, 0.0, -0.3, -0.3, -1.5, 1.27, 1.0, 0.0, 1.0, 0.0]
ARMATURE = [0.614, 0.862, 1.09, 1.09, 1.09, 0.360, 0.614, 0.862, 1.09, 1.09, 1.09, 0.360,
            0.078, 0.078, 0.078, 0.18, 0.18, 0.18, 0.18, 0.0032, 0.0032, 0.0032, 0.0032, 0.0032, 0.0032,
            0.18, 0.18, 0.18, 0.18, 0.0032, 0.0032, 0.0032, 0.0032]


@dataclass
class HeightField:
    """Heightfield ground (gym.add_heightfield; DESIGN.md section 4): vertex (i, j) sits at
    origin + (i row_scale, j column_scale, vertical_scale samples[i, j]), row index i along x and column index j along y
    (Isaac Gym's HeightFieldParams, legged_gym's height_samples[px, py]); each cell is split along its diagonal
    (i, j)-(i+1, j+1); outside the field's x-y rectangle there is no ground.
    friction: the ground's coefficient in place of CoreConfig.friction (None: keep it).
    env_origins: (N, 3) world origins of the envs (None: the usual grid, T:709-718, with z the terrain height there)."""
    samples: np.ndarray
    row_scale: float
    column_scale: float
    vertical_scale: float
    origin: tuple = (0.0, 0.0, 0.0)
    friction: Optional[float] = None
    env_origins: Optional[np.ndarray] = None

    def validate(self):
        s = self.samples
        if not isinstance(s, np.ndarray) or s.dtype != np.int16 or s.ndim != 2 or min(s.shape) < 2:
            raise native.DyrosError("heightfield: samples must be a 2-D int16 array of at least 2 x 2 (rows along x, "
                                    f"columns along y); got {getattr(s, 'dtype', type(s))} {getattr(s, 'shape', '')}")
        for k in ("row_scale", "column_scale", "vertical_scale"):
            v = getattr(self, k)
            if not (np.isfinite(v) and v > 0):
                raise native.DyrosError(f"heightfield: {k} must be positive (got {v})")
        if len(self.origin) != 3 or not np.all(np.isfinite(self.origin)):
            raise native.DyrosError(f"heightfield: origin must be 3 finite numbers (got {self.origin})")
        if self.friction is not None and not (np.isfinite(self.friction) and self.friction >= 0):
            raise native.DyrosError(f"heightfield: friction must be >= 0 (got {self.friction})")

    def height_at(self, x, y):
        """Terrain height at world points (x, y) and whether they lie on the field (same triangles as the kernels)."""
        s = self.samples.astype(np.float64) * self.vertical_scale
        nr, nc = s.shape
        u = (np.asarray(x, np.float64) - self.origin[0]) / self.row_scale
        v = (np.asarray(y, np.float64) - self.origin[1]) / self.column_scale
        inside = (u >= 0) & (v >= 0) & (u <= nr - 1) & (v <= nc - 1)
        u, v = np.where(inside, u, 0.0), np.where(inside, v, 0.0)
        i, j = np.minimum(u.astype(int), nr - 2), np.minimum(v.astype(int), nc - 2)
        fu, fv = u - i, v - j
        h00, h11 = s[i, j], s[i + 1, j + 1]
        lower = fu >= fv
        gu = np.where(lower, s[i + 1, j] - h00, h11 - s[i, j + 1])
        gv = np.where(lower, h11 - s[i + 1, j], s[i, j + 1] - h00)
        return self.origin[2] + h00 + fu * gu + fv * gv, inside


@dataclass
class TerrainCurriculum:
    """Envs on a grid of sub-terrains and the terrain curriculum (legged_gym's _update_terrain_curriculum; DESIGN.md
    section 4, "Curriculum"): env e starts at origins[levels[e], types[e]]. With `curriculum`, every reset moves it one
    level up when it walked farther than move_up_distance from its origin, one level down when it walked less than
    |target_vel| * move_down_scale; past the top level it lands on a random one. The update runs in the reset stage of
    the task kernels (dyros_task_set_terrain_curriculum).
    origins: (num_levels, num_types, 3) world origins of the sub-terrains; types, levels: (N,) integers."""
    origins: np.ndarray
    types: np.ndarray
    levels: np.ndarray
    move_up_distance: float      # terrain_length / 2
    move_down_scale: float       # episode length (s) * 0.5
    curriculum: bool = True      # False: the envs keep their initial sub-terrain (no level updates)

    def validate(self, n: int):
        o = np.asarray(self.origins)
        if o.ndim != 3 or o.shape[2] != 3 or min(o.shape[:2]) < 1 or not np.all(np.isfinite(o)):
            raise native.DyrosError(f"terrain curriculum: origins must be a finite (levels, types, 3) array (got {o.shape})")
        for k, hi in (("types", o.shape[1]), ("levels", o.shape[0])):
            v = np.asarray(getattr(self, k))
            if v.shape != (n,) or not np.issubdtype(v.dtype, np.integer) or v.min() < 0 or v.max() >= hi:
                raise native.DyrosError(f"terrain curriculum: {k} must be ({n},) integers in [0, {hi}) "
                                        f"(got {v.dtype} {v.shape})")
        for k in ("move_up_distance", "move_down_scale"):
            v = getattr(self, k)
            if not (np.isfinite(v) and v >= 0):
                raise native.DyrosError(f"terrain curriculum: {k} must be >= 0 (got {v})")


@dataclass
class CoreConfig:
    """Values of cfg/task/DyrosDynamicWalk.yaml that reach the kernels (SURVEY Appendix A1) plus the
    named model options of SURVEY D2."""
    dt: float = 0.002                    # sim.dt
    substeps: int = 1                    # sim.substeps
    control_freq_inv: int = 2            # env.controlFrequencyInv -> skipframe
    episode_length_s: float = 32.0
    gravity: tuple = (0.0, 0.0, -9.81)
    contact_offset: float = 0.002        # physx.contact_offset
    max_depenetration_velocity: float = 10.0
    num_position_iterations: int = 4
    num_velocity_iterations: int = 1
    contact_erp: float = 0.2
    friction: float = 1.0                # plane 1.0 combined with shape default 1.0
    penalty_stiffness: float = 2.0e5
    penalty_damping: float = 2.0e3
    penalty_max_force: float = 2.0e4
    max_angular_velocity: float = 100.0  # AssetOptions, T:289
    clamp_effort: bool = False
    dof_damping: float = 0.1             # T:365
    dof_vel_limit: float = 4.03          # T:372
    death_cost: float = 0.0
    initial_height: float = 0.93
    env_spacing: float = 5.0
    perturb: bool = True
    randomize: bool = False              # task.randomize (DR re-draw on reset)
    dr_damping_range: tuple = (0.0, 2.9)   # additive, CFG:103-108
    dr_armature_range: tuple = (0.8, 1.2)  # scaling, CFG:109-115
    dr_mass_range: tuple = (0.8, 1.2)      # scaling, setup only, CFG:81-88
    # optional per-env tables (BASELINE configs[3] "friction / PD gains"; commented out in the reference, CFG:89-96):
    dr_friction_range: Optional[tuple] = None  # scaling of `friction` per env -> sim_t["contact_friction"] (N)
    dr_pd_gain_range: Optional[tuple] = None   # scaling of Kp and of Kv per env -> task_t["pd_gain_scale"] (N,2)
    left_foot: str = "L_Foot_Link"
    right_foot: str = "R_Foot_Link"
    solver_bodies: tuple = ("L_Foot_Link", "R_Foot_Link")
    with_rigid_body_state: bool = False  # DyrosDynamicWalk never reads it (T:76,85)
    with_rb_force_tensors: bool = False  # generic apply_rigid_body_force_tensors buffers
    physics_program: str = "roles"       # "roles": one lane per env, warp per role (default); "lanes": 8 lanes per env
    self_collision: bool = True          # create_actor(..., filter 0), T:354: the actor's shapes collide with each other
    heightfield: Optional[HeightField] = None  # ground: None = the plane z = 0 (gym.add_ground), else gym.add_heightfield
    terrain_curriculum: Optional[TerrainCurriculum] = None  # env origins on sub-terrains (+ level updates on reset)
    # (P, 2) points of the height scan in the base's yaw frame (legged_gym's height_points; DESIGN.md section 4, "Height
    # scan"), or None: each observation row gains P terrain heights around the base, on any ground
    height_scan: Optional[np.ndarray] = None
    # critic states (DESIGN.md section 4, "Critic states"): task_t["states_buf"] (N, 487 + P + 31) gains a privileged row
    # per env, written by the observation kernels; the P heights of a height scan then go into it and, only with
    # critic_heights_in_obs, into the observation row as well
    critic_states: bool = False
    critic_heights_in_obs: bool = False


def validate_height_points(points) -> np.ndarray:
    """(P, 2) finite float32 points, 1 <= P <= 1024, or DyrosError."""
    p = np.asarray(points, np.float64)
    if p.ndim != 2 or p.shape[1] != 2 or not 1 <= p.shape[0] <= MAX_HEIGHT_POINTS or not np.all(np.isfinite(p)):
        raise native.DyrosError(f"height scan: points must be a finite (P, 2) array with 1 <= P <= {MAX_HEIGHT_POINTS} "
                                f"(got shape {p.shape})")
    return np.ascontiguousarray(p, np.float32)


def stable_penalty(dt_substep: float, m_ref: float = 0.3):
    """Penalty (non-foot) ground contact is integrated explicitly: stiffness k and damping c are only stable for
    k dt^2 / m <~ 1 and c dt / m <~ 1. Returns (k, c) for a reference link mass, capped at the TOCABI defaults."""
    return min(2.0e5, 0.5 * m_ref / dt_substep ** 2), min(2.0e3, 0.5 * m_ref / dt_substep)


def _np_ptr(a: np.ndarray, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def env_origins(n: int, spacing: float) -> np.ndarray:
    """T:709-718."""
    num_cols = np.floor(np.sqrt(n))
    num_rows = np.ceil(n / num_cols)
    xx, yy = np.meshgrid(np.arange(num_rows), np.arange(num_cols), indexing="ij")
    o = np.zeros((n, 3), dtype=np.float32)
    o[:, 0] = (spacing * xx.flatten()[:n]).astype(np.float32)
    o[:, 1] = (spacing * yy.flatten()[:n]).astype(np.float32)
    return o


_SC_CACHE: dict = {}


def self_collision_tables(t: ModelTables):
    """model/selfcollision.py tables of an articulation, built once per model (rest poses: zero and, for TOCABI, the
    task's initial pose T:95-100)."""
    from .model import selfcollision
    key = (tuple(t.body_names), t.pt_pos.tobytes(), t.cyl_center.tobytes())
    if key not in _SC_CACHE:
        rest = [np.array(INIT_DOF_POS)] if t.num_dofs == ND else []
        try:
            _SC_CACHE[key] = selfcollision.build(t, rest)
        except ValueError:  # primitives this module does not describe (capsules / spheres of the stock Humanoid)
            _SC_CACHE[key] = None
    return _SC_CACHE[key]


def make_model_desc(t: ModelTables, cfg: "CoreConfig"):
    """ModelTables -> DyrosModelDesc (host arrays are returned too: keep them alive during the create call)."""
    keep = []
    f64 = lambda a: keep.append(np.ascontiguousarray(a, dtype=np.float64)) or keep[-1]
    i32 = lambda a: keep.append(np.ascontiguousarray(a, dtype=np.int32)) or keep[-1]
    md = native.DyrosModelDesc()
    md.num_links, md.num_bodies, md.num_dofs = t.num_links, t.num_bodies, t.num_dofs
    solver_ids = [t.body_names.index(n) for n in cfg.solver_bodies]
    pt_solver = np.isin(t.pt_body, solver_ids).astype(np.int32)
    prog = role_programs(t.link_parent, sorted(set(int(l) for l in t.pt_link[pt_solver > 0])))
    md.num_points, md.num_cyls, md.sched_slots = len(t.pt_link), len(t.cyl_link), prog.shape[0]
    vel_limit = np.full(t.num_dofs, cfg.dof_vel_limit)
    for name, arr, ct in [("link_parent", i32(t.link_parent), C.c_int32), ("link_dof", i32(t.link_dof), C.c_int32),
                          ("link_E", f64(t.link_E), C.c_double), ("link_r", f64(t.link_r), C.c_double),
                          ("link_axis", f64(t.link_axis), C.c_double), ("body_link", i32(t.body_link), C.c_int32),
                          ("body_pos", f64(t.body_pos), C.c_double), ("body_rot", f64(t.body_rot), C.c_double),
                          ("body_inertia", f64(t.body_inertia), C.c_double),
                          ("dof_lower", f64(t.dof_lower), C.c_double), ("dof_upper", f64(t.dof_upper), C.c_double),
                          ("dof_vel_limit", f64(vel_limit), C.c_double), ("dof_effort", f64(t.dof_effort), C.c_double),
                          ("dof_stiffness", f64(t.dof_stiffness), C.c_double),
                          ("pt_link", i32(t.pt_link), C.c_int32), ("pt_body", i32(t.pt_body), C.c_int32),
                          ("pt_pos", f64(t.pt_pos), C.c_double), ("pt_radius", f64(t.pt_radius), C.c_double),
                          ("pt_solver", i32(pt_solver), C.c_int32),
                          ("cyl_link", i32(t.cyl_link), C.c_int32), ("cyl_body", i32(t.cyl_body), C.c_int32),
                          ("cyl_center", f64(t.cyl_center), C.c_double), ("cyl_axis", f64(t.cyl_axis), C.c_double),
                          ("cyl_size", f64(t.cyl_size), C.c_double), ("sched", i32(prog), C.c_int32)]:
        setattr(md, name, _np_ptr(arr, ct))
    sc = self_collision_tables(t) if cfg.self_collision else None
    if sc is not None and len(sc.pairs):
        md.sc_num_shapes, md.sc_num_samples, md.sc_num_pairs = sc.num_shapes, len(sc.sample), len(sc.pairs)
        for name, arr, ct in [("sc_shape_kind", i32(sc.shape_kind), C.c_int32), ("sc_shape_link", i32(sc.shape_link), C.c_int32),
                              ("sc_shape_body", i32(sc.shape_body), C.c_int32), ("sc_shape_sample0", i32(sc.shape_sample0), C.c_int32),
                              ("sc_shape_center", f64(sc.shape_center), C.c_double), ("sc_shape_rot", f64(sc.shape_rot), C.c_double),
                              ("sc_shape_size", f64(sc.shape_size), C.c_double), ("sc_sample", f64(sc.sample), C.c_double),
                              ("sc_link_shape0", i32(sc.link_shape0), C.c_int32), ("sc_link_sphere", f64(sc.link_sphere), C.c_double),
                              ("sc_pairs", i32(sc.pairs), C.c_int32)]:
            setattr(md, name, _np_ptr(arr, ct))
    return md, keep


def make_sim_desc(cfg: "CoreConfig", num_envs: int, device_index: int = 0):
    sd = native.DyrosSimDesc()
    sd.num_envs, sd.device = num_envs, device_index
    sd.dt, sd.substeps = cfg.dt, cfg.substeps
    sd.gravity = (C.c_float * 3)(*cfg.gravity)
    sd.contact_offset = cfg.contact_offset
    sd.max_depenetration_velocity = cfg.max_depenetration_velocity
    sd.contact_sweeps = cfg.num_position_iterations + cfg.num_velocity_iterations
    sd.contact_erp = cfg.contact_erp
    sd.friction = cfg.friction
    sd.penalty_stiffness, sd.penalty_damping = cfg.penalty_stiffness, cfg.penalty_damping
    sd.penalty_max_force = cfg.penalty_max_force
    sd.max_angular_velocity = cfg.max_angular_velocity
    sd.clamp_effort = int(cfg.clamp_effort)
    sd.physics_program = {"roles": 0, "lanes": 1}[cfg.physics_program]
    return sd


def measure_fp32_peak(device_index: int = 0, iters: int = 20000) -> float:
    """TFLOP/s of an FFMA-saturation kernel on this GPU (the FP32 roofline denominator, SURVEY section 8d)."""
    out = C.c_double()
    native.check(native.load().dyros_measure_fp32_peak(device_index, iters, C.byref(out)), "dyros_measure_fp32_peak")
    return out.value


class DyrosCore:
    def __init__(self, num_envs: int, device: str = "cuda:0", cfg: Optional[CoreConfig] = None,
                 tables: Optional[ModelTables] = None, seed: int = 42, rank: int = 0, with_task: bool = True):
        """with_task=False builds only the simulator (gym level) and accepts any supported articulation; the
        DyrosDynamicWalk task state needs the 33-DOF / 38-body TOCABI model."""
        if not torch.cuda.is_available():
            raise native.DyrosError("DyrosCore needs a CUDA device (sm_100a); there is no CPU path")
        self.lib = native.load()
        self.cfg = cfg or CoreConfig()
        self.N = int(num_envs)
        hf = self.cfg.heightfield
        if hf is not None:
            hf.validate()
            if self.cfg.physics_program != "roles":
                raise native.DyrosError("heightfield: only the roles physics program has a heightfield ground (the lanes "
                                        "program is plane only)")
            if hf.friction is not None:
                self.cfg = replace(self.cfg, friction=float(hf.friction))
        tc = self.cfg.terrain_curriculum
        if tc is not None:
            if not with_task:
                raise native.DyrosError("terrain curriculum: needs the task (its reset stage moves the envs)")
            tc.validate(int(num_envs))
        self.height_points = None
        if self.cfg.height_scan is not None:
            if not with_task:
                raise native.DyrosError("height scan: needs the task (its observation kernels measure the heights)")
            self.height_points = validate_height_points(self.cfg.height_scan)
        self.num_height_points = 0 if self.height_points is None else len(self.height_points)
        cs = bool(self.cfg.critic_states)
        if cs and not with_task:
            raise native.DyrosError("critic states: need the task (its observation kernels write them)")
        heights_in_obs = not cs or bool(self.cfg.critic_heights_in_obs)
        self.obs_width = NOBS + (self.num_height_points if heights_in_obs else 0)  # columns of obs_buf
        self.states_width = NOBS + self.num_height_points + NPRIV if cs else 0  # columns of states_buf (0: none)
        self.device = torch.device(device)
        self.tables = tables or ModelTables.load(os.path.join(ASSETS, "tocabi_tables.npz"))
        t = self.tables
        self.with_task = with_task
        self.nd, self.nb = t.num_dofs, t.num_bodies
        if with_task and (t.num_dofs != ND or t.num_bodies != NB):
            raise native.DyrosError("DyrosDynamicWalk expects the 33-DOF / 38-body TOCABI model")
        self._keep = []  # host arrays referenced by the descriptors during the create calls
        self.l2_persist = False
        self.sim_handle = C.c_void_p()
        self.task_handle = C.c_void_p()
        torch.cuda.set_device(self.device)
        self._alloc()
        self._pack_state_arena()
        self._create_sim()
        if with_task:
            self._create_task(seed + rank)

    # ------------------------------------------------------------------ buffers
    def _alloc(self):
        N, dev, cfg = self.N, self.device, self.cfg
        nd, nb = self.nd, self.nb
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=dev)
        s: Dict[str, torch.Tensor] = {}
        s["root_states"] = z(N, 13)
        s["dof_state"] = z(N * nd, 2)
        s["net_contact_force"] = z(N * nb, 3)
        s["dof_actuation_force"] = z(N * nd)
        if self.with_task:
            s["dof_damping"] = torch.full((N, nd), cfg.dof_damping, device=dev)
            s["dof_armature"] = torch.tensor(ARMATURE, device=dev).repeat(N, 1).contiguous()
        else:  # the asset's own joint properties (MJCF damping / armature)
            s["dof_damping"] = torch.tensor(self.tables.dof_damping, dtype=torch.float32, device=dev).repeat(N, 1).contiguous()
            s["dof_armature"] = torch.tensor(self.tables.dof_armature, dtype=torch.float32, device=dev).repeat(N, 1).contiguous()
        s["body_mass_scale"] = torch.ones(N, nb, device=dev)
        if cfg.dr_friction_range is not None:
            s["contact_friction"] = torch.full((N,), cfg.friction, device=dev)
        if cfg.with_rigid_body_state:
            s["rigid_body_state"] = z(N * nb, 13)
        if cfg.with_rb_force_tensors:
            s["rb_force"] = z(N * nb, 3)
            s["rb_torque"] = z(N * nb, 3)
        sc = self_collision_tables(self.tables) if cfg.self_collision else None
        if sc is not None and len(sc.pairs):
            s["link_pose"] = z(N, self.tables.num_links, 12)
            s["self_contact_force"] = z(N * nb, 3)
        self.sim_t = s
        s["root_states"][:, 6] = 1.0
        if not self.with_task:
            self.task_t = {}
            return
        tb: Dict[str, torch.Tensor] = {}
        for name, dt, shape in native.TASK_BUFFERS:
            full = tuple(shape[1:]) if (shape and shape[0] is None) else (N,) + tuple(shape)
            tb[name] = torch.zeros(full, dtype=getattr(torch, dt), device=dev)
        if cfg.dr_pd_gain_range is not None:
            tb["pd_gain_scale"] = torch.ones(N, 2, device=dev)
        if self.height_points is not None:  # wider rows; measured_heights (N, P) = legged_gym's self.measured_heights
            tb["obs_buf"] = z(N, self.obs_width)
            tb["measured_heights"] = z(N, self.num_height_points)
            tb["height_points"] = torch.tensor(self.height_points, device=dev)
        if self.states_width:
            tb["states_buf"] = z(N, self.states_width)
        mocap = np.load(os.path.join(ASSETS, "mocap_walk.npy"))
        obs_norm = np.load(os.path.join(ASSETS, "obs_norm.npy"))
        tb["mocap_data"] = torch.tensor(mocap, device=dev).contiguous()
        tb["obs_mean"] = torch.tensor(obs_norm[0], device=dev).contiguous()
        tb["obs_var"] = torch.tensor(obs_norm[1], device=dev).contiguous()
        self.task_t = tb
        # reference initial values (T:87-195, VT:242-255)
        s["root_states"][:, 2] = cfg.initial_height
        s["root_states"][:, 6] = 1.0
        s["dof_state"].view(N, ND, 2)[:, :, 0] = torch.tensor(INIT_DOF_POS, device=dev)
        tb["reset_buf"].fill_(1)
        tb["delay_idx"].fill_(1)
        tb["pert_duration"].fill_(1)
        tb["perturb_timing"].fill_(1)
        tb["motor_constant_scale"].fill_(1.0)
        tc = cfg.terrain_curriculum
        if tc is not None:
            tb["terrain_origins"] = torch.tensor(np.asarray(tc.origins, np.float32), device=dev).contiguous()
            tb["terrain_types"] = torch.tensor(np.asarray(tc.types, np.int32), device=dev)
            tb["terrain_levels"] = torch.tensor(np.asarray(tc.levels, np.int32), device=dev)
            if tc.curriculum:
                tb["terrain_level_mean"] = torch.tensor(float(np.mean(tc.levels)), dtype=torch.float32, device=dev)
        tb["env_origins"].copy_(torch.tensor(self._env_origins()))
        if cfg.heightfield is not None:  # start where the first reset puts the root (T:734-735), not above (0, 0)
            s["root_states"][:, 0:3] = tb["env_origins"]
            s["root_states"][:, 2] += cfg.initial_height
        self.nominal_mass = float(np.float32(self.tables.total_mass()))  # (critic states: total_mass / nominal - 1)
        tb["total_mass"].fill_(self.nominal_mass)
        tb["obs_hist_head"].fill_(19)
        tb["act_hist_head"].fill_(19)

    def _env_origins(self) -> np.ndarray:
        """T:709-718; on a heightfield the given origins, or the grid with z the terrain height there; with a terrain
        curriculum origins[levels, types] (every sub-terrain origin must then lie on the field)."""
        hf, tc = self.cfg.heightfield, self.cfg.terrain_curriculum
        if tc is not None:
            table = np.asarray(tc.origins, np.float32)
            if hf is not None:
                inside = hf.height_at(table[..., 0], table[..., 1])[1]
                if not inside.all():
                    l, t = np.argwhere(~inside)[0]
                    raise native.DyrosError(f"terrain curriculum: the origin of sub-terrain ({l}, {t}) lies outside the field")
            return table[np.asarray(tc.levels), np.asarray(tc.types)]
        if hf is None:
            return env_origins(self.N, self.cfg.env_spacing)
        if hf.env_origins is not None:
            o = np.asarray(hf.env_origins, np.float64)
            if o.shape != (self.N, 3) or not np.all(np.isfinite(o)):
                raise native.DyrosError(f"heightfield: env_origins must be a finite ({self.N}, 3) array (got {o.shape})")
        else:
            o = env_origins(self.N, self.cfg.env_spacing).astype(np.float64)
            o[:, 2] = hf.height_at(o[:, 0], o[:, 1])[0]
        inside = hf.height_at(o[:, 0], o[:, 1])[1]
        if not inside.all():
            e = int(np.flatnonzero(~inside)[0])
            raise native.DyrosError(f"heightfield: the origin of env {e} ({o[e, 0]:.3f}, {o[e, 1]:.3f}) lies outside the "
                                    f"field; {int((~inside).sum())} of {self.N} envs do")
        return o.astype(np.float32)

    def _pack_state_arena(self):
        """Moves every per-env buffer except obs_buf, states_buf and measured_heights (written once per step, never read
        by the step) into ONE contiguous allocation, 256-byte aligned views: the range dyros_sim_set_l2_persistence can
        pin in L2."""
        items = [(d, k) for d in (self.sim_t, self.task_t) for k in d if k not in ("obs_buf", "states_buf", "measured_heights")]
        al = lambda n: (n + 255) & ~255
        total = sum(al(d[k].numel() * d[k].element_size()) for d, k in items)
        self.state_arena = torch.zeros(total, dtype=torch.uint8, device=self.device)
        off = 0
        for d, k in items:
            t = d[k]
            nbytes = t.numel() * t.element_size()
            view = self.state_arena[off:off + nbytes].view(t.dtype).view(t.shape)
            view.copy_(t)
            d[k] = view
            off += al(nbytes)

    def set_l2_persistence(self, on: bool = True, stream: Optional["torch.cuda.Stream"] = None) -> int:
        """Pins the env state (state_arena) in the persisting part of L2 for the kernels launched on `stream` (default:
        the current stream) from now on, including those captured from it into CUDA graphs; returns the bytes of L2 set
        aside. Other kernels' traffic between two env steps then no longer evicts the state."""
        st = stream or torch.cuda.current_stream(self.device)
        out = C.c_size_t(0)
        native.check(self.lib.dyros_sim_set_l2_persistence(
            self.sim_handle, C.c_void_p(self.state_arena.data_ptr() if on else 0),
            C.c_size_t(self.state_arena.numel() if on else 0), C.c_void_p(st.cuda_stream), C.byref(out)),
            "dyros_sim_set_l2_persistence")
        self.l2_persist = bool(on)
        return int(out.value)

    # ------------------------------------------------------------------ native objects
    def _create_sim(self):
        md, keep = make_model_desc(self.tables, self.cfg)
        self._keep.extend(keep)
        sd = make_sim_desc(self.cfg, self.N, self.device.index or 0)
        sb = native.DyrosSimBuffers()
        for n in native.SIM_BUFFERS:
            setattr(sb, n, self.sim_t[n].data_ptr() if n in self.sim_t else None)
        native.check(self.lib.dyros_sim_create(C.byref(sd), C.byref(md), C.byref(sb), C.byref(self.sim_handle)),
                     "dyros_sim_create")
        hf = self.cfg.heightfield
        if hf is not None:
            # (device copy owned by this object: the sim reads it on every step)
            self.field_samples = torch.tensor(np.ascontiguousarray(hf.samples), dtype=torch.int16, device=self.device)
            d = native.DyrosHeightField()
            d.samples = self.field_samples.data_ptr()
            d.num_rows, d.num_columns = hf.samples.shape
            d.row_scale, d.column_scale, d.vertical_scale = hf.row_scale, hf.column_scale, hf.vertical_scale
            d.origin = (C.c_float * 3)(*hf.origin)
            native.check(self.lib.dyros_sim_set_heightfield(self.sim_handle, C.byref(d)), "dyros_sim_set_heightfield")

    def _create_task(self, seed: int):
        t, cfg = self.tables, self.cfg
        keep = self._keep
        f32 = lambda a: keep.append(np.ascontiguousarray(a, dtype=np.float32)) or keep[-1]
        td = native.DyrosTaskDesc()
        td.skipframe = cfg.control_freq_inv
        td.max_episode_length = cfg.episode_length_s / (cfg.dt * cfg.control_freq_inv)  # T:35
        td.death_cost, td.initial_height = cfg.death_cost, cfg.initial_height
        td.perturb, td.randomize = int(cfg.perturb), int(cfg.randomize)
        td.dr_damping_base = cfg.dof_damping
        td.dr_damping_lo, td.dr_damping_hi = cfg.dr_damping_range
        td.dr_armature_lo, td.dr_armature_hi = cfg.dr_armature_range
        arm = np.ascontiguousarray(ARMATURE, dtype=np.float64)
        keep.append(arm)
        td.dr_armature_base = _np_ptr(arm, C.c_double)
        td.dr_friction_base = cfg.friction
        td.dr_friction_lo, td.dr_friction_hi = cfg.dr_friction_range or (0.0, 0.0)
        td.dr_pd_gain_lo, td.dr_pd_gain_hi = cfg.dr_pd_gain_range or (0.0, 0.0)
        td.mocap_rows = int(self.task_t["mocap_data"].shape[0])
        kp = (torch.tensor(KP, dtype=torch.float32) / 9.0).numpy()  # T:58-63 in float32 as torch does
        kv = (torch.tensor(KV, dtype=torch.float32) / 3.0).numpy()  # T:65-70
        td.kp, td.kv = _np_ptr(f32(kp), C.c_float), _np_ptr(f32(kv), C.c_float)
        td.action_high = _np_ptr(f32(ACTION_HIGH), C.c_float)
        td.initial_dof_pos = _np_ptr(f32(INIT_DOF_POS), C.c_float)
        td.left_foot_body = t.body_names.index(cfg.left_foot)
        td.right_foot_body = t.body_names.index(cfg.right_foot)
        td.pelvis_body = 0
        td.seed = seed
        tbuf = native.DyrosTaskBuffers()
        for n, _, _ in native.TASK_BUFFERS:
            setattr(tbuf, n, self.task_t[n].data_ptr())
        for n in native.TASK_SHARED:
            setattr(tbuf, n, self.task_t[n].data_ptr())
        for n, _, _ in native.TASK_OPTIONAL:
            setattr(tbuf, n, self.task_t[n].data_ptr() if n in self.task_t else None)
        native.check(self.lib.dyros_task_create(self.sim_handle, C.byref(td), C.byref(tbuf), C.byref(self.task_handle)),
                     "dyros_task_create")
        tc = cfg.terrain_curriculum
        if tc is not None and tc.curriculum:
            tb = self.task_t
            d = native.DyrosTerrainCurriculum()
            d.origins, d.levels, d.types = (tb[k].data_ptr() for k in ("terrain_origins", "terrain_levels", "terrain_types"))
            d.num_levels, d.num_types = tb["terrain_origins"].shape[:2]
            d.move_up_distance, d.move_down_scale = tc.move_up_distance, tc.move_down_scale
            d.level_mean = tb["terrain_level_mean"].data_ptr()
            native.check(self.lib.dyros_task_set_terrain_curriculum(self.task_handle, C.byref(d)),
                         "dyros_task_set_terrain_curriculum")
        if self.height_points is not None:
            d = native.DyrosHeightScan()
            d.points, d.num_points = self.task_t["height_points"].data_ptr(), self.num_height_points
            d.base_offset, d.scale = HEIGHT_SCAN_BASE_OFFSET, HEIGHT_SCAN_SCALE
            d.measured_heights = self.task_t["measured_heights"].data_ptr()
            native.check(self.lib.dyros_task_set_height_scan(self.task_handle, C.byref(d)), "dyros_task_set_height_scan")
        if self.states_width:
            d = native.DyrosCriticStates()
            d.states = self.task_t["states_buf"].data_ptr()
            d.heights_in_obs = int(bool(cfg.critic_heights_in_obs))
            d.nominal_mass = self.nominal_mass
            native.check(self.lib.dyros_task_set_critic_states(self.task_handle, C.byref(d)), "dyros_task_set_critic_states")

    def close(self):
        if getattr(self, "task_handle", None) and self.task_handle.value:
            self.lib.dyros_task_destroy(self.task_handle)
            self.task_handle = C.c_void_p()
        if getattr(self, "sim_handle", None) and self.sim_handle.value:
            self.lib.dyros_sim_destroy(self.sim_handle)
            self.sim_handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ calls
    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_noise_injection(self, **tensors):
        """Test mode (SURVEY A6): env-indexed draws replacing the Philox streams. Call with no arguments to
        return to the production streams. The tensors must stay alive until replaced."""
        inj = native.DyrosNoiseInjection()
        self._inj_keep = tensors
        for k, v in tensors.items():
            if k not in native.NOISE_FIELDS:
                raise KeyError(k)
            assert v.is_cuda and v.is_contiguous()
            setattr(inj, k, v.data_ptr())
        native.check(self.lib.dyros_task_set_noise_injection(self.task_handle, C.byref(inj) if tensors else None),
                     "dyros_task_set_noise_injection")

    def _actions_ptr(self, actions: torch.Tensor):
        # a pinned host tensor is read by the kernel directly over PCIe (unified addressing: same pointer on the device)
        on_dev = actions.device == self.device or (actions.device.type == "cpu" and actions.is_pinned())
        if not on_dev or actions.dtype != torch.float32 or not actions.is_contiguous() or tuple(actions.shape) != (self.N, NA):
            raise native.DyrosError(f"actions must be a contiguous float32 ({self.N},{NA}) tensor on {self.device} "
                                    f"or in pinned host memory")
        return C.c_void_p(actions.data_ptr())

    def step(self, actions: torch.Tensor):
        """Whole VecTask.step (VT:293-344) as dyros_task_step."""
        native.check(self.lib.dyros_task_step(self.task_handle, self._actions_ptr(actions), self._stream), "dyros_task_step")

    def pack_results(self, dst: torch.Tensor):
        """obs | rew | reset | time_outs of the last step into one contiguous device block (dyros_task_pack_results)."""
        if dst.device != self.device or not dst.is_contiguous() or dst.numel() * dst.element_size() < self.result_bytes():
            raise native.DyrosError(f"pack_results needs a contiguous block of {self.result_bytes()} bytes on {self.device}")
        native.check(self.lib.dyros_task_pack_results(self.task_handle, C.c_void_p(dst.data_ptr()), self._stream), "dyros_task_pack_results")

    def set_obs_buf(self, obs: torch.Tensor):
        """Observation buffer of the launches enqueued from now on (dyros_task_set_obs_buf); `obs` may be the head of a
        result block, pack_results on that block then only adds rew / reset / time_outs."""
        need = self.N * self.obs_width * 4
        if obs.device != self.device or not obs.is_contiguous() or obs.numel() * obs.element_size() < need:
            raise native.DyrosError(f"set_obs_buf needs a contiguous block of {need} bytes on {self.device}")
        native.check(self.lib.dyros_task_set_obs_buf(self.task_handle, C.c_void_p(obs.data_ptr())), "dyros_task_set_obs_buf")

    def result_offsets(self):
        """Byte offsets of rew, reset and time_outs in a pack_results block, and its size: obs (N, obs_width) f32 |
        rew (N) f32 | reset (N) i64 | time_outs (N) i64, the i64 part 8-byte aligned."""
        N = self.N
        rew = N * self.obs_width * 4
        rst = (rew + N * 4 + 7) & ~7
        return rew, rst, rst + N * 8, rst + N * 16

    def result_bytes(self) -> int:
        return self.result_offsets()[3]

    def step_launches(self) -> int:
        return int(self.lib.dyros_task_step_launches(self.task_handle))

    def simulate(self, apply_wrench: bool = False):
        native.check(self.lib.dyros_simulate(self.sim_handle, int(apply_wrench), self._stream), "dyros_simulate")

    def launch_info(self) -> dict:
        out = (C.c_int32 * 4)()
        native.check(self.lib.dyros_sim_launch_info(self.sim_handle, C.byref(out)), "dyros_sim_launch_info")
        return {"envs_per_cta": out[0], "ctas": out[1], "threads_per_cta": out[2], "smem_bytes": out[3]}

    def self_collision(self):
        native.check(self.lib.dyros_self_collision(self.sim_handle, self._stream), "dyros_self_collision")

    def refresh_dof_force(self, out: torch.Tensor):
        native.check(self.lib.dyros_refresh_dof_force(self.sim_handle, C.c_void_p(out.data_ptr()), self._stream), "dyros_refresh_dof_force")

    def refresh_force_sensors(self, sensor_body: torch.Tensor, sensor_pose: torch.Tensor, out: torch.Tensor):
        native.check(self.lib.dyros_refresh_force_sensors(self.sim_handle, C.c_void_p(sensor_body.data_ptr()),
                                                          C.c_void_p(sensor_pose.data_ptr()), int(sensor_body.numel()),
                                                          C.c_void_p(out.data_ptr()), self._stream), "dyros_refresh_force_sensors")

    def refresh_rigid_body_state(self):
        native.check(self.lib.dyros_refresh_rigid_body_state(self.sim_handle, self._stream), "dyros_refresh_rigid_body_state")

    def set_state_indexed(self, ids32: torch.Tensor, count: int):
        native.check(self.lib.dyros_set_state_indexed(self.sim_handle, C.c_void_p(ids32.data_ptr()), int(count),
                                                      self._stream), "dyros_set_state_indexed")

    def prologue(self, actions):
        native.check(self.lib.dyros_task_prologue(self.task_handle, self._actions_ptr(actions), self._stream), "prologue")

    def task_physics(self):
        native.check(self.lib.dyros_task_physics(self.task_handle, self._stream), "task_physics")

    def task_physics_kernel(self):
        """Measurement aid: the physics launch alone; `self_collision()` completes what `task_physics()` does."""
        native.check(self.lib.dyros_task_physics_kernel(self.task_handle, self._stream), "task_physics_kernel")

    def flush_l2(self, buf: "torch.Tensor", value: int = 0):
        """Measurement aid: overwrites `buf` (larger than the L2) with a kernel that keeps the step kernels' L1 / shared
        memory split (dyros_flush_l2)."""
        native.check(self.lib.dyros_flush_l2(C.c_void_p(buf.data_ptr()), C.c_size_t(buf.numel() * buf.element_size()),
                                            int(value) & 0xFF, self._stream), "flush_l2")

    def task_physics_trace(self) -> "torch.Tensor":
        """Profiling aid: runs the fused physics launch and returns clock64() marks of CTA 0, (skipframe, roles, 32)."""
        buf = torch.zeros(self.cfg.control_freq_inv, native.DYROS_LANES, 32, dtype=torch.int64, device=self.device)
        native.check(self.lib.dyros_task_physics_trace(self.task_handle, C.c_void_p(buf.data_ptr()), self._stream), "trace")
        return buf

    def prologue_physics(self, actions, trace: bool = False):
        """The first launch of the fused step on its own (prologue + physics); with `trace` returns the clock64() marks."""
        buf = None
        if trace:
            buf = torch.zeros(self.cfg.control_freq_inv, native.DYROS_LANES, 32, dtype=torch.int64, device=self.device)
        native.check(self.lib.dyros_task_prologue_physics(self.task_handle, self._actions_ptr(actions),
                                                          C.c_void_p(buf.data_ptr()) if trace else None, self._stream),
                     "prologue_physics")
        return buf

    def post_step(self):
        """The launches of `step` after `prologue_physics` (fused post-physics kernel + cross-env pass)."""
        native.check(self.lib.dyros_task_post_step(self.task_handle, self._stream), "dyros_task_post_step")

    def substep_torque(self):
        native.check(self.lib.dyros_task_substep_torque(self.task_handle, self._stream), "substep_torque")

    def sensor_noise(self, k: int):
        native.check(self.lib.dyros_task_sensor_noise(self.task_handle, int(k), self._stream), "sensor_noise")

    def epilogue(self):
        native.check(self.lib.dyros_task_epilogue(self.task_handle, self._stream), "epilogue")

    def check_termination(self):
        native.check(self.lib.dyros_task_check_termination(self.task_handle, self._stream), "check_termination")

    def compute_reward(self):
        native.check(self.lib.dyros_task_compute_reward(self.task_handle, self._stream), "compute_reward")

    def compact_resets(self):
        native.check(self.lib.dyros_task_compact_resets(self.task_handle, self._stream), "compact_resets")

    def reset_idx(self, env_ids: Optional[torch.Tensor] = None):
        """env_ids None = the list dyros_task_compact_resets produced (count read on the device)."""
        if env_ids is None:
            rc = self.lib.dyros_task_reset_idx(self.task_handle, None, -1, self._stream)
        else:
            assert env_ids.dtype == torch.int64 and env_ids.is_cuda and env_ids.is_contiguous()
            rc = self.lib.dyros_task_reset_idx(self.task_handle, C.c_void_p(env_ids.data_ptr()), int(env_ids.numel()),
                                               self._stream)
        native.check(rc, "reset_idx")

    def compute_observations(self):
        native.check(self.lib.dyros_task_compute_observations(self.task_handle, self._stream), "compute_observations")

    def late_update(self):
        native.check(self.lib.dyros_task_late_update(self.task_handle, self._stream), "late_update")

    def end_step(self):
        native.check(self.lib.dyros_task_end_step(self.task_handle, self._stream), "end_step")

    # ------------------------------------------------------------------ history views in reference layout
    def obs_history_linear(self) -> torch.Tensor:
        """(N, 740) oldest-first, as the reference's obs_history (T:783)."""
        h, head = self.task_t["obs_history"], self.task_t["obs_hist_head"].long()
        idx = (head[:, None] + 1 + torch.arange(20, device=self.device)[None, :]) % 20
        return torch.gather(h, 1, idx[:, :, None].expand(-1, -1, 37)).reshape(self.N, 740)

    def action_history_linear(self) -> torch.Tensor:
        h, head = self.task_t["action_history"], self.task_t["act_hist_head"].long()
        idx = (head[:, None] + 1 + torch.arange(20, device=self.device)[None, :]) % 20
        return torch.gather(h, 1, idx[:, :, None].expand(-1, -1, 13)).reshape(self.N, 260)
