"""`gymapi` facade: the subset of Isaac Gym's Python API that the DyrosDynamicWalk path calls, backed by
libdyros_b200.so instead of gym_38.so -> libcarb.gym.plugin.so -> PhysX.

Replaces python/isaacgym/gymapi.py (loader of the closed native module, gymapi.py:32-101) for one asset class
(a floating-base tree of hinge joints loaded from MJCF, one actor per env). Method names, argument order and
return conventions follow docs/api/python/gym_py.html and docs/_sources/programming/tensors.rst.txt (DOCT):
setters / refresh return bool, create_sim returns None on failure (vec_task.py:270-273), tensors are described by
`Tensor` descriptors that gymtorch.wrap_tensor turns into torch tensors (gymtorch.py:61-106).

Semantics chosen where the GPU and CPU pipelines of the reference differ: immediate ("CPU pipeline") visibility of
set_*_tensor_indexed (SURVEY A7/D3). Buffers are allocated once at prepare_sim and every acquire_* returns a view of
the same storage, so refresh_* are no-ops that return True (except rigid_body_state, which runs its FK kernel).
"""
from __future__ import annotations

import os
from dataclasses import replace
from typing import List, Optional

import numpy as np
import torch

from . import native
from .core import ARMATURE, ASSETS, CoreConfig, DyrosCore, HeightField, stable_penalty
from .model.mjcf import load_mjcf
from .model.tables import ModelTables, build_tables

SIM_PHYSX, SIM_FLEX = 0, 1
UP_AXIS_Y, UP_AXIS_Z = 0, 1
ENV_SPACE, LOCAL_SPACE, GLOBAL_SPACE = 0, 1, 2
DOF_MODE_NONE, DOF_MODE_POS, DOF_MODE_VEL, DOF_MODE_EFFORT = 0, 1, 2, 3
MESH_NONE, MESH_COLLISION, MESH_VISUAL, MESH_VISUAL_AND_COLLISION = 0, 1, 2, 3
DTYPE_FLOAT32, DTYPE_UINT32, DTYPE_UINT64, DTYPE_UINT8, DTYPE_INT16 = 0, 1, 2, 3, 4
CC_NEVER, CC_LAST_SUBSTEP, CC_ALL_SUBSTEPS = 0, 1, 2
INVALID_HANDLE = -1
KEY_ESCAPE, KEY_V = 256, 86


def ContactCollection(value: int) -> int:
    """gymapi.ContactCollection(int) as vec_task.py:461 calls it (an enum in the reference; the value is what matters)."""
    if int(value) not in (CC_NEVER, CC_LAST_SUBSTEP, CC_ALL_SUBSTEPS):
        raise ValueError(f"ContactCollection({value})")
    return int(value)


class CameraProperties:
    pass


# The native core behind prepare_sim and the test "is a CUDA device there". Tests that exercise only the Python surface
# of this facade (tests/test_reference_on_facade.py runs the UNMODIFIED reference task on it) substitute both.
_core_factory = None
_device_available = torch.cuda.is_available


class Vec3:
    def __init__(self, x=0.0, y=0.0, z=0.0):
        self.x, self.y, self.z = float(x), float(y), float(z)

    def __repr__(self):
        return f"Vec3({self.x}, {self.y}, {self.z})"


class Quat:
    def __init__(self, x=0.0, y=0.0, z=0.0, w=1.0):
        self.x, self.y, self.z, self.w = float(x), float(y), float(z), float(w)


class Transform:
    def __init__(self, p: Optional[Vec3] = None, r: Optional[Quat] = None):
        self.p, self.r = p or Vec3(), r or Quat()


class PlaneParams:
    def __init__(self):
        self.normal = Vec3(0.0, 1.0, 0.0)
        self.distance = 0.0
        self.static_friction = 1.0
        self.dynamic_friction = 1.0
        self.restitution = 0.0
        self.segmentation_id = 0


class HeightFieldParams:
    """gymapi.HeightFieldParams: the samples are (nbRows, nbColumns), row index along x, column index along y; vertex
    (i, j) at transform.p + (i row_scale, j column_scale, vertical_scale h[i, j]). transform.r must be the identity."""
    def __init__(self):
        self.nbRows = 0
        self.nbColumns = 0
        self.column_scale = 1.0
        self.row_scale = 1.0
        self.vertical_scale = 1.0
        self.transform = Transform()
        self.static_friction = 1.0
        self.dynamic_friction = 1.0
        self.restitution = 0.0
        self.segmentation_id = 0


class TriangleMeshParams:
    def __init__(self):
        self.nb_vertices = 0
        self.nb_triangles = 0
        self.transform = Transform()
        self.static_friction = 1.0
        self.dynamic_friction = 1.0
        self.restitution = 0.0


class AssetOptions:
    def __init__(self):
        self.angular_damping = 0.5
        self.linear_damping = 0.0
        self.max_angular_velocity = 64.0
        self.max_linear_velocity = 1000.0
        self.default_dof_drive_mode = DOF_MODE_NONE
        self.fix_base_link = False
        self.collapse_fixed_joints = False
        self.armature = 0.0
        self.density = 1000.0
        self.disable_gravity = False
        self.flip_visual_attachments = False
        self.thickness = 0.02
        self.use_mesh_materials = False


class PhysXParams:
    def __init__(self):
        self.solver_type = 1
        self.num_position_iterations = 4
        self.num_velocity_iterations = 1
        self.num_threads = 0
        self.use_gpu = True
        self.num_subscenes = 0
        self.contact_offset = 0.02
        self.rest_offset = 0.001
        self.bounce_threshold_velocity = 0.2
        self.max_depenetration_velocity = 100.0
        self.default_buffer_size_multiplier = 2.0
        self.max_gpu_contact_pairs = 1024 * 1024
        self.contact_collection = CC_ALL_SUBSTEPS
        self.always_use_articulations = False
        self.friction_offset_threshold = 0.04
        self.friction_correlation_distance = 0.025


class FlexParams:
    pass


class SimParams:
    def __init__(self):
        self.dt = 1.0 / 60.0
        self.substeps = 2
        self.up_axis = UP_AXIS_Y
        self.gravity = Vec3(0.0, -9.8, 0.0)
        self.use_gpu_pipeline = False
        self.num_client_threads = 0
        self.physx = PhysXParams()
        self.flex = FlexParams()


class RigidBodyProperties:
    def __init__(self, mass=0.0, com=None, inertia=None):
        self.mass = float(mass)
        self.com = com or Vec3()
        self.inertia = inertia
        self.invMass = 1.0 / mass if mass > 0 else 0.0
        self.flags = 0


class RigidShapeProperties:
    def __init__(self, friction=1.0, rolling_friction=0.0, torsion_friction=0.0, restitution=0.0, compliance=0.0,
                 thickness=0.0, contact_offset=0.02, rest_offset=0.0, filter=0):
        self.friction, self.rolling_friction, self.torsion_friction = friction, rolling_friction, torsion_friction
        self.restitution, self.compliance, self.thickness = restitution, compliance, thickness
        self.contact_offset, self.rest_offset, self.filter = contact_offset, rest_offset, filter


class Tensor:
    """Tensor descriptor (docs/api/python/struct_py.html `Tensor`; GymTensor.h:33-41). `torch_tensor` keeps the
    storage alive; gymtorch.wrap_tensor returns it."""

    def __init__(self, t: torch.Tensor, own_data: bool = False):
        self.torch_tensor = t
        self.data_address = t.data_ptr()
        self.device = t.device.index if t.is_cuda else -1
        self.dtype = {torch.float32: DTYPE_FLOAT32, torch.int32: DTYPE_UINT32, torch.int64: DTYPE_UINT64,
                      torch.uint8: DTYPE_UINT8, torch.int16: DTYPE_INT16}.get(t.dtype, DTYPE_FLOAT32)
        self.shape = tuple(t.shape)
        self.own_data = own_data

    @property
    def data_ptr(self):
        return self.data_address

    @property
    def ndim(self):
        return len(self.shape)


DOF_PROPS_DTYPE = np.dtype([("hasLimits", "?"), ("lower", "f4"), ("upper", "f4"), ("driveMode", "i4"), ("velocity", "f4"),
                            ("effort", "f4"), ("stiffness", "f4"), ("damping", "f4"), ("friction", "f4"), ("armature", "f4")])


class ActuatorProperties:
    """get_asset_actuator_properties (tasks/humanoid.py:159-160): the MJCF motors; `motor_effort` = gear / ctrlrange bound."""

    def __init__(self, motor_effort: float, name: str = ""):
        self.motor_effort, self.name = float(motor_effort), name
        self.lower_control_limit, self.upper_control_limit = -1.0, 1.0


class ForceSensorProperties:
    def __init__(self):
        self.enable_forward_dynamics_forces = True
        self.enable_constraint_solver_forces = True
        self.use_world_frame = False


class Asset:
    def __init__(self, tables: ModelTables, options: AssetOptions, name: str):
        self.tables, self.options, self.name = tables, options, name
        self.force_sensors: List[tuple] = []  # (body index, Transform), create_asset_force_sensor


class Env:
    def __init__(self, sim: "Sim", index: int):
        self.sim, self.index = sim, index
        self.actor_names: List[str] = []

    def __index__(self):
        return self.index

    def __int__(self):
        return self.index


class Sim:
    def __init__(self, compute_device: int, params: SimParams):
        self.compute_device, self.params = compute_device, params
        self.plane: Optional[PlaneParams] = None
        self.heightfield: Optional[HeightField] = None  # add_heightfield (a sim has one ground: plane or heightfield)
        self.asset: Optional[Asset] = None
        self.envs: List[Env] = []
        self.start_poses: List[Transform] = []
        self.dof_props: List[np.ndarray] = []
        self.mass_scale: List[np.ndarray] = []
        self.shape_friction: List[float] = []
        self.core: Optional[DyrosCore] = None
        self.frame_count = 0
        self.pending_wrench = False
        self._descs = {}
        # collision filter of create_actor (docs/_sources/programming/assets.rst.txt:107-109: two shapes collide unless
        # their filter masks share a bit; 0 = the actor's shapes collide with each other, as T:354 asks; a non-zero mask
        # on every shape, e.g. 1, switches self-collision off). -1 (filters from the asset file) is read as 0: the MJCF
        # files of this path carry none.
        self.self_collision = True


def _cfg_from_sim(sim: Sim) -> CoreConfig:
    p = sim.params
    cfg = CoreConfig(dt=p.dt, substeps=p.substeps, gravity=(p.gravity.x, p.gravity.y, p.gravity.z),
                     contact_offset=p.physx.contact_offset, max_depenetration_velocity=p.physx.max_depenetration_velocity,
                     num_position_iterations=p.physx.num_position_iterations,
                     num_velocity_iterations=p.physx.num_velocity_iterations,
                     with_rigid_body_state=True, with_rb_force_tensors=True, self_collision=sim.self_collision)
    cfg.penalty_stiffness, cfg.penalty_damping = stable_penalty(p.dt / p.substeps)
    if sim.plane is not None:
        cfg.friction = float(sim.plane.dynamic_friction)  # shape friction default 1.0 (SURVEY D2)
    if sim.heightfield is not None:
        cfg.friction = float(sim.heightfield.friction)    # combined with the shapes as the plane's
        # (the envs sit where create_actor put them: their origins are the actors' start positions on the field)
        pos = np.array([[tf.p.x, tf.p.y, 0.0] for tf in sim.start_poses], np.float64).reshape(-1, 3)
        pos[:, 2] = sim.heightfield.height_at(pos[:, 0], pos[:, 1])[0]
        cfg.heightfield = replace(sim.heightfield, env_origins=pos)
    if sim.asset is not None:
        cfg.max_angular_velocity = float(sim.asset.options.max_angular_velocity)
    return cfg


class Gym:
    """What `gymapi.acquire_gym()` returns (vec_task.py:181)."""

    # ------------------------------------------------------------------ setup (vec_task.py:270, T:199-385)
    def create_sim(self, compute_device: int = 0, graphics_device: int = -1, type: int = SIM_PHYSX,
                   params: Optional[SimParams] = None):
        if type != SIM_PHYSX or not _device_available():
            print("*** Failed to create sim: only SIM_PHYSX-style simulation on a CUDA device is implemented")
            return None
        params = params or SimParams()
        if params.up_axis != UP_AXIS_Z:
            print("*** Failed to create sim: only up_axis z is implemented (T:200)")
            return None
        return Sim(int(compute_device), params)

    def destroy_sim(self, sim: Sim):
        if sim.core is not None:
            sim.core.close()
            sim.core = None

    def add_ground(self, sim: Sim, params: PlaneParams):
        if sim.heightfield is not None:
            raise native.DyrosError("add_ground: the sim already has a heightfield ground (one ground per sim)")
        n = params.normal
        if (round(n.x, 6), round(n.y, 6), round(n.z, 6)) != (0.0, 0.0, 1.0) or params.distance != 0.0:
            raise native.DyrosError("add_ground: only the z = 0 plane with normal +z is implemented (T:227-235)")
        sim.plane = params

    def add_heightfield(self, sim: Sim, heightSamples, params: HeightFieldParams):
        """The ground of the sim becomes a heightfield (legged_gym terrain, mesh_type 'heightfield'): int16 samples of
        shape (nbRows, nbColumns), or their row-major flattening. Outside the field there is no ground."""
        if sim.plane is not None or sim.heightfield is not None:
            raise native.DyrosError("add_heightfield: the sim already has a ground (one ground per sim: a plane or a "
                                    "heightfield)")
        if sim.core is not None:
            raise native.DyrosError("add_heightfield: call it before prepare_sim")
        r = params.transform.r
        if (round(r.x, 6), round(r.y, 6), round(r.z, 6), round(abs(r.w), 6)) != (0.0, 0.0, 0.0, 1.0):
            raise native.DyrosError("add_heightfield: only an identity transform.r is implemented (the field is axis-aligned)")
        a = np.asarray(heightSamples)
        if a.dtype != np.int16:
            raise native.DyrosError(f"add_heightfield: samples must be int16 (got {a.dtype})")
        if a.size != int(params.nbRows) * int(params.nbColumns):
            raise native.DyrosError(f"add_heightfield: {a.size} samples for nbRows x nbColumns = {params.nbRows} x {params.nbColumns}")
        p = params.transform.p
        hf = HeightField(np.ascontiguousarray(a.reshape(int(params.nbRows), int(params.nbColumns))), float(params.row_scale),
                         float(params.column_scale), float(params.vertical_scale), (p.x, p.y, p.z),
                         friction=float(params.dynamic_friction))
        hf.validate()
        sim.heightfield = hf

    def add_triangle_mesh(self, sim: Sim, vertices, triangles, params: "TriangleMeshParams"):
        raise native.DyrosError("add_triangle_mesh: triangle-mesh ground is not implemented (it needs a general mesh "
                                "narrow phase); use add_heightfield (mesh_type 'heightfield') or add_ground")

    def load_asset(self, sim: Sim, rootpath: str, filename: str, options: Optional[AssetOptions] = None):
        options = options or AssetOptions()
        path = os.path.join(rootpath, filename)
        bundled = {"dyros_tocabi.xml": "tocabi_tables.npz", "nv_humanoid.xml": "humanoid_tables.npz"}
        if os.path.isfile(path):
            model = load_mjcf(path, infer_missing_inertia=os.path.basename(filename) != "dyros_tocabi.xml",
                              geom_density=options.density)
            tables = build_tables(model, solver_bodies=[b.name for b in model.bodies if _is_foot(b.name)], vel_limit=1.0e3)
        elif os.path.basename(filename) in bundled:
            tables = ModelTables.load(os.path.join(ASSETS, bundled[os.path.basename(filename)]))  # bundled import of the same MJCF
        else:
            print(f"*** Failed to load asset {path}")
            return None
        if sim.asset is not None and sim.asset.tables.body_names != tables.body_names:
            raise native.DyrosError("load_asset: one asset class per sim (one articulation per env) is implemented")
        sim.asset = Asset(tables, options, os.path.basename(filename))
        return sim.asset

    def get_asset_rigid_body_count(self, asset: Asset) -> int:
        return asset.tables.num_bodies

    def get_asset_dof_count(self, asset: Asset) -> int:
        return asset.tables.num_dofs

    def get_asset_joint_count(self, asset: Asset) -> int:
        return asset.tables.num_bodies - 1  # every non-root body has one joint (hinge or fixed)

    def get_asset_rigid_body_names(self, asset: Asset):
        return list(asset.tables.body_names)

    def get_asset_dof_names(self, asset: Asset):
        return list(asset.tables.dof_names)

    def find_asset_rigid_body_index(self, asset: Asset, name: str) -> int:
        return asset.tables.body_names.index(name) if name in asset.tables.body_names else INVALID_HANDLE

    def find_asset_dof_index(self, asset: Asset, name: str) -> int:
        return asset.tables.dof_names.index(name) if name in asset.tables.dof_names else INVALID_HANDLE

    def get_asset_actuator_properties(self, asset: Asset):
        t = asset.tables
        return [ActuatorProperties(float(t.dof_effort[d]), t.dof_names[d]) for d in range(t.num_dofs)]

    def get_asset_actuator_count(self, asset: Asset) -> int:
        return asset.tables.num_dofs

    def create_asset_force_sensor(self, asset: Asset, body_idx: int, local_pose: Optional[Transform] = None, props=None) -> int:
        """tasks/humanoid.py:163-168. Returns the sensor index."""
        if not (0 <= int(body_idx) < asset.tables.num_bodies):
            return INVALID_HANDLE
        asset.force_sensors.append((int(body_idx), local_pose or Transform()))
        return len(asset.force_sensors) - 1

    def get_asset_force_sensor_count(self, asset: Asset) -> int:
        return len(asset.force_sensors)

    def enable_actor_dof_force_sensors(self, env: Env, handle: int) -> bool:
        return True  # the DOF force tensor is always available (tasks/humanoid.py:196)

    def create_env(self, sim: Sim, lower: Vec3, upper: Vec3, num_per_row: int) -> Env:
        if sim.core is not None:
            raise native.DyrosError("create_env after prepare_sim is not supported")
        e = Env(sim, len(sim.envs))
        sim.envs.append(e)
        return e

    def create_actor(self, env: Env, asset: Asset, pose: Transform, name: str = "", group: int = -1, filter: int = -1,
                     segmentationId: int = 0) -> int:
        sim = env.sim
        if env.actor_names:
            raise native.DyrosError("create_actor: one actor per env is implemented (T:354)")
        env.actor_names.append(name)
        if filter > 0:
            sim.self_collision = False
        t = asset.tables
        sim.start_poses.append(pose)
        props = np.zeros(t.num_dofs, dtype=DOF_PROPS_DTYPE)
        props["hasLimits"] = True
        props["lower"], props["upper"] = t.dof_lower, t.dof_upper
        props["driveMode"] = asset.options.default_dof_drive_mode
        props["velocity"] = 1.0e3
        props["effort"] = t.dof_effort
        props["damping"] = t.dof_damping
        props["armature"] = np.maximum(t.dof_armature, asset.options.armature)
        sim.dof_props.append(props)
        sim.mass_scale.append(np.ones(t.num_bodies, dtype=np.float32))
        return 0

    def set_rigid_body_color(self, *a, **k):
        return None  # headless: no visuals

    def get_actor_dof_properties(self, env: Env, handle: int) -> np.ndarray:
        return env.sim.dof_props[env.index].copy()

    def set_actor_dof_properties(self, env: Env, handle: int, props) -> bool:
        sim = env.sim
        cur = sim.dof_props[env.index]
        for f in DOF_PROPS_DTYPE.names:
            try:
                cur[f] = np.asarray(props[f])
            except (KeyError, ValueError, IndexError):
                pass
        if sim.core is not None:  # live update of this env's rows (the DR path of VT:655-721)
            dev = sim.core.device
            sim.core.sim_t["dof_damping"][env.index] = torch.tensor(np.ascontiguousarray(cur["damping"]), device=dev)
            sim.core.sim_t["dof_armature"][env.index] = torch.tensor(np.ascontiguousarray(cur["armature"]), device=dev)
        return True

    def get_actor_rigid_body_properties(self, env: Env, handle: int):
        t = env.sim.asset.tables
        sc = env.sim.mass_scale[env.index]
        return [RigidBodyProperties(mass=float(t.body_inertia[b, 0] * sc[b])) for b in range(t.num_bodies)]

    def set_actor_rigid_body_properties(self, env: Env, handle: int, props, recomputeInertia: bool = True) -> bool:
        """Mass scaling with the inertia tensor scaled proportionally (recomputeInertia=True, gymutil.py:513)."""
        sim = env.sim
        t = sim.asset.tables
        base = t.body_inertia[:, 0]
        # (gymutil.apply_random_samples leaves a 1-element array in `mass`: gymutil.py:607-619)
        mass = [float(np.ravel(props[b].mass)[0]) for b in range(t.num_bodies)]
        sc = np.array([mass[b] / base[b] if base[b] > 0 else 1.0 for b in range(t.num_bodies)], dtype=np.float32)
        sim.mass_scale[env.index] = sc
        if sim.core is not None:
            sim.core.sim_t["body_mass_scale"][env.index] = torch.tensor(sc, device=sim.core.device)
        return True

    def get_actor_tendon_properties(self, env: Env, handle: int):
        return []  # no tendons in the supported asset class (gymutil.py:487-503 builds its maps with these names)

    def set_actor_tendon_properties(self, env: Env, handle: int, props) -> bool:
        return True

    def get_actor_rigid_shape_properties(self, env: Env, handle: int):
        """One entry per collision shape; `friction` is the coefficient the ground contacts of this env use."""
        sim = env.sim
        mu = float(sim.shape_friction[env.index]) if env.index < len(sim.shape_friction) else 1.0
        return [RigidShapeProperties(friction=mu) for _ in range(self.get_actor_rigid_shape_count(env, handle))]

    def set_actor_rigid_shape_properties(self, env: Env, handle: int, props) -> bool:
        """The ground contact uses ONE coefficient per env (DyrosSimBuffers.contact_friction): the mean over the shapes."""
        sim = env.sim
        mu = float(np.mean([p.friction for p in props])) if len(props) else 1.0
        while len(sim.shape_friction) <= env.index:
            sim.shape_friction.append(1.0)
        sim.shape_friction[env.index] = mu
        if sim.core is not None and "contact_friction" in sim.core.sim_t:
            ground = sim.heightfield.friction if sim.heightfield is not None else (
                sim.plane.dynamic_friction if sim.plane is not None else 1.0)
            plane = float(ground)
            sim.core.sim_t["contact_friction"][env.index] = plane * mu
        return True

    def get_actor_count(self, env: Env) -> int:
        return len(env.actor_names)

    def get_actor_handle(self, env: Env, index: int) -> int:
        return index

    def get_actor_name(self, env: Env, handle: int) -> str:
        return env.actor_names[handle]

    def find_actor_handle(self, env: Env, name: str) -> int:
        return env.actor_names.index(name) if name in env.actor_names else INVALID_HANDLE

    def get_actor_rigid_body_count(self, env: Env, handle: int) -> int:
        return env.sim.asset.tables.num_bodies

    def get_actor_dof_count(self, env: Env, handle: int) -> int:
        return env.sim.asset.tables.num_dofs

    def get_actor_rigid_shape_count(self, env: Env, handle: int) -> int:
        t = env.sim.asset.tables
        return len(t.pt_link) // 8 + len(t.cyl_link)

    def find_actor_rigid_body_handle(self, env: Env, handle: int, name: str) -> int:
        return self.find_asset_rigid_body_index(env.sim.asset, name)

    def get_env_count(self, sim: Sim) -> int:
        return len(sim.envs)

    def get_env(self, sim: Sim, i: int) -> Env:
        return sim.envs[i]

    def get_sim_actor_count(self, sim: Sim) -> int:
        return len(sim.envs)

    def get_sim_dof_count(self, sim: Sim) -> int:
        return len(sim.envs) * sim.asset.tables.num_dofs

    def get_sim_rigid_body_count(self, sim: Sim) -> int:
        return len(sim.envs) * sim.asset.tables.num_bodies

    def get_frame_count(self, sim: Sim) -> int:
        return sim.frame_count

    def get_sim_params(self, sim: Sim) -> SimParams:
        return sim.params

    def set_sim_params(self, sim: Sim, params: SimParams):
        if sim.core is not None:
            g0, g1 = sim.params.gravity, params.gravity
            if (g0.x, g0.y, g0.z) != (g1.x, g1.y, g1.z) or params.dt != sim.params.dt:
                raise native.DyrosError("set_sim_params: dt / gravity are fixed once the sim is prepared")
        sim.params = params

    def prepare_sim(self, sim: Sim) -> bool:
        """vec_task.py:196: allocate the tensor-API buffers and build the native sim."""
        if sim.core is not None:
            return True
        if sim.asset is None or not sim.envs or (sim.plane is None and sim.heightfield is None):
            print("*** prepare_sim: need a ground (plane or heightfield), an asset and at least one env")
            return False
        N = len(sim.envs)
        if any(len(e.actor_names) != 1 for e in sim.envs):
            print("*** prepare_sim: every env needs exactly one actor")
            return False
        cfg = _cfg_from_sim(sim)
        vel = np.stack([p["velocity"] for p in sim.dof_props])
        cfg.dof_vel_limit = float(min(vel.min(), 1.0e9))
        t = sim.asset.tables
        cfg.solver_bodies = tuple(n for n in t.body_names if _is_foot(n))
        try:  # the DyrosDynamicWalk task buffers exist only for the TOCABI tree; any other articulation is simulator-only
            core = (_core_factory or DyrosCore)(N, f"cuda:{sim.compute_device}", cfg, tables=t, with_task=_is_tocabi(t))
        except native.DyrosError as e:
            print(f"*** prepare_sim: {e}")
            return False
        dev = core.device
        core.sim_t["dof_damping"].copy_(torch.tensor(np.stack([p["damping"] for p in sim.dof_props]), device=dev))
        core.sim_t["dof_armature"].copy_(torch.tensor(np.stack([p["armature"] for p in sim.dof_props]), device=dev))
        core.sim_t["body_mass_scale"].copy_(torch.tensor(np.stack(sim.mass_scale), device=dev))
        root = np.zeros((N, 13), np.float32)
        for i, tf in enumerate(sim.start_poses):
            root[i, 0:3] = (tf.p.x, tf.p.y, tf.p.z)
            root[i, 3:7] = (tf.r.x, tf.r.y, tf.r.z, tf.r.w)
        core.sim_t["root_states"].copy_(torch.tensor(root, device=dev))
        core.sim_t["dof_state"].zero_()
        sim.core = core
        return True

    # ------------------------------------------------------------------ tensor API (DOCT)
    def _desc(self, sim: Sim, name: str) -> Tensor:
        if sim.core is None:
            raise native.DyrosError(f"acquire_{name}: call prepare_sim first (DOCT:30-44)")
        if name not in sim._descs:
            sim._descs[name] = Tensor(sim.core.sim_t[name])
        return sim._descs[name]

    def acquire_actor_root_state_tensor(self, sim: Sim) -> Tensor:
        return self._desc(sim, "root_states")

    def acquire_dof_state_tensor(self, sim: Sim) -> Tensor:
        return self._desc(sim, "dof_state")

    def acquire_rigid_body_state_tensor(self, sim: Sim) -> Tensor:
        return self._desc(sim, "rigid_body_state")

    def acquire_net_contact_force_tensor(self, sim: Sim) -> Tensor:
        return self._desc(sim, "net_contact_force")

    def acquire_dof_force_tensor(self, sim: Sim) -> Tensor:
        """(num_dofs,) generalised force at every DOF (tasks/humanoid.py:85); filled by refresh_dof_force_tensor."""
        if sim.core is None:
            raise native.DyrosError("acquire_dof_force_tensor: call prepare_sim first (DOCT:30-44)")
        if "dof_force" not in sim.core.sim_t:
            sim.core.sim_t["dof_force"] = torch.zeros(len(sim.envs) * sim.asset.tables.num_dofs, device=sim.core.device)
        return self._desc(sim, "dof_force")

    def refresh_dof_force_tensor(self, sim: Sim) -> bool:
        if sim.core is None or "dof_force" not in sim.core.sim_t:
            return False
        sim.core.refresh_dof_force(sim.core.sim_t["dof_force"])
        return True

    def acquire_force_sensor_tensor(self, sim: Sim) -> Tensor:
        """(num_envs * sensors_per_env, 6) [force, torque] in the sensor frames (tasks/humanoid.py:80-83)."""
        if sim.core is None:
            raise native.DyrosError("acquire_force_sensor_tensor: call prepare_sim first (DOCT:30-44)")
        ns = len(sim.asset.force_sensors)
        if ns == 0:
            return Tensor(torch.zeros(0, 6, device=sim.core.device))  # wrap_tensor prints "Can't create empty tensor" (GTC:40-45)
        if "force_sensor" not in sim.core.sim_t:
            dev = sim.core.device
            sim.core.sim_t["force_sensor"] = torch.zeros(len(sim.envs) * ns, 6, device=dev)
            sim.core.sim_t["sensor_body"] = torch.tensor([b for b, _ in sim.asset.force_sensors], dtype=torch.int32, device=dev)
            sim.core.sim_t["sensor_pose"] = torch.tensor([[tf.p.x, tf.p.y, tf.p.z, tf.r.x, tf.r.y, tf.r.z, tf.r.w]
                                                          for _, tf in sim.asset.force_sensors], dtype=torch.float32, device=dev)
        return self._desc(sim, "force_sensor")

    def refresh_force_sensor_tensor(self, sim: Sim) -> bool:
        if sim.core is None or "force_sensor" not in sim.core.sim_t:
            return False
        t = sim.core.sim_t
        sim.core.refresh_force_sensors(t["sensor_body"], t["sensor_pose"], t["force_sensor"])
        return True

    def refresh_actor_root_state_tensor(self, sim: Sim) -> bool:
        return sim.core is not None

    def refresh_dof_state_tensor(self, sim: Sim) -> bool:
        return sim.core is not None

    def refresh_net_contact_force_tensor(self, sim: Sim) -> bool:
        return sim.core is not None

    def refresh_rigid_body_state_tensor(self, sim: Sim) -> bool:
        if sim.core is None:
            return False
        sim.core.refresh_rigid_body_state()
        return True

    @staticmethod
    def _src(desc) -> torch.Tensor:
        return desc.torch_tensor if isinstance(desc, Tensor) else desc

    def _copy_in(self, sim: Sim, name: str, desc, shape) -> bool:
        if sim.core is None:
            return False
        src, dst = self._src(desc), sim.core.sim_t[name]
        if src.numel() != dst.numel() or src.dtype != dst.dtype:
            return False
        if src.data_ptr() != dst.data_ptr():
            dst.copy_(src.reshape(dst.shape))
        return True

    def set_dof_actuation_force_tensor(self, sim: Sim, desc) -> bool:
        """(num_dofs,) N*m in dof-state order (DOCT:300-311)."""
        return self._copy_in(sim, "dof_actuation_force", desc, None)

    def set_dof_state_tensor(self, sim: Sim, desc) -> bool:
        return self._copy_in(sim, "dof_state", desc, None)

    def set_actor_root_state_tensor(self, sim: Sim, desc) -> bool:
        return self._copy_in(sim, "root_states", desc, None)

    def _set_indexed(self, sim: Sim, name: str, desc, ids_desc, count: int, rows_per_actor: int) -> bool:
        """Full tensor + int32 actor ids (DOCT:141-147, 176-180)."""
        if sim.core is None:
            return False
        ids = self._src(ids_desc)
        if ids.dtype != torch.int32 or count < 0 or count > ids.numel():
            return False
        src, dst = self._src(desc), sim.core.sim_t[name]
        if src.numel() != dst.numel():
            return False
        sim.core.set_state_indexed(ids, count)
        if src.data_ptr() != dst.data_ptr() and count > 0:
            idx = ids[:count].long()
            N = sim.core.N
            dst.view(N, rows_per_actor, -1)[idx] = src.reshape(N, rows_per_actor, -1)[idx]
        return True

    def set_dof_state_tensor_indexed(self, sim: Sim, desc, ids_desc, count: int) -> bool:
        return self._set_indexed(sim, "dof_state", desc, ids_desc, count, sim.asset.tables.num_dofs)

    def set_actor_root_state_tensor_indexed(self, sim: Sim, desc, ids_desc, count: int) -> bool:
        return self._set_indexed(sim, "root_states", desc, ids_desc, count, 1)

    def apply_rigid_body_force_tensors(self, sim: Sim, force=None, torque=None, space: int = ENV_SPACE) -> bool:
        """(num_bodies,3) each, at the bodies' centres of mass, for the next time step only (DOCT:322-335).
        Envs have zero extents (T:341-349), so ENV_SPACE and GLOBAL_SPACE coincide; LOCAL_SPACE is not implemented."""
        if sim.core is None or space == LOCAL_SPACE:
            return False
        for name, d in (("rb_force", force), ("rb_torque", torque)):
            dst = sim.core.sim_t[name]
            if d is None:
                dst.zero_()
            else:
                src = self._src(d)
                if src.numel() != dst.numel():
                    return False
                dst.copy_(src.reshape(dst.shape))
        sim.pending_wrench = True
        return True

    def simulate(self, sim: Sim) -> None:
        """One time step dt in `substeps` sub-steps (gym_py.html simulate; T:525)."""
        if sim.core is None:
            raise native.DyrosError("simulate: call prepare_sim first")
        sim.core.simulate(apply_wrench=sim.pending_wrench)
        sim.pending_wrench = False
        sim.frame_count += 1

    def fetch_results(self, sim: Sim, wait: bool) -> None:
        if wait and sim.core is not None and sim.core.device.type == "cuda":
            torch.cuda.current_stream(sim.core.device).synchronize()

    # ------------------------------------------------------------------ viewer (headless only, vec_task.py:212-231)
    def create_viewer(self, *a, **k):
        return None

    def viewer_camera_look_at(self, *a, **k):
        return None

    def subscribe_viewer_keyboard_event(self, *a, **k):
        return None

    def step_graphics(self, *a, **k):
        return None

    def poll_viewer_events(self, *a, **k):
        return None

    def query_viewer_has_closed(self, *a, **k):
        return False


def _is_foot(body_name: str) -> bool:
    """Bodies whose ground contact is constraint-solved: `*_Foot_Link` (TOCABI), `right_foot` / `left_foot` (Humanoid)."""
    import re
    return re.search(r"(^|_)foot(_link)?$", body_name, re.IGNORECASE) is not None


def _is_tocabi(t: ModelTables) -> bool:
    return t.num_dofs == 33 and t.num_bodies == 38


_GYM: Optional[Gym] = None


def acquire_gym() -> Gym:
    global _GYM
    if _GYM is None:
        _GYM = Gym()
    return _GYM
