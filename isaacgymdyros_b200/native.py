"""ctypes binding of libdyros_b200.so (C ABI: include/dyros_b200.h).

The structures below mirror the header member for member. There is no CPU fallback: if the shared
library is missing, `load()` raises and every caller fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
ABI_VERSION = 3  # include/dyros_b200.h DYROS_ABI_VERSION: struct layouts below mirror that header
LIB_PATH = os.environ.get("DYROS_B200_LIB", os.path.join(_HERE, "libdyros_b200.so"))  # override: A/B builds only
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "dyros_b200.h")

i32, f32, f64, u64 = C.c_int32, C.c_float, C.c_double, C.c_uint64
P_i32, P_i64, P_f32, P_f64 = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_float), C.POINTER(C.c_double)
DYROS_LANES = 4


class DyrosModelDesc(C.Structure):
    _fields_ = [(n, i32) for n in ("num_links", "num_bodies", "num_dofs", "num_points", "num_cyls", "sched_slots")] + [
        ("link_parent", P_i32), ("link_dof", P_i32), ("link_E", P_f64), ("link_r", P_f64), ("link_axis", P_f64),
        ("body_link", P_i32), ("body_pos", P_f64), ("body_rot", P_f64), ("body_inertia", P_f64),
        ("dof_lower", P_f64), ("dof_upper", P_f64), ("dof_vel_limit", P_f64), ("dof_effort", P_f64), ("dof_stiffness", P_f64),
        ("pt_link", P_i32), ("pt_body", P_i32), ("pt_pos", P_f64), ("pt_radius", P_f64), ("pt_solver", P_i32),
        ("cyl_link", P_i32), ("cyl_body", P_i32), ("cyl_center", P_f64), ("cyl_axis", P_f64), ("cyl_size", P_f64),
        ("sched", P_i32),
        ("sc_num_shapes", i32), ("sc_num_samples", i32), ("sc_num_pairs", i32),
        ("sc_shape_kind", P_i32), ("sc_shape_link", P_i32), ("sc_shape_body", P_i32), ("sc_shape_sample0", P_i32),
        ("sc_shape_center", P_f64), ("sc_shape_rot", P_f64), ("sc_shape_size", P_f64), ("sc_sample", P_f64),
        ("sc_link_shape0", P_i32), ("sc_link_sphere", P_f64), ("sc_pairs", P_i32)]


class DyrosSimDesc(C.Structure):
    _fields_ = [("num_envs", i32), ("device", i32), ("dt", f64), ("substeps", i32), ("gravity", f32 * 3),
                ("contact_offset", f32), ("max_depenetration_velocity", f32), ("contact_sweeps", i32),
                ("contact_erp", f32), ("friction", f32), ("penalty_stiffness", f32), ("penalty_damping", f32),
                ("penalty_max_force", f32), ("max_angular_velocity", f32), ("clamp_effort", i32), ("physics_program", i32)]


SIM_BUFFERS = ["root_states", "dof_state", "net_contact_force", "rigid_body_state", "dof_actuation_force", "rb_force",
               "rb_torque", "dof_damping", "dof_armature", "body_mass_scale", "contact_friction", "link_pose", "self_contact_force"]


class DyrosHeightField(C.Structure):
    _fields_ = [("samples", C.c_void_p), ("num_rows", i32), ("num_columns", i32), ("row_scale", f32),
                ("column_scale", f32), ("vertical_scale", f32), ("origin", f32 * 3)]


class DyrosSimBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in SIM_BUFFERS]


# (name, torch dtype name, trailing shape); N is prepended unless the shape starts with None. (obs_buf is (N, 487 + P)
# with a height scan of P points: DyrosCore._alloc)
TASK_BUFFERS = [
    ("obs_buf", "float32", (487,)), ("rew_buf", "float32", ()), ("reset_buf", "int64", ()),
    ("timeout_buf", "int64", ()), ("progress_buf", "int64", ()), ("randomize_buf", "int64", ()),
    ("stacked_rewards", "float32", (15,)), ("reset_env_ids", "int64", ()), ("reset_env_ids32", "int32", ()),
    ("reset_count", "int32", (None, 1)),
    ("actions", "float32", (13,)), ("actions_pre", "float32", (13,)), ("time", "float32", ()),
    ("init_mocap_data_idx", "int32", ()), ("mocap_data_idx", "int32", ()), ("target_data_qpos", "float32", (33,)),
    ("target_data_force", "float32", (2,)), ("action_torque", "float32", (12,)),
    ("action_torque_pre", "float32", (12,)), ("motor_constant_scale", "float32", (12,)),
    ("action_log", "float32", (6, 12)), ("delay_idx", "int32", ()), ("simul_len", "int32", ()),
    ("qpos_noise", "float32", (33,)), ("qvel_noise", "float32", (33,)), ("qpos_pre", "float32", (33,)),
    ("qpos_bias", "float32", (12,)), ("quat_bias", "float32", (3,)), ("target_vel", "float32", (2,)),
    ("pre_joint_velocity_states", "float32", (33,)), ("contact_forces_pre", "float32", (38, 3)),
    ("total_mass", "float32", ()), ("env_origins", "float32", (3,)), ("epi_len", "float32", ()),
    ("epi_len_log", "float32", ()), ("contact_reward_sum", "float32", ()), ("contact_reward_mean", "float32", ()),
    ("perturbation_count", "int32", ()), ("pert_duration", "int32", ()), ("pert_on", "int32", ()),
    ("impulse", "int32", ()), ("magnitude", "float32", ()), ("phase", "float32", ()), ("perturb_timing", "int32", ()),
    ("perturb_start", "int32", (None, 1)), ("push_force", "float32", (3,)),
    ("obs_history", "float32", (20, 37)), ("action_history", "float32", (20, 13)),
    ("obs_hist_head", "int32", ()), ("act_hist_head", "int32", ()), ("reset_seq", "int32", ()),
]
TASK_SHARED = ["mocap_data", "obs_mean", "obs_var"]
TASK_OPTIONAL = [("pd_gain_scale", "float32", (2,))]  # allocated on request (CoreConfig.dr_pd_gain_range), else NULL


class DyrosTaskBuffers(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n, _, _ in TASK_BUFFERS] + [(n, C.c_void_p) for n in TASK_SHARED]
                + [(n, C.c_void_p) for n, _, _ in TASK_OPTIONAL])


class DyrosTaskDesc(C.Structure):
    _fields_ = [("skipframe", i32), ("max_episode_length", f32), ("death_cost", f32), ("initial_height", f32),
                ("perturb", i32), ("randomize", i32), ("dr_damping_base", f32), ("dr_damping_lo", f32),
                ("dr_damping_hi", f32), ("dr_armature_lo", f32), ("dr_armature_hi", f32), ("dr_armature_base", P_f64),
                ("dr_friction_base", f32), ("dr_friction_lo", f32), ("dr_friction_hi", f32),
                ("dr_pd_gain_lo", f32), ("dr_pd_gain_hi", f32),
                ("mocap_rows", i32), ("kp", P_f32), ("kv", P_f32), ("action_high", P_f32), ("initial_dof_pos", P_f32),
                ("left_foot_body", i32), ("right_foot_body", i32), ("pelvis_body", i32), ("seed", u64)]


class DyrosTerrainCurriculum(C.Structure):
    _fields_ = [("origins", C.c_void_p), ("levels", C.c_void_p), ("types", C.c_void_p), ("num_levels", i32),
                ("num_types", i32), ("move_up_distance", f32), ("move_down_scale", f32), ("level_mean", C.c_void_p)]


class DyrosHeightScan(C.Structure):
    _fields_ = [("points", C.c_void_p), ("num_points", i32), ("base_offset", f32), ("scale", f32),
                ("measured_heights", C.c_void_p)]


class DyrosCriticStates(C.Structure):
    _fields_ = [("states", C.c_void_p), ("heights_in_obs", i32), ("nominal_mass", f32)]


NOISE_FIELDS = ["qpos_normal", "vel_u", "reset_f", "reset_i", "pert_i", "pert_f", "dr_u"]


class DyrosNoiseInjection(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in NOISE_FIELDS]


class DyrosPpoBuffers(C.Structure):
    _fields_ = [("N", i32), ("H", i32), ("gamma", f32), ("tau", f32), ("e_clip", f32), ("critic_coef", f32),
                ("reward_scale", f32), ("value_bootstrap", i32), ("seed", u64)] + [
        (n, C.c_void_p) for n in ("obs", "actions", "mus", "neglogp", "values", "rewards", "dones", "advantages", "returns",
                                  "cur_reward", "cur_length", "ep_stats", "step", "global_step")] + [("obs_dim", i32)]


class DyrosPpoNet(C.Structure):
    _fields_ = [("hidden", i32), ("inputs", i32)] + [(n, C.c_void_p) for n in ("w0", "b0", "w1", "b1", "wh", "bh", "gw0", "gw1", "gwh", "gb0", "gb1", "gbh")]


class DyrosPpoPeers(C.Structure):
    _fields_ = [("world", i32), ("rank", i32), ("stride", i32), ("grad", (C.c_void_p * 2) * 8), ("flags", C.c_void_p * 8),
                ("epoch", C.c_void_p), ("ticket", C.c_void_p), ("sum", (C.c_void_p * 2) * 8), ("flags2", C.c_void_p * 8),
                ("pnorm", C.c_void_p * 8)]


_VP, _INT = C.c_void_p, C.c_int
_PB = C.POINTER(DyrosPpoBuffers)
_PN = C.POINTER(DyrosPpoNet)
SIGNATURES = {
    "dyros_ppo_act": (_INT, [_PB, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "dyros_ppo_reward": (_INT, [_PB, _VP, _VP, _VP, _VP]),
    "dyros_ppo_gae": (_INT, [_PB, _VP, _VP, _VP]),
    "dyros_ppo_loss_grad": (_INT, [_PB, _INT, _INT, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "dyros_ppo_adam": (_INT, [_VP, _VP, _VP, _VP, _INT, _INT, f32, f32, _VP, _VP, _VP, f32, f32, f32, f32, f32, _INT, _VP]),
    "dyros_ppo_cast_obs": (_INT, [_PB, _VP, _VP, _VP, _VP]),
    "dyros_ppo_bias_relu": (_INT, [_VP, _VP, _INT, _INT, _VP]),
    "dyros_ppo_relu_bwd": (_INT, [_VP, _VP, _VP, _INT, _INT, _VP]),
    "dyros_ppo_act_packed": (_INT, [_PB, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "dyros_ppo_loss_grad_packed": (_INT, [_PB, _INT, _INT, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "dyros_ppo_pack_params": (_INT, [_PN, _VP, _VP]),
    "dyros_ppo_unpack_grads": (_INT, [_PN, _VP, _VP, _VP]),
    "dyros_ppo_pack_params_ac": (_INT, [_PN, _INT, _VP, _VP]),
    "dyros_ppo_unpack_grads_ac": (_INT, [_PN, _INT, _VP, _VP, _VP]),
    "dyros_peer_alloc": (_INT, [C.c_size_t, C.POINTER(_VP), C.c_char_p]),
    "dyros_peer_open": (_INT, [C.c_char_p, C.POINTER(_VP)]),
    "dyros_peer_close": (_INT, [_VP]),
    "dyros_peer_free": (_INT, [_VP]),
    "dyros_ppo_unpack_grads_peers": (_INT, [_PN, C.POINTER(DyrosPpoPeers), _VP]),
    "dyros_ppo_unpack_grads_peers_ac": (_INT, [_PN, _INT, C.POINTER(DyrosPpoPeers), _VP]),
    "dyros_ppo_reduce_peers": (_INT, [C.POINTER(DyrosPpoPeers), _VP, _INT, _INT, _VP, _VP]),
    "dyros_ppo_reduce_scatter_peers": (_INT, [C.POINTER(DyrosPpoPeers), _VP, _INT, _INT, _VP]),
    "dyros_ppo_all_gather_peers": (_INT, [C.POINTER(DyrosPpoPeers), _VP, _INT, _VP, _VP]),
    "dyros_ppo_adam_packed": (_INT, [_PN, _VP, _VP, _VP, _VP, f32, f32, _INT, _VP, _VP, _VP, f32, f32, f32, f32, f32, _INT, _VP]),
    "dyros_ppo_adam_packed_ac": (_INT, [_PN, _INT, _VP, _VP, _VP, _VP, f32, f32, _INT, _VP, _VP, _VP, f32, f32, f32, f32, f32, _INT,
                                        _VP]),
    "dyros_last_error": (C.c_char_p, []),
    "dyros_abi_version": (_INT, []),
    "dyros_sim_set_l2_persistence": (_INT, [_VP, _VP, C.c_size_t, _VP, C.POINTER(C.c_size_t)]),
    "dyros_sim_create": (_INT, [C.POINTER(DyrosSimDesc), C.POINTER(DyrosModelDesc), C.POINTER(DyrosSimBuffers), C.POINTER(_VP)]),
    "dyros_sim_destroy": (_INT, [_VP]),
    "dyros_simulate": (_INT, [_VP, _INT, _VP]),
    "dyros_refresh_rigid_body_state": (_INT, [_VP, _VP]),
    "dyros_self_collision": (_INT, [_VP, _VP]),
    "dyros_set_state_indexed": (_INT, [_VP, _VP, _INT, _VP]),
    "dyros_refresh_dof_force": (_INT, [_VP, _VP, _VP]),
    "dyros_refresh_force_sensors": (_INT, [_VP, _VP, _VP, _INT, _VP, _VP]),
    "dyros_measure_fp32_peak": (_INT, [_INT, _INT, C.POINTER(C.c_double)]),
    "dyros_flush_l2": (_INT, [C.c_void_p, C.c_size_t, _INT, C.c_void_p]),
    "dyros_sim_launch_info": (_INT, [_VP, C.POINTER(C.c_int32 * 4)]),
    "dyros_sim_set_heightfield": (_INT, [_VP, C.POINTER(DyrosHeightField)]),
    "dyros_task_create": (_INT, [_VP, C.POINTER(DyrosTaskDesc), C.POINTER(DyrosTaskBuffers), C.POINTER(_VP)]),
    "dyros_task_destroy": (_INT, [_VP]),
    "dyros_task_set_noise_injection": (_INT, [_VP, C.POINTER(DyrosNoiseInjection)]),
    "dyros_task_set_terrain_curriculum": (_INT, [_VP, C.POINTER(DyrosTerrainCurriculum)]),
    "dyros_task_set_height_scan": (_INT, [_VP, C.POINTER(DyrosHeightScan)]),
    "dyros_task_set_critic_states": (_INT, [_VP, C.POINTER(DyrosCriticStates)]),
    "dyros_task_prologue": (_INT, [_VP, _VP, _VP]),
    "dyros_task_physics": (_INT, [_VP, _VP]),
    "dyros_task_physics_kernel": (_INT, [_VP, _VP]),
    "dyros_task_physics_trace": (_INT, [_VP, _VP, _VP]),
    "dyros_task_prologue_physics": (_INT, [_VP, _VP, _VP, _VP]),
    "dyros_task_substep_torque": (_INT, [_VP, _VP]),
    "dyros_task_sensor_noise": (_INT, [_VP, _INT, _VP]),
    "dyros_task_epilogue": (_INT, [_VP, _VP]),
    "dyros_task_check_termination": (_INT, [_VP, _VP]),
    "dyros_task_compute_reward": (_INT, [_VP, _VP]),
    "dyros_task_compact_resets": (_INT, [_VP, _VP]),
    "dyros_task_reset_idx": (_INT, [_VP, _VP, _INT, _VP]),
    "dyros_task_compute_observations": (_INT, [_VP, _VP]),
    "dyros_task_late_update": (_INT, [_VP, _VP]),
    "dyros_task_end_step": (_INT, [_VP, _VP]),
    "dyros_task_step": (_INT, [_VP, _VP, _VP]),
    "dyros_task_step_launches": (_INT, [_VP]),
    "dyros_task_post_step": (_INT, [_VP, _VP]),
    "dyros_task_pack_results": (_INT, [_VP, _VP, _VP]),
    "dyros_task_set_obs_buf": (_INT, [_VP, _VP]),
}


def header_symbols(path: str = HEADER_PATH):
    """Every function the public header declares (used by the CPU test that checks the exports)."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dyros_[a-z0-9_]+)\s*\(", src)))


class DyrosError(RuntimeError):
    pass


_LIB = None


def load(path: str = LIB_PATH):
    """Load the native library (built by `make -C isaacgymdyros_b200/csrc` / __graft_entry__.build())."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.isfile(path):
        raise DyrosError(f"{path} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
                         f"g.build()'). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.dyros_abi_version() != ABI_VERSION:
        raise DyrosError("libdyros_b200.so ABI version mismatch")
    _LIB = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().dyros_last_error()
        raise DyrosError(f"{what}: {msg.decode() if msg else 'unknown error'}")
