/* dyros_b200.h -- C ABI of libdyros_b200.so (hand-written sm_100a CUDA behind the Isaac Gym tensor API).
 *
 * Drop-in boundary for ONE hot path of kdh0429/IsaacGymDyros: the per-step vectorised environment
 * behind `python train.py task=DyrosDynamicWalk`.  Paths below are relative to the reference root:
 *   T  = python/IsaacGymEnvs/isaacgymenvs/tasks/dyros_dynamic_walk.py
 *   VT = python/IsaacGymEnvs/isaacgymenvs/tasks/base/vec_task.py
 *   DOCT = docs/_sources/programming/tensors.rst.txt   (Isaac Gym tensor API contract)
 *
 * Conventions
 *   - Every pointer in DyrosSimBuffers / DyrosTaskBuffers is a DEVICE pointer into memory owned by the
 *     caller (torch allocations); the library keeps the pointers, never frees them, and allocates only
 *     its own constant model tables at create time (no allocation after dyros_sim_create).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  No call synchronises the
 *     host; every call is capturable in a CUDA graph.
 *   - Return value: 0 = ok, non-zero = error; dyros_last_error() gives the message (thread-local).
 *   - Tensor layouts are the reference's: root (N,13) [pos3, quat xyzw, linvel3, angvel3] DOCT:50-62;
 *     dof_state (N*nd,2) [pos,vel] DOCT:154-156; net contact force (N*nb,3) DOCT:267-279;
 *     actuation force (N*nd) DOCT:300-311; reset/progress/timeout/randomize buffers int64 VT:248-255.
 */
#ifndef DYROS_B200_H
#define DYROS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DYROS_ABI_VERSION 3  /* 3: DyrosTaskBuffers.reset_seq, DyrosSimDesc.physics_program (later additions within 3, a no-op for zero-initialised structs: DyrosPpoNet.inputs, DyrosPpoBuffers.obs_dim); 2: contact_friction, pd_gain_scale, dr_friction_*, dr_pd_gain_*, pack_results, set_obs_buf, post_step */
#define DYROS_MAX_LINKS 40
#define DYROS_MAX_BODIES 48
#define DYROS_LANES 4 /* roles (warps) per env group in the physics kernel */

typedef struct DyrosSim DyrosSim;   /* replaces the `sim` handle of gym.create_sim (VT:270) */
typedef struct DyrosTask DyrosTask; /* per-env task state of DyrosDynamicWalk (T:58-195) */

/* Flat model tables (host pointers, float64/int32; see isaacgymdyros_b200/model/tables.py).
 * Replaces what gym.load_asset + create_actor build inside the closed importer (T:293, T:354). */
typedef struct {
  int32_t num_links, num_bodies, num_dofs, num_points, num_cyls, sched_slots;
  const int32_t* link_parent; /* [nl] */
  const int32_t* link_dof;    /* [nl] */
  const double* link_E;       /* [nl*9] */
  const double* link_r;       /* [nl*3] */
  const double* link_axis;    /* [nl*3] */
  const int32_t* body_link;   /* [nb] */
  const double* body_pos;     /* [nb*3] */
  const double* body_rot;     /* [nb*9] */
  const double* body_inertia; /* [nb*10] */
  const double* dof_lower;    /* [nd] */
  const double* dof_upper;    /* [nd] */
  const double* dof_vel_limit;/* [nd]  dof_prop['velocity'], T:372 */
  const double* dof_effort;   /* [nd]  MJCF ctrlrange; used only if clamp_effort */
  const double* dof_stiffness;/* [nd]  joint spring about q = 0 (MJCF joint stiffness; NULL = none) */
  const int32_t* pt_link;     /* [np] */
  const int32_t* pt_body;     /* [np] */
  const double* pt_pos;       /* [np*3] */
  const double* pt_radius;    /* [np] */
  const int32_t* pt_solver;   /* [np] 1 = ground contact of this point is constraint-solved (sole corners), 0 = penalty */
  const int32_t* cyl_link;    /* [nc] */
  const int32_t* cyl_body;    /* [nc] */
  const double* cyl_center;   /* [nc*3] */
  const double* cyl_axis;     /* [nc*3] */
  const double* cyl_size;     /* [nc*2] radius, half height */
  const int32_t* sched;       /* [sched_slots*DYROS_LANES] role programs: column r = links of role r, ascending, -1 padded
                                 (model/tables.py::role_programs) */
  /* self-collision tables (model/selfcollision.py; all NULL / 0 = no self-collision): exact shapes + sample spheres per
   * link, bounding spheres of the links, candidate link pairs. Reference: create_actor(..., group i, filter 0), T:354. */
  int32_t sc_num_shapes, sc_num_samples, sc_num_pairs;
  const int32_t* sc_shape_kind;    /* [ns] 0 = box, 1 = cylinder, 2 = capsule (a sphere when its half height is 0) */
  const int32_t* sc_shape_link;    /* [ns] shapes are grouped by link */
  const int32_t* sc_shape_body;    /* [ns] */
  const int32_t* sc_shape_sample0; /* [ns+1] sample range of each shape */
  const double* sc_shape_center;   /* [ns*3] link frame */
  const double* sc_shape_rot;      /* [ns*9] row-major, columns = shape axes in the link frame (cylinder: column 2 = axis) */
  const double* sc_shape_size;     /* [ns*3] box half extents | cylinder / capsule radius, half height, 0 */
  const double* sc_sample;         /* [nsamp*4] link-frame position, radius */
  const int32_t* sc_link_shape0;   /* [nl+1] */
  const double* sc_link_sphere;    /* [nl*4] link-frame centre, radius (broad phase of the oracle; the kernel uses the shapes' own spheres) */
  const int32_t* sc_pairs;         /* [np*2] candidate link pairs i < j */
} DyrosModelDesc;

/* gymapi.SimParams / PhysXParams subset that reaches the solver (VT:423-471, DyrosDynamicWalk.yaml:37-56)
 * plus the named model options of SURVEY D2. */
typedef struct {
  int32_t num_envs;
  int32_t device;
  double dt;                /* sim.dt = 0.002 (double: derived constants are formed in double as Python does) */
  int32_t substeps;         /* sim.substeps = 1 (sub-steps inside one gym.simulate) */
  float gravity[3];
  float contact_offset;     /* physx.contact_offset 0.002 */
  float max_depenetration_velocity; /* 10 */
  int32_t contact_sweeps;   /* fixed PGS sweeps = physx.num_position_iterations + num_velocity_iterations (4+1) */
  float contact_erp;        /* fraction of penetration removed per sub-step through the velocity bias (DESIGN.md) */
  float friction;           /* combined plane/shape friction, terrain_cfg.py:7-8 -> 1.0 */
  float penalty_stiffness;  /* ground contact of non-solved points (N/m) */
  float penalty_damping;    /* (N s/m) */
  float penalty_max_force;  /* clamp of one penalty point's normal force (N) */
  float max_angular_velocity; /* AssetOptions.max_angular_velocity T:289 */
  int32_t clamp_effort;     /* clamp actuation to MJCF ctrlrange (SURVEY D2; default 0) */
  int32_t physics_program;  /* mapping of gym.simulate to the GPU: 0 = one lane per env, one warp per role (default, the
                               faster one at <= 28 envs per SM); 1 = 8 lanes per env with column-distributed articulated
                               inertias. Same model, same results up to float rounding (DESIGN.md section 4). */
} DyrosSimDesc;

/* Device buffers behind the gym tensor API (all owned by the caller). */
typedef struct {
  float* root_states;        /* (N,13)      acquire_actor_root_state_tensor  T:73 */
  float* dof_state;          /* (N*nd,2)    acquire_dof_state_tensor         T:74 */
  float* net_contact_force;  /* (N*nb,3)    acquire_net_contact_force_tensor T:75 */
  float* rigid_body_state;   /* (N*nb,13)   acquire_rigid_body_state_tensor  T:76 (may be NULL) */
  float* dof_actuation_force;/* (N*nd)      set_dof_actuation_force_tensor   T:520 */
  float* rb_force;           /* (N*nb,3)    apply_rigid_body_force_tensors   T:502 (may be NULL) */
  float* rb_torque;          /* (N*nb,3)    (may be NULL) */
  float* dof_damping;        /* (N,nd) per-env dof_prop['damping']  T:365 + DR */
  float* dof_armature;       /* (N,nd) per-env dof_prop['armature'] T:366-371 + DR */
  float* body_mass_scale;    /* (N,nb) per-env rigid_body_properties.mass scaling (setup-only DR) */
  float* contact_friction;   /* (N) per-env friction coefficient of the ground contacts, replaces DyrosSimDesc.friction
                                (DR of rigid_shape_properties.friction, DyrosDynamicWalk.yaml:89-96); may be NULL */
  float* link_pose;          /* (N,nl,12) world rotation (row-major) and origin of every link at the start of the LAST
                                sub-step of a simulate call: what the contact forces of that sub-step are computed from;
                                written by the physics kernels for the self-collision pass; may be NULL (no self-collision) */
  float* self_contact_force; /* (N*nb,3) net self-contact force per body of the last sub-step (also added into
                                net_contact_force); may be NULL */
} DyrosSimBuffers;

/* Per-env task state (names = the reference attributes, T:87-195; internal integers are int32). */
typedef struct {
  /* VecTask API buffers (VT:242-255) */
  float* obs_buf;            /* (N,487); (N,487+P) with a height scan of P points (dyros_task_set_height_scan) */
  float* rew_buf;            /* (N) */
  int64_t* reset_buf;        /* (N) */
  int64_t* timeout_buf;      /* (N) */
  int64_t* progress_buf;     /* (N) */
  int64_t* randomize_buf;    /* (N) */
  float* stacked_rewards;    /* (N,15) extras["stacked_rewards"] T:415-427 */
  int64_t* reset_env_ids;    /* (N) compacted ascending ids, T:554 */
  int32_t* reset_env_ids32;  /* (N) int32 copy, T:737,745 */
  int32_t* reset_count;      /* (1) */
  /* task attributes */
  float* actions;            /* (N,13) */
  float* actions_pre;        /* (N,13) */
  float* time;               /* (N) */
  int32_t* init_mocap_data_idx; /* (N) */
  int32_t* mocap_data_idx;   /* (N) */
  float* target_data_qpos;   /* (N,33) */
  float* target_data_force;  /* (N,2) */
  float* action_torque;      /* (N,12) */
  float* action_torque_pre;  /* (N,12) */
  float* motor_constant_scale; /* (N,12) */
  float* action_log;         /* (N,6,12) delay ring, linear layout as T:166 */
  int32_t* delay_idx;        /* (N) delay_idx_tensor[:,1] */
  int32_t* simul_len;        /* (N) simul_len_tensor[:,1] */
  float* qpos_noise;         /* (N,33) */
  float* qvel_noise;         /* (N,33) */
  float* qpos_pre;           /* (N,33) */
  float* qpos_bias;          /* (N,12) */
  float* quat_bias;          /* (N,3) */
  float* target_vel;         /* (N,2) */
  float* pre_joint_velocity_states; /* (N,33) */
  float* contact_forces_pre; /* (N,38,3) */
  float* total_mass;         /* (N) */
  float* env_origins;        /* (N,3) */
  float* epi_len;            /* (N) */
  float* epi_len_log;        /* (N) */
  float* contact_reward_sum; /* (N) */
  float* contact_reward_mean;/* (N) */
  int32_t* perturbation_count; /* (N) */
  int32_t* pert_duration;    /* (N) */
  int32_t* pert_on;          /* (N) 0/1 */
  int32_t* impulse;          /* (N) */
  float* magnitude;          /* (N) */
  float* phase;              /* (N) */
  int32_t* perturb_timing;   /* (N) */
  int32_t* perturb_start;    /* (1) sticky curriculum flag, T:489-490 */
  float* push_force;         /* (N,3) pelvis force for the next substep, forces[:,pelvis,:] T:498-499 */
  float* obs_history;        /* (N,20,37) ring; slot (head+1+j)%20 = reference history position j */
  float* action_history;     /* (N,20,13) ring */
  int32_t* obs_hist_head;    /* (N) newest slot */
  int32_t* act_hist_head;    /* (N) newest slot */
  int32_t* reset_seq;        /* (N) resets of this env so far: part of the Philox counter of reset_idx, so that two resets of
                                one env inside one step epoch (reset_done() + a termination) draw different values, T:611-665 */
  /* shared tables */
  const float* mocap_data;   /* (3600,36) T:112-113 */
  const float* obs_mean;     /* (37) */
  const float* obs_var;      /* (37) */
  float* pd_gain_scale;      /* (N,2) per-env scale of Kp, Kv in the upper-body PD of T:506 (DR of the PD gains,
                                BASELINE configs[3]; the reference has no such table: NULL = gains as in T:58-70) */
} DyrosTaskBuffers;

/* Constants of the task (SURVEY Appendix A1). */
typedef struct {
  int32_t skipframe;         /* controlFrequencyInv = 2 */
  float max_episode_length;  /* 8000.0 */
  float death_cost;          /* 0.0 */
  float initial_height;      /* 0.93 */
  int32_t perturb;           /* env.perturbation */
  int32_t randomize;         /* task.randomize: re-draw damping/armature on reset (VT:519-733) */
  float dr_damping_base, dr_damping_lo, dr_damping_hi;  /* 0.1, +U[0,2.9] */
  float dr_armature_lo, dr_armature_hi;                 /* xU[0.8,1.2] of the base table */
  const double* dr_armature_base;                       /* [nd] host pointer, T:366-371 */
  /* optional DR re-drawn on reset next to damping / armature (lo == hi == 0: leave the table alone):
   * contact_friction = dr_friction_base * U[lo,hi] (DyrosDynamicWalk.yaml:89-96, "scaling");
   * pd_gain_scale[:,0] and [:,1] = two independent U[lo,hi] */
  float dr_friction_base, dr_friction_lo, dr_friction_hi;
  float dr_pd_gain_lo, dr_pd_gain_hi;
  int32_t mocap_rows;        /* 3600 */
  const float* kp;           /* [33] host, already /9 in float32 (T:58-63) */
  const float* kv;           /* [33] host, already /3 in float32 (T:65-70) */
  const float* action_high;  /* [33] host (T:296-301) */
  const float* initial_dof_pos; /* [33] host (T:95-100) */
  int32_t left_foot_body, right_foot_body, pelvis_body; /* find_asset_rigid_body_index T:304-306 */
  uint64_t seed;             /* Philox key (config.yaml:11 seed 42 + rank) */
} DyrosTaskDesc;

/* Test-mode noise injection: env-indexed draws replacing the Philox streams (SURVEY A6). Any NULL
 * member keeps its production stream. */
typedef struct {
  const float* qpos_normal;  /* (skipframe,N,33) outputs of torch.normal(0,0.00016/3) T:528 */
  const float* vel_u;        /* (N,6)  torch.rand T:766 */
  const float* reset_f;      /* (N,32) [qpos_bias u12, quat_bias u3, ft u2(unused), vel_mag, vel_theta, mocap, motor u12, pad2] */
  const int64_t* reset_i;    /* (N,2)  [delay, perturb_timing] T:652,665 */
  const int64_t* pert_i;     /* (N,2)  [impulse, duration] T:440-441 */
  const float* pert_f;       /* (N,1)  T:443 */
  const float* dr_u;         /* (N,66) [damping u33, armature u33] */
} DyrosNoiseInjection;

const char* dyros_last_error(void);
int dyros_abi_version(void);

/* --- gym level (replaces gym.create_sim / prepare_sim / simulate, VT:270, VT:196, T:525) --- */
int dyros_sim_create(const DyrosSimDesc* desc, const DyrosModelDesc* model, const DyrosSimBuffers* buf, DyrosSim** out);
int dyros_sim_destroy(DyrosSim* sim);
/* gym.simulate: one time step dt (in `substeps` sub-steps) from dof_actuation_force (+ pending rb_force/torque
 * when apply_wrench != 0, consumed by the first sub-step, DOCT:322-335). */
int dyros_simulate(DyrosSim* sim, int apply_wrench, void* stream);
/* Self-collision pass (actor created with collision filter 0, T:354): detects contacts between the shapes of
 * non-adjacent links from link_pose, writes self_contact_force and adds it into net_contact_force, so that
 * collision_true (T:590, T:937) sees them. dyros_simulate and dyros_task_step run it themselves when the model carries
 * self-collision tables and both buffers are given; exported for callers that stage the step (after
 * dyros_task_physics_kernel). It ADDS into net_contact_force: once per physics launch. */
int dyros_self_collision(DyrosSim* sim, void* stream);
/* gym.refresh_rigid_body_state_tensor: forward kinematics into rigid_body_state (DOCT:193-207). */
int dyros_refresh_rigid_body_state(DyrosSim* sim, void* stream);
/* gym.refresh_dof_force_tensor (tasks/humanoid.py:85,245; DOCT "DOF forces"): (N*nd) generalised force at every DOF =
 * applied actuation + passive joint spring and damper on the current state, into the caller's buffer. */
int dyros_refresh_dof_force(DyrosSim* sim, float* dof_force, void* stream);
/* gym.refresh_force_sensor_tensor (tasks/humanoid.py:80,167-168,243): per env and sensor [force 3, torque 3] in the sensor
 * frame: the net contact force on the sensor's body (torque entries zero: the contact model keeps no line of action).
 * sensor_body (ns) int32 and sensor_pose (ns,7) [pos3, quat xyzw] are device arrays describing the asset's sensors;
 * refreshes rigid_body_state first (the sensor frames come from it). */
int dyros_refresh_force_sensors(DyrosSim* sim, const int32_t* sensor_body, const float* sensor_pose, int num_sensors,
                                float* sensor_out, void* stream);
/* gym.set_dof_state_tensor_indexed / set_actor_root_state_tensor_indexed (T:738,746): buffers are the live state
 * already (immediate CPU-pipeline semantics, SURVEY D3); validates the ids and returns. */
int dyros_set_state_indexed(DyrosSim* sim, const int32_t* env_ids, int count, void* stream);

/* Measurement aid (no reference counterpart): FFMA-saturation micro-benchmark giving the FP32 roofline denominator
 * that MEASURED_PEAKS.json lacks (SURVEY section 8d). Synchronous; returns TFLOP/s (FMA = 2 FLOP). */
int dyros_measure_fp32_peak(int device, int iters, double* tflops_out);
/* Measurement aid (no reference counterpart): overwrites [buf, buf+bytes) on `stream`, to evict the L2 between timed
 * steps with a kernel that keeps the SMs' L1 / shared-memory split of the step kernels (a fill launched by another
 * library reconfigures the SMs, and the ~25 us of the switch back would land inside the next timed step). */
int dyros_flush_l2(void* buf, size_t bytes, int value, void* stream);
/* Optional: keep the env state resident in the set-aside (persisting) part of the B200's 126 MB L2. [base, base+bytes)
 * is the one contiguous range holding the per-env buffers (the caller allocates them from one arena); kernels launched
 * on `stream` afterwards, and kernel nodes captured from it into CUDA graphs, access that range with the persisting
 * property, so traffic of other kernels (a policy network between two env steps, an L2 flush) does not evict it.
 * bytes = 0 switches the window off and resets the persisting lines. *set_aside_out (may be NULL) receives the size of
 * the set-aside region actually configured (device limit: cudaDevAttrMaxPersistingL2CacheSize). */
int dyros_sim_set_l2_persistence(DyrosSim* sim, void* base, size_t bytes, void* stream, size_t* set_aside_out);
/* Physics launch geometry chosen at create time: envs per CTA, CTAs, threads per CTA, dynamic shared memory bytes. */
int dyros_sim_launch_info(DyrosSim* sim, int32_t out[4]);

/* gym.add_heightfield (legged_gym terrain, mesh_type 'heightfield'): the ground of the sim becomes a heightfield instead
 * of the plane z = 0. Vertex (i, j) sits at (origin.x + i row_scale, origin.y + j column_scale,
 * origin.z + vertical_scale samples[i, j]); each cell is split along the diagonal (i, j)-(i+1, j+1); outside the
 * field's x-y rectangle there is no ground (DESIGN.md section 4). The contact friction stays DyrosSimDesc.friction /
 * contact_friction. `samples` is a caller-owned DEVICE buffer that must stay alive and unchanged while the sim uses it.
 * NULL switches back to the plane. The launch geometry stays as it is. Not for physics_program 1. */
typedef struct {
  const int16_t* samples;     /* (num_rows, num_columns) row-major device array; row index along x, column along y */
  int32_t num_rows, num_columns;  /* >= 2 each */
  float row_scale, column_scale, vertical_scale;  /* > 0 (m per sample step / per sample unit) */
  float origin[3];            /* world position of vertex (0, 0) at sample value 0 (HeightFieldParams.transform.p) */
} DyrosHeightField;
int dyros_sim_set_heightfield(DyrosSim* sim, const DyrosHeightField* field);

/* gym.add_triangle_mesh (legged_gym terrain, mesh_type 'trimesh'): the ground of the sim becomes a triangle mesh. Vertex v
 * sits at vertices[v] + origin (only a translation, as for the heightfield); triangle (a, b, c) has the face normal
 * normalize((b - a) x (c - a)), its front the counter-clockwise side. A sphere of centre c and radius r (r = 0 for box
 * corners and cylinder rim points) touches the nearest triangle (ties: the lowest index) with gap s - r, s the distance
 * signed by the face normal; a point farther than the query margin M = contact_offset + the model's largest point radius
 * + 0.1 m from every triangle has no ground (DESIGN.md section 4, "Triangle-mesh ground"). The library copies the mesh
 * into its own device memory and builds a bucket grid over it; zero-area triangles are dropped. One ground per sim: a sim
 * with a heightfield refuses a mesh and the other way round. The lanes program (physics_program 1) has no mesh ground.
 * NULL switches back to the plane z = 0, frees the mesh and restores DyrosSimDesc.friction. While the mesh is set, the
 * contact friction of envs without a contact_friction table is dynamic_friction. */
typedef struct {
  const float* vertices;      /* (num_vertices, 3) HOST array */
  const uint32_t* triangles;  /* (num_triangles, 3) HOST array of vertex indices */
  int64_t num_vertices, num_triangles;
  float origin[3];            /* TriangleMeshParams.transform.p */
  float dynamic_friction;     /* TriangleMeshParams.dynamic_friction, >= 0 */
} DyrosTriangleMesh;
int dyros_sim_set_triangle_mesh(DyrosSim* sim, const DyrosTriangleMesh* mesh);
/* The sim's mesh ground: out[0] device bytes allocated, out[1] zero-area triangles dropped, out[2] triangles kept,
 * out[3] buckets of the grid (all 0 without a mesh). */
int dyros_sim_triangle_mesh_info(DyrosSim* sim, int64_t out[4]);

/* --- task level (bodies of DyrosDynamicWalk methods) --- */
int dyros_task_create(DyrosSim* sim, const DyrosTaskDesc* desc, const DyrosTaskBuffers* buf, DyrosTask** out);
int dyros_task_destroy(DyrosTask* task);
int dyros_task_set_noise_injection(DyrosTask* task, const DyrosNoiseInjection* inj);
/* Terrain curriculum (legged_gym's _update_terrain_curriculum; DESIGN.md section 4, "Curriculum"). Every reset of env e,
 * fused or staged or through dyros_task_reset_idx, first moves the env one level up when its root has walked farther than
 * move_up_distance from env_origins[e] in x-y, else one level down when it walked less than |target_vel[e]| *
 * move_down_scale; a level past the top is redrawn uniformly over [0, num_levels) (reset_f column 30), a level below 0
 * stays 0. env_origins[e] then becomes origins[levels[e], types[e]] and the root is placed there. The end-of-step pass
 * writes the mean of `levels` over all envs to level_mean. All pointers are caller-owned DEVICE memory that must stay
 * alive while the task uses them. NULL switches the curriculum off. Call before a CUDA graph of the step is captured:
 * captured launches keep the setting they were captured with. */
typedef struct {
  const float* origins;      /* (num_levels, num_types, 3) world origin of each sub-terrain */
  int32_t* levels;           /* (N) terrain level of each env, in [0, num_levels); updated on every reset */
  const int32_t* types;      /* (N) terrain type (column) of each env, in [0, num_types) */
  int32_t num_levels, num_types;  /* >= 1 each */
  float move_up_distance;    /* terrain_length / 2 */
  float move_down_scale;     /* episode length (s) * 0.5 */
  float* level_mean;         /* (1) mean level after each step's resets; may be NULL */
} DyrosTerrainCurriculum;
int dyros_task_set_terrain_curriculum(DyrosTask* task, const DyrosTerrainCurriculum* curriculum);
/* Height scan (legged_gym's measure_heights; DESIGN.md section 4, "Height scan"): the observation row gains P columns,
 * obs[e, 487 + k] = clip(root_z - base_offset - h_k, -1, 1) * scale. h_k is the terrain height under point k, the point
 * (points[k].x, points[k].y, 0) of the base's yaw frame carried to the world: rotated by the yaw of the root quaternion,
 * shifted by the root's x-y. On a heightfield h_k is the lowest of the three samples legged_gym reads at the clamped
 * cell index (not the triangle the physics touches); on the plane it is 0. The heights are those of the root the rest
 * of the row describes (post-reset for an env reset in the step). measured_heights, if given, receives h_k in m.
 * The field is the sim's at each launch (dyros_sim_set_heightfield). From this call on, obs_buf and every later
 * dyros_task_set_obs_buf target must hold N*(487+P) floats, and dyros_task_pack_results writes the wider rows. Call
 * before a CUDA graph of the step is captured: captured launches keep the setting they were captured with. NULL
 * switches the scan off (rows of 487 floats again). All pointers are caller-owned DEVICE memory that must stay alive
 * while the task uses them. */
typedef struct {
  const float* points;       /* (P,2) x, y in the base's yaw frame (m) */
  int32_t num_points;        /* P, 1..1024 */
  float base_offset;         /* 0.5 */
  float scale;               /* obs_scales.height_measurements, 5.0 */
  float* measured_heights;   /* (N,P) h_k in m; may be NULL */
  /* the samples h_k is read from: NULL = the sim's heightfield at each launch (0 on the plane); non-NULL = this field
   * (validated and copied at this call; its samples stay caller-owned device memory), e.g. the samples a triangle-mesh
   * ground was made from (legged_gym reads height_samples with mesh_type 'trimesh') */
  const DyrosHeightField* field;
} DyrosHeightScan;
int dyros_task_set_height_scan(DyrosTask* task, const DyrosHeightScan* scan);
/* Critic states (DESIGN.md section 4, "Critic states"): a privileged row per env for an asymmetric critic, written by
 * the observation kernels beside the observation row, from the same post-reset root. With P the points of the height
 * scan (0 without one), row e of `states` (N, S), S = 487 + P + 31, holds
 *   0..486      the observation row's first 487 columns, bit for bit;
 *   487..486+P  the height-scan columns clip(root_z - base_offset - h_k, -1, 1) * scale;
 *   then 31 privileged columns, each clipped to [-5, 5]: root linear velocity (world, no noise) x 2, root angular
 *   velocity x 0.25, net contact force of the left and right foot x 1e-3, push_force x 1e-2 (these two 0 at an episode
 *   start, epi_len == 0), motor_constant_scale - 1 (12), total_mass / nominal_mass - 1, the env's ground friction - 1
 *   (contact_friction[e], else the sim's friction), pd_gain_scale - 1 (2; 0 without the table).
 * With states set and heights_in_obs == 0, the heights go into the state row ONLY: obs_buf rows (and the rows of
 * dyros_task_pack_results) are 487 floats wide. With heights_in_obs != 0 they go into both rows (487 + P). `states`
 * must hold N*S floats for the height scan in force at each launch. Call before a CUDA graph of the step is captured.
 * NULL, or a NULL `states`, switches the rows off. `states` is caller-owned DEVICE memory that must stay alive while
 * the task uses it. */
typedef struct {
  float* states;             /* (N, 487 + P + 31), 4-byte aligned */
  int32_t heights_in_obs;    /* 0: the heights go into the state row only */
  float nominal_mass;        /* > 0: the total mass the model was built with */
} DyrosCriticStates;
int dyros_task_set_critic_states(DyrosTask* task, const DyrosCriticStates* states);
int dyros_task_prologue(DyrosTask* task, const float* actions, void* stream);      /* VT:307 + T:449-502 */
/* T:504-530 in one launch: skipframe x (substep torque, gym.simulate, sensor noise); what dyros_task_step uses. */
int dyros_task_physics(DyrosTask* task, void* stream);
/* Measurement aid: the physics launch of dyros_task_physics alone (without the self-collision pass that follows it;
 * dyros_self_collision completes the step), so that the dominant kernel can be timed by itself. */
int dyros_task_physics_kernel(DyrosTask* task, void* stream);
/* Profiling aid: dyros_task_physics that also writes clock64() at the phase boundaries of CTA 0 into `trace`
 * (device buffer of skipframe * DYROS_LANES * 32 int64; see physics_roles.cuh for the mark ids). */
int dyros_task_physics_trace(DyrosTask* task, int64_t* trace, void* stream);
/* The first launch of dyros_task_step on its own: dyros_task_prologue + dyros_task_physics in one kernel (the
 * prologue runs on the I/O warps while the role warps start the first sub-step). `trace` may be NULL. */
int dyros_task_prologue_physics(DyrosTask* task, const float* actions, int64_t* trace, void* stream);
int dyros_task_substep_torque(DyrosTask* task, void* stream);                      /* T:505-520 -> dof_actuation_force */
int dyros_task_sensor_noise(DyrosTask* task, int substep, void* stream);           /* T:528-530 */
int dyros_task_epilogue(DyrosTask* task, void* stream);                            /* T:532-541 + VT:325 + T:544-545 */
int dyros_task_check_termination(DyrosTask* task, void* stream);                   /* T:581-596 */
int dyros_task_compute_reward(DyrosTask* task, void* stream);                      /* T:387-428, T:802-947 */
int dyros_task_compact_resets(DyrosTask* task, void* stream);                      /* T:554 nonzero + curriculum gate sums T:489 */
int dyros_task_reset_idx(DyrosTask* task, const int64_t* env_ids, int count, void* stream); /* T:598-669; env_ids NULL = use compacted list */
int dyros_task_compute_observations(DyrosTask* task, void* stream);                /* T:750-796 */
int dyros_task_late_update(DyrosTask* task, void* stream);                         /* T:560-563 */
/* End of a staged step: the cross-env curriculum gate of T:489 (evaluated for the next step) + RNG epoch bump. */
int dyros_task_end_step(DyrosTask* task, void* stream);
/* Whole VecTask.step (VT:293-344) in the fewest launches; same results as the staged calls, except that the compacted
 * id list of T:554 (reset_env_ids / reset_count), which the fused step does not need, is left to
 * dyros_task_compact_resets. */
int dyros_task_step(DyrosTask* task, const float* actions, void* stream);
/* The launches of dyros_task_step after dyros_task_prologue_physics, on their own (T:532-563 fused + the cross-env
 * pass): dyros_task_prologue_physics followed by dyros_task_post_step is dyros_task_step. */
int dyros_task_post_step(DyrosTask* task, void* stream);
/* Number of kernel launches dyros_task_step enqueues (for bench.py's gpu_launches). */
int dyros_task_step_launches(DyrosTask* task);
/* What VecTask.step returns (VT:336-344: obs_dict["obs"], rew_buf, reset_buf, extras["time_outs"]) gathered into ONE
 * contiguous device block `dst`, 16-byte aligned, with W = 487 (+ P with a height scan):
 * obs (N,W) f32 | rew (N) f32 | [4 bytes of padding if N*(W+1) is odd] | reset (N) i64 | time_outs (N) i64,
 * i.e. the i64 part starts at N*(W+1)*4 rounded up to a multiple of 8 (N*488*4 without a scan). A host-side
 * caller then moves the block with a single device->host copy on its own stream while the next step runs. */
int dyros_task_pack_results(DyrosTask* task, void* dst, void* stream);
/* Re-points the observation buffer (DyrosTaskBuffers.obs_buf, (N,487) f32, or (N,487+P) with a height scan; 16-byte
 * aligned) for the launches enqueued
 * from now on; launches already enqueued or captured in a CUDA graph keep the pointer they were given. With obs_buf
 * set to a result block, dyros_task_pack_results on that block only adds rew / reset / time_outs. */
int dyros_task_set_obs_buf(DyrosTask* task, float* obs_buf);

/* --- on-device PPO around the env step (SURVEY 8f-1; reference: learning/rl_games_custom/a2c_common_dyros.py = A2C,
 *     a2c_continuous_seperate.py = AG, models_dyros.py = MD, cfg/train/DyrosDynamicWalkPPO.yaml = PPO) ---
 * Rollout buffers are ENV-major, (N, H, .): a minibatch of the update (rl_games slices the swap_and_flatten01 layout,
 * A2C:703) is a contiguous block of rows. All pointers are device pointers owned by the caller. */
typedef struct {
  int32_t N, H;               /* envs, horizon_length (PPO:85) */
  float gamma, tau;           /* PPO:66-67 */
  float e_clip, critic_coef;  /* PPO:84, PPO:88 */
  float reward_scale;         /* reward_shaper.scale_value, PPO:64 */
  int32_t value_bootstrap;    /* PPO:61 */
  uint64_t seed;              /* Philox key of the action noise */
  float* obs;                 /* (N,H,W) fp32 rows, W = obs_dim (the fp32 path; the packed path keeps bf16 rows) A2C:639 */
  float* actions;             /* (N,H,13) */
  float* mus;                 /* (N,H,13) */
  float* neglogp;             /* (N,H) */
  float* values;              /* (N,H) */
  float* rewards;             /* (N,H) shaped, A2C:654-661 */
  float* dones;               /* (N,H) 0/1, self.dones before the step, A2C:640 */
  float* advantages;          /* (N,H) A2C:485-500 */
  float* returns;             /* (N,H) A2C:692 */
  float* cur_reward;          /* (N) A2C:663 */
  float* cur_length;          /* (N) A2C:664 */
  float* ep_stats;            /* (3) sums over finished episodes: reward, length, count (A2C:676-677) */
  int32_t* step;              /* (1) slot of the next rollout step, 0..H-1 */
  uint64_t* global_step;      /* (1) rollout steps so far (Philox counter) */
  int32_t obs_dim;            /* W, columns of an observation row: 487 + P with a height scan of P points; 0 means 487.
                               * Appended in ABI 3: a zero-initialised struct keeps the 487 layout. Negative: refused. */
} DyrosPpoBuffers;
/* get_action_values + the experience_buffer updates of one rollout step (A2C:633-647, MD:28-58): samples the actions
 * from N(mu, exp(logstd)), computes their neglogp (MD:60-63), records obs / done / mu / value / action / neglogp at slot
 * *step, and hands the actions to the env (`actions_env`, (N,13)). inject_normal (H,N,13) replaces the Philox draws (tests). */
int dyros_ppo_act(const DyrosPpoBuffers* b, const float* mu, const float* value, const float* logstd, const float* obs,
                  const int64_t* reset_buf, float* actions_env, const float* inject_normal, void* stream);
/* after VecTask.step: shaped reward with the time-out bootstrap (A2C:654-661), episode statistics (A2C:663-684); advances *step. */
int dyros_ppo_reward(const DyrosPpoBuffers* b, const float* rew, const int64_t* timeout, const int64_t* reset_buf, void* stream);
/* discount_values (A2C:485-500) and returns = advantages + values (A2C:692). */
int dyros_ppo_gae(const DyrosPpoBuffers* b, const float* last_values, const int64_t* last_reset, void* stream);
/* calc_gradients up to the network outputs (AG:108-160) for rows [row0, row0+mb): d loss / d mu, d loss / d value, and the
 * logged means accumulated into stats[4] = {actor loss, critic loss, kl, clip fraction}. adv_norm: normalised advantages (A2C:944). */
int dyros_ppo_loss_grad(const DyrosPpoBuffers* b, int row0, int mb, const float* mu, const float* value, const float* logstd,
                        const float* adv_norm, float* dmu, float* dvalue, float* stats, void* stream);
/* optimizer_actor + optimizer_critic (AG:50-54) on flat buffers, with clip_grad_norm_ of the actor part (AG:179) and the
 * 1/world averaging of all-reduced gradient sums (AG:161-163). lr_dev[2] = {actor, critic} rates and step_dev live on the
 * device; after the update the actor's rate follows rl_games' LinearScheduler, stepped per minibatch as the reference
 * does (A2C:888-892; lr_max_steps = max_epochs, 0 = constant rate). */
int dyros_ppo_adam(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int n_actor, int n, float grad_scale,
                   float max_norm, float* norm2_scratch, float* lr_dev, int32_t* step_dev, float beta1, float beta2,
                   float eps, float lr0, float lr_min, int lr_max_steps, void* stream);


/* ---- packed bf16 path of the two MLPs (network_builder_dyros.py:129-216: separate W-H-H actor and critic): one batch-2
 * problem in GEMM layout, net 0 = actor, net 1 = critic. The caller runs the 8 batched GEMMs of a minibatch with a
 * library (3 forward: x W0^T, h0 W1^T, h1 Wh^T; 5 backward); these entry points are everything between them. Weights
 * and activations bf16 (where the reference trains under fp16 autocast + GradScaler, PPO:59), biases, bias gradients,
 * master parameters, Adam moments fp32. The flat master layout (dyros_ppo_adam's buffers) is, per net,
 * [W0 (H x W), b0 (H), W1 (H x H), b1 (H), Wh (nout x H), bh (nout)], nout = 13 (actor) then 1 (critic).
 * W is the input width and K0 = round_up(W, 8) the padded one: a GEMM's rows must be a multiple of 8 elements for the
 * library's tensor-core kernels (an odd leading dimension falls back to its slow align-1 kernels), so W0 and the bf16
 * observation rows x_step / x_roll are K0 wide, with columns W..K0-1 zero. W = 487: K0 = 488; W = 674: K0 = 680. */
typedef struct DyrosPpoNet {
  int32_t hidden;        /* H, a multiple of 8 (256: PPO:28-35) */
  int32_t inputs;        /* W; 0 means 487. Added in ABI 3 in the padding before w0: sizeof and every other offset are
                          * unchanged, and a zero-initialised struct keeps the 487 layout. Negative: refused. */
  void* w0;              /* bf16 [2][H][K0]: W inputs padded to K0 (columns W..K0-1 are zero) */
  float* b0;             /* [2][H] */
  void* w1;              /* bf16 [2][H][H] */
  float* b1;             /* [2][H] */
  void* wh;              /* bf16 [2][16][H]: rows 0..12 of net 0 = mu, row 0 of net 1 = value, the rest zero */
  float* bh;             /* [2][16] */
  void* gw0;             /* bf16 gradients in the same layouts (GEMM outputs) */
  void* gw1;
  void* gwh;
  float* gb0;            /* fp32 bias gradients, accumulated by dyros_ppo_relu_bwd / dyros_ppo_loss_grad_packed, */
  float* gb1;            /* zeroed by dyros_ppo_unpack_grads */
  float* gbh;
} DyrosPpoNet;
/* obs (N,W) fp32 -> bf16 rows of width K0 (W = b->obs_dim, columns W..K0-1 written as zero): x_step (N,K0) for this
 * step's policy forward and, if x_roll is given, row e*H + *step of the env-major rollout store (N*H,K0). */
int dyros_ppo_cast_obs(const DyrosPpoBuffers* b, const float* obs, void* x_step, void* x_roll, void* stream);
/* t [2][rows][H] bf16 = relu(t + bias [2][H]) in place (the hidden layers' activation, network_builder_dyros.py:132-146). */
int dyros_ppo_bias_relu(void* t, const float* bias, int rows, int hidden, void* stream);
/* g [2][rows][H] bf16 = (h > 0 ? g : 0) in place; gbias [2][H] += column sums of the result. */
int dyros_ppo_relu_bwd(void* g, const void* h, float* gbias, int rows, int hidden, void* stream);
/* dyros_ppo_act on the packed head output out [2][N][16] bf16 (without bias) and bh [2][16]; does not store obs. */
int dyros_ppo_act_packed(const DyrosPpoBuffers* b, const void* out, const float* bh, const float* logstd, const int64_t* reset_buf,
                         float* actions_env, const float* inject_normal, void* stream);
/* dyros_ppo_loss_grad on the packed head output of rows [row0, row0+mb): writes dout [2][mb][16] bf16, accumulates gbh,
 * refreshes the rows' stored mu (dataset.update_mu_sigma, A2C:884) and stats[4]. */
int dyros_ppo_loss_grad_packed(const DyrosPpoBuffers* b, int row0, int mb, const void* out, const float* bh, const float* logstd,
                               const float* adv_norm, void* dout, float* gbh, float* stats, void* stream);
/* flat fp32 master parameters -> packed weights / biases (after every optimiser step). */
int dyros_ppo_pack_params(const DyrosPpoNet* net, const float* flat, void* stream);
/* packed gradients -> flat fp32 master gradient (what the all-reduce and the optimiser see); zeroes gb0 / gb1 / gbh.
 * norm2_accum (optional): += squared norm of the actor's gradients (the clip_grad_norm_ reduction of AG:179 folded in;
 * only meaningful when no all-reduce follows, i.e. on a single rank). */
int dyros_ppo_unpack_grads(const DyrosPpoNet* net, float* flat_grad, float* norm2_accum, void* stream);
/* dyros_ppo_adam that also refreshes the packed copy of every parameter it updates (dyros_ppo_pack_params folded in).
 * norm_done != 0: norm2_scratch already holds the squared norm of the actor's (unscaled) gradients. */
int dyros_ppo_adam_packed(const DyrosPpoNet* net, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float grad_scale,
                          float max_norm, int norm_done, float* norm2_scratch, float* lr_dev, int32_t* step_dev, float beta1, float beta2,
                          float eps, float lr0, float lr_min, int lr_max_steps, void* stream);
/* Asymmetric critic (DESIGN.md section 9): the same three calls for a critic of input width critic_inputs = Wc wider
 * than the actor's Wa = net->inputs (0: Wc = Wa, exactly the calls above; otherwise Wc >= Wa, or refused). The flat
 * master layout then holds the actor's W0 as H x Wa and the critic's as H x Wc; both packed W0 blocks share the leading
 * dimension K0 = round_up(Wc, 8), so one bf16 input row of width K0 (the state row: its first Wa columns are the
 * actor's observation) feeds both nets in one batched GEMM. Columns Wa..K0-1 of the actor's W0 are never written and
 * stay zero: the actor is blind to the critic's extra columns. Run dyros_ppo_cast_obs / dyros_ppo_act with
 * obs_dim = Wc on the state rows. */
int dyros_ppo_pack_params_ac(const DyrosPpoNet* net, int critic_inputs, const float* flat, void* stream);
int dyros_ppo_unpack_grads_ac(const DyrosPpoNet* net, int critic_inputs, float* flat_grad, float* norm2_accum, void* stream);
int dyros_ppo_adam_packed_ac(const DyrosPpoNet* net, int critic_inputs, float* params, const float* grads, float* exp_avg,
                             float* exp_avg_sq, float grad_scale, float max_norm, int norm_done, float* norm2_scratch, float* lr_dev,
                             int32_t* step_dev, float beta1, float beta2, float eps, float lr0, float lr_min, int lr_max_steps,
                             void* stream);

/* ---- gradient exchange over peer memory (NVLink / NVSwitch): the Horovod all-reduce of AG:161-173 folded into the
 * optimiser's kernels. Every rank allocates two flat gradient buffers of `stride` floats (stride >= n, a multiple of 4,
 * the second right after the first) and 8 flag words, zero-initialised, and maps its peers' allocations into its own
 * address space (CUDA IPC); `grad[r][p]` / `flags[r]` are those addresses as seen from THIS process. One process per GPU,
 * one node, at most 8 ranks. */
typedef struct DyrosPpoPeers {
  int32_t world, rank;
  int32_t stride;            /* floats between a rank's two gradient buffers */
  float* grad[8][2];         /* [rank][parity of the minibatch counter] */
  uint32_t* flags[8];        /* [rank] -> that rank's 8 flag words: flags[r][q] = minibatches rank q has published to rank r */
  uint32_t* epoch;           /* local (1): minibatches finished; advanced by dyros_ppo_reduce_peers / dyros_ppo_all_gather_peers */
  uint32_t* ticket;          /* local (4): zero-initialised scratch */
  /* two-phase exchange only (dyros_ppo_reduce_scatter_peers + dyros_ppo_all_gather_peers); may be NULL otherwise */
  float* sum[8][2];          /* [rank][parity]: `stride` floats, of which the rank writes ITS slice of the summed gradient */
  uint32_t* flags2[8];       /* [rank] -> 8 more flag words: "rank q has published its summed slice" */
  float* pnorm[8];           /* [rank] -> 2 floats [parity]: squared norm of the actor entries of the rank's slice */
} DyrosPpoPeers;
/* Peer-shareable device memory for the exchange (cudaMalloc + CUDA IPC). dyros_peer_alloc: `bytes` of zeroed memory on
 * the current device and its 64-byte IPC handle (to be sent to the other ranks of the node by any host channel).
 * dyros_peer_open: maps another rank's allocation for kernels of the CURRENT device (enables the NVLink peer path).
 * dyros_peer_close / dyros_peer_free undo them. */
int dyros_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int dyros_peer_open(const unsigned char* handle64, void** ptr);
int dyros_peer_close(void* ptr);
int dyros_peer_free(void* ptr);
/* dyros_ppo_unpack_grads into this rank's buffer of the current parity. */
int dyros_ppo_unpack_grads_peers(const DyrosPpoNet* net, const DyrosPpoPeers* peers, void* stream);
int dyros_ppo_unpack_grads_peers_ac(const DyrosPpoNet* net, int critic_inputs, const DyrosPpoPeers* peers, void* stream);
/* Publishes this rank's buffer, waits for every rank's, and writes the SUM over ranks (in rank order: bit-identical on
 * every rank) to flat_grad_sum (local, n floats); norm2_accum += squared norm of its first n_actor entries. */
int dyros_ppo_reduce_peers(const DyrosPpoPeers* peers, float* flat_grad_sum, int n, int n_actor, float* norm2_accum, void* stream);
/* The same exchange in two phases, each rank reading 2 x (world-1)/world of a buffer instead of (world-1) buffers:
 * reduce-scatter (rank r sums slice r of all ranks' buffers, in rank order, into flat_grad_sum and its published `sum`
 * buffer) and all-gather (every rank copies the other ranks' summed slices; norm2_accum += the slices' partial norms in
 * rank order). Call one after the other on the same stream. */
int dyros_ppo_reduce_scatter_peers(const DyrosPpoPeers* peers, float* flat_grad_sum, int n, int n_actor, void* stream);
int dyros_ppo_all_gather_peers(const DyrosPpoPeers* peers, float* flat_grad_sum, int n, float* norm2_accum, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DYROS_B200_H */
