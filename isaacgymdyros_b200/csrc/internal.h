// Internal (non-ABI) structures shared by capi.cu, task_kernels.cu and physics_kernels.cu.
#pragma once
#include "common.cuh"

namespace dyros {

constexpr int ND = 33, NB = 38, NA = 13, NOBS1 = 37, NHIS = 10, NSKIP = 2, NSLOT = NHIS * NSKIP;  // T:36-43
constexpr int NOBS = (NOBS1 + NA) * (NHIS - 1) + NOBS1;                                           // 487
constexpr int LOG_DEPTH = 6;                                                                      // T:166

// float32 device copies of the model tables (see model/tables.py for the meaning of each array) plus
// tables derived at create time (children lists, per-link candidate ranges, foot chains)
constexpr int MAX_CHAIN = 8;   // links between the feet's common ancestor and a solver (foot) link / the base and that ancestor
constexpr int MAX_FEET = 2;    // solver links
constexpr int MAX_SOLVER_PTS = 8;  // candidate solver points per foot
constexpr int MAX_ACTIVE_PTS = 4;  // active (constraint-solved) points per foot and sub-step
// record of one link in the flattened role programs (word offsets; ints and floats share the table)
constexpr int REC_WORDS = 44, MAX_LINK_BODIES = 3, MAX_LINK_CHILDREN = 3, REC_FOREIGN = 1 << 30;
// (44 words: a multiple of 4 so that the 3-vectors below sit on 16-byte boundaries, and 44 mod 32 = 12 so that the 8
//  lanes of a group reading 8 consecutive records hit 8 different shared-memory banks)
constexpr int R_LINK = 0, R_PARENT = 1, R_FLAGS = 2, R_DOF = 3, R_NBODY = 4, R_BODY0 = 5, R_NCHILD = 8, R_CHILD0 = 9,
              R_AXIS = 12, R_R = 16, R_E = 20, R_REACH = 32, R_PT0 = 33, R_PT1 = 34, R_CYL0 = 35, R_CYL1 = 36,
              R_VLIM = 37, R_LO = 38, R_UP = 39, R_EFF = 40, R_FOOT = 41, R_STIFF = 42, R_CSLOT = 43;
constexpr int RF_PARENT_FOREIGN = 1, RF_PARENT_BASE = 2;
constexpr int RF_PUBLISH = 4;  // a child of the link lives in another role: its stage flags are read there
constexpr int RF_KEEP = 8;     // a child of the link in the SAME role is not the role's next link: results go through the block
constexpr int SC_MAX_SHAPES = 96;         // self-collision: collision primitives of one articulation
constexpr int SC_MAX_SHAPE_SAMPLES = 8;
constexpr int SC_SWEEP_BATCH = 128;       // k_self_collision tests shape pairs in batches of 4 rounds x 32 lanes   // sample spheres of one primitive (a box has its 8 corners)
constexpr int MAX_CSLOTS = 8;  // links whose parent is not the role's previous link (R_CSLOT: their index, else -1)
struct DevModel {
  int nl, nb, nd, np, nc, T;
  const int* link_parent;
  const int* link_dof;
  const float* link_E;
  const float* link_r;
  const float* link_axis;
  const int* link_child_start;  // [nl+1]
  const int* link_children;     // [nl-1] ascending link order inside each parent
  const int* link_body_start;   // [nl+1]
  const int* link_bodies;       // [nb] bodies grouped by link
  const int* body_link;
  const float* body_pos;
  const float* body_rot;
  const float* body_inertia;
  const float* dof_lower;
  const float* dof_upper;
  const float* dof_vel_limit;
  const float* dof_effort;
  const float* dof_stiffness;   // [nd] joint spring about q = 0
  const int* link_pt_start;     // [nl+1] penalty points grouped by link
  const int* pt_body;           // [npp]
  const float* pt_pos;          // [npp*3]
  const float* pt_radius;       // [npp]
  const int* link_cyl_start;    // [nl+1]
  const int* cyl_body;
  const float* cyl_center;
  const float* cyl_axis;
  const float* cyl_size;
  const int* sched;             // [T*DYROS_LANES]
  const float* link_reach;      // [nl] bounding radius of the link's penalty candidates about its origin
  // self-collision tables (see DyrosModelDesc), packed for k_self_collision, which stages all of them in shared memory:
  //   pair   [np] link i | link j << 8 | (bit c set: chunk c of `sp` holds shape pairs of this link pair) << 16
  //   lsph   [nl*4] float: bounding sphere of the link's shapes (link frame)
  //   sp     [nq_padded] uint16: shape a | shape b << 8: the shape pairs of every candidate link pair, flattened in the
  //          order of `pair`, cut into at most 16 chunks of sc_chunk pairs (a multiple of SC_SWEEP_BATCH)
  //   shape  [ns*16] float: centre 3, rot 9 (row-major, columns = axes), size 3, bounding radius about the centre
  //   meta   [ns*2] link | body << 8 | kind << 16, first sample | number of samples << 16
  //   sample [nsamp*4] float: position in the link frame, radius
  int sc_ns, sc_nsamp, sc_np, sc_nq, sc_nq_padded, sc_chunk;
  const int* sc_hot;
  int sc_hot_words, sc_o_pair, sc_o_lsph, sc_o_sp, sc_o_shape, sc_o_meta, sc_o_sample;
  const void* blob;             // base of the packed tables; [blob, blob + hot_bytes) is what the kernel stages in smem
  int hot_bytes;
  // word offsets of the hot tables inside the staged prefix (same order as the pointers above)
  int o_parent, o_dof, o_E, o_r, o_axis, o_child_start, o_children, o_body_start, o_bodies, o_body_inertia, o_lower,
      o_upper, o_vel_limit, o_effort, o_pt_start, o_cyl_start, o_sched, o_reach, o_role_of, o_dof_link;
  int o_foot_pts;   // hot: [MAX_FEET][MAX_SOLVER_PTS][4] = candidate position (3) and radius of the solver points
  int o_foot_body;  // hot: [MAX_FEET][MAX_SOLVER_PTS] body index of each candidate
  int base_role, foot_role[MAX_FEET], role_len[DYROS_LANES];
  // flattened role programs: one record of REC_WORDS words per link, base first, then role 0's links in order, ...
  int o_prog, prog_start[DYROS_LANES], chain_rec[MAX_FEET][MAX_CHAIN];
  int lca, shared_len, shared[MAX_CHAIN], shared_rec[MAX_CHAIN];  // base -> common ancestor of the feet (0 = the base itself)
  int n_xchild[DYROS_LANES], xchild[DYROS_LANES][8];  // children of the role's links that live in other roles
  int num_feet;
  int foot_link[MAX_FEET];
  int chain_len[MAX_FEET];
  int chain[MAX_FEET][MAX_CHAIN];      // base child ... foot link
  int foot_npts[MAX_FEET];
  int foot_pt_body[MAX_FEET][MAX_SOLVER_PTS];
  float foot_pt_pos[MAX_FEET][MAX_SOLVER_PTS][3];
  float foot_pt_radius[MAX_FEET][MAX_SOLVER_PTS];
};

// The ground of the physics kernels' role program (physics_roles.cuh), a compile-time parameter: the plane z = 0 with
// normal +z, or a heightfield (DESIGN.md section 4).
struct PlaneGround {
  static constexpr bool kField = false;
};
struct FieldGround {
  static constexpr bool kField = true;
  const int16_t* s;        // (nr, nc) samples, row-major: row i along x, column j along y (device memory)
  int nr, nc;              // >= 2 each
  float ox, oy, oz;        // transform.p
  float dx, dy, dz;        // row_scale, column_scale, vertical_scale
  float zmax;              // height of the highest vertex
  float cull;              // 1 / (smallest n_z of any triangle) >= 1: see link_ext_wrench
};

// The height scan of the observation kernels (DESIGN.md section 4, "Height scan"), a compile-time parameter of
// k_post_fused and k_compute_observations like the ground of the physics kernels: none (rows of NOBS floats), or P
// terrain heights around the base appended to each row.
struct NoScan {
  static constexpr bool kOn = false;
};
struct HeightScan {
  static constexpr bool kOn = true;
  const float2* points;    // (P) x-y in the base's yaw frame (device memory)
  int P;                   // 1..1024
  float base_offset, scale;
  float* measured;         // (N, P) heights in m, or NULL
  int has_field;           // 0: the plane z = 0 (every height 0)
  FieldGround f;           // the sim's heightfield when has_field
};

// The critic's state row (DESIGN.md section 4, "Critic states"), a second compile-time parameter of the same kernels:
// none, or rows of S = NOBS + P + kPrivCols floats written beside the observation rows: the observation row's NOBS
// columns, the P heights of a height scan, then the privileged block.
constexpr int kPrivCols = 31;
struct NoStates {
  static constexpr bool kOn = false;
};
struct CriticStates {
  static constexpr bool kOn = true;
  float* states;           // (N, S) (device memory)
  int S;                   // NOBS + P + kPrivCols
  int priv;                // first column of the privileged block: NOBS + P
  int obs_w;               // columns of the observation row: NOBS, or NOBS + P with the heights in it
  int heights_in_obs;      // the heights go into the observation row as well
  float nominal_mass;      // total_mass / nominal_mass - 1 is column priv + 27
  float mu;                // the sim's friction, for an env without a contact_friction table
};

struct SimParams {
  int N;
  float dt;       // dt / substeps: the integration step of one sub-step
  int substeps;
  float g[3];
  float contact_offset, max_depen_vel, erp, mu, pen_k, pen_c, pen_fmax, max_ang_vel;
  int sweeps, clamp_effort;
  int sc_hits_cap;  // capacity of k_self_collision's hit list (smaller than the array only in tests)
};

// task constants; every derived value is formed in double on the host the way Python forms it, then cast once
struct TaskParams {
  int N, skipframe, perturb, randomize, mocap_rows;
  int mocap_data_num;       // 3599, T:114
  float period;             // float32(3599*0.0005), T:116
  float cycle_dt;           // float32(0.0005), T:115
  float dt;                 // float32(sim dt), T:529
  float dt_policy;          // float32(dt*skipframe), T:540
  float time_gain;          // float32(5*dt_policy), T:541
  float pert_period;        // float32(8/dt_policy), T:495
  float max_len_m1;         // float32(max_episode_length-1), T:594 / VT:325
  float gate_len;           // max_episode_length - 8/dt_policy, T:489
  float death_cost, initial_height;
  float noise_std;          // float32(0.00016/3.0), T:528
  float dr_damping_base, dr_damping_lo, dr_damping_hi, dr_armature_lo, dr_armature_hi;
  float dr_friction_base, dr_friction_lo, dr_friction_hi, dr_pd_gain_lo, dr_pd_gain_hi;
  int lfoot, rfoot, pelvis;
  // integer bounds of the randint draws, formed on the host in double exactly as Python forms them from dt / dt_policy
  int delay_lo, delay_hi;   // 1+int(0.002/dt), 1+round(0.01/dt), T:652
  int timing_hi;            // int(8/dt_policy), T:665
  int dur_lo, dur_hi;       // int(0.1/dt_policy), int(1/dt_policy), T:441
  uint64_t seed;
  // small device tables
  const float* kp;
  const float* kv;
  const float* action_high;
  const float* reset_dof_pos;   // clamp(initial_dof_pos, lower, upper), T:742
  const float* init_dof_pos;
  const float* armature_base;
  uint64_t* step_counter;       // device, Philox epoch; bumped once per step by the cross-env pass
  unsigned long long* tail;     // device [4]: fixed-point sums of the two gate means, CTA ticket of the fused post-physics
                                // launch, sum of the terrain levels (curriculum)
  unsigned* scan_state;         // device [2 + ceil(N/1024)]: tile ticket, tiles finished, per-tile counts of the id compaction
};

struct Sim {
  SimParams p;
  DevModel m;
  DyrosSimBuffers b;
  void* dev_blob = nullptr;  // one allocation holding every model table
  int device = 0;
  int sm_count = 148;
  int program = 0;           // physics program: 0 = one lane per env, warp per role (physics_roles.cuh); 1 = 8 lanes per env (physics_lanes.cuh)
  int envs_per_block = 0;    // physics kernel: envs per CTA
  size_t phys_smem = 0;      // dynamic shared memory of one physics CTA
  bool has_field = false;    // ground: false = the plane z = 0, true = the heightfield `field` (dyros_sim_set_heightfield)
  FieldGround field{};
};

struct Task {
  Sim* sim;
  TaskParams p;
  DyrosTaskBuffers b;
  DyrosNoiseInjection inj;
  DyrosTerrainCurriculum cur{};  // dyros_task_set_terrain_curriculum; levels == NULL: off
  DyrosHeightScan scan{};        // dyros_task_set_height_scan; num_points == 0: off
  DyrosCriticStates crit{};      // dyros_task_set_critic_states; states == NULL: off
  void* dev_blob = nullptr;
  // the heights of a height scan go into the observation row unless critic states take them alone
  int obs_width() const { return NOBS + (!crit.states || crit.heights_in_obs ? scan.num_points : 0); }
  int states_width() const { return NOBS + scan.num_points + kPrivCols; }
};

// launchers (task_kernels.cu)
int launch_prologue(Task* t, const float* actions, cudaStream_t s);
int launch_substep_torque(Task* t, cudaStream_t s);
int launch_sensor_noise(Task* t, int substep, cudaStream_t s);
int launch_epilogue(Task* t, cudaStream_t s);
int launch_check_termination(Task* t, cudaStream_t s);
int launch_compute_reward(Task* t, cudaStream_t s);
int launch_crossenv(Task* t, bool compact, bool gate, bool bump, cudaStream_t s, bool pdl = false);
int launch_reset_idx(Task* t, const int64_t* env_ids, int count, cudaStream_t s);
int launch_compute_observations(Task* t, cudaStream_t s);
int launch_late_update(Task* t, cudaStream_t s);
int launch_post_fused(Task* t, cudaStream_t s, bool pdl = false, bool tail = false);
int launch_pack_results(Task* t, float* dst, cudaStream_t s);  // rows of t->obs_width() floats
// launchers (physics_kernels.cu)
int physics_configure(Sim* sim);  // chooses envs_per_block / shared memory, sets the kernel attributes
int launch_simulate(Sim* sim, int apply_wrench, const float* push_force, cudaStream_t s);
int launch_refresh_rigid_body_state(Sim* sim, cudaStream_t s);
int launch_refresh_dof_force(Sim* sim, float* out, cudaStream_t s);
int configure_physics_aux_kernels();
int launch_fill(void* buf, size_t bytes, int value, cudaStream_t s);
int configure_task_kernels();
int launch_self_collision(Sim* sim, cudaStream_t s, bool pdl = false);
inline bool has_self_collision(const Sim* sim) { return sim->m.sc_np > 0 && sim->b.link_pose && sim->b.self_contact_force; }
int launch_refresh_force_sensors(Sim* sim, const int32_t* sensor_body, const float* sensor_pose, int ns, float* out, cudaStream_t s);
// skipframe x (torque, simulate, sensor noise) in one launch; with `actions` the policy-step prologue runs in it too
int launch_task_physics(Task* t, cudaStream_t s, long long* trace = nullptr, bool pdl = false, const float* actions = nullptr);
int measure_fp32_peak(int device, int iters, double* tflops_out);
int physics_step_threads(const Sim* sim);  // threads of a k_step_physics CTA (role warps + I/O warps)
// the multi-lane variant (physics_lanes_kernels.cu)
int physics_configure_lanes(Sim* sim);
int launch_simulate_lanes(Sim* sim, int apply_wrench, const float* push_force, cudaStream_t s);
int launch_task_physics_lanes(Task* t, cudaStream_t s, long long* trace, bool pdl, const float* actions);
int physics_step_threads_lanes(const Sim* sim);

}  // namespace dyros
