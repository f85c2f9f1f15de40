// C ABI of libdyros_b200.so (include/dyros_b200.h): object lifetime, model-table upload, parameter
// derivation and the per-call launch sequences. No kernel lives here.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <new>
#include <string>
#include <vector>

#include "host_model.h"
#include "internal.h"
#include "mesh_grid.h"

namespace dyros {

static thread_local std::string g_error;
void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
}

#define REQUIRE(cond, ...)      \
  do {                          \
    if (!(cond)) {              \
      set_error(__VA_ARGS__);   \
      return 1;                 \
    }                           \
  } while (0)

static int build_sim(const DyrosSimDesc* d, const DyrosModelDesc* m, const DyrosSimBuffers* b, Sim** out) {
  REQUIRE(d && m && b && out, "dyros_sim_create: null argument");
  REQUIRE(d->num_envs > 0, "dyros_sim_create: num_envs must be positive (got %d)", d->num_envs);
  REQUIRE(d->substeps >= 1 && d->dt > 0, "dyros_sim_create: need dt > 0 and substeps >= 1");
  REQUIRE(d->physics_program == 0 || d->physics_program == 1, "dyros_sim_create: physics_program %d (0 = roles, 1 = lanes)", d->physics_program);
  REQUIRE(d->contact_sweeps >= 0 && d->contact_sweeps <= 64, "dyros_sim_create: contact_sweeps %d", d->contact_sweeps);
  REQUIRE(b->root_states && b->dof_state && b->net_contact_force && b->dof_actuation_force && b->dof_damping &&
              b->dof_armature && b->body_mass_scale,
          "dyros_sim_create: a required device buffer is NULL");
  Sim* sim = new (std::nothrow) Sim();
  REQUIRE(sim, "out of host memory");
  sim->device = d->device;
  sim->program = d->physics_program;
  fill_sim_params(d, sim->p);
  sim->desc_mu = sim->p.mu;
  for (int i = 0; i < m->num_points; ++i) sim->max_radius = std::max(sim->max_radius, (float)m->pt_radius[i]);
  sim->b = *b;
  Blob bl;
  ModelOffsets off;
  std::string err = build_model_tables(m, bl, sim->m, off);
  if (!err.empty()) {
    set_error("dyros_sim_create: %s", err.c_str());
    delete sim;
    return 1;
  }
  cudaError_t e = cudaSetDevice(d->device);
  if (e == cudaSuccess) e = cudaMalloc(&sim->dev_blob, bl.host.size());
  if (e == cudaSuccess) e = cudaMemcpy(sim->dev_blob, bl.host.data(), bl.host.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error("dyros_sim_create: CUDA error while uploading the model: %s", cudaGetErrorString(e));
    if (sim->dev_blob) cudaFree(sim->dev_blob);
    delete sim;
    return 1;
  }
  resolve_model(sim->m, off, sim->dev_blob);
  int dev_sms = 0;
  if (cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, d->device) == cudaSuccess && dev_sms > 0)
    sim->sm_count = dev_sms;
  if (physics_configure(sim) || configure_physics_aux_kernels()) {
    cudaFree(sim->dev_blob);
    delete sim;
    return 1;
  }
  *out = sim;
  return 0;
}

static int build_task(Sim* sim, const DyrosTaskDesc* d, const DyrosTaskBuffers* b, Task** out) {
  REQUIRE(sim && d && b && out, "dyros_task_create: null argument");
  REQUIRE(sim->m.nd == ND && sim->m.nb == NB, "dyros_task_create: DyrosDynamicWalk needs %d DOF / %d bodies (model has %d / %d)",
          ND, NB, sim->m.nd, sim->m.nb);
  REQUIRE(d->skipframe >= 1 && d->skipframe <= 8, "dyros_task_create: skipframe %d", d->skipframe);
  REQUIRE(d->kp && d->kv && d->action_high && d->initial_dof_pos, "dyros_task_create: missing gain/limit tables");
  REQUIRE(d->mocap_rows >= 2 && b->mocap_data && b->obs_mean && b->obs_var, "dyros_task_create: missing shared tables");
  // every per-env pointer is required (names: DyrosTaskBuffers)
  const void* req[] = {b->obs_buf, b->rew_buf, b->reset_buf, b->timeout_buf, b->progress_buf, b->randomize_buf,
                       b->stacked_rewards, b->reset_env_ids, b->reset_env_ids32, b->reset_count, b->actions,
                       b->actions_pre, b->time, b->init_mocap_data_idx, b->mocap_data_idx, b->target_data_qpos,
                       b->target_data_force, b->action_torque, b->action_torque_pre, b->motor_constant_scale,
                       b->action_log, b->delay_idx, b->simul_len, b->qpos_noise, b->qvel_noise, b->qpos_pre,
                       b->qpos_bias, b->quat_bias, b->target_vel, b->pre_joint_velocity_states, b->contact_forces_pre,
                       b->total_mass, b->env_origins, b->epi_len, b->epi_len_log, b->contact_reward_sum,
                       b->contact_reward_mean, b->perturbation_count, b->pert_duration, b->pert_on, b->impulse,
                       b->magnitude, b->phase, b->perturb_timing, b->perturb_start, b->push_force, b->obs_history,
                       b->action_history, b->obs_hist_head, b->act_hist_head, b->reset_seq};
  for (size_t i = 0; i < sizeof(req) / sizeof(req[0]); ++i)
    REQUIRE(req[i], "dyros_task_create: DyrosTaskBuffers member #%zu is NULL", i);
  Task* t = new (std::nothrow) Task();
  REQUIRE(t, "out of host memory");
  t->sim = sim;
  t->b = *b;
  memset(&t->inj, 0, sizeof(t->inj));
  TaskParams& p = t->p;
  memset(&p, 0, sizeof(p));
  // Constants are formed in double exactly as the reference's Python forms them, then cast once (SURVEY A1).
  const double dt = (double)sim->p.dt * sim->p.substeps;  // gym.simulate advances sim.dt, T:118
  const double dt_sim = std::round(dt * 1e9) / 1e9;       // undo the float round trip of SimParams.dt (0.002)
  const double dt_policy = dt_sim * d->skipframe;         // T:120
  p.N = sim->p.N;
  p.skipframe = d->skipframe;
  p.perturb = d->perturb;
  p.randomize = d->randomize;
  p.mocap_rows = d->mocap_rows;
  p.mocap_data_num = d->mocap_rows - 1;                         // T:114
  p.cycle_dt = (float)0.0005;                                   // T:115
  p.period = (float)((double)p.mocap_data_num * 0.0005);        // T:116
  p.dt = (float)dt_sim;                                         // T:529
  p.dt_policy = (float)dt_policy;                               // T:540
  p.time_gain = (float)(5 * dt_policy);                         // T:541
  p.pert_period = (float)(8 / dt_policy);                       // T:495
  p.max_len_m1 = (float)((double)d->max_episode_length - 1);    // T:594, VT:325
  p.gate_len = (float)((double)d->max_episode_length - 8 / dt_policy);  // T:489
  p.death_cost = d->death_cost;
  p.initial_height = d->initial_height;
  p.noise_std = (float)(0.00016 / 3.0);                         // T:528
  p.dr_damping_base = d->dr_damping_base;
  p.dr_damping_lo = d->dr_damping_lo;
  p.dr_damping_hi = d->dr_damping_hi;
  p.dr_armature_lo = d->dr_armature_lo;
  p.dr_armature_hi = d->dr_armature_hi;
  p.dr_friction_base = d->dr_friction_base;
  p.dr_friction_lo = d->dr_friction_lo;
  p.dr_friction_hi = d->dr_friction_hi;
  p.dr_pd_gain_lo = d->dr_pd_gain_lo;
  p.dr_pd_gain_hi = d->dr_pd_gain_hi;
  p.lfoot = d->left_foot_body;
  p.rfoot = d->right_foot_body;
  p.pelvis = d->pelvis_body;
  p.seed = d->seed;
  // Python: int() truncates, round() is half-to-even; all on the double dt / dt_policy (never on their float32 casts:
  // float(0.002) = 0.00200000009 would turn int(0.002/dt) into 0)
  p.delay_lo = 1 + (int)(0.002 / dt_sim);                 // T:652
  p.delay_hi = 1 + (int)std::nearbyint(0.01 / dt_sim);    // T:652
  p.timing_hi = (int)(8.0 / dt_policy);                   // T:665
  p.dur_lo = (int)(0.1 / dt_policy);                      // T:441
  p.dur_hi = (int)(1.0 / dt_policy);                      // T:441
  if (!(p.delay_hi == LOG_DEPTH && p.delay_lo >= 0 && p.delay_lo < p.delay_hi && p.timing_hi > 0 && p.dur_lo < p.dur_hi)) {
    set_error("dyros_task_create: dt %.6g / skipframe %d unsupported: the actuation-delay ring is compiled for "
              "round(0.01/dt)+1 == %d (T:166), and the draw ranges of T:441,652,665 must be non-empty", dt_sim,
              d->skipframe, LOG_DEPTH);
    delete t;
    return 1;
  }
  REQUIRE(p.lfoot >= 0 && p.lfoot < NB && p.rfoot >= 0 && p.rfoot < NB && p.pelvis >= 0 && p.pelvis < NB,
          "dyros_task_create: body index out of range");

  std::vector<float> lower(ND), upper(ND), reset_pos(ND), arm(ND, 0.f);
  if (cudaMemcpy(lower.data(), sim->m.dof_lower, ND * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(upper.data(), sim->m.dof_upper, ND * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess) {
    set_error("dyros_task_create: cannot read back dof limits");
    delete t;
    return 1;
  }
  for (int i = 0; i < ND; ++i)  // tensor_clamp(initial_dof_pos, lower, upper): max(min(x, upper), lower), TU:208, T:742
    reset_pos[i] = std::max(std::min(d->initial_dof_pos[i], upper[i]), lower[i]);
  if (d->dr_armature_base)
    for (int i = 0; i < ND; ++i) arm[i] = (float)d->dr_armature_base[i];
  Blob bl;
  size_t o_kp = bl.add_f32(d->kp, ND), o_kv = bl.add_f32(d->kv, ND), o_ah = bl.add_f32(d->action_high, ND);
  size_t o_rp = bl.add_f32(reset_pos.data(), ND), o_ip = bl.add_f32(d->initial_dof_pos, ND), o_ar = bl.add_f32(arm.data(), ND);
  unsigned long long zero = 0;
  size_t o_ct = bl.add(&zero, sizeof(zero));
  unsigned long long zeros4[4] = {0, 0, 0, 0};
  size_t o_tail = bl.add(zeros4, sizeof(zeros4));
  std::vector<unsigned> scan0(2 + (size_t)(sim->p.N + 1023) / 1024, 0u);
  size_t o_scan = bl.add(scan0.data(), scan0.size() * sizeof(unsigned));
  cudaError_t e = cudaMalloc(&t->dev_blob, bl.host.size());
  if (e == cudaSuccess) e = cudaMemcpy(t->dev_blob, bl.host.data(), bl.host.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error("dyros_task_create: CUDA error: %s", cudaGetErrorString(e));
    if (t->dev_blob) cudaFree(t->dev_blob);
    delete t;
    return 1;
  }
  void* base = t->dev_blob;
  p.kp = at<float>(base, o_kp); p.kv = at<float>(base, o_kv); p.action_high = at<float>(base, o_ah);
  p.reset_dof_pos = at<float>(base, o_rp); p.init_dof_pos = at<float>(base, o_ip); p.armature_base = at<float>(base, o_ar);
  p.step_counter = const_cast<uint64_t*>(at<uint64_t>(base, o_ct));
  p.tail = const_cast<unsigned long long*>(at<unsigned long long>(base, o_tail));
  p.scan_state = const_cast<unsigned*>(at<unsigned>(base, o_scan));
  if (configure_task_kernels()) {
    delete t;
    return 1;
  }
  *out = t;
  return 0;
}

}  // namespace dyros

using namespace dyros;

extern "C" {

const char* dyros_last_error(void) { return g_error.c_str(); }
int dyros_abi_version(void) { return DYROS_ABI_VERSION; }

int dyros_sim_create(const DyrosSimDesc* desc, const DyrosModelDesc* model, const DyrosSimBuffers* buf, DyrosSim** out) {
  Sim* s = nullptr;
  int rc = build_sim(desc, model, buf, &s);
  if (rc == 0) *out = reinterpret_cast<DyrosSim*>(s);
  return rc;
}
int dyros_sim_destroy(DyrosSim* sim) {
  Sim* s = reinterpret_cast<Sim*>(sim);
  if (!s) return 0;
  if (s->dev_blob) cudaFree(s->dev_blob);
  if (s->mesh_blob) cudaFree(s->mesh_blob);
  delete s;
  return 0;
}
#define SIM_OR_FAIL(fn)                           \
  Sim* s = reinterpret_cast<Sim*>(sim);           \
  if (!s) {                                       \
    set_error(fn ": sim is NULL");                \
    return 1;                                     \
  }
#define TASK_OR_FAIL(fn)                          \
  Task* t = reinterpret_cast<Task*>(task);        \
  if (!t) {                                       \
    set_error(fn ": task is NULL");               \
    return 1;                                     \
  }

int dyros_simulate(DyrosSim* sim, int apply_wrench, void* stream) {
  SIM_OR_FAIL("dyros_simulate");
  if (apply_wrench && !(s->b.rb_force && s->b.rb_torque)) {
    set_error("dyros_simulate: apply_wrench set but rb_force / rb_torque buffers are NULL");
    return 1;
  }
  if (launch_simulate(s, apply_wrench, nullptr, (cudaStream_t)stream)) return 1;
  return launch_self_collision(s, (cudaStream_t)stream);
}
int dyros_self_collision(DyrosSim* sim, void* stream) {
  SIM_OR_FAIL("dyros_self_collision");
  if (!has_self_collision(s)) {
    set_error("dyros_self_collision: the model has no self-collision tables, or link_pose / self_contact_force is NULL");
    return 1;
  }
  return launch_self_collision(s, (cudaStream_t)stream);
}
int dyros_refresh_rigid_body_state(DyrosSim* sim, void* stream) {
  SIM_OR_FAIL("dyros_refresh_rigid_body_state");
  if (!s->b.rigid_body_state) {
    set_error("dyros_refresh_rigid_body_state: rigid_body_state buffer is NULL");
    return 1;
  }
  return launch_refresh_rigid_body_state(s, (cudaStream_t)stream);
}
int dyros_refresh_dof_force(DyrosSim* sim, float* dof_force, void* stream) {
  SIM_OR_FAIL("dyros_refresh_dof_force");
  if (!dof_force) {
    set_error("dyros_refresh_dof_force: output buffer is NULL");
    return 1;
  }
  return launch_refresh_dof_force(s, dof_force, (cudaStream_t)stream);
}
int dyros_refresh_force_sensors(DyrosSim* sim, const int32_t* sensor_body, const float* sensor_pose, int num_sensors,
                                float* sensor_out, void* stream) {
  SIM_OR_FAIL("dyros_refresh_force_sensors");
  if (!sensor_body || !sensor_pose || !sensor_out || num_sensors < 1) {
    set_error("dyros_refresh_force_sensors: null argument or no sensors");
    return 1;
  }
  if (!s->b.rigid_body_state) {
    set_error("dyros_refresh_force_sensors: the sim was created without a rigid_body_state buffer (sensor frames come from it)");
    return 1;
  }
  if (launch_refresh_rigid_body_state(s, (cudaStream_t)stream)) return 1;
  return launch_refresh_force_sensors(s, sensor_body, sensor_pose, num_sensors, sensor_out, (cudaStream_t)stream);
}
int dyros_set_state_indexed(DyrosSim* sim, const int32_t* env_ids, int count, void* stream) {
  SIM_OR_FAIL("dyros_set_state_indexed");
  (void)stream;
  if (count < 0 || count > s->p.N || (count > 0 && !env_ids)) {
    set_error("dyros_set_state_indexed: count %d outside [0,%d] or NULL ids", count, s->p.N);
    return 1;
  }
  return 0;  // buffers are the live state (immediate CPU-pipeline semantics)
}

int dyros_measure_fp32_peak(int device, int iters, double* tflops_out) {
  if (!tflops_out || iters < 1) {
    set_error("dyros_measure_fp32_peak: bad arguments");
    return 1;
  }
  return measure_fp32_peak(device, iters, tflops_out);
}
int dyros_flush_l2(void* buf, size_t bytes, int value, void* stream) {
  if (!buf || (reinterpret_cast<uintptr_t>(buf) & 15)) {
    set_error("dyros_flush_l2: NULL or unaligned buffer");
    return 1;
  }
  return launch_fill(buf, bytes, value, (cudaStream_t)stream);
}
int dyros_sim_set_l2_persistence(DyrosSim* sim, void* base, size_t bytes, void* stream, size_t* set_aside_out) {
  SIM_OR_FAIL("dyros_sim_set_l2_persistence");
  cudaStream_t st = (cudaStream_t)stream;
  cudaStreamAttrValue attr;
  memset(&attr, 0, sizeof(attr));
  size_t set_aside = 0;
  if (base && bytes) {
    int max_persist = 0, max_window = 0;
    DY_CUDA(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, s->device));
    DY_CUDA(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, s->device));
    if (max_persist <= 0 || max_window <= 0) {
      set_error("dyros_sim_set_l2_persistence: the device has no persisting L2 cache");
      return 1;
    }
    set_aside = std::min(bytes, (size_t)max_persist);
    DY_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside));
    const size_t window = std::min(bytes, (size_t)max_window);
    attr.accessPolicyWindow.base_ptr = base;
    attr.accessPolicyWindow.num_bytes = window;
    // fraction of the window that gets the persisting property: what fits the set-aside part of L2
    attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)set_aside / (double)window);
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  } else {
    attr.accessPolicyWindow.num_bytes = 0;  // window off
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
  }
  DY_CUDA(cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr));
  if (!(base && bytes)) DY_CUDA(cudaCtxResetPersistingL2Cache());
  if (set_aside_out) *set_aside_out = set_aside;
  return 0;
}
int dyros_sim_launch_info(DyrosSim* sim, int32_t out[4]) {
  SIM_OR_FAIL("dyros_sim_launch_info");
  if (!out) {
    set_error("dyros_sim_launch_info: out is NULL");
    return 1;
  }
  out[0] = s->envs_per_block;
  out[1] = (s->p.N + s->envs_per_block - 1) / s->envs_per_block;
  out[2] = physics_step_threads(s);
  out[3] = (int32_t)s->phys_smem;
  return 0;
}

int dyros_sim_set_heightfield(DyrosSim* sim, const DyrosHeightField* f) {
  SIM_OR_FAIL("dyros_sim_set_heightfield");
  if (!f) {
    s->has_field = false;
    s->field = FieldGround{};
    return 0;
  }
  REQUIRE(s->program == 0, "dyros_sim_set_heightfield: the lanes physics program (physics_program 1) has no heightfield "
                           "ground; use the roles program (0)");
  REQUIRE(!s->has_mesh, "dyros_sim_set_heightfield: the sim already has a triangle-mesh ground (one ground per sim)");
  REQUIRE(f->samples, "dyros_sim_set_heightfield: samples is NULL");
  REQUIRE(f->num_rows >= 2 && f->num_columns >= 2, "dyros_sim_set_heightfield: need at least 2 x 2 samples (got %d x %d)",
          f->num_rows, f->num_columns);
  REQUIRE(f->row_scale > 0 && f->column_scale > 0 && f->vertical_scale > 0 && std::isfinite(f->row_scale) &&
              std::isfinite(f->column_scale) && std::isfinite(f->vertical_scale),
          "dyros_sim_set_heightfield: row_scale, column_scale and vertical_scale must be positive");
  REQUIRE(std::isfinite(f->origin[0]) && std::isfinite(f->origin[1]) && std::isfinite(f->origin[2]),
          "dyros_sim_set_heightfield: origin must be finite");
  // highest vertex and steepest triangle (for the conservative per-link reach cull), from a host copy of the samples
  const size_t n = (size_t)f->num_rows * f->num_columns;
  std::vector<int16_t> h(n);
  DY_CUDA(cudaSetDevice(s->device));
  DY_CUDA(cudaMemcpy(h.data(), f->samples, n * sizeof(int16_t), cudaMemcpyDeviceToHost));
  const double dz = f->vertical_scale;
  double top = -1e300, gmax = 0;
  for (size_t k = 0; k < n; ++k) top = std::max(top, dz * h[k]);
  for (int i = 0; i + 1 < f->num_rows; ++i)
    for (int j = 0; j + 1 < f->num_columns; ++j) {
      const size_t c = (size_t)i * f->num_columns + j;
      const double h00 = dz * h[c], h10 = dz * h[c + f->num_columns], h01 = dz * h[c + 1], h11 = dz * h[c + f->num_columns + 1];
      for (int t = 0; t < 2; ++t) {  // the two triangles of the cell (physics_roles.cuh field_query)
        const double sx = (t == 0 ? h10 - h00 : h11 - h01) / f->row_scale, sy = (t == 0 ? h11 - h10 : h01 - h00) / f->column_scale;
        gmax = std::max(gmax, sx * sx + sy * sy);
      }
    }
  FieldGround g{};
  g.s = f->samples;
  g.nr = f->num_rows;
  g.nc = f->num_columns;
  g.ox = f->origin[0];
  g.oy = f->origin[1];
  g.oz = f->origin[2];
  g.dx = f->row_scale;
  g.dy = f->column_scale;
  g.dz = f->vertical_scale;
  g.zmax = (float)(f->origin[2] + top) + 1e-4f;                     // (rounded up: the cull stays conservative)
  g.cull = (float)std::sqrt(1 + gmax) * (1 + 1e-5f);                 // 1 / smallest n_z
  s->has_field = true;  // (same launch geometry as the plane: the env scratch block is the same size)
  s->field = g;
  return 0;
}

static void free_mesh(Sim* s) {
  if (s->mesh_blob) cudaFree(s->mesh_blob);
  s->mesh_blob = nullptr;
  s->has_mesh = false;
  s->mesh = MeshGround{};
  s->mesh_bytes = 0;
  s->mesh_dropped = 0;
  s->mesh_kept = 0;
  s->p.mu = s->desc_mu;
}

// Copies the mesh and builds its bucket grid (mesh_grid.h), then uploads both in one allocation.
int dyros_sim_set_triangle_mesh(DyrosSim* sim, const DyrosTriangleMesh* mesh) {
  SIM_OR_FAIL("dyros_sim_set_triangle_mesh");
  if (!mesh) {
    DY_CUDA(cudaSetDevice(s->device));
    free_mesh(s);
    return 0;
  }
  REQUIRE(s->program == 0, "dyros_sim_set_triangle_mesh: the lanes physics program (physics_program 1) has no "
                           "triangle-mesh ground; use the roles program (0)");
  REQUIRE(!s->has_field, "dyros_sim_set_triangle_mesh: the sim already has a heightfield ground (one ground per sim)");
  MeshGrid mg;
  const std::string err = build_mesh_grid(mesh, (double)s->p.contact_offset + s->max_radius + kMeshDepthAllowance, mg);
  REQUIRE(err.empty(), "dyros_sim_set_triangle_mesh: %s", err.c_str());
  const size_t b_tri = mg.tri.size() * sizeof(float4), b_cell = mg.cell.size() * sizeof(int4), b_list = mg.list.size() * sizeof(int);
  DY_CUDA(cudaSetDevice(s->device));
  free_mesh(s);
  void* blob = nullptr;
  DY_CUDA(cudaMalloc(&blob, b_tri + b_cell + b_list));
  char* base = static_cast<char*>(blob);
  cudaError_t e = cudaMemcpy(base, mg.tri.data(), b_tri, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(base + b_tri, mg.cell.data(), b_cell, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && b_list) e = cudaMemcpy(base + b_tri + b_cell, mg.list.data(), b_list, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(blob);
    set_error("dyros_sim_set_triangle_mesh: CUDA error while uploading the mesh: %s", cudaGetErrorString(e));
    return 1;
  }
  MeshGround g = mg.g;
  g.tri = reinterpret_cast<const float4*>(base);
  g.cell = reinterpret_cast<const int4*>(base + b_tri);
  g.list = reinterpret_cast<const int*>(base + b_tri + b_cell);
  s->mesh_blob = blob;
  s->mesh_bytes = b_tri + b_cell + b_list;
  s->mesh_dropped = mg.dropped;
  s->mesh_kept = mg.kept;
  s->mesh = g;
  s->has_mesh = true;  // (same launch geometry as the plane: the env scratch block is the same size)
  s->p.mu = mesh->dynamic_friction;
  return 0;
}
int dyros_sim_triangle_mesh_info(DyrosSim* sim, int64_t out[4]) {
  SIM_OR_FAIL("dyros_sim_triangle_mesh_info");
  REQUIRE(out, "dyros_sim_triangle_mesh_info: out is NULL");
  out[0] = (int64_t)s->mesh_bytes;
  out[1] = s->mesh_dropped;
  out[2] = s->mesh_kept;
  out[3] = s->has_mesh ? (int64_t)s->mesh.gx * s->mesh.gy : 0;
  return 0;
}

int dyros_task_create(DyrosSim* sim, const DyrosTaskDesc* desc, const DyrosTaskBuffers* buf, DyrosTask** out) {
  Task* t = nullptr;
  int rc = build_task(reinterpret_cast<Sim*>(sim), desc, buf, &t);
  if (rc == 0) *out = reinterpret_cast<DyrosTask*>(t);
  return rc;
}
int dyros_task_destroy(DyrosTask* task) {
  Task* t = reinterpret_cast<Task*>(task);
  if (!t) return 0;
  if (t->dev_blob) cudaFree(t->dev_blob);
  delete t;
  return 0;
}
int dyros_task_set_noise_injection(DyrosTask* task, const DyrosNoiseInjection* inj) {
  TASK_OR_FAIL("dyros_task_set_noise_injection");
  if (inj) t->inj = *inj;
  else memset(&t->inj, 0, sizeof(t->inj));
  if ((t->inj.pert_i != nullptr) != (t->inj.pert_f != nullptr)) {
    set_error("dyros_task_set_noise_injection: pert_i and pert_f must be given together");
    memset(&t->inj, 0, sizeof(t->inj));
    return 1;
  }
  return 0;
}
int dyros_task_set_terrain_curriculum(DyrosTask* task, const DyrosTerrainCurriculum* c) {
  TASK_OR_FAIL("dyros_task_set_terrain_curriculum");
  if (!c) {
    t->cur = DyrosTerrainCurriculum{};
    return 0;
  }
  REQUIRE(c->origins && c->levels && c->types, "dyros_task_set_terrain_curriculum: origins, levels and types must be given");
  REQUIRE(c->num_levels >= 1 && c->num_types >= 1, "dyros_task_set_terrain_curriculum: need num_levels >= 1 and num_types >= 1 "
          "(got %d, %d)", c->num_levels, c->num_types);
  REQUIRE(std::isfinite(c->move_up_distance) && c->move_up_distance >= 0 && std::isfinite(c->move_down_scale) &&
              c->move_down_scale >= 0,
          "dyros_task_set_terrain_curriculum: move_up_distance and move_down_scale must be finite and >= 0");
  // the kernel indexes origins with levels / types: check them once here, from host copies
  const int N = t->p.N;
  const size_t no = (size_t)c->num_levels * c->num_types * 3;
  std::vector<int32_t> lv(N), ty(N);
  std::vector<float> org(no);
  DY_CUDA(cudaSetDevice(t->sim->device));
  DY_CUDA(cudaMemcpy(lv.data(), c->levels, N * sizeof(int32_t), cudaMemcpyDeviceToHost));
  DY_CUDA(cudaMemcpy(ty.data(), c->types, N * sizeof(int32_t), cudaMemcpyDeviceToHost));
  DY_CUDA(cudaMemcpy(org.data(), c->origins, no * sizeof(float), cudaMemcpyDeviceToHost));
  for (int e = 0; e < N; ++e) {
    REQUIRE(lv[e] >= 0 && lv[e] < c->num_levels, "dyros_task_set_terrain_curriculum: level %d of env %d outside [0, %d)",
            lv[e], e, c->num_levels);
    REQUIRE(ty[e] >= 0 && ty[e] < c->num_types, "dyros_task_set_terrain_curriculum: type %d of env %d outside [0, %d)",
            ty[e], e, c->num_types);
  }
  for (size_t i = 0; i < no; ++i)
    REQUIRE(std::isfinite(org[i]), "dyros_task_set_terrain_curriculum: origins must be finite");
  t->cur = *c;
  return 0;
}
int dyros_task_set_height_scan(DyrosTask* task, const DyrosHeightScan* sc) {
  TASK_OR_FAIL("dyros_task_set_height_scan");
  if (!sc) {
    t->scan = DyrosHeightScan{};
    t->scan_own_field = false;
    return 0;
  }
  REQUIRE(sc->points && (reinterpret_cast<uintptr_t>(sc->points) & 7) == 0,
          "dyros_task_set_height_scan: points is NULL or not 8-byte aligned");
  REQUIRE(sc->num_points >= 1 && sc->num_points <= 1024, "dyros_task_set_height_scan: num_points %d outside [1, 1024]",
          sc->num_points);
  REQUIRE(std::isfinite(sc->base_offset) && std::isfinite(sc->scale),
          "dyros_task_set_height_scan: base_offset and scale must be finite");
  std::vector<float> pts((size_t)sc->num_points * 2);
  DY_CUDA(cudaSetDevice(t->sim->device));
  DY_CUDA(cudaMemcpy(pts.data(), sc->points, pts.size() * sizeof(float), cudaMemcpyDeviceToHost));
  for (float v : pts) REQUIRE(std::isfinite(v), "dyros_task_set_height_scan: points must be finite");
  FieldGround g{};
  if (const DyrosHeightField* f = sc->field) {
    REQUIRE(f->samples && f->num_rows >= 2 && f->num_columns >= 2,
            "dyros_task_set_height_scan: field needs samples of at least 2 x 2");
    REQUIRE(f->row_scale > 0 && f->column_scale > 0 && f->vertical_scale > 0 && std::isfinite(f->row_scale) &&
                std::isfinite(f->column_scale) && std::isfinite(f->vertical_scale) && std::isfinite(f->origin[0]) &&
                std::isfinite(f->origin[1]) && std::isfinite(f->origin[2]),
            "dyros_task_set_height_scan: field scales must be positive and its origin finite");
    g.s = f->samples;
    g.nr = f->num_rows;
    g.nc = f->num_columns;
    g.ox = f->origin[0];
    g.oy = f->origin[1];
    g.oz = f->origin[2];
    g.dx = f->row_scale;
    g.dy = f->column_scale;
    g.dz = f->vertical_scale;
  }
  t->scan = *sc;
  t->scan.field = nullptr;  // (copied into scan_field: the caller's struct need not outlive this call)
  t->scan_own_field = sc->field != nullptr;
  t->scan_field = g;
  return 0;
}
int dyros_task_set_critic_states(DyrosTask* task, const DyrosCriticStates* cs) {
  TASK_OR_FAIL("dyros_task_set_critic_states");
  if (!cs || !cs->states) {
    t->crit = DyrosCriticStates{};
    return 0;
  }
  REQUIRE((reinterpret_cast<uintptr_t>(cs->states) & 3) == 0, "dyros_task_set_critic_states: states is not 4-byte aligned");
  REQUIRE(std::isfinite(cs->nominal_mass) && cs->nominal_mass > 0.f,
          "dyros_task_set_critic_states: nominal_mass must be finite and positive (got %g)", (double)cs->nominal_mass);
  t->crit = *cs;
  return 0;
}
int dyros_task_prologue(DyrosTask* task, const float* actions, void* stream) {
  TASK_OR_FAIL("dyros_task_prologue");
  if (!actions) {
    set_error("dyros_task_prologue: actions is NULL");
    return 1;
  }
  return launch_prologue(t, actions, (cudaStream_t)stream);
}
int dyros_task_physics(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_physics");
  if (launch_task_physics(t, (cudaStream_t)stream)) return 1;
  return launch_self_collision(t->sim, (cudaStream_t)stream);
}
int dyros_task_physics_kernel(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_physics_kernel");
  return launch_task_physics(t, (cudaStream_t)stream);
}
int dyros_task_physics_trace(DyrosTask* task, int64_t* trace, void* stream) {
  TASK_OR_FAIL("dyros_task_physics_trace");
  if (!trace) {
    set_error("dyros_task_physics_trace: trace buffer is NULL");
    return 1;
  }
  if (launch_task_physics(t, (cudaStream_t)stream, reinterpret_cast<long long*>(trace))) return 1;
  return launch_self_collision(t->sim, (cudaStream_t)stream);
}
int dyros_task_prologue_physics(DyrosTask* task, const float* actions, int64_t* trace, void* stream) {
  TASK_OR_FAIL("dyros_task_prologue_physics");
  if (!actions) {
    set_error("dyros_task_prologue_physics: actions is NULL");
    return 1;
  }
  if (launch_task_physics(t, (cudaStream_t)stream, reinterpret_cast<long long*>(trace), false, actions)) return 1;
  return launch_self_collision(t->sim, (cudaStream_t)stream);
}
int dyros_task_substep_torque(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_substep_torque");
  return launch_substep_torque(t, (cudaStream_t)stream);
}
int dyros_task_sensor_noise(DyrosTask* task, int substep, void* stream) {
  TASK_OR_FAIL("dyros_task_sensor_noise");
  if (substep < 0 || substep >= t->p.skipframe) {
    set_error("dyros_task_sensor_noise: substep %d outside [0,%d)", substep, t->p.skipframe);
    return 1;
  }
  return launch_sensor_noise(t, substep, (cudaStream_t)stream);
}
int dyros_task_epilogue(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_epilogue");
  return launch_epilogue(t, (cudaStream_t)stream);
}
int dyros_task_check_termination(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_check_termination");
  return launch_check_termination(t, (cudaStream_t)stream);
}
int dyros_task_compute_reward(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_compute_reward");
  return launch_compute_reward(t, (cudaStream_t)stream);
}
int dyros_task_compact_resets(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_compact_resets");
  return launch_crossenv(t, true, false, false, (cudaStream_t)stream);
}
int dyros_task_reset_idx(DyrosTask* task, const int64_t* env_ids, int count, void* stream) {
  TASK_OR_FAIL("dyros_task_reset_idx");
  if (env_ids && (count < 0 || count > t->p.N)) {
    set_error("dyros_task_reset_idx: count %d outside [0,%d]", count, t->p.N);
    return 1;
  }
  return launch_reset_idx(t, env_ids, env_ids ? count : -1, (cudaStream_t)stream);
}
int dyros_task_compute_observations(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_compute_observations");
  return launch_compute_observations(t, (cudaStream_t)stream);
}
int dyros_task_late_update(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_late_update");
  return launch_late_update(t, (cudaStream_t)stream);
}
int dyros_task_end_step(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_end_step");
  return launch_crossenv(t, false, true, true, (cudaStream_t)stream);
}

int dyros_task_step(DyrosTask* task, const float* actions, void* stream) {
  TASK_OR_FAIL("dyros_task_step");
  if (!actions) {
    set_error("dyros_task_step: actions is NULL");
    return 1;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // the kernels use programmatic dependent launch: their CTAs get resident and run their preamble while the previous
  // kernel drains (common.cuh); the data dependency is enforced by griddepcontrol.wait inside each kernel
  if (launch_task_physics(t, st, nullptr, true, actions)) return 1;  // prologue folded into the physics launch
  if (launch_self_collision(t->sim, st, true)) return 1;             // (no launch unless the model carries the tables)
  // ... and the cross-env pass (gate of T:489, Philox epoch) into the post-physics launch: its last CTA does it. The
  // compacted id list of T:554 is not needed by the fused step (every env resets itself): dyros_task_compact_resets
  // produces it on demand.
  return launch_post_fused(t, st, true, true);
}
int dyros_task_post_step(DyrosTask* task, void* stream) {
  TASK_OR_FAIL("dyros_task_post_step");
  return launch_post_fused(t, (cudaStream_t)stream, true, true);
}
int dyros_task_step_launches(DyrosTask* task) {
  TASK_OR_FAIL("dyros_task_step_launches");
  return has_self_collision(t->sim) ? 3 : 2;  // prologue + fused physics, [self-collision], fused post-physics (+ cross-env pass)
}
int dyros_task_set_obs_buf(DyrosTask* task, float* obs_buf) {
  TASK_OR_FAIL("dyros_task_set_obs_buf");
  if (!obs_buf || (reinterpret_cast<uintptr_t>(obs_buf) & 15)) {
    set_error("dyros_task_set_obs_buf: obs_buf is NULL or not 16-byte aligned");
    return 1;
  }
  t->b.obs_buf = obs_buf;
  return 0;
}
int dyros_task_pack_results(DyrosTask* task, void* dst, void* stream) {
  TASK_OR_FAIL("dyros_task_pack_results");
  if (!dst || (reinterpret_cast<uintptr_t>(dst) & 15)) {
    set_error("dyros_task_pack_results: dst is NULL or not 16-byte aligned");
    return 1;
  }
  return launch_pack_results(t, static_cast<float*>(dst), (cudaStream_t)stream);
}

}  // extern "C"
