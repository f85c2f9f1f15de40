// Stages of the per-step task logic that run both as their own kernels (task_kernels.cu, one warp per env) and
// inside the fused physics kernel (physics_kernels.cu, DYROS_LANES lanes per env). Arithmetic uses the
// non-contracting intrinsics so that both compilation units (with and without -fmad) produce the same bits,
// and the same float32 results as the reference's op-by-op torch code.
#pragma once
#include "internal.h"

namespace dyros {

struct TK {
  TaskParams p;
  DyrosTaskBuffers b;
  DyrosSimBuffers s;
  DyrosNoiseInjection j;
  DyrosTerrainCurriculum c;  // levels == NULL: no curriculum
};
// (host) the argument of every task kernel and of the fused physics step
inline TK make_tk(const Task* t) {
  TK k;
  k.p = t->p;
  k.b = t->b;
  k.s = t->sim->b;
  k.j = t->inj;
  k.c = t->cur;
  return k;
}

// JU:374-395 with x_dot_0 = x_dot_f = 0.0 (T:458-461), reference operation order. The terms that depend on the knot
// times only (tt^2, tt^3 and the reference's literal 0/tt, 0/tt^2) are computed by cubic_knots once per env: a zero
// numerator sends the IEEE division down its slow path, which is not something to repeat for each of the 35 columns.
struct CubicKnots {
  float t0, tf, tt2, tt3, z1, z2;  // z1 = 0/tt, z2 = 0/tt^2
};
__device__ __forceinline__ CubicKnots cubic_knots(float t0, float tf) {
  float tt = __fsub_rn(tf, t0);
  float tt2 = __fmul_rn(tt, tt);
  // 0/x in IEEE arithmetic is a zero with the sign of x (NaN for x = 0 or NaN): no need to run a division for it
  auto zero_over = [](float x) { return (x == 0.0f || x != x) ? __int_as_float(0x7fffffff) : copysignf(0.0f, x); };
  return CubicKnots{t0, tf, tt2, __fmul_rn(tt2, tt), zero_over(tt), zero_over(tt2)};
}
__device__ __forceinline__ float cubic0(float time, const CubicKnots& kn, float x0, float xf) {
  float e = __fsub_rn(time, kn.t0);
  float tx = __fsub_rn(xf, x0);
  float c = __fadd_rn(x0, __fmul_rn(0.0f, e));
  float a2 = __fsub_rn(__fsub_rn(__fdiv_rn(__fmul_rn(3.0f, tx), kn.tt2), kn.z1), kn.z1);
  c = __fadd_rn(c, __fmul_rn(__fmul_rn(a2, e), e));
  float a3 = __fadd_rn(__fdiv_rn(__fmul_rn(-2.0f, tx), kn.tt3), kn.z2);
  c = __fadd_rn(c, __fmul_rn(__fmul_rn(__fmul_rn(a3, e), e), e));
  float xt = (time > kn.tf) ? xf : x0;
  if (kn.t0 <= time && time <= kn.tf) xt = c;
  return xt;
}

// push schedule of one env (T:489-502, T:438-447): one thread
__device__ __forceinline__ void stage_push_schedule(const TK& k, int e) {
  const TaskParams& P = k.p;
  float fx = 0.f, fy = 0.f;
  if (*k.b.perturb_start) {                                                     // T:492
    int on = k.b.pert_on[e], cnt = k.b.perturbation_count[e], dur = k.b.pert_duration[e];
    float mag = k.b.magnitude[e], ph = k.b.phase[e];
    if (py_fmodf(k.b.epi_len[e], P.pert_period) == (float)k.b.perturb_timing[e]) {  // T:495
      int imp;
      float u;
      if (k.j.pert_i) {
        imp = (int)k.j.pert_i[(size_t)e * 2];
        dur = (int)k.j.pert_i[(size_t)e * 2 + 1];
        u = k.j.pert_f[e];
      } else {
        uint4 r = draw4(P.seed, *P.step_counter, e, kSitePert, 0);
        imp = 50 + (int)(r.x % 200u);                                           // T:440 randint(50,250)
        dur = P.dur_lo + (int)(r.y % (uint32_t)(P.dur_hi - P.dur_lo));          // T:441
        u = u01(r.z);
      }
      on = 1;                                                                   // T:439
      mag = __fdiv_rn((float)imp, __fmul_rn((float)dur, P.dt_policy));          // T:442
      ph = __fmul_rn(__fmul_rn(u, 2.0f), 3.14159265358979f);                    // T:443
      k.b.impulse[e] = imp;
      k.b.pert_duration[e] = dur;
      k.b.magnitude[e] = mag;
      k.b.phase[e] = ph;
    }
    if (on) cnt += 1;                                                           // T:497
    if (on) {                                                                   // T:498-499
      fx = __fmul_rn(mag, cosf(ph));
      fy = __fmul_rn(mag, sinf(ph));
    }
    if (cnt == dur) {                                                           // T:500-501, T:445-447
      on = 0;
      cnt = 0;
    }
    k.b.pert_on[e] = on;
    k.b.perturbation_count[e] = cnt;
  }
  k.b.push_force[(size_t)e * 3 + 0] = fx;
  k.b.push_force[(size_t)e * 3 + 1] = fy;
  k.b.push_force[(size_t)e * 3 + 2] = 0.f;
}

// VT:307 clamp + T:449-468 + push schedule T:489-502, T:438-447; one warp per env. Runs as its own kernel
// (k_prologue) and on the I/O warps of the fused physics kernel.
__device__ __forceinline__ void stage_prologue(const TK& k, const float* __restrict__ actions_in, int e, int lane) {
  const TaskParams& P = k.p;
  float time = k.b.time[e];
  int init = k.b.init_mocap_data_idx[e];
  float local_time = py_fmodf(time, P.period);                                                          // T:450
  float lt_init = py_fmodf(__fadd_rn(local_time, __fmul_rn((float)init, P.cycle_dt)), P.period);        // T:451
  int idx = (int)(((long long)init + (long long)__fdiv_rn(local_time, P.cycle_dt)) % P.mocap_data_num);  // T:452
  if (lane == 0) k.b.mocap_data_idx[e] = idx;
  const float* r0 = k.b.mocap_data + (size_t)idx * 36;
  const float* r1 = r0 + 36;
  const CubicKnots kn = cubic_knots(r0[0], r1[0]);
  for (int c = lane; c < 35; c += 32) {                                           // T:458-461
    float v = cubic0(lt_init, kn, r0[1 + c], r1[1 + c]);
    if (c < ND) k.b.target_data_qpos[(size_t)e * ND + c] = v;
    else k.b.target_data_force[(size_t)e * 2 + (c - ND)] = v;
  }
  if (lane < NA) {
    float a = actions_in[(size_t)e * NA + lane];
    a = (a < -1.0f) ? -1.0f : ((a > 1.0f) ? 1.0f : a);                            // VT:307 (NaN passes through)
    if (lane == NA - 1) a = __fmul_rn((a > 0.0f) ? 1.0f : 0.0f, a);               // T:464-465
    k.b.actions[(size_t)e * NA + lane] = a;
    int head = (k.b.act_hist_head[e] + 1) % NSLOT;                                // T:466 as a ring push
    k.b.action_history[((size_t)e * NSLOT + head) * NA + lane] = a;
    if (lane < 12)                                                                // T:468
      k.b.action_torque[(size_t)e * 12 + lane] =
          __fmul_rn(__fmul_rn(a, k.b.motor_constant_scale[(size_t)e * 12 + lane]), P.action_high[lane]);
    __syncwarp(0x1fffu);
    if (lane == 0) k.b.act_hist_head[e] = head;
  }
  if (lane == 0) stage_push_schedule(k, e);
}

// The same stage for a contiguous slab of envs [e0, e0 + nenv), thread `tid` of `nthreads` cooperating threads. The
// warp-per-env form above is a serial chain of dependent loads per env; here the per-env scalars (phase time, mocap
// row, knot times) are computed once by one thread per env and parked in `pro` (shared memory, 8 words per env), and
// the (env, column) items of the cubic targets and of the action block then need one batch of independent loads each.
// Same arithmetic, same bits. `group_sync` is a barrier of the cooperating threads; `after_env_phase` runs at the end,
// after the push schedule (it stages the push).
constexpr int kSlabMaxEnvs = 32;
template <class GroupSync, class AfterEnvPhase>
__device__ __forceinline__ void stage_prologue_slab(const TK& k, const float* __restrict__ actions_in, int e0, int nenv, int tid,
                                                    int nthreads, float (*pro)[8], GroupSync group_sync,
                                                    AfterEnvPhase after_env_phase) {
  const TaskParams& P = k.p;
  const FastDiv d35(35), dNA(NA);
  constexpr int THREADS = 128;
  constexpr int IT_A = (kSlabMaxEnvs * NA + THREADS - 1) / THREADS;  // action items per thread
  // ---- first round trip: everything that depends on nothing is requested at once: the action block of this thread's
  //      items (VT:307, T:464-468) and, on the per-env threads, the phase time
  float act[IT_A], mcs[IT_A];
  int hd[IT_A];
#pragma unroll
  for (int j = 0; j < IT_A; ++j) {
    int it = tid + j * nthreads;
    it = it < nenv * NA ? it : 0;
    const int le = dNA.div(it), lane = it - le * NA, e = e0 + le;
    act[j] = actions_in[(size_t)e * NA + lane];
    hd[j] = k.b.act_hist_head[e];
    mcs[j] = k.b.motor_constant_scale[(size_t)e * 12 + (lane < 12 ? lane : 0)];
  }
  const bool env_thread = tid < nenv;
  const int ee = e0 + (env_thread ? tid : 0);
  const float time = k.b.time[ee];
  const int init = k.b.init_mocap_data_idx[ee];
  const int head0 = k.b.act_hist_head[ee];
  if (env_thread) {                                                               // T:450-452
    float local_time = py_fmodf(time, P.period);
    float lt_init = py_fmodf(__fadd_rn(local_time, __fmul_rn((float)init, P.cycle_dt)), P.period);
    int idx = (int)(((long long)init + (long long)__fdiv_rn(local_time, P.cycle_dt)) % P.mocap_data_num);
    k.b.mocap_data_idx[ee] = idx;
    // ---- second round trip (per-env threads): the knot times of the mocap row
    const float t0 = k.b.mocap_data[(size_t)idx * 36], tf = k.b.mocap_data[(size_t)(idx + 1) * 36];
    pro[tid][0] = lt_init;
    pro[tid][1] = __int_as_float(idx);
    const CubicKnots kn = cubic_knots(t0, tf);
    pro[tid][2] = kn.t0; pro[tid][3] = kn.tf; pro[tid][4] = kn.tt2; pro[tid][5] = kn.tt3; pro[tid][6] = kn.z1; pro[tid][7] = kn.z2;
  }
#pragma unroll
  for (int j = 0; j < IT_A; ++j) {
    const int it = tid + j * nthreads;
    if (it < nenv * NA) {
      const int le = dNA.div(it), lane = it - le * NA, e = e0 + le;
      float a = act[j];
      a = (a < -1.0f) ? -1.0f : ((a > 1.0f) ? 1.0f : a);
      if (lane == NA - 1) a = __fmul_rn((a > 0.0f) ? 1.0f : 0.0f, a);
      k.b.actions[(size_t)e * NA + lane] = a;
      const int head = (hd[j] + 1) % NSLOT;
      k.b.action_history[((size_t)e * NSLOT + head) * NA + lane] = a;
      if (lane < 12) k.b.action_torque[(size_t)e * 12 + lane] = __fmul_rn(__fmul_rn(a, mcs[j]), P.action_high[lane]);
    }
  }
  group_sync();  // pro[] complete; every action item has read act_hist_head
  if (env_thread) k.b.act_hist_head[ee] = (head0 + 1) % NSLOT;
  // ---- third round trip: the columns of the two mocap rows, B (env, column) items per thread in flight
  constexpr int B = 4;
#pragma unroll 1
  for (int it0 = tid; it0 < nenv * 35; it0 += nthreads * B) {                     // T:458-461
    float x0[B], xf[B];
#pragma unroll
    for (int j = 0; j < B; ++j) {
      int it = it0 + j * nthreads;
      it = it < nenv * 35 ? it : 0;
      const int le = d35.div(it), c = it - le * 35;
      const float* r0 = k.b.mocap_data + (size_t)__float_as_int(pro[le][1]) * 36;
      x0[j] = r0[1 + c];
      xf[j] = r0[36 + 1 + c];
    }
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const int it = it0 + j * nthreads;
      if (it < nenv * 35) {
        const int le = d35.div(it), c = it - le * 35, e = e0 + le;
        const CubicKnots kn{pro[le][2], pro[le][3], pro[le][4], pro[le][5], pro[le][6], pro[le][7]};
        float v = cubic0(pro[le][0], kn, x0[j], xf[j]);
        if (c < ND) k.b.target_data_qpos[(size_t)e * ND + c] = v;
        else k.b.target_data_force[(size_t)e * 2 + (c - ND)] = v;
      }
    }
  }
  // ---- the push schedule (T:489-502) last: nothing in the torque stage depends on it, and the role warps need the
  //      staged push no earlier than the torques
  if (env_thread) stage_push_schedule(k, ee);
  group_sync();
  after_env_phase();
}

// T:505-520: upper-body PD, actuation-delay ring, the 33 torques of set_dof_actuation_force_tensor.
// LANES lanes of one env cooperate; `lane` in [0, LANES). Ends with the lanes in sync.
template <int LANES, class Sync>
__device__ __forceinline__ void stage_substep_torque(const TK& k, int e, int lane, Sync& sync, bool live = true) {
  const float* ds = k.s.dof_state + (size_t)e * ND * 2;
  float* out = k.s.dof_actuation_force + (size_t)e * ND;
  {  // T:506; loads of all iterations are issued before the first use (trip count is a compile-time constant)
    constexpr int IT = (ND - 12 + LANES - 1) / LANES;
    float pos[IT], vel[IT], tgt[IT], kp[IT], kv[IT];
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      int d = 12 + lane + it * LANES;
      int dc = d < ND ? d : ND - 1;
      pos[it] = ds[2 * dc];
      vel[it] = ds[2 * dc + 1];
      tgt[it] = k.b.target_data_qpos[(size_t)e * ND + dc];
      // optional per-env gain scales (DR of the PD gains); a scale of 1 leaves the reference's product unchanged
      kp[it] = k.b.pd_gain_scale ? __fmul_rn(k.p.kp[dc], k.b.pd_gain_scale[(size_t)e * 2]) : k.p.kp[dc];
      kv[it] = k.b.pd_gain_scale ? __fmul_rn(k.p.kv[dc], k.b.pd_gain_scale[(size_t)e * 2 + 1]) : k.p.kv[dc];
    }
#pragma unroll
    for (int it = 0; it < IT; ++it) {
      int d = 12 + lane + it * LANES;
      if (d < ND && live) out[d] = __fadd_rn(__fmul_rn(kp[it], __fsub_rn(tgt[it], pos[it])), __fmul_rn(kv[it], -vel[it]));
    }
  }
  int sl = k.b.simul_len[e] + 1;                                                  // T:513-514
  sl = sl > LOG_DEPTH ? LOG_DEPTH : (sl < 0 ? 0 : sl);
  int dl = k.b.delay_idx[e];
  for (int j = lane; j < 12; j += LANES) {
    float* lg = k.b.action_log + (size_t)e * LOG_DEPTH * 12 + j;
    float v[LOG_DEPTH];
#pragma unroll
    for (int i = 0; i < LOG_DEPTH - 1; ++i) v[i] = lg[(i + 1) * 12];              // T:511
    v[LOG_DEPTH - 1] = k.b.action_torque[(size_t)e * 12 + j];                     // T:512
#pragma unroll
    for (int i = 0; i < LOG_DEPTH; ++i)
      if (live) lg[i * 12] = v[i];
    int pick = (sl > dl) ? dl : (LOG_DEPTH - sl);                                 // T:515-519
    float r = v[0];
#pragma unroll
    for (int i = 1; i < LOG_DEPTH; ++i) r = (pick == i) ? v[i] : r;
    if (live) out[j] = r;                                                         // T:520
  }
  sync();
  if (lane == 0 && live) k.b.simul_len[e] = sl;
}

// T:528-530
template <int LANES>
__device__ __forceinline__ void stage_sensor_noise(const TK& k, int substep, int e, int lane, bool live = true) {
  const float* ds = k.s.dof_state + (size_t)e * ND * 2;
  constexpr int IT = (ND + LANES - 1) / LANES;
  float pos[IT], pre[IT], nz[IT];
  const bool inject = k.j.qpos_normal != nullptr;
  const uint64_t epoch = inject ? 0 : *k.p.step_counter;
#pragma unroll
  for (int it = 0; it < IT; ++it) {  // all loads first
    int d = lane + it * LANES;
    int dc = d < ND ? d : ND - 1;
    pos[it] = ds[2 * dc];
    pre[it] = k.b.qpos_pre[(size_t)e * ND + dc];
    nz[it] = inject ? k.j.qpos_normal[((size_t)substep * k.p.N + e) * ND + dc] : 0.f;
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    int d = lane + it * LANES;
    if (d < ND && live) {
      float n = nz[it];
      if (!inject) {
        uint4 r = draw4(k.p.seed, epoch, e, kSiteQposNoise, substep * 64 + (d >> 1));  // one draw per pair of DOFs
        float2 nn = normal01_pair(r.x, r.y);
        n = __fmul_rn((d & 1) ? nn.y : nn.x, k.p.noise_std);
      }
      n = (n < -0.00016f) ? -0.00016f : ((n > 0.00016f) ? 0.00016f : n);
      float qn = __fadd_rn(pos[it], n);
      size_t i = (size_t)e * ND + d;
      k.b.qvel_noise[i] = __fdiv_rn(__fsub_rn(qn, pre[it]), k.p.dt);
      k.b.qpos_noise[i] = qn;
      k.b.qpos_pre[i] = qn;
    }
  }
}

// ---- CTA-cooperative variants for a contiguous slab of envs [e0, e0 + nenv): thread `tid` of `nthreads`, one
//      element per thread and iteration, so every global access is coalesced; the loads of all iterations are issued
//      before the first use (MAXE bounds the slab). Same arithmetic, same bits as the per-env variants.
//      `tau_sink(le, d, v)` additionally receives every torque (the fused kernel feeds its scratch blocks with it).
struct TorqueSlabArgs {  // the handful of pointers the torque stage touches (passed by value to a non-inlined function)
  const float* dof_state;
  float* dof_actuation_force;
  const float* target_data_qpos;
  const float* kp;
  const float* kv;
  int* simul_len;
  const int* delay_idx;
  float* action_log;
  const float* action_torque;
  const float* pd_gain_scale;  // (N,2) or NULL
};
struct NoiseSlabArgs {
  const float* qpos_normal;  // injected draws or NULL
  float* qpos_pre;
  float* qvel_noise;
  float* qpos_noise;
  const uint64_t* step_counter;
  uint64_t seed;
  float noise_std, dt;
  int N;
};
__device__ __forceinline__ TorqueSlabArgs torque_args(const TK& k) {
  return TorqueSlabArgs{k.s.dof_state, k.s.dof_actuation_force, k.b.target_data_qpos, k.p.kp, k.p.kv, k.b.simul_len,
                        k.b.delay_idx, k.b.action_log, k.b.action_torque, k.b.pd_gain_scale};
}
__device__ __forceinline__ NoiseSlabArgs noise_args(const TK& k) {
  return NoiseSlabArgs{k.j.qpos_normal, k.b.qpos_pre, k.b.qvel_noise, k.b.qpos_noise, k.p.step_counter, k.p.seed,
                       k.p.noise_std, k.p.dt, k.p.N};
}
// `state_of(le, d, which)` supplies the joint angle (which = 0) / velocity (1): global dof_state or the fused kernel's
// scratch blocks.
// Split in two: the part below reads simul_len, stage_simul_len_update (after a barrier of the cooperating threads)
// advances it. `tid` of `nthreads` = 128 VIRTUAL threads: a single warp runs it as four chunks of 32.
template <class Sink, class StateFn>
__device__ __forceinline__ void stage_substep_torque_cta(const TorqueSlabArgs& k, int e0, int nenv, int tid, int nthreads,
                                                         Sink tau_sink, StateFn state_of) {
  constexpr int NU = ND - 12;
  constexpr int THREADS = 128;
  const FastDiv dNU(NU), d12(12);
  constexpr int IT_PD = (kSlabMaxEnvs * NU + THREADS - 1) / THREADS, IT_RG = (kSlabMaxEnvs * 12 + THREADS - 1) / THREADS;
  {
    float pos[IT_PD], vel[IT_PD], tgt[IT_PD], kp[IT_PD], kv[IT_PD];
#pragma unroll
    for (int it = 0; it < IT_PD; ++it) {                                          // T:506, loads
      int idx = tid + it * nthreads;
      idx = idx < nenv * NU ? idx : 0;
      int le = dNU.div(idx), d = 12 + idx - le * NU;
      size_t e = (size_t)(e0 + le);
      pos[it] = state_of(le, d, 0);
      vel[it] = state_of(le, d, 1);
      tgt[it] = k.target_data_qpos[e * ND + d];
      kp[it] = k.pd_gain_scale ? __fmul_rn(k.kp[d], k.pd_gain_scale[e * 2]) : k.kp[d];
      kv[it] = k.pd_gain_scale ? __fmul_rn(k.kv[d], k.pd_gain_scale[e * 2 + 1]) : k.kv[d];
    }
#pragma unroll
    for (int it = 0; it < IT_PD; ++it) {
      int idx = tid + it * nthreads;
      if (idx < nenv * NU) {
        int le = dNU.div(idx), d = 12 + idx - le * NU;
        float t = __fadd_rn(__fmul_rn(kp[it], __fsub_rn(tgt[it], pos[it])), __fmul_rn(kv[it], -vel[it]));
        k.dof_actuation_force[(size_t)(e0 + le) * ND + d] = t;
        tau_sink(le, d, t);
      }
    }
  }
  {
    float v[IT_RG][LOG_DEPTH];
    int sl[IT_RG], dl[IT_RG];
#pragma unroll
    for (int it = 0; it < IT_RG; ++it) {                                          // loads
      int idx = tid + it * nthreads;
      idx = idx < nenv * 12 ? idx : 0;
      int le = d12.div(idx), j = idx - le * 12;
      size_t e = (size_t)(e0 + le);
      sl[it] = k.simul_len[e];
      dl[it] = k.delay_idx[e];
      const float* lg = k.action_log + e * LOG_DEPTH * 12 + j;
#pragma unroll
      for (int i = 0; i < LOG_DEPTH - 1; ++i) v[it][i] = lg[(i + 1) * 12];        // T:511
      v[it][LOG_DEPTH - 1] = k.action_torque[e * 12 + j];                       // T:512
    }
#pragma unroll
    for (int it = 0; it < IT_RG; ++it) {
      int idx = tid + it * nthreads;
      if (idx < nenv * 12) {
        int le = d12.div(idx), j = idx - le * 12;
        size_t e = (size_t)(e0 + le);
        int s1 = sl[it] + 1;                                                      // T:513-514
        s1 = s1 > LOG_DEPTH ? LOG_DEPTH : (s1 < 0 ? 0 : s1);
        float* lg = k.action_log + e * LOG_DEPTH * 12 + j;
#pragma unroll
        for (int i = 0; i < LOG_DEPTH; ++i) lg[i * 12] = v[it][i];
        int pick = (s1 > dl[it]) ? dl[it] : (LOG_DEPTH - s1);                     // T:515-519
        float r = v[it][0];
#pragma unroll
        for (int i = 1; i < LOG_DEPTH; ++i) r = (pick == i) ? v[it][i] : r;
        k.dof_actuation_force[e * ND + j] = r;                                  // T:520
        tau_sink(le, j, r);
      }
    }
  }
}
__device__ __forceinline__ void stage_simul_len_update(const TorqueSlabArgs& k, int e0, int nenv, int tid, int nthreads) {
#pragma unroll 1
  for (int le = tid; le < nenv; le += nthreads) {
    int s1 = k.simul_len[e0 + le] + 1;
    k.simul_len[e0 + le] = s1 > LOG_DEPTH ? LOG_DEPTH : (s1 < 0 ? 0 : s1);
  }
}

// T:528-530 for a slab; `pos_of(le, d)` supplies the fresh joint angle (from shared memory in the fused kernel).
// One thread handles a pair of DOFs (one Philox draw and one Box-Muller transform per pair).
template <class PosFn>
__device__ __forceinline__ void stage_sensor_noise_cta(const NoiseSlabArgs& k, int substep, int e0, int nenv, int tid, int nthreads, PosFn pos_of) {
  constexpr int THREADS = 128;
  constexpr int NP = (ND + 1) / 2;
  constexpr int IT = (kSlabMaxEnvs * NP + THREADS - 1) / THREADS;
  const FastDiv dNP(NP);
  const bool inject = k.qpos_normal != nullptr;
  const uint64_t epoch = inject ? 0 : *k.step_counter;
  float pre[IT][2], nz[IT][2];
#pragma unroll
  for (int it = 0; it < IT; ++it) {  // loads
    int idx = tid + it * nthreads;
    idx = idx < nenv * NP ? idx : 0;
    int le = dNP.div(idx), pr = idx - le * NP;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int d = 2 * pr + h;
      d = d < ND ? d : ND - 1;
      pre[it][h] = k.qpos_pre[(size_t)(e0 + le) * ND + d];
      nz[it][h] = inject ? k.qpos_normal[((size_t)substep * k.N + e0 + le) * ND + d] : 0.f;
    }
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    int idx = tid + it * nthreads;
    if (idx < nenv * NP) {
      int le = dNP.div(idx), pr = idx - le * NP;
      float2 nn = make_float2(0.f, 0.f);
      if (!inject) {
        nn = draw_normal_pair(k.seed, epoch, e0 + le, kSiteQposNoise, substep * 64 + pr);
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        int d = 2 * pr + h;
        if (d < ND) {
          size_t i = (size_t)(e0 + le) * ND + d;
          float n = inject ? nz[it][h] : __fmul_rn(h ? nn.y : nn.x, k.noise_std);
          n = (n < -0.00016f) ? -0.00016f : ((n > 0.00016f) ? 0.00016f : n);
          float qn = __fadd_rn(pos_of(le, d), n);
          k.qvel_noise[i] = __fdiv_rn(__fsub_rn(qn, pre[it][h]), k.dt);
          k.qpos_noise[i] = qn;
          k.qpos_pre[i] = qn;
        }
      }
    }
  }
}

}  // namespace dyros
