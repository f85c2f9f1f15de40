// K2/K3/K4: the bodies of DyrosDynamicWalk's per-step methods as sm_100a kernels (one warp per env).
//
// Compiled with -fmad=false: the reference computes every float32 op separately (CPU torch / op-by-op
// ATen), and parity is judged at 1e-5 relative with bit-exact masks, so no FMA contraction here.
// Citations: T = tasks/dyros_dynamic_walk.py, VT = tasks/base/vec_task.py, JU = utils/torch_jit_utils.py,
// TU = isaacgym/torch_utils.py (all under the reference's python/ tree).
#include "task_stages.cuh"

namespace dyros {

constexpr int kWarpsPerBlock = 8;

// ------------------------------------------------------------------ small math (TU / JU restated)
// JU:142-160 with a = identity: |vec(a (x) conj(q))| through the TU:20-40 product, then 2*asin(min(.,1))
__device__ __forceinline__ float quat_err_identity(const float* q) {
  float x2 = -q[0], y2 = -q[1], z2 = -q[2], w2 = q[3];
  const float x1 = 0.f, y1 = 0.f, z1 = 0.f, w1 = 1.f;
  float ww = (z1 + x1) * (x2 + y2);
  float yy = (w1 - y1) * (w2 + z2);
  float zz = (w1 + y1) * (w2 - z2);
  float xx = ww + yy + zz;
  float qq = 0.5f * (xx + (z1 - x1) * (x2 - y2));
  float x = qq - xx + (x1 + w1) * (x2 + w2);
  float y = qq - yy + (w1 - x1) * (y2 + z2);
  float z = qq - zz + (z1 + y1) * (w2 - x2);
  float n = sqrtf(x * x + y * y + z * z);
  return 2.0f * asinf(fminf(n, 1.0f));
}

// TU:228-273 quat2euler (xyzw) -> component `which` (0:x 1:y 2:z)
__device__ __forceinline__ float quat2euler_comp(const float* q, int which) {
  float w = q[3], x = q[0], y = q[1], z = q[2];
  float m00 = w * w + x * x - y * y - z * z;
  float m01 = 2.f * x * y - 2.f * w * z;
  float m10 = 2.f * x * y + 2.f * w * z;
  float m11 = w * w - x * x + y * y - z * z;
  float m20 = 2.f * x * z - 2.f * w * y;
  float m21 = 2.f * y * z + 2.f * w * x;
  float m22 = w * w - x * x - y * y + z * z;
  float cy = sqrtf(m00 * m00 + m10 * m10);
  bool cond = cy > (float)(2.220446049250313e-16 * 4);
  // one atan2f for whichever component the lane wants (lanes with different `which` do not diverge):
  // 2: cond ? atan2(m10, m00) : atan2(-m01, m11); 1: atan2(-m20, cy); 0: cond ? atan2(m21, m22) : 0 (= atan2(0, 1))
  float ay = which == 2 ? (cond ? m10 : -m01) : (which == 1 ? -m20 : (cond ? m21 : 0.0f));
  float ax = which == 2 ? (cond ? m00 : m11) : (which == 1 ? cy : (cond ? m22 : 1.0f));
  return atan2f(ay, ax);
}

__device__ __forceinline__ bool collision_true(const TK& k, int e, int lane) {
  // T:590 / T:937: any non-foot body with |F| > 1
  bool hit = false;
  for (int b = lane; b < NB; b += kWarp) {
    if (b == k.p.lfoot || b == k.p.rfoot) continue;
    const float* f = k.s.net_contact_force + ((size_t)e * NB + b) * 3;
    float n = sqrtf(f[0] * f[0] + f[1] * f[1] + f[2] * f[2]);
    hit |= n > 1.0f;
  }
  return __any_sync(kFull, hit);
}

// ------------------------------------------------------------------ stages (device functions, one warp per env)
struct WarpSyncT {
  __device__ __forceinline__ void operator()() const { __syncwarp(); }
};

// T:532-541, VT:325, T:544-545
__device__ void stage_epilogue(const TK& k, int e, int lane) {
  if (lane != 0) return;
  k.b.epi_len[e] = k.b.epi_len[e] + 1.0f;
  float t = k.b.time[e] + k.p.dt_policy;
  t = t + k.p.time_gain * k.b.actions[(size_t)e * NA + NA - 1];
  k.b.time[e] = t;
  long long pr = k.b.progress_buf[e];
  k.b.timeout_buf[e] = ((float)pr >= k.p.max_len_m1) ? 1 : 0;
  k.b.progress_buf[e] = pr + 1;
  k.b.randomize_buf[e] = k.b.randomize_buf[e] + 1;
}

// T:581-596 ; returns the reset flag (warp-uniform)
// `shared` (fused kernel): hands the collision flag and the orientation error on to the reward stage, which needs
// the same two quantities of the same (pre-reset) state.
struct TermShared {
  bool col;
  float qe;
};
__device__ int stage_check_termination(const TK& k, int e, int lane, TermShared* shared = nullptr) {
  float qe = quat_err_identity(k.s.root_states + (size_t)e * 13 + 3);
  int reset = (fabsf(qe) > 0.5f) ? 1 : 0;
  if ((float)k.b.progress_buf[e] >= k.p.max_len_m1) reset = 1;
  const bool col = collision_true(k, e, lane);
  if (shared) {
    shared->col = col;
    shared->qe = qe;
  }
  if (col) reset = 1;
  if (lane == 0) k.b.reset_buf[e] = reset;
  return reset;
}

// T:387-428 + T:802-947, in two parts: the warp-wide reductions over the joints, and the scalar terms (one thread per
// env: the fused kernel runs them for all envs of a CTA side by side in one warp instead of on lane 0 of each).
struct RewardSums {
  float s_qpos, s_qvel, s_qacc, s_tq, s_tqd, qe;
  bool col;
};
__device__ RewardSums reward_sums(const TK& k, int e, int lane, const TermShared* shared = nullptr) {
  const float* root = k.s.root_states + (size_t)e * 13;
  const float* ds = k.s.dof_state + (size_t)e * ND * 2;
  float s_qpos = 0.f, s_qvel = 0.f, s_qacc = 0.f, s_tq = 0.f, s_tqd = 0.f;
  for (int d = lane; d < ND; d += kWarp) {
    float pos = ds[2 * d], vel = ds[2 * d + 1];
    float a = k.b.target_data_qpos[(size_t)e * ND + d] - pos;
    float b = 0.0f - vel;
    float c = vel - k.b.pre_joint_velocity_states[(size_t)e * ND + d];
    s_qpos += a * a;
    s_qvel += b * b;
    s_qacc += c * c;
  }
  if (lane < 12) {
    float a = k.b.actions[(size_t)e * NA + lane], ap = k.b.actions_pre[(size_t)e * NA + lane];
    float t = a * 333.0f, td = (a - ap) * 333.0f;
    s_tq = t * t;
    s_tqd = td * td;
  }
  RewardSums o;
  o.s_qpos = warp_sum(s_qpos);
  o.s_qvel = warp_sum(s_qvel);
  o.s_qacc = warp_sum(s_qacc);
  o.s_tq = warp_sum(s_tq);
  o.s_tqd = warp_sum(s_tqd);
  o.col = shared ? shared->col : collision_true(k, e, lane);
  o.qe = shared ? shared->qe : quat_err_identity(root + 3);
  return o;
}
__device__ void reward_scalar(const TK& k, int e, const RewardSums& in) {
  const float* root = k.s.root_states + (size_t)e * 13;
  const float s_qpos = in.s_qpos, s_qvel = in.s_qvel, s_qacc = in.s_qacc, s_tq = in.s_tq, s_tqd = in.s_tqd, qe = in.qe;
  const bool col = in.col;
  float r[14];
  r[0] = 0.3f * expf(-13.2f * fabsf(qe));                                          // T:835
  float n;
  n = sqrtf(s_qpos); r[1] = 0.35f * expf(-2.0f * (n * n));                         // T:837
  n = sqrtf(s_qvel); r[2] = 0.05f * expf(-0.01f * (n * n));                        // T:839
  const float* F = k.s.net_contact_force + (size_t)e * NB * 3;
  const float* Fp = k.b.contact_forces_pre + (size_t)e * NB * 3;
  const float *lf = F + k.p.lfoot * 3, *rf = F + k.p.rfoot * 3, *lfp = Fp + k.p.lfoot * 3, *rfp = Fp + k.p.rfoot * 3;
  float dl0 = lf[0] - lfp[0], dl1 = lf[1] - lfp[1], dl2 = lf[2] - lfp[2];
  float dr0 = rf[0] - rfp[0], dr1 = rf[1] - rfp[1], dr2 = rf[2] - rfp[2];
  r[9] = 0.2f * expf(-0.01f * (sqrtf(dl0 * dl0 + dl1 * dl1 + dl2 * dl2) + sqrtf(dr0 * dr0 + dr1 * dr1 + dr2 * dr2)));  // T:858
  r[4] = 0.05f * expf(-0.01f * sqrtf(s_tq));                                        // T:861
  r[5] = 0.6f * expf(-0.01f * sqrtf(s_tqd));                                        // T:863
  n = sqrtf(s_qacc); r[7] = 0.05f * expf(-20.0f * (n * n));                        // T:865
  float vx = k.b.target_vel[(size_t)e * 2] - root[7], vy = k.b.target_vel[(size_t)e * 2 + 1] - root[8];
  n = sqrtf(vx * vx + vy * vy); r[6] = 0.3f * expf(-3.0f * (n * n));               // T:867
  bool lc = lf[2] > 1.0f, rc = rf[2] > 1.0f;                                       // T:869-870
  int idx = k.b.mocap_data_idx[e];
  bool DSP = ((3300 <= idx) && (idx < 3600)) || (idx < 300) || ((1500 <= idx) && (idx < 2100));
  bool RSSP = (300 <= idx) && (idx < 1500);
  bool LSSP = (2100 <= idx) && (idx < 3300);
  bool sync = (DSP && rc && lc) || (RSSP && rc && !lc) || (LSSP && !rc && lc);     // T:882-889
  r[8] = sync ? 0.2f : 0.0f;
  k.b.contact_reward_sum[e] = k.b.contact_reward_sum[e] + r[8];                    // T:891
  r[10] = 0.0f;                                                                    // T:893
  float m = k.b.total_mass[e];
  float thr = (float)(1.4 * 9.81) * m;                                             // T:895
  bool thres = (lf[2] > thr) || (rf[2] > thr);
  r[11] = thres ? -0.2f : 0.0f;                                                    // T:898
  float cl = fmaxf(lf[2] - thr, 0.0f), cr = fmaxf(rf[2] - thr, 0.0f);
  float pen = 0.1f * expf(-0.007f * (sqrtf(cl * cl) + sqrtf(cr * cr)));            // T:900-901
  r[3] = thres ? pen : 0.1f;                                                       // T:902
  float dthr = (float)(0.2 * 9.81) * m / 1.0f;                                     // T:904
  bool tdiff = (fabsf(lf[2] - lfp[2]) > dthr) || (fabsf(rf[2] - rfp[2]) > dthr);
  r[12] = tdiff ? -0.05f : 0.0f;                                                   // T:907
  float ws = m / 104.48f;                                                          // T:917
  const float* ft = k.b.target_data_force + (size_t)e * 2;
  r[13] = 0.1f * expf(-0.001f * fabsf(lf[2] + ws * ft[0])) + 0.1f * expf(-0.001f * fabsf(rf[2] + ws * ft[1]));  // T:918-919
  float total = r[0] + r[1] + r[2] + r[3] + r[4] + r[5] + r[6] + r[7] + r[8] + r[9] + r[10] + r[11] + r[12] + r[13];  // T:932-934
  if (col) total = k.p.death_cost;                                                 // T:942
  if (fabsf(qe) > 0.5f) total = k.p.death_cost;                                    // T:943
  k.b.rew_buf[e] = total;
  float* st = k.b.stacked_rewards + (size_t)e * 15;
#pragma unroll
  for (int i = 0; i < 14; ++i) st[i] = col ? k.p.death_cost : r[i];                // T:945
  st[14] = (*k.b.perturb_start) ? 1.0f : 0.0f;                                     // T:415
}
__device__ void stage_compute_reward(const TK& k, int e, int lane, const TermShared* shared = nullptr) {
  RewardSums sums = reward_sums(k, e, lane, shared);
  if (lane == 0) reward_scalar(k, e, sums);
}

// Terrain curriculum of one resetting env (legged_gym _update_terrain_curriculum; DESIGN.md section 4, "Curriculum"),
// one thread: the new level from the root and the target_vel of the ending episode, then the env's new origin.
__device__ __forceinline__ void stage_terrain_level(const TK& k, int e, uint64_t step) {
  const DyrosTerrainCurriculum& C = k.c;
  const float* root = k.s.root_states + (size_t)e * 13;
  float* org = k.b.env_origins + (size_t)e * 3;
  const float dx = root[0] - org[0], dy = root[1] - org[1];
  const float d = sqrtf(dx * dx + dy * dy);
  const float tvx = k.b.target_vel[(size_t)e * 2], tvy = k.b.target_vel[(size_t)e * 2 + 1];
  const bool up = d > C.move_up_distance;
  const bool down = !up && d < sqrtf(tvx * tvx + tvy * tvy) * C.move_down_scale;
  int lvl = C.levels[e] + (up ? 1 : 0) - (down ? 1 : 0);
  if (lvl >= C.num_levels) {  // past the top: a uniform level, from reset_f column 30
    const float u = k.j.reset_f ? k.j.reset_f[(size_t)e * 32 + 30] : u01(draw4(k.p.seed, step, e, kSiteResetF, 7).z);
    lvl = min((int)(u * (float)C.num_levels), C.num_levels - 1);
  }
  lvl = max(lvl, 0);
  C.levels[e] = lvl;
  const float* o = C.origins + ((size_t)lvl * C.num_types + C.types[e]) * 3;
  org[0] = o[0];
  org[1] = o[1];
  org[2] = o[2];
}

// T:598-669, T:720-748 (+ DR re-draw of damping/armature, VT:519-733 / gymutil.py:584-619)
__device__ void stage_reset_env(const TK& k, int e, int lane) {
  const TaskParams& P = k.p;
  // Philox epoch of this reset: the step epoch, plus the env's own count of explicit resets since the last step so that
  // an env reset twice within one epoch (reset_done() then a termination; repeated reset_idx calls) draws afresh
  const uint64_t step = *P.step_counter + ((uint64_t)k.b.reset_seq[e] << 40);
  // VT:540-544: only envs whose randomize_buf reached the frequency (1) are re-randomised; the buffer is cleared below
  const bool dr = P.randomize && k.b.randomize_buf[e] >= 1;
  __syncwarp();
  // --- draws (env-indexed). reset_f columns: see DyrosNoiseInjection
  auto uf = [&](int col) -> float {
    if (k.j.reset_f) return k.j.reset_f[(size_t)e * 32 + col];
    uint4 r = draw4(P.seed, step, e, kSiteResetF, col >> 2);
    uint32_t w = (col & 3) == 0 ? r.x : (col & 3) == 1 ? r.y : (col & 3) == 2 ? r.z : r.w;
    return u01(w);
  };
  for (int d = lane; d < ND; d += kWarp) {
    size_t i = (size_t)e * ND + d;
    k.b.qpos_noise[i] = P.init_dof_pos[d];                                         // T:611
    k.b.qpos_pre[i] = P.init_dof_pos[d];                                           // T:612
    k.b.qvel_noise[i] = 0.f;                                                       // T:613
    k.s.dof_state[2 * i] = P.reset_dof_pos[d];                                     // T:742
    k.s.dof_state[2 * i + 1] = 0.f;                                                // T:743
    k.b.pre_joint_velocity_states[i] = 0.f;                                        // T:635
    if (dr) {                                                                      // CFG:103-115, re-drawn on reset
      float u0, u1;
      if (k.j.dr_u) {
        u0 = k.j.dr_u[(size_t)e * 66 + d];
        u1 = k.j.dr_u[(size_t)e * 66 + 33 + d];
      } else {
        uint4 r = draw4(P.seed, step, e, kSiteDR, d);
        u0 = u01(r.x);
        u1 = u01(r.y);
      }
      k.s.dof_damping[i] = P.dr_damping_base + (P.dr_damping_lo + u0 * (P.dr_damping_hi - P.dr_damping_lo));
      k.s.dof_armature[i] = P.armature_base[d] * (P.dr_armature_lo + u1 * (P.dr_armature_hi - P.dr_armature_lo));
    }
  }
  // optional tables of the same randomisation pass (DyrosDynamicWalk.yaml:89-96 friction; PD gains: BASELINE configs[3]);
  // with injected DR draws (tests) they are left alone
  if (dr && !k.j.dr_u && lane == 0) {
    uint4 r = draw4(P.seed, step, e, kSiteDR, 64);
    if (k.s.contact_friction && P.dr_friction_hi > 0.f)
      k.s.contact_friction[e] = P.dr_friction_base * (P.dr_friction_lo + u01(r.x) * (P.dr_friction_hi - P.dr_friction_lo));
    if (k.b.pd_gain_scale && P.dr_pd_gain_hi > 0.f) {
      k.b.pd_gain_scale[(size_t)e * 2] = P.dr_pd_gain_lo + u01(r.y) * (P.dr_pd_gain_hi - P.dr_pd_gain_lo);
      k.b.pd_gain_scale[(size_t)e * 2 + 1] = P.dr_pd_gain_lo + u01(r.z) * (P.dr_pd_gain_hi - P.dr_pd_gain_lo);
    }
  }
  if (lane < 12) {
    k.b.qpos_bias[(size_t)e * 12 + lane] = uf(lane) * 6.28f / 100.f - (float)(3.14 / 100);        // T:615
    k.b.motor_constant_scale[(size_t)e * 12 + lane] = uf(18 + lane) * 0.4f + 0.8f;                // T:645
    k.b.action_torque_pre[(size_t)e * 12 + lane] = 0.f;                                            // T:636
  }
  if (lane < 3) k.b.quat_bias[(size_t)e * 3 + lane] = uf(12 + lane) * 6.28f / 150.f - (float)(3.14 / 150);  // T:616
  if (k.c.levels) {  // before the root and target_vel are overwritten below
    if (lane == 0) stage_terrain_level(k, e, step);
    __syncwarp();
  }
  if (lane < 13) {                                                                 // T:734-735
    float v = 0.f;
    if (lane < 3) v = k.b.env_origins[(size_t)e * 3 + lane];
    if (lane == 2) v = P.initial_height + v;
    if (lane == 6) v = 1.f;
    k.s.root_states[(size_t)e * 13 + lane] = v;
  }
  for (int i = lane; i < NB * 3; i += kWarp)                                       // T:638
    k.b.contact_forces_pre[(size_t)e * NB * 3 + i] = k.s.net_contact_force[(size_t)e * NB * 3 + i];
  for (int i = lane; i < LOG_DEPTH * 12; i += kWarp) k.b.action_log[(size_t)e * LOG_DEPTH * 12 + i] = 0.f;  // T:651
  for (int i = lane; i < NSLOT * NOBS1; i += kWarp) k.b.obs_history[(size_t)e * NSLOT * NOBS1 + i] = 0.f;   // T:668
  for (int i = lane; i < NSLOT * NA; i += kWarp) k.b.action_history[(size_t)e * NSLOT * NA + i] = 0.f;       // T:669
  if (lane == 0) {
    float vel_mag = uf(15) * 0.8f;                                                 // T:624
    float vel_theta = uf(16) * 0.0f;                                               // T:625
    k.b.target_vel[(size_t)e * 2] = vel_mag * cosf(vel_theta);                     // T:626-628
    k.b.target_vel[(size_t)e * 2 + 1] = vel_mag * sinf(vel_theta);
    k.b.init_mocap_data_idx[e] = (uf(17) > 0.5f) ? 0 : 1800;                       // T:630-632
    k.b.time[e] = 0.f;                                                             // T:642
    k.b.progress_buf[e] = 0;                                                       // T:648
    k.b.reset_buf[e] = 1;                                                          // T:649
    int delay, timing;
    if (k.j.reset_i) {
      delay = (int)k.j.reset_i[(size_t)e * 2];
      timing = (int)k.j.reset_i[(size_t)e * 2 + 1];
    } else {
      uint4 r = draw4(P.seed, step, e, kSiteResetI, 0);
      delay = P.delay_lo + (int)(r.x % (uint32_t)(P.delay_hi - P.delay_lo));       // T:652
      timing = (int)(r.y % (uint32_t)P.timing_hi);                                 // T:665
    }
    k.b.delay_idx[e] = delay;
    float el = k.b.epi_len[e];
    k.b.contact_reward_mean[e] = k.b.contact_reward_sum[e] / el;                   // T:654
    k.b.contact_reward_sum[e] = 0.f;                                               // T:655
    k.b.simul_len[e] = 0;                                                          // T:657
    k.b.epi_len_log[e] = el;                                                       // T:658
    k.b.epi_len[e] = 0.f;                                                          // T:659
    k.b.perturbation_count[e] = 0;                                                 // T:663
    k.b.pert_on[e] = 0;                                                            // T:664
    k.b.perturb_timing[e] = timing;                                                // T:665
    if (dr) k.b.randomize_buf[e] = 0;                                              // VT:540-544 (frequency 1)
    k.b.reset_seq[e] = k.b.reset_seq[e] + 1;
  }
}

// Width of an observation row: NOBS, plus the P heights of a height scan
__host__ __device__ constexpr int obs_width(const NoScan&) { return NOBS; }
__host__ __device__ inline int obs_width(const HeightScan& sc) { return NOBS + sc.P; }

// Height scan of one env (DESIGN.md section 4, "Height scan": legged_gym's _get_heights, quat_apply_yaw and the height
// term of compute_observations), one warp: lane l takes points l, l + 32, ...; the sample gathers of up to kScanBatch
// points per lane (all of them for P <= 256) are issued before the first is used. (x, y, z) is the root's position,
// (qz, qw) the z and w components of its quaternion, `ob` the env's observation row (columns NOBS + k are written).
// kStates: the columns go to the state row `sr` as well, and to `ob` only if it is not NULL.
constexpr int kScanBatch = 8;
template <bool kStates = false>
__device__ __forceinline__ void stage_height_scan(const HeightScan& sc, int e, int lane, float x, float y, float z,
                                                  float qz, float qw, float* ob, float* sr = nullptr) {
  const float n = fmaxf(sqrtf(qz * qz + qw * qw), 1e-9f);  // TU normalize of the quaternion with x = y = 0
  const float yz = qz / n, yw = qw / n;
  const float zb = z - sc.base_offset;
  const FieldGround& f = sc.f;
  float* mh = sc.measured ? sc.measured + (size_t)e * sc.P : nullptr;
  for (int k0 = 0; k0 < sc.P; k0 += kWarp * kScanBatch) {
    int s0[kScanBatch], s1[kScanBatch], s2[kScanBatch];
#pragma unroll
    for (int b = 0; b < kScanBatch; ++b) {
      const int k = min(k0 + lane + b * kWarp, sc.P - 1);  // (past the end: a repeat of the last point, not stored)
      const float2 p = __ldg(sc.points + k);
      // TU quat_apply((0, 0, yz, yw), (p.x, p.y, 0)) = v + w t + cross(xyz, t), t = cross(xyz, v) * 2; the left-out
      // terms have a zero factor and add exact zeros
      const float tx = -(yz * p.y) * 2.0f, ty = (yz * p.x) * 2.0f;
      const float wx = ((p.x + yw * tx) - yz * ty) + x;
      const float wy = ((p.y + yw * ty) + yz * tx) + y;
      s0[b] = s1[b] = s2[b] = 0;
      if (sc.has_field) {  // cell index trunc((w - p) / scale), clamped to the field: off it, the edge's samples
        const int px = (int)fminf(fmaxf((wx - f.ox) / f.dx, 0.0f), (float)(f.nr - 2));
        const int py = (int)fminf(fmaxf((wy - f.oy) / f.dy, 0.0f), (float)(f.nc - 2));
        const int16_t* c = f.s + (size_t)px * f.nc + py;
        s0[b] = __ldg(c);
        s1[b] = __ldg(c + f.nc);
        s2[b] = __ldg(c + 1);
      }
    }
#pragma unroll
    for (int b = 0; b < kScanBatch; ++b) {
      const int k = k0 + lane + b * kWarp;
      if (k < sc.P) {
        const float h = sc.has_field ? f.oz + f.dz * (float)min(min(s0[b], s1[b]), s2[b]) : 0.0f;  // plane: 0
        const float v = fminf(fmaxf(zb - h, -1.0f), 1.0f) * sc.scale;
        if constexpr (kStates) {
          if (ob) ob[NOBS + k] = v;
          sr[NOBS + k] = v;
        } else {
          ob[NOBS + k] = v;
        }
        if (mh) mh[k] = h;
      }
    }
  }
}

// Privileged block of the state row (DESIGN.md section 4, "Critic states"): lane c < kPrivCols writes column
// st.priv + c of `sr` from the post-reset state in global memory; `start`: the env is at an episode start (T:785), where
// the contact-force and push columns are 0. Every column is clipped to [-5, 5] (fminf / fmaxf: a NaN becomes -5).
__device__ __forceinline__ void stage_critic_privileged(const TK& k, const CriticStates& st, int e, int lane, bool start,
                                                        float* sr) {
  if (lane >= kPrivCols) return;
  const size_t E = (size_t)e;
  float v;
  if (lane < 3) v = __fmul_rn(k.s.root_states[E * 13 + 7 + lane], 2.0f);                  // linear velocity (world)
  else if (lane < 6) v = __fmul_rn(k.s.root_states[E * 13 + 7 + lane], 0.25f);           // angular velocity (world)
  else if (lane < 12) {                                                                  // foot contact forces
    const int b = lane < 9 ? k.p.lfoot : k.p.rfoot, c = lane < 9 ? lane - 6 : lane - 9;
    v = start ? 0.0f : __fmul_rn(k.s.net_contact_force[(E * NB + b) * 3 + c], 1e-3f);
  } else if (lane < 15) v = start ? 0.0f : __fmul_rn(k.b.push_force[E * 3 + (lane - 12)], 1e-2f);  // pelvis push
  else if (lane < 27) v = __fsub_rn(k.b.motor_constant_scale[E * 12 + (lane - 15)], 1.0f);
  else if (lane == 27) v = __fsub_rn(__fdiv_rn(k.b.total_mass[e], st.nominal_mass), 1.0f);
  else if (lane == 28) v = __fsub_rn(k.s.contact_friction ? k.s.contact_friction[e] : st.mu, 1.0f);
  else v = k.b.pd_gain_scale ? __fsub_rn(k.b.pd_gain_scale[E * 2 + (lane - 29)], 1.0f) : 0.0f;
  sr[st.priv + lane] = fminf(fmaxf(v, -5.0f), 5.0f);
}

// T:750-796 (history kept as rings, see DyrosTaskBuffers), then the height scan if there is one, then the privileged
// block of the critic states if they are on
template <class Scan, class St>
__device__ void stage_compute_observations(const TK& k, int e, int lane, const Scan& sc, const St& st) {
  const TaskParams& P = k.p;
  const float* root = k.s.root_states + (size_t)e * 13;
  float time = k.b.time[e];
  float time2idx = py_fmodf(time, P.period) / P.cycle_dt;                                           // T:762
  float phase = py_fmodf((float)k.b.init_mocap_data_idx[e] + time2idx, (float)P.mocap_data_num) / (float)P.mocap_data_num;  // T:763
  float ang = (float)(2 * 3.14159265358979) * phase;
  int head = (k.b.obs_hist_head[e] + 1) % NSLOT;
  bool start = k.b.epi_len[e] == 0.0f;                                                              // T:785
  float* hist = k.b.obs_history + (size_t)e * NSLOT * NOBS1;
  for (int i = lane; i < NOBS1; i += kWarp) {
    float v;
    if (i < 3) v = quat2euler_comp(root + 3, i) + k.b.quat_bias[(size_t)e * 3 + i];                 // T:753-757
    else if (i < 15) v = k.b.qpos_noise[(size_t)e * ND + (i - 3)] + k.b.qpos_bias[(size_t)e * 12 + (i - 3)];
    else if (i < 27) v = k.b.qvel_noise[(size_t)e * ND + (i - 15)];
    else if (i == 27) v = sinf(ang);                                                                // T:764
    else if (i == 28) v = cosf(ang);                                                                // T:765
    else if (i < 31) v = k.b.target_vel[(size_t)e * 2 + (i - 29)];
    else {
      int c = i - 31;
      float u;
      if (k.j.vel_u) u = k.j.vel_u[(size_t)e * 6 + c];
      else {
        uint4 r = draw4(P.seed, *P.step_counter, e, kSiteVelNoise, c);
        u = u01(r.x);
      }
      v = root[7 + c] + (u * 0.05f - 0.025f);                                                       // T:766,774
    }
    float nv = (v - k.b.obs_mean[i]) / sqrtf(k.b.obs_var[i] + 1e-8f * 1.0f);                        // T:776-777
    if (start) {
      for (int sl = 0; sl < NSLOT; ++sl) hist[sl * NOBS1 + i] = nv;                                 // T:786-787
    } else {
      hist[head * NOBS1 + i] = nv;                                                                  // T:783
    }
  }
  __syncwarp();
  if (lane == 0) k.b.obs_hist_head[e] = head;
  float* ob;
  if constexpr (St::kOn) ob = k.b.obs_buf + (size_t)e * st.obs_w;
  else if constexpr (Scan::kOn) ob = k.b.obs_buf + (size_t)e * obs_width(sc);
  else ob = k.b.obs_buf + (size_t)e * NOBS;  // (spelt out: the default instantiation keeps its instruction stream)
  float* sr = nullptr;
  if constexpr (St::kOn) sr = st.states + (size_t)e * st.S;
  const float* ah = k.b.action_history + (size_t)e * NSLOT * NA;
  int ahead = k.b.act_hist_head[e];
  // gather: all loads first (the compiler cannot reorder them across the stores itself), then the stores
  constexpr int IT = (NOBS + kWarp - 1) / kWarp;
  float vals[IT];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    int o = lane + it * kWarp;
    o = o < NOBS ? o : NOBS - 1;
    float v;
    if (o < NOBS1 * NHIS) {                                                                         // T:789-791
      int i = o / NOBS1, j = o - i * NOBS1;
      int pos = NSKIP * (i + 1) - 1;
      v = hist[((head + 1 + pos) % NSLOT) * NOBS1 + j];
    } else {                                                                                        // T:793-796
      int q = o - NOBS1 * NHIS;
      int i = q / NA, j = q - i * NA;
      int pos = NSKIP * (i + 1);
      v = ah[((ahead + 1 + pos) % NSLOT) * NA + j];
    }
    vals[it] = v;
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    int o = lane + it * kWarp;
    if (o < NOBS) {
      ob[o] = vals[it];
      if constexpr (St::kOn) sr[o] = vals[it];  // the state row's prefix: a second store of the same value
    }
  }
  if constexpr (Scan::kOn) {
    if constexpr (St::kOn)
      stage_height_scan<true>(sc, e, lane, root[0], root[1], root[2], root[5], root[6], st.heights_in_obs ? ob : nullptr, sr);
    else
      stage_height_scan(sc, e, lane, root[0], root[1], root[2], root[5], root[6], ob);
  }
  if constexpr (St::kOn) stage_critic_privileged(k, st, e, lane, start, sr);
}

// T:560-563 (loads of all four copies are issued before the first store)
__device__ void stage_late_update(const TK& k, int e, int lane) {
  const float* ds = k.s.dof_state + (size_t)e * ND * 2;
  constexpr int ITC = (NB * 3 + kWarp - 1) / kWarp;
  float vel[2], cf[ITC], at = 0.f, ac = 0.f;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    int d = lane + it * kWarp;
    vel[it] = ds[2 * (d < ND ? d : ND - 1) + 1];
  }
#pragma unroll
  for (int it = 0; it < ITC; ++it) {
    int i = lane + it * kWarp;
    cf[it] = k.s.net_contact_force[(size_t)e * NB * 3 + (i < NB * 3 ? i : NB * 3 - 1)];
  }
  if (lane < 12) at = k.b.action_torque[(size_t)e * 12 + lane];
  if (lane < NA) ac = k.b.actions[(size_t)e * NA + lane];
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    int d = lane + it * kWarp;
    if (d < ND) k.b.pre_joint_velocity_states[(size_t)e * ND + d] = vel[it];
  }
  if (lane < 12) k.b.action_torque_pre[(size_t)e * 12 + lane] = at;
  if (lane < NA) k.b.actions_pre[(size_t)e * NA + lane] = ac;
#pragma unroll
  for (int it = 0; it < ITC; ++it) {
    int i = lane + it * kWarp;
    if (i < NB * 3) k.b.contact_forces_pre[(size_t)e * NB * 3 + i] = cf[it];
  }
}

// ------------------------------------------------------------------ kernels
#define ENV_LANE()                                                   \
  int lane = threadIdx.x & 31;                                       \
  int e = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);          \
  if (e >= k.p.N) return;

__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_prologue(TK k, const float* __restrict__ actions) {
  pdl_launch_dependents();
  ENV_LANE();
  stage_prologue(k, actions, e, lane);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_substep_torque(TK k) {
  ENV_LANE();
  WarpSyncT sync;
  stage_substep_torque<32>(k, e, lane, sync);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_sensor_noise(TK k, int substep) {
  ENV_LANE();
  stage_sensor_noise<32>(k, substep, e, lane);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_epilogue(TK k) {
  ENV_LANE();
  stage_epilogue(k, e, lane);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_check_termination(TK k) {
  ENV_LANE();
  stage_check_termination(k, e, lane);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_compute_reward(TK k) {
  ENV_LANE();
  stage_compute_reward(k, e, lane);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_reset_idx(TK k, const int64_t* __restrict__ ids, int count) {
  int lane = threadIdx.x & 31;
  int w = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  int n = count >= 0 ? count : *k.b.reset_count;
  if (w >= n || w >= k.p.N) return;
  long long e = ids[w];
  if (e < 0 || e >= k.p.N) return;
  stage_reset_env(k, (int)e, lane);
}
template <class Scan, class St>
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_compute_observations(TK k, Scan sc, St st) {
  ENV_LANE();
  stage_compute_observations(k, e, lane, sc, st);
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_late_update(TK k) {
  ENV_LANE();
  stage_late_update(k, e, lane);
}
// one L2 prefetch per 128-byte line of [p, p + bytes), spread over the lanes of a warp
__device__ __forceinline__ void prefetch_rows_l2(const void* p, int bytes, int lane) {
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(p) & ~uintptr_t(127);
  const int lines = (int)((reinterpret_cast<uintptr_t>(p) + bytes + 127 - a0) >> 7);
  for (int i = lane; i < lines; i += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(a0 + (uintptr_t)i * 128));
}

// Inputs of the observation / late-update stages of one env, one value per lane (registers). Loaded once up front and,
// for an env that resets in this step, once more after the reset has rewritten them.
struct ObsIn {
  float root;        // lane < 13: root_states[lane]
  float qn, qv, qb;  // lane < 12: qpos_noise, qvel_noise, qpos_bias
  float quatb;       // lane < 3
  float vel0, vel1;  // joint velocity of DOF lane and of DOF 32 (late update)
  float tv;          // lane < 2: target_vel
  float time;
  int init_idx;
};
__device__ __forceinline__ ObsIn load_obs_in(const TK& k, int e, int lane) {
  ObsIn in;
  in.root = lane < 13 ? k.s.root_states[(size_t)e * 13 + lane] : 0.f;
  const int l12 = lane < 12 ? lane : 11;
  in.qn = k.b.qpos_noise[(size_t)e * ND + l12];
  in.qv = k.b.qvel_noise[(size_t)e * ND + l12];
  in.qb = k.b.qpos_bias[(size_t)e * 12 + l12];
  in.quatb = k.b.quat_bias[(size_t)e * 3 + (lane < 3 ? lane : 2)];
  const float2* ds2 = reinterpret_cast<const float2*>(k.s.dof_state + (size_t)e * ND * 2);
  in.vel0 = ds2[lane].y;
  in.vel1 = ds2[32].y;
  in.tv = k.b.target_vel[(size_t)e * 2 + (lane & 1)];
  in.time = k.b.time[e];
  in.init_idx = k.b.init_mocap_data_idx[e];
  return in;
}

// post_physics_step in one launch: epilogue, termination, reward, reset, observations, late update (T:532-563), one
// warp per env, written as ONE stage: every input of every stage is requested up front (one round of independent,
// coalesced loads; a second one for the history rows, whose addresses depend on the ring heads), all arithmetic then
// runs on registers, and the results go out at the end. The arithmetic is that of the staged kernels above, operation
// for operation (tests/test_env_step_gpu.py pins the two bit for bit). The scalar reward terms are computed by every
// lane of the warp from broadcast values: no regrouping through shared memory, no CTA barrier.
// Reward/termination read the pre-reset state, observations the post-reset state (SURVEY A3). Of contact_forces_pre only
// the two foot rows are maintained here: they are all the reward reads (T:858-859, T:904-907).
// The two means of the curriculum gate (T:489) are formed from fixed-point terms summed in 64-bit integers, so that the
// result does not depend on the order of summation: k_crossenv and this launch (atomics across CTAs) give the same
// bits. epi_len_log holds whole numbers (exact at 2^-20), contact_reward_mean lies in [0, 1].
__device__ __forceinline__ long long gate_term0(float epi_len_log) { return __double2ll_rn((double)epi_len_log * 1048576.0); }
__device__ __forceinline__ long long gate_term1(float contact_reward_mean) { return __double2ll_rn((double)contact_reward_mean * 1099511627776.0); }
__device__ __forceinline__ bool gate_open(const TaskParams& P, long long s0, long long s1) {  // T:489
  return (float)((double)s0 / 1048576.0 / P.N) > P.gate_len && (float)((double)s1 / 1099511627776.0 / P.N) > 0.165f;
}

// 4 warps per CTA, 7 CTAs per SM: 4096 envs (1024 CTAs) are resident on 148 SMs in ONE wave at <= 73 registers per thread
// (instantiated without and with the height scan, which runs last, from the post-reset root of the observation stage,
// and without and with the critic states, whose privileged block runs after it)
constexpr int kPostWarps = 4;
template <class Scan, class St>
__global__ void __launch_bounds__(kPostWarps * 32, 7) k_post_fused(TK k, int tail, Scan sc, St st) {
  __shared__ long long gate_acc[2][kPostWarps];
  __shared__ int level_acc[kPostWarps];
  pdl_launch_dependents();
  pdl_wait();
  const TaskParams& P = k.p;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int e = blockIdx.x * kPostWarps + w;
  const int live_warps = min(kPostWarps, P.N - (int)blockIdx.x * kPostWarps);  // warps of this CTA that hold an env
  if (e >= P.N) return;
  {
    const size_t E = (size_t)e;
    // ================================================================ loads, round 1 (independent of each other)
    ObsIn in = load_obs_in(k, e, lane);
    const float2* ds2 = reinterpret_cast<const float2*>(k.s.dof_state + E * ND * 2);
    const float2 dsA = ds2[lane], dsB = ds2[32];                   // DOF lane, DOF 32
    const float tqA = k.b.target_data_qpos[E * ND + lane], tqB = k.b.target_data_qpos[E * ND + 32];
    const float pjA = k.b.pre_joint_velocity_states[E * ND + lane], pjB = k.b.pre_joint_velocity_states[E * ND + 32];
    const int l13 = lane < NA ? lane : NA - 1, l12 = lane < 12 ? lane : 11;
    const float act = k.b.actions[E * NA + l13], actp = k.b.actions_pre[E * NA + l13];
    const float atq = k.b.action_torque[E * 12 + l12];
    const float* F = k.s.net_contact_force + E * NB * 3;
    const int bB = lane + 32 < NB ? lane + 32 : NB - 1;            // second body of this lane (lanes 0..5)
    const float fA0 = F[3 * lane], fA1 = F[3 * lane + 1], fA2 = F[3 * lane + 2];
    const float fB0 = F[3 * bB], fB1 = F[3 * bB + 1], fB2 = F[3 * bB + 2];
    const float* Fp = k.b.contact_forces_pre + E * NB * 3;
    const float lfp0 = Fp[P.lfoot * 3], lfp1 = Fp[P.lfoot * 3 + 1], lfp2 = Fp[P.lfoot * 3 + 2];
    const float rfp0 = Fp[P.rfoot * 3], rfp1 = Fp[P.rfoot * 3 + 1], rfp2 = Fp[P.rfoot * 3 + 2];
    const float epi0 = k.b.epi_len[e];
    const long long pr = k.b.progress_buf[e], rnd = k.b.randomize_buf[e];
    const float crs = k.b.contact_reward_sum[e], mass = k.b.total_mass[e];
    const int midx = k.b.mocap_data_idx[e];
    const float ft0 = k.b.target_data_force[E * 2], ft1 = k.b.target_data_force[E * 2 + 1];
    const int ohead0 = k.b.obs_hist_head[e], ahead = k.b.act_hist_head[e];
    const int pstart = *k.b.perturb_start;
    float ell = k.b.epi_len_log[e], crm = k.b.contact_reward_mean[e];  // terms of the curriculum gate (T:489)
    const int iA = lane, iB = lane + 32 < NOBS1 ? lane + 32 : NOBS1 - 1;  // observation components of this lane
    const float meanA = k.b.obs_mean[iA], varA = k.b.obs_var[iA], meanB = k.b.obs_mean[iB], varB = k.b.obs_var[iB];
    float velu = 0.f;                                               // T:766 draw of component 31 + c (lanes 31 and 0..4)
    if (k.j.vel_u) velu = k.j.vel_u[E * 6 + (lane == 31 ? 0 : (lane < 5 ? lane + 1 : 0))];
    // ================================================================ loads, round 2: history rows of the gather
    // T:789-796 frame by frame: lane j holds component j (and, lanes 0..4, component 32 + j) of each of the 9 older
    // observation frames and, lanes 0..12, of the 9 older actions; this step's frame (position 19) stays in registers
    const int head = (ohead0 + 1) % NSLOT;
    const float* hist = k.b.obs_history + E * NSLOT * NOBS1;
    const float* ah = k.b.action_history + E * NSLOT * NA;
    float hA[NHIS - 1], hB[NHIS - 1], hC[NHIS - 1];
#pragma unroll
    for (int i = 0; i < NHIS - 1; ++i) {
      const float* row = hist + ((head + 1 + NSKIP * (i + 1) - 1) % NSLOT) * NOBS1;   // T:789-791, position 2(i+1)-1
      hA[i] = row[lane];
      hB[i] = row[iB];
      hC[i] = ah[((ahead + 1 + NSKIP * (i + 1)) % NSLOT) * NA + l13];                 // T:793-796, position 2(i+1)
    }
    // ================================================================ epilogue (T:532-541, VT:325, T:544-545)
    const float a12 = __shfl_sync(kFull, act, NA - 1);
    float epi = epi0 + 1.0f;
    float t = in.time + P.dt_policy;
    t = t + P.time_gain * a12;
    const int timeout = ((float)pr >= P.max_len_m1) ? 1 : 0;
    const long long progress = pr + 1;
    long long randomize = rnd + 1;
    // ================================================================ termination (T:581-596)
    float quat[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) quat[i] = __shfl_sync(kFull, in.root, 3 + i);
    const float qe = quat_err_identity(quat);
    int reset = (fabsf(qe) > 0.5f) ? 1 : 0;
    if ((float)progress >= P.max_len_m1) reset = 1;
    bool hit = false;                                               // T:590 / T:937: any non-foot body with |F| > 1
    if (lane != P.lfoot && lane != P.rfoot) hit |= sqrtf(fA0 * fA0 + fA1 * fA1 + fA2 * fA2) > 1.0f;
    if (lane + 32 < NB && lane + 32 != P.lfoot && lane + 32 != P.rfoot) hit |= sqrtf(fB0 * fB0 + fB1 * fB1 + fB2 * fB2) > 1.0f;
    const bool col = __any_sync(kFull, hit);
    if (col) reset = 1;
    // ================================================================ reward (T:387-428, T:802-947)
    float s_qpos, s_qvel, s_qacc, s_tq = 0.f, s_tqd = 0.f;
    {
      float a = tqA - dsA.x, b = 0.0f - dsA.y, c = dsA.y - pjA;
      s_qpos = a * a; s_qvel = b * b; s_qacc = c * c;
      if (lane == 0) {                                              // DOF 32 rides on lane 0, after DOF 0
        a = tqB - dsB.x; b = 0.0f - dsB.y; c = dsB.y - pjB;
        s_qpos += a * a; s_qvel += b * b; s_qacc += c * c;
      }
      if (lane < 12) {
        const float tt = act * 333.0f, td = (act - actp) * 333.0f;
        s_tq = tt * tt;
        s_tqd = td * td;
      }
    }
    s_qpos = warp_sum(s_qpos); s_qvel = warp_sum(s_qvel); s_qacc = warp_sum(s_qacc); s_tq = warp_sum(s_tq); s_tqd = warp_sum(s_tqd);
    // the scalar terms, by every lane from broadcast values (reward_scalar, operation for operation)
    const float lf0 = __shfl_sync(kFull, fA0, P.lfoot), lf1 = __shfl_sync(kFull, fA1, P.lfoot), lf2 = __shfl_sync(kFull, fA2, P.lfoot);
    const float rf0 = __shfl_sync(kFull, fA0, P.rfoot), rf1 = __shfl_sync(kFull, fA1, P.rfoot), rf2 = __shfl_sync(kFull, fA2, P.rfoot);
    const float rootvx = __shfl_sync(kFull, in.root, 7), rootvy = __shfl_sync(kFull, in.root, 8);
    const float tvx = __shfl_sync(kFull, in.tv, 0), tvy = __shfl_sync(kFull, in.tv, 1);
    float r[14];
    float total;
    {
      r[0] = 0.3f * expf(-13.2f * fabsf(qe));                                         // T:835
      float n;
      n = sqrtf(s_qpos); r[1] = 0.35f * expf(-2.0f * (n * n));                        // T:837
      n = sqrtf(s_qvel); r[2] = 0.05f * expf(-0.01f * (n * n));                       // T:839
      const float dl0 = lf0 - lfp0, dl1 = lf1 - lfp1, dl2 = lf2 - lfp2;
      const float dr0 = rf0 - rfp0, dr1 = rf1 - rfp1, dr2 = rf2 - rfp2;
      r[9] = 0.2f * expf(-0.01f * (sqrtf(dl0 * dl0 + dl1 * dl1 + dl2 * dl2) + sqrtf(dr0 * dr0 + dr1 * dr1 + dr2 * dr2)));  // T:858
      r[4] = 0.05f * expf(-0.01f * sqrtf(s_tq));                                       // T:861
      r[5] = 0.6f * expf(-0.01f * sqrtf(s_tqd));                                       // T:863
      n = sqrtf(s_qacc); r[7] = 0.05f * expf(-20.0f * (n * n));                       // T:865
      const float vx = tvx - rootvx, vy = tvy - rootvy;
      n = sqrtf(vx * vx + vy * vy); r[6] = 0.3f * expf(-3.0f * (n * n));              // T:867
      const bool lc = lf2 > 1.0f, rc = rf2 > 1.0f;                                    // T:869-870
      const bool DSP = ((3300 <= midx) && (midx < 3600)) || (midx < 300) || ((1500 <= midx) && (midx < 2100));
      const bool RSSP = (300 <= midx) && (midx < 1500);
      const bool LSSP = (2100 <= midx) && (midx < 3300);
      const bool sync = (DSP && rc && lc) || (RSSP && rc && !lc) || (LSSP && !rc && lc);  // T:882-889
      r[8] = sync ? 0.2f : 0.0f;
      r[10] = 0.0f;                                                                   // T:893
      const float thr = (float)(1.4 * 9.81) * mass;                                   // T:895
      const bool thres = (lf2 > thr) || (rf2 > thr);
      r[11] = thres ? -0.2f : 0.0f;                                                   // T:898
      const float cl = fmaxf(lf2 - thr, 0.0f), cr = fmaxf(rf2 - thr, 0.0f);
      const float pen = 0.1f * expf(-0.007f * (sqrtf(cl * cl) + sqrtf(cr * cr)));     // T:900-901
      r[3] = thres ? pen : 0.1f;                                                      // T:902
      const float dthr = (float)(0.2 * 9.81) * mass / 1.0f;                           // T:904
      const bool tdiff = (fabsf(lf2 - lfp2) > dthr) || (fabsf(rf2 - rfp2) > dthr);
      r[12] = tdiff ? -0.05f : 0.0f;                                                  // T:907
      const float ws = mass / 104.48f;                                                // T:917
      r[13] = 0.1f * expf(-0.001f * fabsf(lf2 + ws * ft0)) + 0.1f * expf(-0.001f * fabsf(rf2 + ws * ft1));  // T:918-919
      total = r[0] + r[1] + r[2] + r[3] + r[4] + r[5] + r[6] + r[7] + r[8] + r[9] + r[10] + r[11] + r[12] + r[13];  // T:932-934
      if (col) total = P.death_cost;                                                  // T:942
      if (fabsf(qe) > 0.5f) total = P.death_cost;                                     // T:943
    }
    {
      float stv = col ? P.death_cost : 0.f;                                           // T:945
#pragma unroll
      for (int i = 0; i < 14; ++i)
        if (lane == i && !col) stv = r[i];
      if (lane == 14) stv = pstart ? 1.0f : 0.0f;                                     // T:415
      if (lane < 15) k.b.stacked_rewards[E * 15 + lane] = stv;
    }
    // ================================================================ stores of the scalar state; reset (T:598-669)
    if (lane == 0) {
      k.b.rew_buf[e] = total;
      k.b.timeout_buf[e] = timeout;
      k.b.reset_buf[e] = reset;
      k.b.contact_reward_sum[e] = crs + r[8];                                          // T:891
    }
    if (reset) {
      // the reset stage reads what the epilogue wrote: publish it first, then let it rewrite the env (rare: the stage is
      // the staged kernel's, from and to global memory), then fetch the rewritten inputs of the observation stage again
      if (lane == 0) {
        k.b.epi_len[e] = epi;
        k.b.time[e] = t;
        k.b.progress_buf[e] = progress;
        k.b.randomize_buf[e] = randomize;
      }
      __syncwarp();
      stage_reset_env(k, e, lane);
      __syncwarp();
      in = load_obs_in(k, e, lane);
      t = in.time;
      epi = k.b.epi_len[e];
      ell = k.b.epi_len_log[e];
      crm = k.b.contact_reward_mean[e];
#pragma unroll
      for (int i = 0; i < NHIS - 1; ++i) hA[i] = hB[i] = hC[i] = 0.f;                  // T:668-669: histories zeroed
    } else if (lane == 0) {
      k.b.epi_len[e] = epi;
      k.b.time[e] = t;
      k.b.progress_buf[e] = progress;
      k.b.randomize_buf[e] = randomize;
    }
    // ================================================================ cross-env pass of the fused step
    // (what k_crossenv does for the staged one, minus the id list): gate sums by 64-bit integer atomics, one pair per
    // CTA; the last CTA to take a ticket decides the gate and bumps the Philox epoch. Placed HERE, before the
    // observation stage and its 2 KB of stores per env, so that the fence below has little to wait for and the ticket
    // traffic overlaps the rest of the kernel: every draw of this launch that uses the epoch is either behind us (reset)
    // or uses the copy taken now.
    const uint64_t epoch = *P.step_counter;
    if (tail) {
      const bool gate = P.perturb != 0;
      const bool lmean = k.c.levels && k.c.level_mean;  // mean terrain level: an integer sum, order-free like the gate's
      if (gate && lane == 0) {
        gate_acc[0][w] = gate_term0(ell);  // (post-reset values, as k_crossenv reads them)
        gate_acc[1][w] = gate_term1(crm);
      }
      if (lmean && lane == 0) level_acc[w] = k.c.levels[e];  // (post-reset level: written by this thread)
      asm volatile("bar.sync 1, %0;" ::"r"(live_warps * 32) : "memory");
      if (threadIdx.x == 0) {
        if (gate) {
          long long a = 0, b = 0;
          for (int i = 0; i < live_warps; ++i) {
            a += gate_acc[0][i];
            b += gate_acc[1][i];
          }
          atomicAdd(P.tail + 0, (unsigned long long)a);
          atomicAdd(P.tail + 1, (unsigned long long)b);
        }
        if (lmean) {
          long long l = 0;
          for (int i = 0; i < live_warps; ++i) l += level_acc[i];
          atomicAdd(P.tail + 3, (unsigned long long)l);
        }
        if (gate || lmean) __threadfence();  // the sums before the ticket
        if (atomicAdd(P.tail + 2, 1ull) == gridDim.x - 1) {  // every CTA has published its sums and taken its epoch copy
          __threadfence();
          if (gate) {
            const long long s0 = (long long)atomicExch(P.tail + 0, 0ull), s1 = (long long)atomicExch(P.tail + 1, 0ull);
            if (gate_open(P, s0, s1)) *k.b.perturb_start = 1;  // T:489-490 (sticky)
          }
          if (lmean) *k.c.level_mean = (float)((double)(long long)atomicExch(P.tail + 3, 0ull) / P.N);
          P.tail[2] = 0;
          *P.step_counter = epoch + 1;
        }
      }
    }
    // ================================================================ observations (T:750-796)
    const float time2idx = py_fmodf(t, P.period) / P.cycle_dt;                         // T:762
    const float phase = py_fmodf((float)in.init_idx + time2idx, (float)P.mocap_data_num) / (float)P.mocap_data_num;  // T:763
    const float ang = (float)(2 * 3.14159265358979) * phase;
    const bool start = epi == 0.0f;                                                    // T:785
#pragma unroll
    for (int i = 0; i < 4; ++i) quat[i] = __shfl_sync(kFull, in.root, 3 + i);
    // (shuffles are executed by all lanes: gather every lane's sources first, then select)
    const float tv0n = __shfl_sync(kFull, in.tv, 0), tv1n = __shfl_sync(kFull, in.tv, 1);
    const float qb_for_A = __shfl_sync(kFull, in.qb, (lane - 3) & 31), qn_for_A = __shfl_sync(kFull, in.qn, (lane - 3) & 31);
    const float qv_for_A = __shfl_sync(kFull, in.qv, (lane - 15) & 31);
    const float rootv_for_A = __shfl_sync(kFull, in.root, 7);       // component 31 = root[7] (lane 31)
    const float rootv_for_B = __shfl_sync(kFull, in.root, (8 + lane) & 31);  // components 32..36 = root[8..12] (lanes 0..4)
    // T:766: one draw per velocity component c = 0..5, held by lane 31 (component 31) and lanes 0..4 (32..36)
    const int cdraw = lane == 31 ? 0 : (lane < 5 ? lane + 1 : 0);
    float vnoise = velu;
    if (!k.j.vel_u) vnoise = u01(draw4(P.seed, epoch, e, kSiteVelNoise, cdraw).x);
    vnoise = vnoise * 0.05f - 0.025f;
    float vA, vB = 0.f;
    if (iA < 3) vA = quat2euler_comp(quat, iA) + in.quatb;                             // T:753-757 (quat_bias[lane], lane < 3)
    else if (iA < 15) vA = qn_for_A + qb_for_A;
    else if (iA < 27) vA = qv_for_A;
    else if (iA == 27) vA = sinf(ang);                                                 // T:764
    else if (iA == 28) vA = cosf(ang);                                                 // T:765
    else if (iA < 31) vA = iA == 29 ? tv0n : tv1n;
    else vA = rootv_for_A + vnoise;                                                    // T:766,774 (component 31)
    if (lane < NOBS1 - 32) vB = rootv_for_B + vnoise;                                  // components 32..36
    const float nvA = (vA - meanA) / sqrtf(varA + 1e-8f * 1.0f);                       // T:776-777
    const float nvB = (vB - meanB) / sqrtf(varB + 1e-8f * 1.0f);
    {
      float* hw = k.b.obs_history + E * NSLOT * NOBS1;
      if (start) {
        for (int sl = 0; sl < NSLOT; ++sl) {                                           // T:786-787
          hw[sl * NOBS1 + iA] = nvA;
          if (lane < NOBS1 - 32) hw[sl * NOBS1 + lane + 32] = nvB;
        }
      } else {
        hw[head * NOBS1 + iA] = nvA;                                                   // T:783
        if (lane < NOBS1 - 32) hw[head * NOBS1 + lane + 32] = nvB;
      }
      if (lane == 0) k.b.obs_hist_head[e] = head;
    }
    {
      float* ob;                                                                       // (with critic states the heights may
      if constexpr (St::kOn) ob = k.b.obs_buf + E * st.obs_w;                          //  live in the state row only)
      else ob = k.b.obs_buf + E * obs_width(sc);
#pragma unroll
      for (int i = 0; i < NHIS; ++i) {                                                 // T:789-791
        const bool newest = start || i == NHIS - 1;                                    // (T:786-787: at an episode start every slot holds this frame)
        ob[NOBS1 * i + lane] = newest ? nvA : hA[i < NHIS - 1 ? i : 0];
        if (lane < NOBS1 - 32) ob[NOBS1 * i + 32 + lane] = newest ? nvB : hB[i < NHIS - 1 ? i : 0];
      }
#pragma unroll
      for (int i = 0; i < NHIS - 1; ++i)                                               // T:793-796
        if (lane < NA) ob[NOBS1 * NHIS + NA * i + lane] = hC[i];
      if constexpr (St::kOn) {  // the state row's prefix: the same registers stored a second time
        float* sr = st.states + E * st.S;
#pragma unroll
        for (int i = 0; i < NHIS; ++i) {
          const bool newest = start || i == NHIS - 1;
          sr[NOBS1 * i + lane] = newest ? nvA : hA[i < NHIS - 1 ? i : 0];
          if (lane < NOBS1 - 32) sr[NOBS1 * i + 32 + lane] = newest ? nvB : hB[i < NHIS - 1 ? i : 0];
        }
#pragma unroll
        for (int i = 0; i < NHIS - 1; ++i)
          if (lane < NA) sr[NOBS1 * NHIS + NA * i + lane] = hC[i];
      }
    }
    // ================================================================ late update (T:560-563)
    k.b.pre_joint_velocity_states[E * ND + lane] = in.vel0;
    if (lane == 0) k.b.pre_joint_velocity_states[E * ND + 32] = in.vel1;
    if (lane < 12) k.b.action_torque_pre[E * 12 + lane] = atq;
    if (lane < NA) k.b.actions_pre[E * NA + lane] = act;
    if (lane == P.lfoot || lane == P.rfoot) {                                          // the rows the reward reads
      float* o = k.b.contact_forces_pre + E * NB * 3 + 3 * lane;
      o[0] = fA0; o[1] = fA1; o[2] = fA2;
    }
    // ================================================================ height scan (DESIGN.md section 4)
    if constexpr (Scan::kOn) {
      const float rx = __shfl_sync(kFull, in.root, 0), ry = __shfl_sync(kFull, in.root, 1), rz = __shfl_sync(kFull, in.root, 2);
      if constexpr (St::kOn)
        stage_height_scan<true>(sc, e, lane, rx, ry, rz, quat[2], quat[3],
                                st.heights_in_obs ? k.b.obs_buf + E * st.obs_w : nullptr, st.states + E * st.S);
      else
        stage_height_scan(sc, e, lane, rx, ry, rz, quat[2], quat[3], k.b.obs_buf + E * obs_width(sc));
    }
    // ================================================================ privileged block of the critic states (section 4)
    if constexpr (St::kOn) stage_critic_privileged(k, st, e, lane, start, st.states + E * st.S);
  }
}

// Cross-env pass: (a) reset_buf.nonzero() -> ascending ids (T:554) by warp ballot + prefix scan, multi-CTA;
// (b) the curriculum gate means of T:489 (order-free fixed-point sums) and the mean terrain level; (c) Philox epoch bump.
//
// Compaction: a CTA takes a tile of kScanTile consecutive envs (tile index = an atomic ticket, so a tile only ever waits
// for tiles whose CTAs are already running); thread t reads reset_buf[tile * kScanTile + t] (coalesced), a warp ballot
// gives every lane its rank inside the warp (popc of the lower lanes' bits) and the warp its count, a shuffle scan of
// the 32 warp counts gives the offsets inside the tile, and the tile's offset in the output is the sum of the counts of
// the tiles before it: every tile publishes its count as soon as it has it (decoupled: nobody waits for a prefix, only
// for counts), and warp 0 of tile i sums the i counts before it, 32 at a time. ids come out ascending, exactly
// reset_buf.nonzero(); the int32 copy (T:737,745) is written alongside. The last CTA to finish writes nothing but the
// clean-up (ticket, status words) for the next launch, decides the gate and bumps the epoch.
constexpr int kScanTile = 1024;
__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__global__ void __launch_bounds__(kScanTile) k_crossenv(TK k, int do_compact, int do_gate, int do_bump) {
  __shared__ int warp_cnt[kScanTile / 32];
  __shared__ long long red[2][kScanTile / 32];
  __shared__ int level_red[kScanTile / 32];
  __shared__ int s_tile, s_prefix;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int N = k.p.N, ntiles = (N + kScanTile - 1) / kScanTile;
  unsigned* ticket = k.p.scan_state;      // [0] next tile, [1] tiles finished, [2 + t] count of tile t, + 1 (0 = not yet)
  unsigned* status = k.p.scan_state + 2;
  pdl_wait();
  if (tid == 0) s_tile = (int)atomicAdd(ticket, 1u);
  __syncthreads();
  const int tile = s_tile;
  const int e = tile * kScanTile + tid;
  const bool valid = e < N;
  const bool gate = do_gate && k.p.perturb;
  const bool flag = do_compact && valid && k.b.reset_buf[e] != 0;
  const unsigned bal = __ballot_sync(kFull, flag);
  const int rank = __popc(bal & ((1u << lane) - 1u));
  long long s0 = (gate && valid) ? gate_term0(k.b.epi_len_log[e]) : 0;  // fixed-point terms: see gate_term0 / gate_term1
  long long s1 = (gate && valid) ? gate_term1(k.b.contact_reward_mean[e]) : 0;
  const bool lmean = do_gate && k.c.levels && k.c.level_mean;  // mean terrain level (as k_post_fused: an integer sum)
  int lv = (lmean && valid) ? k.c.levels[e] : 0;
  if (gate) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(kFull, s0, o);
      s1 += __shfl_xor_sync(kFull, s1, o);
    }
  }
  if (lmean) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lv += __shfl_xor_sync(kFull, lv, o);
  }
  if (lane == 0) {
    warp_cnt[w] = __popc(bal);
    red[0][w] = s0;
    red[1][w] = s1;
    level_red[w] = lv;
  }
  __syncthreads();
  if (w == 0) {
    // exclusive scan of the warp counts; the tile's count goes out at once
    const int v = warp_cnt[lane];
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += t;
    }
    warp_cnt[lane] = inc - v;
    const int total = __shfl_sync(kFull, inc, 31);
    if (lane == 0) atomicExch(status + tile, (unsigned)total + 1u);
    // offset of the tile = sum of the counts of the tiles before it
    int before = 0;
    for (int t = lane; t < tile; t += 32) {
      unsigned c;
      while ((c = ld_acquire_gpu_u32(status + t)) == 0u) __nanosleep(20);
      before += (int)(c - 1u);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(kFull, before, o);
    if (lane == 0) {
      s_prefix = before;
      if (do_compact && tile == ntiles - 1) *k.b.reset_count = before + total;
    }
    if (gate) {
      long long a = red[0][lane], b = red[1][lane];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(kFull, a, o);
        b += __shfl_xor_sync(kFull, b, o);
      }
      if (lane == 0) {
        atomicAdd(k.p.tail + 0, (unsigned long long)a);
        atomicAdd(k.p.tail + 1, (unsigned long long)b);
      }
    }
    if (lmean) {
      long long l = level_red[lane];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(kFull, l, o);
      if (lane == 0) atomicAdd(k.p.tail + 3, (unsigned long long)l);
    }
  }
  __syncthreads();
  if (flag) {
    const int pos = s_prefix + warp_cnt[w] + rank;
    k.b.reset_env_ids[pos] = e;
    k.b.reset_env_ids32[pos] = e;
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(ticket + 1, 1u) == (unsigned)ntiles - 1u) {  // every tile is done: clean up for the next launch
      __threadfence();
      for (int t = 0; t < ntiles; ++t) status[t] = 0u;
      ticket[0] = 0u;
      ticket[1] = 0u;
      if (gate) {
        const long long a = (long long)atomicExch(k.p.tail + 0, 0ull), b = (long long)atomicExch(k.p.tail + 1, 0ull);
        if (gate_open(k.p, a, b)) *k.b.perturb_start = 1;  // T:489-490 (sticky)
      }
      if (lmean) *k.c.level_mean = (float)((double)(long long)atomicExch(k.p.tail + 3, 0ull) / N);
      if (do_bump) *k.p.step_counter = *k.p.step_counter + 1;
    }
  }
}


// ------------------------------------------------------------------ results of a step -> one contiguous block
// Layout of `dst`: obs (N,W) f32 | rew (N) f32 | reset (N) i64 | time_outs (N) i64, W = NOBS (+ P with a height scan);
// the i64 part starts at N*(W+1)*4 rounded up to a multiple of 8 (N*488*4 for W = NOBS). The host-facing
// step (DyrosDynamicWalk.step_async) hands this block to the copy engine as ONE device->host transfer on a second
// stream, so the next step may overwrite obs_buf / rew_buf / reset_buf / timeout_buf (VT:336-344) while the block is still in flight.
__global__ void __launch_bounds__(256) k_pack_results(TK k, float* __restrict__ dst, int W) {
  const int N = k.p.N;
  const size_t n_obs = (size_t)N * W;
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  const size_t n4 = n_obs / 4;  // obs_buf and dst are 16-byte aligned (torch allocations)
  const float4* src4 = reinterpret_cast<const float4*>(k.b.obs_buf);
  float4* dst4 = reinterpret_cast<float4*>(dst);
  if (k.b.obs_buf != dst) {  // (dyros_task_set_obs_buf(dst): the observation kernel has written the block itself)
    // Both sides of this copy are touched once per step: L2 evict-first, so that the 16 MB streamed here do not linger
    // in L2 at the expense of the env state (measured: plain loads / stores cost the next step 75 us, with the hints
    // 50 us; the pipelined host step therefore avoids this branch altogether, profiles/r1j_step_async.txt)
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    for (size_t i = tid; i < n4; i += nth) {
      float4 v;
      asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                   : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(src4 + i), "l"(pol));
      asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                   ::"l"(dst4 + i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
    }
    for (size_t i = n4 * 4 + tid; i < n_obs; i += nth) dst[i] = k.b.obs_buf[i];
  }
  float* rew = dst + n_obs;
  long long* rst = reinterpret_cast<long long*>(dst + ((n_obs + N + 1) & ~(size_t)1));
  for (size_t e = tid; e < (size_t)N; e += nth) {
    rew[e] = k.b.rew_buf[e];
    rst[e] = k.b.reset_buf[e];
    rst[N + e] = k.b.timeout_buf[e];
  }
}

// ------------------------------------------------------------------ launchers
static inline HeightScan make_scan(const Task* t) {
  HeightScan sc;
  sc.points = reinterpret_cast<const float2*>(t->scan.points);
  sc.P = t->scan.num_points;
  sc.base_offset = t->scan.base_offset;
  sc.scale = t->scan.scale;
  sc.measured = t->scan.measured_heights;
  sc.has_field = t->sim->has_field ? 1 : 0;  // the sim's ground at this launch (dyros_sim_set_heightfield)
  sc.f = t->sim->field;
  return sc;
}
static inline CriticStates make_states(const Task* t) {
  CriticStates st;
  st.states = t->crit.states;
  st.S = t->states_width();
  st.priv = NOBS + t->scan.num_points;
  st.obs_w = t->obs_width();
  st.heights_in_obs = t->crit.heights_in_obs ? 1 : 0;
  st.nominal_mass = t->crit.nominal_mass;
  st.mu = t->sim->p.mu;
  return st;
}
static inline int env_grid(int N) { return (N + kWarpsPerBlock - 1) / kWarpsPerBlock; }
#define LAUNCH_ENV(kern, ...)                                                    \
  kern<<<env_grid(t->p.N), kWarpsPerBlock * 32, 0, s>>>(make_tk(t), ##__VA_ARGS__); \
  DY_LAUNCH_CHECK();                                                             \
  return 0;

int launch_prologue(Task* t, const float* actions, cudaStream_t s) { LAUNCH_ENV(k_prologue, actions) }
int launch_substep_torque(Task* t, cudaStream_t s) { LAUNCH_ENV(k_substep_torque) }
int launch_sensor_noise(Task* t, int substep, cudaStream_t s) { LAUNCH_ENV(k_sensor_noise, substep) }
int launch_epilogue(Task* t, cudaStream_t s) { LAUNCH_ENV(k_epilogue) }
int launch_check_termination(Task* t, cudaStream_t s) { LAUNCH_ENV(k_check_termination) }
int launch_compute_reward(Task* t, cudaStream_t s) { LAUNCH_ENV(k_compute_reward) }
int launch_compute_observations(Task* t, cudaStream_t s) {
  if (t->crit.states) {
    if (t->scan.num_points) { LAUNCH_ENV((k_compute_observations<HeightScan, CriticStates>), make_scan(t), make_states(t)) }
    LAUNCH_ENV((k_compute_observations<NoScan, CriticStates>), NoScan(), make_states(t))
  }
  if (t->scan.num_points) { LAUNCH_ENV((k_compute_observations<HeightScan, NoStates>), make_scan(t), NoStates()) }
  LAUNCH_ENV((k_compute_observations<NoScan, NoStates>), NoScan(), NoStates())
}
int launch_late_update(Task* t, cudaStream_t s) { LAUNCH_ENV(k_late_update) }
int configure_task_kernels() {
  DY_CUDA(prefer_max_smem_carveout(k_prologue)); DY_CUDA(prefer_max_smem_carveout(k_substep_torque));
  DY_CUDA(prefer_max_smem_carveout(k_sensor_noise)); DY_CUDA(prefer_max_smem_carveout(k_epilogue));
  DY_CUDA(prefer_max_smem_carveout(k_check_termination)); DY_CUDA(prefer_max_smem_carveout(k_compute_reward));
  DY_CUDA(prefer_max_smem_carveout((k_compute_observations<NoScan, NoStates>)));
  DY_CUDA(prefer_max_smem_carveout((k_compute_observations<HeightScan, NoStates>)));
  DY_CUDA(prefer_max_smem_carveout((k_compute_observations<NoScan, CriticStates>)));
  DY_CUDA(prefer_max_smem_carveout((k_compute_observations<HeightScan, CriticStates>)));
  DY_CUDA(prefer_max_smem_carveout(k_late_update));
  DY_CUDA(prefer_max_smem_carveout(k_reset_idx)); DY_CUDA(prefer_max_smem_carveout(k_pack_results));
  DY_CUDA(prefer_max_smem_carveout((k_post_fused<NoScan, NoStates>)));
  DY_CUDA(prefer_max_smem_carveout((k_post_fused<HeightScan, NoStates>)));
  DY_CUDA(prefer_max_smem_carveout((k_post_fused<NoScan, CriticStates>)));
  DY_CUDA(prefer_max_smem_carveout((k_post_fused<HeightScan, CriticStates>)));
  DY_CUDA(prefer_max_smem_carveout(k_crossenv));
  return 0;
}
int launch_post_fused(Task* t, cudaStream_t s, bool pdl, bool tail) {
  const dim3 grid((t->p.N + kPostWarps - 1) / kPostWarps), block(kPostWarps * 32);
  if (t->crit.states) {
    if (t->scan.num_points)
      DY_CUDA(launch_kernel(k_post_fused<HeightScan, CriticStates>, grid, block, 0, s, pdl, make_tk(t), (int)tail, make_scan(t),
                            make_states(t)));
    else
      DY_CUDA(launch_kernel(k_post_fused<NoScan, CriticStates>, grid, block, 0, s, pdl, make_tk(t), (int)tail, NoScan(),
                            make_states(t)));
  } else if (t->scan.num_points) {
    DY_CUDA(launch_kernel(k_post_fused<HeightScan, NoStates>, grid, block, 0, s, pdl, make_tk(t), (int)tail, make_scan(t), NoStates()));
  } else {
    DY_CUDA(launch_kernel(k_post_fused<NoScan, NoStates>, grid, block, 0, s, pdl, make_tk(t), (int)tail, NoScan(), NoStates()));
  }
  return 0;
}
int launch_reset_idx(Task* t, const int64_t* env_ids, int count, cudaStream_t s) {
  if (count == 0) return 0;
  const int64_t* ids = env_ids ? env_ids : t->b.reset_env_ids;
  int n = count >= 0 ? count : t->p.N;
  k_reset_idx<<<env_grid(n), kWarpsPerBlock * 32, 0, s>>>(make_tk(t), ids, count);
  DY_LAUNCH_CHECK();
  return 0;
}
int launch_pack_results(Task* t, float* dst, cudaStream_t s) {
  // a multiple of the SM count; 8 MB at N = 4096: ~13 float4 per thread
  k_pack_results<<<148 * 4, 256, 0, s>>>(make_tk(t), dst, t->obs_width());
  DY_LAUNCH_CHECK();
  return 0;
}
int launch_crossenv(Task* t, bool compact, bool gate, bool bump, cudaStream_t s, bool pdl) {
  const int ntiles = (t->p.N + kScanTile - 1) / kScanTile;
  DY_CUDA(launch_kernel(k_crossenv, dim3(ntiles), dim3(kScanTile), 0, s, pdl, make_tk(t), (int)compact, (int)gate, (int)bump));
  return 0;
}

}  // namespace dyros
