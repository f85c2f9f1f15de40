// K1, multi-lane variant (DyrosSimDesc.physics_program = 1; the default is the one-lane-per-env role program of
// physics_kernels.cu: at 28 envs per SM the multi-lane mapping measured SLOWER, 158 vs 87 us per launch at 4096 envs,
// profiles/r2b_*; DESIGN.md section 4 has the numbers and the reasons. Kept selectable, built and parity-tested.)
// gym.simulate as one kernel launch, multi-lane (physics_lanes.cuh): 8 lanes per env, 4 envs per warp, one warp
// per role and group of 4 envs; up to 28 envs per CTA (7 groups x 4 role warps = 28 warps, + 4 I/O warps in the fused
// step = 1024 threads, one CTA per SM: N = 4096 is a single wave on 148 SMs). The per-env scratch blocks, the hot model
// tables and the dataflow flags live in dynamic shared memory.
#include "physics_lanes.cuh"
#include "task_stages.cuh"

namespace dyros {
using namespace ln;
namespace lanes_impl {

__device__ __forceinline__ int ld_acquire_shared(const int* p) {
  int v;
  asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_shared(int* p, int v) {
  asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}

// Flags between the role warps of a group of envs: the producer's lanes finish their shared-memory writes, lane 0
// publishes with release; the consumer's lanes spin with acquire.
struct LaneSync {
  int lane;
  long long* trace;  // profiling aid: clock64() at the phase boundaries of one warp per role (NULL in production)
  __device__ __forceinline__ void mark(int id) const {
    if (trace && lane == 0) trace[id] = clock64();
  }
  __device__ __forceinline__ void signal(int* f, int v) const {
    __syncwarp();
    if (lane == 0) st_release_shared(f, v);
  }
  // every lane polls (one broadcast load per iteration): the loop branch is warp-uniform, so the warp never splits
  // into a lane-0 group and a rest group that would then run the following phase twice
  // 7 warps share a scheduler here: a waiting warp backs off between polls instead of taking issue slots from the
  // warps it is waiting for (measured without the back-off: 38 % of the executed instructions were polls)
  __device__ __forceinline__ void wait(const int* f, int v) const {
    while (ld_acquire_shared(f) < v) __nanosleep(40);
    __syncwarp();
  }
  // for flags published by the I/O warps: back off between polls
  __device__ __forceinline__ void wait_io(const int* f, int v) const {
    while (ld_acquire_shared(f) < v) __nanosleep(100);
    __syncwarp();
  }
};

constexpr int kMaxPhysSmem = 227 * 1024 - 1024;  // dynamic part; 1 KiB is left for static shared memory (k_step_physics: 1 KiB)
constexpr int kEnvsPerWarp = 32 / LPE;           // 4
constexpr int kMaxQuads = 7;                     // groups of 4 envs per CTA
constexpr int kMaxEpb = kMaxQuads * kEnvsPerWarp;
constexpr int kIoThreads = 128;
constexpr int kSlabVThreads = 128;               // virtual thread count the slab stages of task_stages.cuh are written for
static_assert(kMaxEpb <= kSlabMaxEnvs, "slab stages are sized for kSlabMaxEnvs envs per CTA");
static_assert(DYROS_LANES == 4, "four roles per group of envs");

struct PhysCta {
  const float* hot;
  int* ioflags;   // CTA-wide flags of the I/O warps
  int* qflags;    // flags of this warp's group of envs
  float* envs;    // scratch blocks of the CTA's envs
  float* sm;      // this lane group's env scratch block
  int role, lane, quad, e, nrole;  // nrole: threads of the role warps
  bool active;    // this warp's group holds at least one env
  bool live;      // this lane group's env is a real one (padding groups shadow the last env of their warp)
  Ln g;
};
__device__ __forceinline__ int nquads_of(int epb) { return (epb + kEnvsPerWarp - 1) / kEnvsPerWarp; }

// Common prologue of the physics kernels: stage the hot tables, clear the flags, locate the lane group's env.
__device__ __forceinline__ PhysCta phys_cta_setup(const DevModel& m, const SimParams& p, float* smem, int epb, int es) {
  {  // 16-byte cp.async: in flight together with the state copies issued after griddepcontrol.wait (the caller waits)
    const char* src = reinterpret_cast<const char*>(m.blob);
    for (int i = threadIdx.x; i < m.hot_bytes / 16; i += blockDim.x)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem) + i * 16), "l"(src + (size_t)i * 16)
                   : "memory");
  }
  const int nq = nquads_of(epb);
  int* flags = reinterpret_cast<int*>(smem + m.hot_bytes / 4);
  for (int i = threadIdx.x; i < IOF_COUNT + nq * QF_COUNT; i += blockDim.x) flags[i] = 0;
  pdl_launch_dependents();
  pdl_wait();  // everything above is independent of the previous kernel of the step (model tables only)
  PhysCta c;
  c.hot = smem;
  c.ioflags = flags;
  c.envs = smem + m.hot_bytes / 4 + IOF_COUNT + nq * QF_COUNT;
  c.nrole = nq * DYROS_LANES * 32;
  const int w = threadIdx.x >> 5;
  c.lane = threadIdx.x & 31;
  c.quad = (w >> 2) < nq ? (w >> 2) : 0;
  // roles rotate from group to group, so that every scheduler (warp index mod 4) gets warps of all four roles
  c.role = (w + (w >> 2)) & (DYROS_LANES - 1);
  c.qflags = flags + IOF_COUNT + c.quad * QF_COUNT;
  c.g = make_ln(c.lane);
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  c.active = c.quad * kEnvsPerWarp < nenv;
  int le = c.quad * kEnvsPerWarp + (c.lane >> 3);
  c.live = le < nenv;
  le = le < nenv ? le : nenv - 1;  // padding groups shadow the last env (same warp: same values, in lockstep; no global writes)
  c.e = e0 + le;
  c.sm = c.envs + (size_t)le * es;
  return c;
}

__device__ __forceinline__ EnvIO env_io(const DevModel& m, const DyrosSimBuffers& b, int e, bool live) {
  EnvIO io;
  io.contact = b.net_contact_force + (size_t)e * m.nb * 3;
  io.rb_force = nullptr;
  io.rb_torque = nullptr;
  io.push = false;
  io.link_pose = nullptr;
  io.live = live;
  return io;
}

// ---- CTA-cooperative, coalesced slab copies between the API tensors and the env scratch blocks. The envs of a CTA
//      are contiguous in every tensor, so thread t handles words t, t + nthreads, ... of each slab. Inputs go through
//      cp.async (LDGSTS, 4-byte): every word is copied straight to its scattered place in shared memory without a
//      register round trip, all copies of all slabs are in flight together and the CTA pays one memory latency.
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
// one L2 prefetch per 128-byte line of a contiguous slab (thread tid takes lines tid, tid + nthreads, ...); rolled: this
// runs once per launch and should cost as few instruction-cache lines as possible
__device__ __forceinline__ void slab_prefetch_l2(const void* base, unsigned bytes, int tid, int nthreads) {
  const char* p = static_cast<const char*>(base);
#pragma unroll 1
  for (unsigned off = tid * 128u; off < bytes; off += nthreads * 128u) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// The copies below are issued by thread `tid` of `nthreads` cooperating threads; the caller waits with
// cp_async_wait_all() and then synchronises the cooperating threads.
// (1) joint state, mass scales and root: once per launch (they stay in the scratch blocks)
__device__ __forceinline__ void slab_stage_state(const DevModel& m, const DyrosSimBuffers& b, const float* hot, float* envs, int es,
                                                 int e0, int nenv, int tid, int nthreads, float mu) {
  const int nd = m.nd, nb = m.nb, xoff = m.nl * LB;
#pragma unroll 1
  for (int le = tid; le < nenv; le += nthreads) {  // per-env friction (DR) or the sim's coefficient
    if (b.contact_friction) cp_async4(envs + le * es + xoff + X_MU, b.contact_friction + e0 + le);
    else envs[le * es + xoff + X_MU] = mu;
  }
  const int* dof_link = reinterpret_cast<const int*>(hot) + m.o_dof_link;
  const FastDiv d2nd(2 * nd), dnb(nb), d13(13);  // slabs are < 2^20 / divisor words (checked at create)
  {
    const float* src = b.dof_state + (size_t)e0 * nd * 2;
#pragma unroll 1
    for (int i = tid; i < nenv * nd * 2; i += nthreads) {
      int le = d2nd.div(i), w = i - le * 2 * nd;
      cp_async4(envs + le * es + dof_link[w >> 1] * LB + ((w & 1) ? B_QD : B_Q), src + i);
    }
  }
  {
    const float* src = b.body_mass_scale + (size_t)e0 * nb;
#pragma unroll 1
    for (int i = tid; i < nenv * nb; i += nthreads) {
      int le = dnb.div(i);
      cp_async4(envs + le * es + xoff + X_MASS + (i - le * nb), src + i);
    }
  }
  {
    const float* src = b.root_states + (size_t)e0 * 13;
#pragma unroll 1
    for (int i = tid; i < nenv * 13; i += nthreads) {
      int le = d13.div(i);
      cp_async4(envs + le * es + xoff + X_ROOT + (i - le * 13), src + i);
    }
  }
}
// (2) per sub-step, needed by the own-terms phase: the push, and the zeroed net contact forces (THIS sub-step only)
__device__ __forceinline__ void slab_stage_pre(const DevModel& m, const DyrosSimBuffers& b, const float* push, float* envs, int es,
                                               int e0, int nenv, int tid, int nthreads) {
  const int nb = m.nb, xoff = m.nl * LB;
  const FastDiv d3(3);
#pragma unroll 1
  for (int i = tid; i < nenv * 3; i += nthreads) {
    int le = d3.div(i);
    if (push) cp_async4(envs + le * es + xoff + X_PUSH + (i - le * 3), push + (size_t)e0 * 3 + i);
    else envs[le * es + xoff + X_PUSH + (i - le * 3)] = 0.f;
  }
  float* cf = b.net_contact_force + (size_t)e0 * nb * 3;
  const int nw = nenv * nb * 3;
  if (((reinterpret_cast<uintptr_t>(cf) | (uintptr_t)(nw * 4)) & 15) == 0) {  // the usual case: 16-byte stores
#pragma unroll 1
    for (int i = tid; i < nw / 4; i += nthreads) reinterpret_cast<float4*>(cf)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
#pragma unroll 1
    for (int i = tid; i < nw; i += nthreads) cf[i] = 0.f;
  }
}
// (3) per sub-step, needed by pass 2: damping and armature (their slots are reused by the recursion) and the torque
__device__ __forceinline__ void slab_stage_dofpar(const DevModel& m, const DyrosSimBuffers& b, const float* hot, float* envs, int es,
                                                  int e0, int nenv, bool with_tau, int tid, int nthreads) {
  const int nd = m.nd;
  const int* dof_link = reinterpret_cast<const int*>(hot) + m.o_dof_link;
  const FastDiv dnd(nd);
  const float* tau = b.dof_actuation_force + (size_t)e0 * nd;
  const float* dmp = b.dof_damping + (size_t)e0 * nd;
  const float* arm = b.dof_armature + (size_t)e0 * nd;
#pragma unroll 1
  for (int i = tid; i < nenv * nd; i += nthreads) {
    int le = dnd.div(i), d = i - le * nd;
    float* L = envs + le * es + dof_link[d] * LB + B_SC;
    if (with_tau) cp_async4(L + 0, tau + i);
    cp_async4(L + 1, dmp + i);
    cp_async4(L + 2, arm + i);
  }
}

__device__ __forceinline__ void slab_store_outputs(const DevModel& m, const DyrosSimBuffers& b, const float* hot,
                                                   const float* envs, int es, int e0, int nenv, int tid, int nthreads) {
  const int nd = m.nd, xoff = m.nl * LB;
  const int* dof_link = reinterpret_cast<const int*>(hot) + m.o_dof_link;
  const FastDiv d2nd(2 * nd), d13(13);
  float* ds = b.dof_state + (size_t)e0 * nd * 2;
#pragma unroll 2
  for (int i = tid; i < nenv * nd * 2; i += nthreads) {
    int le = d2nd.div(i), w = i - le * 2 * nd;
    ds[i] = envs[le * es + dof_link[w >> 1] * LB + ((w & 1) ? B_QD : B_Q)];
  }
  float* rs = b.root_states + (size_t)e0 * 13;
#pragma unroll 1
  for (int i = tid; i < nenv * 13; i += nthreads) {
    int le = d13.div(i);
    rs[i] = envs[le * es + xoff + X_ROOT + (i - le * 13)];
  }
}

// The task's slab stages are compiled as separate functions so that their (large, short-lived) register arrays do not
// raise the register pressure of the role programs. `tid0` of `nreal` real threads act as kSlabVThreads virtual threads.
__device__ __noinline__ void torque_stage_slab(TorqueSlabArgs k, int e0, int nenv, float* envs, int es, const int* dof_link,
                                               int tid0, int nreal) {
  // joint state comes from the scratch blocks; the torques go to the API tensor and straight into the scratch blocks
#pragma unroll 1
  for (int vt = tid0; vt < kSlabVThreads; vt += nreal)
    stage_substep_torque_cta(
        k, e0, nenv, vt, kSlabVThreads, [&](int le, int d, float v) { envs[le * es + dof_link[d] * LB + B_SC] = v; },
        [&](int le, int d, int which) { return envs[le * es + dof_link[d] * LB + (which ? B_QD : B_Q)]; });
}
__device__ __noinline__ void noise_stage_slab(NoiseSlabArgs k, int substep, int e0, int nenv, const float* envs, int es,
                                              const int* dof_link, int tid0, int nreal) {
  // sensor noise reads the fresh joint angles from the scratch blocks
#pragma unroll 1
  for (int vt = tid0; vt < kSlabVThreads; vt += nreal)
    stage_sensor_noise_cta(k, substep, e0, nenv, vt, kSlabVThreads,
                           [&](int le, int d) { return envs[le * es + dof_link[d] * LB + B_Q]; });
}

__global__ void __launch_bounds__(kMaxQuads * DYROS_LANES * 32) k_simulate_lanes(DevModel m, SimParams p, DyrosSimBuffers b,
                                                                          const float* __restrict__ push, int apply_wrench, int epb, int es) {
  extern __shared__ __align__(16) float smem[];
  PhysCta c = phys_cta_setup(m, p, smem, epb, es);
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  float* envs = c.envs;
  EnvIO io = env_io(m, b, c.e, c.live);
  // applied wrenches act over the whole simulate() call, i.e. all of its sub-steps (gym_py.html apply_rigid_body_force_tensors)
  io.push = push != nullptr;
  io.rb_force = apply_wrench ? b.rb_force + (size_t)c.e * m.nb * 3 : nullptr;
  io.rb_torque = apply_wrench ? b.rb_torque + (size_t)c.e * m.nb * 3 : nullptr;
  LaneSync sync{c.lane, nullptr};
  for (int s = 0; s < p.substeps; ++s) {
    // (first sub-step: the staged tables are still in flight, dof_link is read from the global copy)
    const float* tab = s == 0 ? reinterpret_cast<const float*>(m.blob) : c.hot;
    if (s == 0) slab_stage_state(m, b, tab, envs, es, e0, nenv, threadIdx.x, blockDim.x, p.mu);
    slab_stage_pre(m, b, push, envs, es, e0, nenv, threadIdx.x, blockDim.x);
    slab_stage_dofpar(m, b, tab, envs, es, e0, nenv, true, threadIdx.x, blockDim.x);
    cp_async_wait_all();
    __syncthreads();
    io.link_pose = (s + 1 == p.substeps && b.link_pose) ? b.link_pose + (size_t)c.e * m.nl * 12 : nullptr;
    if (c.active) env_substep_lanes(io, c.sm, c.qflags, c.ioflags, s, c.hot, m, p, c.role, sync, c.g, false);
    __syncthreads();
    if (s + 1 == p.substeps) slab_store_outputs(m, b, c.hot, envs, es, e0, nenv, threadIdx.x, blockDim.x);
  }
}

constexpr int kStepThreadsMax = kMaxQuads * DYROS_LANES * 32 + kIoThreads;  // 1024
__device__ __forceinline__ void io_group_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kIoThreads) : "memory"); }

// The physics part of one policy step in ONE launch: skipframe x (PD + delay torque, gym.simulate, sensor noise),
// i.e. the loop body of T:504-530 with the three gym calls of T:520-526 folded in; with `actions` also the part of
// pre_physics_step before that loop (T:449-502).
// The first nrole threads run the role programs; the last 4 warps are the I/O group: while the roles are in pass 1 of a
// sub-step it zeroes the contact forces and stages the push (F_IO_PRE), draws the sensor noise of the PREVIOUS policy
// sub-step (which only reads the joint angles, untouched until the roles' last pass), evaluates the torque stage and
// re-stages damping and armature (F_IO_TAU, consumed by pass 2), so none of this sits on the roles' critical path.
__global__ void __launch_bounds__(kStepThreadsMax) k_step_physics_lanes(DevModel m, SimParams p, TK k, int epb, int es, long long* trace,
                                                                   const float* __restrict__ actions) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float pro[kSlabMaxEnvs][8];  // per-env scalars of the prologue (stage_prologue_slab)
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[24] = clock64();  // kernel entry (profiling)
  PhysCta c = phys_cta_setup(m, p, smem, epb, es);
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[25] = clock64();  // tables staged, previous kernel done
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  float* envs = c.envs;
  const int nthreads = blockDim.x;
  const bool io_group = (int)threadIdx.x >= c.nrole;
  const int it = threadIdx.x - c.nrole;  // thread index within the I/O group
  EnvIO io = env_io(m, k.s, c.e, c.live);
  // trace layout: [sub-step][role][32 marks], taken by the role warps of the first group of CTA 0
  LaneSync sync{c.lane, (trace && blockIdx.x == 0 && !io_group && c.quad == 0 && (threadIdx.x >> 7) == 0) ? trace + c.role * 32 : nullptr};
  const int* dof_link = reinterpret_cast<const int*>(c.hot) + m.o_dof_link;
  // (profiling: marks 18.. of role 0's row are the I/O group's phase boundaries)
  auto io_mark = [&](int s, int id) {
    if (trace && blockIdx.x == 0 && it == 0) trace[(size_t)s * DYROS_LANES * 32 + id] = clock64();
  };
  // per sub-step, I/O group: the push (every sub-step of the first simulate of the policy step, T:502 vs T:504) and the
  // zeroed contact forces
  auto stage_pre = [&](int s, int ss, int epoch) {
    slab_stage_pre(m, k.s, s == 0 ? k.b.push_force : nullptr, envs, es, e0, nenv, it, kIoThreads);
    cp_async_wait_all();
    io_group_sync();
    if (it == 0) st_release_shared(c.ioflags + F_IO_PRE, epoch + 1);
    io_mark(s, 19);
  };
  // Start-up. The two groups do not meet at a full barrier: the I/O group arrives (non-blocking) at barrier 3 once its
  // share of the model tables has landed and goes straight on to the prologue, which needs nothing from the role
  // warps; the role warps stage the state and wait at barrier 3 for the tables; the I/O group waits for the staged
  // state (barrier 4, where the role warps only arrive) before the first torque stage, which reads it.
  if (io_group) {
    {  // with a cold L2, pull in what the torque and noise stages will read
      const size_t e = (size_t)e0;
      slab_prefetch_l2(k.b.action_log + e * LOG_DEPTH * 12, (unsigned)nenv * LOG_DEPTH * 12 * 4, it, kIoThreads);
      slab_prefetch_l2(k.b.qpos_pre + e * ND, (unsigned)nenv * ND * 4, it, kIoThreads);
      slab_prefetch_l2(k.s.dof_damping + e * ND, (unsigned)nenv * ND * 4, it, kIoThreads);
      slab_prefetch_l2(k.s.dof_armature + e * ND, (unsigned)nenv * ND * 4, it, kIoThreads);
      if (!actions) {
        slab_prefetch_l2(k.b.target_data_qpos + e * ND, (unsigned)nenv * ND * 4, it, kIoThreads);
        slab_prefetch_l2(k.b.action_torque + e * 12, (unsigned)nenv * 12 * 4, it, kIoThreads);
      }
    }
    cp_async_wait_all();  // this thread's share of the tables
    asm volatile("bar.arrive 3, %0;" ::"r"(nthreads) : "memory");
    io_mark(0, 18);
    if (actions) {  // the policy-step prologue (T:449-502) of the CTA's envs; the push it decides is staged at its end
      stage_prologue_slab(k, actions, e0, nenv, it, kIoThreads, pro, [] { io_group_sync(); }, [&] { stage_pre(0, 0, 0); });
      io_group_sync();
    }
    asm volatile("bar.sync 4, %0;" ::"r"(nthreads) : "memory");
  } else {
    // joint state, root and mass scales are staged once and then live in the scratch blocks for the whole launch; the
    // torque and noise stages read them there, and only the final state is written back
    // (the staged tables are still in flight: dof_link is read from the global copy here)
    slab_stage_state(m, k.s, reinterpret_cast<const float*>(m.blob), envs, es, e0, nenv, threadIdx.x, c.nrole, p.mu);
    cp_async_wait_all();  // this thread's share of the tables and of the state
    asm volatile("bar.sync 3, %0;" ::"r"(nthreads) : "memory");
    asm volatile("bar.arrive 4, %0;" ::"r"(nthreads) : "memory");
  }
  int epoch = 0;
  for (int s = 0; s < k.p.skipframe; ++s) {
    for (int ss = 0; ss < p.substeps; ++ss, ++epoch) {
      if (io_group) {
        if (epoch > 0) io_mark(s, 18);
        if (!(actions && epoch == 0)) stage_pre(s, ss, epoch);  // (epoch 0 with a prologue: done above)
        io_mark(s, 20);
        // damping / armature (and, after the first sub-step of a policy step, the unchanged torque) are copied while
        // the torque stage runs: the copies only touch their own slots
        slab_stage_dofpar(m, k.s, c.hot, envs, es, e0, nenv, ss > 0, it, kIoThreads);
        if (ss == 0) {
          torque_stage_slab(torque_args(k), e0, nenv, envs, es, dof_link, it, kIoThreads);
          io_group_sync();  // every thread has read simul_len
          stage_simul_len_update(torque_args(k), e0, nenv, it, kIoThreads);
        }
        io_mark(s, 21);
        cp_async_wait_all();
        io_group_sync();
        if (it == 0) st_release_shared(c.ioflags + F_IO_TAU, epoch + 1);
        io_mark(s, 22);
        // off the critical path: the sensor noise of the previous policy sub-step
        if (ss == 0 && s > 0) noise_stage_slab(noise_args(k), s - 1, e0, nenv, envs, es, dof_link, it, kIoThreads);
        io_group_sync();
        if (it == 0) st_release_shared(c.ioflags + F_IO_DONE, epoch + 1);
        if (s + 1 == k.p.skipframe && ss + 1 == p.substeps) {
          // idle from here on: request the rows the post-physics launch will read and this launch never touched
          // (history rings, previous-step copies), so that with a cold L2 it finds them in L2 instead of in HBM
          const size_t e = (size_t)e0;
          slab_prefetch_l2(k.b.obs_history + e * NSLOT * NOBS1, (unsigned)nenv * NSLOT * NOBS1 * 4, it, kIoThreads);
          slab_prefetch_l2(k.b.action_history + e * NSLOT * NA, (unsigned)nenv * NSLOT * NA * 4, it, kIoThreads);
          slab_prefetch_l2(k.b.contact_forces_pre + e * NB * 3, (unsigned)nenv * NB * 3 * 4, it, kIoThreads);
          slab_prefetch_l2(k.b.pre_joint_velocity_states + e * ND, (unsigned)nenv * ND * 4, it, kIoThreads);
          slab_prefetch_l2(k.b.actions_pre + e * NA, (unsigned)nenv * NA * 4, it, kIoThreads);
          slab_prefetch_l2(k.b.qpos_bias + e * 12, (unsigned)nenv * 12 * 4, it, kIoThreads);
        }
      } else {
        io.push = s == 0;
        io.link_pose = (s + 1 == k.p.skipframe && ss + 1 == p.substeps && k.s.link_pose) ? k.s.link_pose + (size_t)c.e * m.nl * 12 : nullptr;
        sync.mark(13);
        if (c.active) env_substep_lanes(io, c.sm, c.qflags, c.ioflags, epoch, c.hot, m, p, c.role, sync, c.g, true);
      }
      __syncthreads();
    }
    if (s + 1 == k.p.skipframe) {  // last policy sub-step: its noise stage on the I/O group, the state write-back on the role warps
      if (io_group) noise_stage_slab(noise_args(k), s, e0, nenv, envs, es, dof_link, it, kIoThreads);
      else slab_store_outputs(m, k.s, c.hot, envs, es, e0, nenv, threadIdx.x, c.nrole);
    }
    sync.mark(15);
    if (sync.trace) sync.trace += DYROS_LANES * 32;
  }
  __syncthreads();
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[26] = clock64();  // all outputs written (profiling)
}

}  // namespace lanes_impl
using namespace lanes_impl;

static size_t phys_smem_bytes_lanes(const Sim* sim, int epb) {
  const int nq = (epb + kEnvsPerWarp - 1) / kEnvsPerWarp;
  return (size_t)sim->m.hot_bytes + ((size_t)IOF_COUNT + (size_t)nq * QF_COUNT + (size_t)epb * env_scratch_floats(sim->m.nl, sim->m.nb)) * sizeof(float);
}

int physics_configure_lanes(Sim* sim) {
  int epb = (sim->p.N + sim->sm_count - 1) / sim->sm_count;  // one wave when it fits
  epb = std::max(epb, 8);
  epb = std::min(epb, kMaxEpb);
  while (epb > 1 && phys_smem_bytes_lanes(sim, epb) > (size_t)kMaxPhysSmem) --epb;
  if (phys_smem_bytes_lanes(sim, epb) > (size_t)kMaxPhysSmem) {
    set_error("physics_configure: one env needs %zu bytes of shared memory", phys_smem_bytes_lanes(sim, 1));
    return 1;
  }
  sim->envs_per_block = epb;
  sim->phys_smem = phys_smem_bytes_lanes(sim, epb);
  DY_CUDA(cudaFuncSetAttribute(k_simulate_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPhysSmem));
  DY_CUDA(cudaFuncSetAttribute(k_step_physics_lanes, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPhysSmem));
  return 0;
}

int physics_role_threads_lanes(const Sim* sim) { return ((sim->envs_per_block + kEnvsPerWarp - 1) / kEnvsPerWarp) * DYROS_LANES * 32; }
int physics_step_threads_lanes(const Sim* sim) { return physics_role_threads_lanes(sim) + kIoThreads; }

int launch_simulate_lanes(Sim* sim, int apply_wrench, const float* push, cudaStream_t s) {
  const int epb = sim->envs_per_block;
  const int grid = (sim->p.N + epb - 1) / epb;
  k_simulate_lanes<<<grid, physics_role_threads_lanes(sim), sim->phys_smem, s>>>(sim->m, sim->p, sim->b, push, apply_wrench, epb,
                                                                     env_scratch_floats(sim->m.nl, sim->m.nb));
  DY_LAUNCH_CHECK();
  return 0;
}

int launch_task_physics_lanes(Task* t, cudaStream_t s, long long* trace, bool pdl, const float* actions) {
  Sim* sim = t->sim;
  const int epb = sim->envs_per_block;
  const int grid = (sim->p.N + epb - 1) / epb;
  TK k;
  k.p = t->p;
  k.b = t->b;
  k.s = sim->b;
  k.j = t->inj;
  k.c = t->cur;
  DY_CUDA(launch_kernel(k_step_physics_lanes, dim3(grid), dim3(physics_step_threads_lanes(sim)), sim->phys_smem, s, pdl, sim->m, sim->p, k, epb,
                        env_scratch_floats(sim->m.nl, sim->m.nb), trace, actions));
  return 0;
}

}  // namespace dyros
