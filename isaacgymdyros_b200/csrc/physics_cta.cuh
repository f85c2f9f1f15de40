// The CTA layer shared by the two physics programs' kernels (physics_kernels.cu: the role program of physics_roles.cuh,
// one lane per env; physics_lanes_kernels.cu: the multi-lane program of physics_lanes.cuh): shared-memory flags, the
// coalesced slab copies between the API tensors and the env scratch blocks, the task's slab stages, and the bodies of
// the two launches, gym.simulate (simulate_body) and the fused policy step (step_physics_body).
// What differs between the programs is a compile-time scratch layout `L` (RolesScratch, LanesScratch: word offsets in
// an env's scratch block) and what the kernels pass in: the role-thread count, the I/O flags, the barrier count and one
// sub-step of the role program (a callable for simulate_body, the program's role_substep for step_physics_body).
#pragma once
#include <type_traits>

#include "task_stages.cuh"

namespace dyros {

constexpr int kMaxPhysSmem = 227 * 1024 - 1024;  // dynamic part; 1 KiB is left for static shared memory (k_step_physics: 1 KiB)
constexpr int kIoThreads = 128;                  // the I/O group of the fused step: 4 warps
constexpr int kSlabVThreads = 128;               // virtual thread count the slab stages of task_stages.cuh are written for

__device__ __forceinline__ int ld_acquire_shared(const int* p) {
  int v;
  asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_shared(int* p, int v) {
  asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
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
__device__ __forceinline__ void io_group_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kIoThreads) : "memory"); }

// Named barrier `Id` of all `n` threads of the CTA. A count that is a compile-time constant (std::integral_constant)
// goes into the instruction as an immediate; an int (a CTA whose size is chosen at launch) in a register.
template <int Id, class N>
__device__ __forceinline__ void cta_bar_sync(N n) {
  if constexpr (std::is_integral_v<N>) asm volatile("bar.sync %0, %1;" ::"n"(Id), "r"(n) : "memory");
  else asm volatile("bar.sync %0, %1;" ::"n"(Id), "n"(N::value) : "memory");
}
template <int Id, class N>
__device__ __forceinline__ void cta_bar_arrive(N n) {
  if constexpr (std::is_integral_v<N>) asm volatile("bar.arrive %0, %1;" ::"n"(Id), "r"(n) : "memory");
  else asm volatile("bar.arrive %0, %1;" ::"n"(Id), "n"(N::value) : "memory");
}

// The copies below are issued by thread `tid` of `nthreads` cooperating threads (a CTA's role warps, or the I/O group);
// the caller waits with cp_async_wait_all() and then synchronises the cooperating threads.
// (1) joint state, mass scales and root: once per launch (they stay in the scratch blocks)
template <class L>
__device__ __forceinline__ void slab_stage_state(const DevModel& m, const DyrosSimBuffers& b, const float* hot, float* envs, int es,
                                                 int e0, int nenv, int tid, int nthreads, float mu) {
  const int nd = m.nd, nb = m.nb, xoff = m.nl * L::link;
#pragma unroll 1
  for (int le = tid; le < nenv; le += nthreads) {  // per-env friction (DR) or the sim's coefficient
    if (b.contact_friction) cp_async4(envs + le * es + xoff + L::mu, b.contact_friction + e0 + le);
    else envs[le * es + xoff + L::mu] = mu;
  }
  const int* dof_link = reinterpret_cast<const int*>(hot) + m.o_dof_link;
  const FastDiv d2nd(2 * nd), dnb(nb), d13(13);  // slabs are < 2^20 / divisor words (checked at create)
  {
    const float* src = b.dof_state + (size_t)e0 * nd * 2;
#pragma unroll 1
    for (int i = tid; i < nenv * nd * 2; i += nthreads) {
      int le = d2nd.div(i), w = i - le * 2 * nd;
      cp_async4(envs + le * es + dof_link[w >> 1] * L::link + ((w & 1) ? L::qd : L::q), src + i);
    }
  }
  {
    const float* src = b.body_mass_scale + (size_t)e0 * nb;
#pragma unroll 1
    for (int i = tid; i < nenv * nb; i += nthreads) {
      int le = dnb.div(i);
      cp_async4(envs + le * es + xoff + L::mass + (i - le * nb), src + i);
    }
  }
  {
    const float* src = b.root_states + (size_t)e0 * 13;
#pragma unroll 1
    for (int i = tid; i < nenv * 13; i += nthreads) {
      int le = d13.div(i);
      cp_async4(envs + le * es + xoff + L::root + (i - le * 13), src + i);
    }
  }
}
// (2) per sub-step, needed by the force loop of pass 1: the push, and the zeroed net contact forces (THIS sub-step only)
template <class L>
__device__ __forceinline__ void slab_stage_pre(const DevModel& m, const DyrosSimBuffers& b, const float* push, float* envs, int es,
                                               int e0, int nenv, int tid, int nthreads) {
  const int nb = m.nb, xoff = m.nl * L::link;
  const FastDiv d3(3);
#pragma unroll 1
  for (int i = tid; i < nenv * 3; i += nthreads) {
    int le = d3.div(i);
    if (push) cp_async4(envs + le * es + xoff + L::push + (i - le * 3), push + (size_t)e0 * 3 + i);
    else envs[le * es + xoff + L::push + (i - le * 3)] = 0.f;
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
template <class L>
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
    float* blk = envs + le * es + dof_link[d] * L::link;
    if (with_tau) cp_async4(blk + L::tau, tau + i);
    cp_async4(blk + L::damping, dmp + i);
    cp_async4(blk + L::armature, arm + i);
  }
}

template <class L>
__device__ __forceinline__ void slab_store_outputs(const DevModel& m, const DyrosSimBuffers& b, const float* hot,
                                                   const float* envs, int es, int e0, int nenv, int tid, int nthreads) {
  const int nd = m.nd, xoff = m.nl * L::link;
  const int* dof_link = reinterpret_cast<const int*>(hot) + m.o_dof_link;
  const FastDiv d2nd(2 * nd), d13(13);
  float* ds = b.dof_state + (size_t)e0 * nd * 2;
#pragma unroll 2
  for (int i = tid; i < nenv * nd * 2; i += nthreads) {
    int le = d2nd.div(i), w = i - le * 2 * nd;
    ds[i] = envs[le * es + dof_link[w >> 1] * L::link + ((w & 1) ? L::qd : L::q)];
  }
  float* rs = b.root_states + (size_t)e0 * 13;
#pragma unroll 1
  for (int i = tid; i < nenv * 13; i += nthreads) {
    int le = d13.div(i);
    rs[i] = envs[le * es + xoff + L::root + (i - le * 13)];
  }
}

// The task's slab stages are compiled as separate functions so that their (large, short-lived) register arrays do not
// raise the register pressure of the role programs. `tid0` of `nreal` real threads act as kSlabVThreads virtual threads.
template <class L>
__device__ __noinline__ void torque_stage_slab(TorqueSlabArgs k, int e0, int nenv, float* envs, int es, const int* dof_link,
                                               int tid0, int nreal) {
  // joint state comes from the scratch blocks; the torques go to the API tensor and straight into the scratch blocks
#pragma unroll 1
  for (int vt = tid0; vt < kSlabVThreads; vt += nreal)
    stage_substep_torque_cta(
        k, e0, nenv, vt, kSlabVThreads, [&](int le, int d, float v) { envs[le * es + dof_link[d] * L::link + L::tau] = v; },
        [&](int le, int d, int which) { return envs[le * es + dof_link[d] * L::link + (which ? L::qd : L::q)]; });
}
template <class L>
__device__ __noinline__ void noise_stage_slab(NoiseSlabArgs k, int substep, int e0, int nenv, const float* envs, int es,
                                              const int* dof_link, int tid0, int nreal) {
  // sensor noise reads the fresh joint angles from the scratch blocks
#pragma unroll 1
  for (int vt = tid0; vt < kSlabVThreads; vt += nreal)
    stage_sensor_noise_cta(k, substep, e0, nenv, vt, kSlabVThreads,
                           [&](int le, int d) { return envs[le * es + dof_link[d] * L::link + L::q]; });
}

// gym.simulate as one launch: per sub-step, the `nthreads` threads of the CTA stage the inputs of its envs, then
// `substep(s)` runs sub-step s of the role program on the calling warp; after the last one they write the state back.
// `io` is the calling thread's EnvIO (env `e`): the link poses are exported in the last sub-step. The kernels declare
// `substep` __attribute__((always_inline)): like a __forceinline__ function, it is then inlined before the optimiser
// sees the kernel, which compiles as if the role program were called directly.
template <class L, class IO, class Substep>
__device__ __forceinline__ void simulate_body(const DevModel& m, const SimParams& p, const DyrosSimBuffers& b, const float* push,
                                              const float* hot, float* envs, int es, int e0, int nenv, int nthreads, int e,
                                              IO& io, Substep substep) {
  for (int s = 0; s < p.substeps; ++s) {
    // (first sub-step: the staged tables are still in flight, dof_link is read from the global copy)
    const float* tab = s == 0 ? reinterpret_cast<const float*>(m.blob) : hot;
    if (s == 0) slab_stage_state<L>(m, b, tab, envs, es, e0, nenv, threadIdx.x, nthreads, p.mu);
    slab_stage_pre<L>(m, b, push, envs, es, e0, nenv, threadIdx.x, nthreads);
    slab_stage_dofpar<L>(m, b, tab, envs, es, e0, nenv, true, threadIdx.x, nthreads);
    cp_async_wait_all();
    __syncthreads();
    io.link_pose = (s + 1 == p.substeps && b.link_pose) ? b.link_pose + (size_t)e * m.nl * 12 : nullptr;
    substep(s);
    __syncthreads();
    // (applied wrenches act over the whole simulate() call, i.e. all of its sub-steps: gym_py.html apply_rigid_body_force_tensors)
    if (s + 1 == p.substeps) slab_store_outputs<L>(m, b, hot, envs, es, e0, nenv, threadIdx.x, nthreads);
  }
}

// The physics part of one policy step in ONE launch: skipframe x (PD + delay torque, gym.simulate, sensor noise),
// i.e. the loop body of T:504-530 with the three gym calls of T:520-526 folded in; with `actions` also the part of
// pre_physics_step before that loop (T:449-502).
// The first `nrole` threads run the role programs; the last 4 warps are the I/O group: while the roles are in pass 1 of
// a sub-step it zeroes the contact forces and stages the push (F_IO_PRE), draws the sensor noise of the PREVIOUS policy
// sub-step (which only reads the joint angles, untouched until the roles' last pass), evaluates the torque stage and
// re-stages damping and armature (F_IO_TAU, consumed by pass 2), so none of this sits on the roles' critical path.
// `io_flags` points at the I/O group's flags F_IO_PRE, F_IO_TAU and F_IO_DONE, in this order; `it` is the thread's
// index within the I/O group and `nbar` the CTA size for the named barriers (cta_bar_sync). The role warps run
// role_substep(c, io, sync, m, p, k, s, ss, epoch, extra...), which each program defines for its PhysCta `c`: one
// sub-step of the role program with the calling thread's EnvIO `io`, for sub-step ss of policy sub-step s, `epoch`
// counting the sub-steps of the launch; `sync` also takes the role warps' trace marks. (A function rather than a
// callable as in simulate_body, and `envs` by reference: here, reaching the kernel's locals through one more level of
// indirection changes what the optimiser makes of them, and the kernels would no longer compile to the same code as
// when each program spelt this body out.)
template <class L, class NBar, class Cta, class IO, class Sync, class... Extra>
__device__ __forceinline__ void step_physics_body(const DevModel& m, const SimParams& p, const TK& k, long long* trace,
                                                  const float* __restrict__ actions, float (*pro)[8], const float* hot,
                                                  float* const& envs, int* io_flags, int es, int e0, int nenv, int nrole,
                                                  int it, NBar nbar, bool io_group, Cta& c, IO& io, Sync& sync,
                                                  const Extra&... extra) {
  const int* dof_link = reinterpret_cast<const int*>(hot) + m.o_dof_link;
  // (profiling: marks 18.. of role 0's row are the I/O group's phase boundaries)
  auto io_mark = [&](int s, int id) {
    if (trace && blockIdx.x == 0 && it == 0) trace[(size_t)s * DYROS_LANES * 32 + id] = clock64();
  };
  // per sub-step, I/O group: the push (every sub-step of the first simulate of the policy step, T:502 vs T:504) and the
  // zeroed contact forces
  auto stage_pre = [&](int s, int ss, int epoch) {
    slab_stage_pre<L>(m, k.s, s == 0 ? k.b.push_force : nullptr, envs, es, e0, nenv, it, kIoThreads);
    cp_async_wait_all();
    io_group_sync();
    if (it == 0) st_release_shared(io_flags + 0, epoch + 1);
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
    cta_bar_arrive<3>(nbar);
    io_mark(0, 18);
    if (actions) {  // the policy-step prologue (T:449-502) of the CTA's envs; the push it decides is staged at its end
      stage_prologue_slab(k, actions, e0, nenv, it, kIoThreads, pro, [] { io_group_sync(); }, [&] { stage_pre(0, 0, 0); });
      io_group_sync();
    }
    cta_bar_sync<4>(nbar);
  } else {
    // joint state, root and mass scales are staged once and then live in the scratch blocks for the whole launch; the
    // torque and noise stages read them there, and only the final state is written back
    // (the staged tables are still in flight: dof_link is read from the global copy here)
    slab_stage_state<L>(m, k.s, reinterpret_cast<const float*>(m.blob), envs, es, e0, nenv, threadIdx.x, nrole, p.mu);
    cp_async_wait_all();  // this thread's share of the tables and of the state
    cta_bar_sync<3>(nbar);
    cta_bar_arrive<4>(nbar);
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
        slab_stage_dofpar<L>(m, k.s, hot, envs, es, e0, nenv, ss > 0, it, kIoThreads);
        if (ss == 0) {
          torque_stage_slab<L>(torque_args(k), e0, nenv, envs, es, dof_link, it, kIoThreads);
          io_group_sync();  // every thread has read simul_len
          stage_simul_len_update(torque_args(k), e0, nenv, it, kIoThreads);
        }
        io_mark(s, 21);
        cp_async_wait_all();
        io_group_sync();
        if (it == 0) st_release_shared(io_flags + 1, epoch + 1);
        io_mark(s, 22);
        // off the critical path: the sensor noise of the previous policy sub-step
        if (ss == 0 && s > 0) noise_stage_slab<L>(noise_args(k), s - 1, e0, nenv, envs, es, dof_link, it, kIoThreads);
        io_group_sync();
        if (it == 0) st_release_shared(io_flags + 2, epoch + 1);
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
        role_substep(c, io, sync, m, p, k, s, ss, epoch, extra...);
      }
      __syncthreads();
    }
    if (s + 1 == k.p.skipframe) {  // last policy sub-step: its noise stage on the I/O group, the state write-back on the role warps
      if (io_group) noise_stage_slab<L>(noise_args(k), s, e0, nenv, envs, es, dof_link, it, kIoThreads);
      else slab_store_outputs<L>(m, k.s, hot, envs, es, e0, nenv, threadIdx.x, nrole);
    }
    sync.mark(15);
    if (sync.trace) sync.trace += DYROS_LANES * 32;
  }
  __syncthreads();
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[26] = clock64();  // all outputs written (profiling)
}

// Envs per CTA of a physics program: one wave when it fits, at least 8 and at most `max_epb`, fewer while the CTA's
// shared memory (`smem_bytes`) exceeds kMaxPhysSmem. Sets sim->envs_per_block and sim->phys_smem; 1 when one env does
// not fit.
inline int physics_choose_envs_per_block(Sim* sim, int max_epb, size_t (*smem_bytes)(const Sim*, int)) {
  int epb = (sim->p.N + sim->sm_count - 1) / sim->sm_count;  // one wave when it fits
  epb = std::max(epb, 8);
  epb = std::min(epb, max_epb);
  while (epb > 1 && smem_bytes(sim, epb) > (size_t)kMaxPhysSmem) --epb;
  if (smem_bytes(sim, epb) > (size_t)kMaxPhysSmem) {
    set_error("physics_configure: one env needs %zu bytes of shared memory", smem_bytes(sim, 1));
    return 1;
  }
  sim->envs_per_block = epb;
  sim->phys_smem = smem_bytes(sim, epb);
  return 0;
}

}  // namespace dyros
