// K1, multi-lane variant (DyrosSimDesc.physics_program = 1; the default is the one-lane-per-env role program of
// physics_kernels.cu: at 28 envs per SM the multi-lane mapping measured SLOWER, 158 vs 87 us per launch at 4096 envs,
// profiles/r2b_*; DESIGN.md section 4 has the numbers and the reasons. Kept selectable, built and parity-tested.)
// gym.simulate as one kernel launch, multi-lane (physics_lanes.cuh): 8 lanes per env, 4 envs per warp, one warp
// per role and group of 4 envs; up to 28 envs per CTA (7 groups x 4 role warps = 28 warps, + 4 I/O warps in the fused
// step = 1024 threads, one CTA per SM: N = 4096 is a single wave on 148 SMs). The per-env scratch blocks, the hot model
// tables and the dataflow flags live in dynamic shared memory.
#include "physics_lanes.cuh"
#include "physics_cta.cuh"

namespace dyros {
using namespace ln;
namespace lanes_impl {  // (PhysCta, phys_cta_setup and env_io of the role program are defined in namespace dyros)

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

constexpr int kEnvsPerWarp = 32 / LPE;           // 4
constexpr int kMaxQuads = 7;                     // groups of 4 envs per CTA
constexpr int kMaxEpb = kMaxQuads * kEnvsPerWarp;
static_assert(kMaxEpb <= kSlabMaxEnvs, "slab stages are sized for kSlabMaxEnvs envs per CTA");
static_assert(DYROS_LANES == 4, "four roles per group of envs");
static_assert(F_IO_TAU == F_IO_PRE + 1 && F_IO_DONE == F_IO_PRE + 2, "step_physics_body takes the I/O flags in this order");

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

__global__ void __launch_bounds__(kMaxQuads * DYROS_LANES * 32) k_simulate_lanes(DevModel m, SimParams p, DyrosSimBuffers b,
                                                                          const float* __restrict__ push, int apply_wrench, int epb, int es) {
  extern __shared__ __align__(16) float smem[];
  PhysCta c = phys_cta_setup(m, p, smem, epb, es);
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  EnvIO io = env_io(m, b, c.e, c.live);
  io.push = push != nullptr;
  io.rb_force = apply_wrench ? b.rb_force + (size_t)c.e * m.nb * 3 : nullptr;
  io.rb_torque = apply_wrench ? b.rb_torque + (size_t)c.e * m.nb * 3 : nullptr;
  LaneSync sync{c.lane, nullptr};
  simulate_body<LanesScratch>(m, p, b, push, c.hot, c.envs, es, e0, nenv, blockDim.x, c.e, io, [&](int s) __attribute__((always_inline)) {
    if (c.active) env_substep_lanes(io, c.sm, c.qflags, c.ioflags, s, c.hot, m, p, c.role, sync, c.g, false);
  });
}

constexpr int kStepThreadsMax = kMaxQuads * DYROS_LANES * 32 + kIoThreads;  // 1024

// one sub-step of the role program in the fused step (step_physics_body)
__device__ __forceinline__ void role_substep(PhysCta& c, EnvIO& io, LaneSync& sync, const DevModel& m, const SimParams& p,
                                             const TK& k, int s, int ss, int epoch) {
  io.push = s == 0;
  io.link_pose = (s + 1 == k.p.skipframe && ss + 1 == p.substeps && k.s.link_pose) ? k.s.link_pose + (size_t)c.e * m.nl * 12 : nullptr;
  sync.mark(13);
  if (c.active) env_substep_lanes(io, c.sm, c.qflags, c.ioflags, epoch, c.hot, m, p, c.role, sync, c.g, true);
}

// The fused policy step (step_physics_body): the first c.nrole threads run the role programs, the last 4 warps are the
// I/O group; the CTA's size follows its envs, so its named barriers take blockDim.x.
__global__ void __launch_bounds__(kStepThreadsMax) k_step_physics_lanes(DevModel m, SimParams p, TK k, int epb, int es, long long* trace,
                                                                   const float* __restrict__ actions) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float pro[kSlabMaxEnvs][8];  // per-env scalars of the prologue (stage_prologue_slab)
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[24] = clock64();  // kernel entry (profiling)
  PhysCta c = phys_cta_setup(m, p, smem, epb, es);
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[25] = clock64();  // tables staged, previous kernel done
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  const int nthreads = blockDim.x;
  const bool io_group = (int)threadIdx.x >= c.nrole;
  const int it = threadIdx.x - c.nrole;  // thread index within the I/O group
  EnvIO io = env_io(m, k.s, c.e, c.live);
  // trace layout: [sub-step][role][32 marks], taken by the role warps of the first group of CTA 0
  LaneSync sync{c.lane, (trace && blockIdx.x == 0 && !io_group && c.quad == 0 && (threadIdx.x >> 7) == 0) ? trace + c.role * 32 : nullptr};
  step_physics_body<LanesScratch>(m, p, k, trace, actions, pro, c.hot, c.envs, c.ioflags + F_IO_PRE, es, e0, nenv, c.nrole, it,
                                  nthreads, io_group, c, io, sync);
}

}  // namespace lanes_impl
using namespace lanes_impl;

static size_t phys_smem_bytes_lanes(const Sim* sim, int epb) {
  const int nq = (epb + kEnvsPerWarp - 1) / kEnvsPerWarp;
  return (size_t)sim->m.hot_bytes + ((size_t)IOF_COUNT + (size_t)nq * QF_COUNT + (size_t)epb * env_scratch_floats(sim->m.nl, sim->m.nb)) * sizeof(float);
}

int physics_configure_lanes(Sim* sim) {
  if (physics_choose_envs_per_block(sim, kMaxEpb, phys_smem_bytes_lanes)) return 1;
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
  DY_CUDA(launch_kernel(k_step_physics_lanes, dim3(grid), dim3(physics_step_threads_lanes(sim)), sim->phys_smem, s, pdl, sim->m, sim->p, make_tk(t), epb,
                        env_scratch_floats(sim->m.nl, sim->m.nb), trace, actions));
  return 0;
}

}  // namespace dyros
