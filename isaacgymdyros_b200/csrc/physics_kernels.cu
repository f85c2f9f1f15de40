// K1: gym.simulate as one kernel launch, warp-specialised: one warp per role (physics_roles.cuh), lane = env, up to 32
// envs per CTA (28 for N = 4096, so that one CTA per SM covers the shard in a single wave); the per-env scratch
// blocks, the hot model tables and the dataflow flags live in dynamic shared memory.
#include "physics_roles.cuh"
#include "physics_cta.cuh"

namespace dyros {

// Flags between role warps: the producer's lanes finish their shared-memory writes, lane 0 publishes with release;
// the consumer's lanes spin with acquire.
struct RoleSync {
  int lane;
  long long* trace;  // profiling aid: clock64() at the phase boundaries of one CTA (NULL in production)
  __device__ __forceinline__ void mark(int id) const {
    if (trace && lane == 0) trace[id] = clock64();
  }
  __device__ __forceinline__ void signal(int* f, int v) const {
    __syncwarp();
    if (lane == 0) st_release_shared(f, v);
  }
  // every lane polls (one broadcast load per iteration): the loop branch is warp-uniform, so the warp never splits
  // into a lane-0 group and a rest group that would then run the following phase twice
  __device__ __forceinline__ void wait(const int* f, int v) const {
    while (ld_acquire_shared(f) < v) {
    }
  }
  // for flags published by the I/O warps, which share the schedulers with the role warps: back off between polls so
  // that the waiting warp does not take issue slots from the warp it is waiting for
  __device__ __forceinline__ void wait_io(const int* f, int v) const {
    while (ld_acquire_shared(f) < v) __nanosleep(100);
  }
};

constexpr int kPhysThreads = DYROS_LANES * 32;
static_assert(F_IO_TAU == F_IO_PRE + 1 && F_IO_DONE == F_IO_PRE + 2, "step_physics_body takes the I/O flags in this order");

struct PhysCta {
  const float* hot;
  int* flags;
  real* sm;     // this lane's env scratch block
  int role, lane, e;
  bool live;
};

// Common prologue of the physics kernels: stage the hot tables, clear the flags, locate the lane's env.
// `flag_thread0`: first of the F_COUNT consecutive threads that clear the flags (the fused step lets its I/O group do
// it, which is also the first to publish one).
__device__ __forceinline__ PhysCta phys_cta_setup(const DevModel& m, const SimParams& p, float* smem, int epb, int es,
                                                  int flag_thread0 = 0) {
  {  // 16-byte cp.async: in flight together with the state copies issued after griddepcontrol.wait (the caller waits)
    const char* src = reinterpret_cast<const char*>(m.blob);
    for (int i = threadIdx.x; i < m.hot_bytes / 16; i += blockDim.x)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem) + i * 16), "l"(src + (size_t)i * 16)
                   : "memory");
  }
  int* flags = reinterpret_cast<int*>(smem + m.hot_bytes / 4);
  static_assert(F_COUNT <= kPhysThreads, "one thread per flag");
  if ((int)threadIdx.x >= flag_thread0 && (int)threadIdx.x < flag_thread0 + F_COUNT) flags[threadIdx.x - flag_thread0] = 0;
  pdl_launch_dependents();
  pdl_wait();  // everything above is independent of the previous kernel of the step (model tables only)
  PhysCta c;
  c.hot = smem;
  c.flags = flags;
  c.role = threadIdx.x >> 5;
  c.lane = threadIdx.x & 31;
  const int le = c.lane < epb ? c.lane : epb - 1;  // padding lanes shadow the last env (same values, no global writes)
  int e = blockIdx.x * epb + le;
  c.live = c.lane < epb && e < p.N;
  c.e = e < p.N ? e : p.N - 1;
  c.sm = smem + m.hot_bytes / 4 + ((F_COUNT + 3) & ~3) + (size_t)le * es;
  return c;
}

__device__ __forceinline__ EnvIO env_io(const DevModel& m, const DyrosSimBuffers& b, int e, bool live) {
  EnvIO io;
  io.root = b.root_states + (size_t)e * 13;
  io.dof_state = b.dof_state + (size_t)e * m.nd * 2;
  io.tau = b.dof_actuation_force + (size_t)e * m.nd;
  io.damping = b.dof_damping + (size_t)e * m.nd;
  io.armature = b.dof_armature + (size_t)e * m.nd;
  io.mass_scale = b.body_mass_scale + (size_t)e * m.nb;
  io.friction = b.contact_friction ? b.contact_friction + e : nullptr;
  io.contact = b.net_contact_force + (size_t)e * m.nb * 3;
  io.push = nullptr;
  io.rb_force = nullptr;
  io.rb_torque = nullptr;
  io.link_pose = nullptr;
  io.live = live;
  return io;
}

// (both kernels are instantiated for each ground, PlaneGround and FieldGround: physics_roles.cuh)
template <class Ground>
__global__ void __launch_bounds__(kPhysThreads) k_simulate(DevModel m, SimParams p, DyrosSimBuffers b, const float* __restrict__ push,
                                                           int apply_wrench, int epb, int es, Ground gnd) {
  extern __shared__ __align__(16) float smem[];
  PhysCta c = phys_cta_setup(m, p, smem, epb, es);
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  float* envs = smem + m.hot_bytes / 4 + ((F_COUNT + 3) & ~3);
  EnvIO io = env_io(m, b, c.e, c.live);
  io.push = push ? push + (size_t)c.e * 3 : nullptr;
  io.rb_force = apply_wrench ? b.rb_force + (size_t)c.e * m.nb * 3 : nullptr;
  io.rb_torque = apply_wrench ? b.rb_torque + (size_t)c.e * m.nb * 3 : nullptr;
  RoleSync sync{c.lane, nullptr};
  simulate_body<RolesScratch>(m, p, b, push, c.hot, envs, es, e0, nenv, kPhysThreads, c.e, io, [&](int s) __attribute__((always_inline)) {
    env_substep_role(io, c.sm, c.flags, s, c.hot, m, p, c.role, sync, false, gnd);
  });
}

constexpr int kStepThreads = kPhysThreads + kIoThreads;

// one sub-step of the role program in the fused step (step_physics_body)
template <class Ground>
__device__ __forceinline__ void role_substep(PhysCta& c, EnvIO& io, RoleSync& sync, const DevModel& m, const SimParams& p,
                                             const TK& k, int s, int ss, int epoch, const int& role, const Ground& gnd) {
  io.push = s == 0 ? k.b.push_force : nullptr;  // every sub-step of the first simulate of the policy step (T:502 vs T:504)
  io.link_pose = (s + 1 == k.p.skipframe && ss + 1 == p.substeps && k.s.link_pose) ? k.s.link_pose + (size_t)c.e * m.nl * 12 : nullptr;
  sync.mark(13);
  env_substep_role(io, c.sm, c.flags, epoch, c.hot, m, p, role, sync, true, gnd);
}

// The fused policy step (step_physics_body): warps 0-3 run the role programs, warps 4-7 are the I/O group.
template <class Ground>
__global__ void __launch_bounds__(kStepThreads) k_step_physics(DevModel m, SimParams p, TK k, int epb, int es, long long* trace,
                                                                const float* __restrict__ actions, Ground gnd) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float pro[kSlabMaxEnvs][8];  // per-env scalars of the prologue (stage_prologue_slab)
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[24] = clock64();  // kernel entry (profiling)
  PhysCta c = phys_cta_setup(m, p, smem, epb, es, kPhysThreads);
  if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[25] = clock64();  // tables staged, previous kernel done
  const int e0 = blockIdx.x * epb, nenv = min(epb, p.N - e0);
  float* envs = smem + m.hot_bytes / 4 + ((F_COUNT + 3) & ~3);
  const bool io_group = c.role >= DYROS_LANES;
  const int role = c.role & (DYROS_LANES - 1);
  const int it = threadIdx.x - kPhysThreads;  // thread index within the I/O group
  EnvIO io = env_io(m, k.s, c.e, c.live);
  // trace layout: [sub-step][role][32 marks]
  RoleSync sync{c.lane, (trace && blockIdx.x == 0 && !io_group) ? trace + role * 32 : nullptr};
  step_physics_body<RolesScratch>(m, p, k, trace, actions, pro, c.hot, envs, c.flags + F_IO_PRE, es, e0, nenv, kPhysThreads, it,
                                  std::integral_constant<int, kStepThreads>(), io_group, c, io, sync, role, gnd);
}

static size_t phys_smem_bytes(const Sim* sim, int epb) {
  return (size_t)sim->m.hot_bytes + (((F_COUNT + 3) & ~3) + (size_t)epb * env_scratch_floats(sim->m.nl, sim->m.nb)) * sizeof(float);
}

static int physics_configure_roles(Sim* sim) {
  if (physics_choose_envs_per_block(sim, 32, phys_smem_bytes)) return 1;
  DY_CUDA(cudaFuncSetAttribute(k_simulate<PlaneGround>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPhysSmem));
  DY_CUDA(cudaFuncSetAttribute(k_step_physics<PlaneGround>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPhysSmem));
  DY_CUDA(cudaFuncSetAttribute(k_simulate<FieldGround>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPhysSmem));
  DY_CUDA(cudaFuncSetAttribute(k_step_physics<FieldGround>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPhysSmem));
  return 0;
}

static int launch_simulate_roles(Sim* sim, int apply_wrench, const float* push, cudaStream_t s) {
  const int epb = sim->envs_per_block;
  const int grid = (sim->p.N + epb - 1) / epb;
  if (sim->has_field)
    k_simulate<<<grid, kPhysThreads, sim->phys_smem, s>>>(sim->m, sim->p, sim->b, push, apply_wrench, epb, env_scratch_floats(sim->m.nl, sim->m.nb),
                                                     sim->field);
  else
    k_simulate<<<grid, kPhysThreads, sim->phys_smem, s>>>(sim->m, sim->p, sim->b, push, apply_wrench, epb, env_scratch_floats(sim->m.nl, sim->m.nb),
                                                     PlaneGround());
  DY_LAUNCH_CHECK();
  return 0;
}

static int launch_task_physics_roles(Task* t, cudaStream_t s, long long* trace, bool pdl, const float* actions) {
  Sim* sim = t->sim;
  const int epb = sim->envs_per_block;
  const int grid = (sim->p.N + epb - 1) / epb;
  if (sim->has_field)
    DY_CUDA(launch_kernel(k_step_physics<FieldGround>, dim3(grid), dim3(kStepThreads), sim->phys_smem, s, pdl, sim->m, sim->p,
                          make_tk(t), epb, env_scratch_floats(sim->m.nl, sim->m.nb), trace, actions, sim->field));
  else
    DY_CUDA(launch_kernel(k_step_physics<PlaneGround>, dim3(grid), dim3(kStepThreads), sim->phys_smem, s, pdl, sim->m, sim->p,
                          make_tk(t), epb, env_scratch_floats(sim->m.nl, sim->m.nb), trace, actions, PlaneGround()));
  return 0;
}

// ---- the two physics programs behind one set of entry points (Sim::program: 0 = roles, the default; 1 = lanes)
int physics_configure(Sim* sim) { return sim->program == 1 ? physics_configure_lanes(sim) : physics_configure_roles(sim); }
int launch_simulate(Sim* sim, int apply_wrench, const float* push, cudaStream_t s) {
  return sim->program == 1 ? launch_simulate_lanes(sim, apply_wrench, push, s) : launch_simulate_roles(sim, apply_wrench, push, s);
}
int launch_task_physics(Task* t, cudaStream_t s, long long* trace, bool pdl, const float* actions) {
  return t->sim->program == 1 ? launch_task_physics_lanes(t, s, trace, pdl, actions) : launch_task_physics_roles(t, s, trace, pdl, actions);
}
int physics_step_threads(const Sim* sim) { return sim->program == 1 ? physics_step_threads_lanes(sim) : kStepThreads; }

// FFMA-saturation micro-benchmark: 8 independent accumulator chains per thread.
__global__ void __launch_bounds__(512) k_ffma_peak(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 4
  for (int i = 0; i < iters; ++i) {
    x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
    x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
  }
  float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 123.456f) out[0] = s;  // never true in practice; keeps the chains alive
}

int measure_fp32_peak(int device, int iters, double* tflops_out) {
  DY_CUDA(cudaSetDevice(device));
  int sms = 0;
  DY_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  float* out = nullptr;
  DY_CUDA(cudaMalloc(&out, sizeof(float)));
  cudaEvent_t e0, e1;
  DY_CUDA(cudaEventCreate(&e0));
  DY_CUDA(cudaEventCreate(&e1));
  const int blocks = sms * 4, threads = 512;
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    DY_CUDA(cudaEventRecord(e0));
    k_ffma_peak<<<blocks, threads>>>(out, iters, 0.999f, 0.001f);
    DY_CUDA(cudaEventRecord(e1));
    DY_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    DY_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    double tf = (double)blocks * threads * 8.0 * iters * 2.0 / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *tflops_out = best;
  return 0;
}

// gym.refresh_rigid_body_state_tensor: forward kinematics of every body (tensors.rst.txt:193-207), one thread per env.
__global__ void __launch_bounds__(64) k_rigid_body_state(DevModel m, SimParams p, DyrosSimBuffers b) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.N) return;
  M3 Rw[DYROS_MAX_LINKS];
  V3 pw[DYROS_MAX_LINKS];
  SV v[DYROS_MAX_LINKS];
  const float* root = b.root_states + (size_t)e * 13;
  const float* ds = b.dof_state + (size_t)e * m.nd * 2;
  Rw[0] = quat_to_mat(root[3], root[4], root[5], root[6]);
  pw[0] = ld3_f(root);
  v[0] = SV{mulT(Rw[0], ld3_f(root + 10)), mulT(Rw[0], ld3_f(root + 7))};
  for (int i = 1; i < m.nl; ++i) {
    int pr = m.link_parent[i], d = m.link_dof[i];
    V3 ax = ld3_f(m.link_axis + 3 * i), r = ld3_f(m.link_r + 3 * i);
    float q = ds[2 * d], qd = ds[2 * d + 1];
    M3 E = mul(axis_rot_T(ax, sinf(q), cosf(q)), ld_m3_f(m.link_E + 9 * i));
    v[i] = xform_motion(E, r, v[pr]);
    v[i].w = v[i].w + qd * ax;
    Rw[i] = mulABt(Rw[pr], E);
    pw[i] = pw[pr] + mul(Rw[pr], r);
  }
  for (int bb = 0; bb < m.nb; ++bb) {
    int l = m.body_link[bb];
    V3 bp = ld3_f(m.body_pos + 3 * bb);
    M3 Rb = mul(Rw[l], ld_m3_f(m.body_rot + 9 * bb));
    V3 pos = pw[l] + mul(Rw[l], bp);
    V3 lin = mul(Rw[l], v[l].v + cross(v[l].w, bp));
    V3 ang = mul(Rw[l], v[l].w);
    // rotation -> quaternion xyzw
    const real* a = Rb.a;
    real tr = a[0] + a[4] + a[8], qx, qy, qz, qw;
    if (tr > 0) {
      real s = sqrtf(tr + 1.f) * 2.f;
      qw = 0.25f * s; qx = (a[7] - a[5]) / s; qy = (a[2] - a[6]) / s; qz = (a[3] - a[1]) / s;
    } else if (a[0] > a[4] && a[0] > a[8]) {
      real s = sqrtf(1.f + a[0] - a[4] - a[8]) * 2.f;
      qw = (a[7] - a[5]) / s; qx = 0.25f * s; qy = (a[1] + a[3]) / s; qz = (a[2] + a[6]) / s;
    } else if (a[4] > a[8]) {
      real s = sqrtf(1.f + a[4] - a[0] - a[8]) * 2.f;
      qw = (a[2] - a[6]) / s; qx = (a[1] + a[3]) / s; qy = 0.25f * s; qz = (a[5] + a[7]) / s;
    } else {
      real s = sqrtf(1.f + a[8] - a[0] - a[4]) * 2.f;
      qw = (a[3] - a[1]) / s; qx = (a[2] + a[6]) / s; qy = (a[5] + a[7]) / s; qz = 0.25f * s;
    }
    float* o = b.rigid_body_state + ((size_t)e * m.nb + bb) * 13;
    o[0] = pos.x; o[1] = pos.y; o[2] = pos.z; o[3] = qx; o[4] = qy; o[5] = qz; o[6] = qw;
    o[7] = lin.x; o[8] = lin.y; o[9] = lin.z; o[10] = ang.x; o[11] = ang.y; o[12] = ang.z;
  }
}

// ---------------------------------------------------------------- self-collision (model/selfcollision.py, T:354 filter 0)
// One warp per env, 16 envs per CTA; the CTA stages the packed tables (DevModel::sc_hot, ~13 KB for TOCABI) in shared
// memory while the physics kernel before it drains (PDL).
//   0. the env's link poses -> shared memory (coalesced); world centres of the shapes' bounding spheres;
//   1. (a) the 497 candidate link pairs, one per lane, 4 rounds in flight: overlapping link spheres mark, warp
//      uniformly (redux.or), the chunks of the shape-pair list that hold their shape pairs -- the link pairs are ordered
//      by how often they are near each other, so a standing / walking robot marks 3-5 of 13 chunks; (b) sweep over the
//      shape pairs of the marked chunks (1656 in all for TOCABI), one per lane, 4 rounds in flight: two bounding spheres
//      overlap -> hit list (standing: ~20);
//   2. hit list, one per lane: face-axis separating-axis test of the two oriented bounding boxes (a box is its own, a
//      cylinder's is r x r x h) -> what stays is really close (standing: a few), compacted with a ballot;
//   3. half a warp per surviving shape pair: lane = one sample sphere of one shape against the exact box / cylinder of
//      the other (both ways); a penetrating sample pushes the two bodies apart along the gradient of the signed
//      distance with the penalty stiffness of the ground contacts, accumulated per body in shared memory.
// Every cull is conservative, so the result is that of the plain double loop restated in oracle/selfcollision_oracle.py
// (up to the order of the sums); an env that overflows the hit list is swept again without it, never dropping a contact.
// (Measured dead ends, profiles/r2_self_collision.md: link-level culls that build LISTS of link pairs cost more in list
// handling -- compaction, prefix sums, mapping lanes to shape pairs -- than the sphere tests they save; two warps per env
// only fit one wave at 32 registers; a lane-chunked sweep doubles the shared-memory bank conflicts.)
constexpr int kScEnvs = 16;    // envs (warps) per CTA
constexpr int kScHits = 128;   // shape pairs whose spheres overlap
__device__ __forceinline__ float sc_sdf(int kind, V3 size, V3 x, V3& g) {
  if (kind == 0) {  // box: half extents
    const V3 q = v3(fabsf(x.x) - size.x, fabsf(x.y) - size.y, fabsf(x.z) - size.z);
    const V3 o = v3(fmaxf(q.x, 0.f), fmaxf(q.y, 0.f), fmaxf(q.z, 0.f));
    const float n = sqrtf(dot(o, o));
    const V3 sg = v3(x.x < 0 ? -1.f : 1.f, x.y < 0 ? -1.f : 1.f, x.z < 0 ? -1.f : 1.f);
    if (n > 0.f) {
      g = v3(o.x / n * sg.x, o.y / n * sg.y, o.z / n * sg.z);
      return n;
    }
    // inside: the face that is nearest (first of the largest components, as numpy's argmax)
    if (q.x >= q.y && q.x >= q.z) { g = v3(sg.x, 0, 0); return q.x; }
    if (q.y >= q.z) { g = v3(0, sg.y, 0); return q.y; }
    g = v3(0, 0, sg.z);
    return q.z;
  }
  if (kind == 2) {  // capsule about its z axis (a sphere when the half height is 0): distance to the segment, minus r
    const V3 q = v3(x.x, x.y, x.z - fminf(fmaxf(x.z, -size.y), size.y));
    const float n = sqrtf(dot(q, q));
    g = n > 0.f ? (1.f / n) * q : v3(1.f, 0.f, 0.f);
    return n - size.x;
  }
  const float r = size.x, h = size.y;  // cylinder about its z axis
  const float rho = sqrtf(x.x * x.x + x.y * x.y);
  const float inv = 1.f / fmaxf(rho, 1e-30f);
  const V3 er = v3(x.x * inv, x.y * inv, 0.f), ez = v3(0.f, 0.f, x.z < 0 ? -1.f : 1.f);
  const float qr = rho - r, qz = fabsf(x.z) - h;
  const float o0 = fmaxf(qr, 0.f), o1 = fmaxf(qz, 0.f);
  const float n = sqrtf(o0 * o0 + o1 * o1);
  if (n > 0.f) {
    g = (o0 / n) * er + (o1 / n) * ez;
    return n;
  }
  if (qr > qz) { g = er; return qr; }
  g = ez;
  return qz;
}
struct ScEnv {  // views into the env's block of shared memory (sized by the model: sc_env_bytes)
  float* pose;                // [nl*12]
  float4* link_c;             // [nl]: world centre and radius of each link's bounding sphere
  float4* shape_c;            // [ns+2]: world centre and radius of each shape's bounding sphere; two far-apart dummies
  float* force;               // [nb*3]
  int* count;                 // [0] hits, [1] any contact
  unsigned short* hits;       // [kScHits] shape a | shape b << 8
};
__host__ __device__ inline int sc_align4(int words) { return (words + 3) & ~3; }
__host__ __device__ inline int sc_env_bytes(int nl, int ns, int nb) {
  return 4 * (sc_align4(nl * 12) + nl * 4 + (ns + 2) * 4 + sc_align4(nb * 3) + 4) + 2 * kScHits;
}
__device__ __forceinline__ ScEnv sc_env_views(void* base, int nl, int ns, int nb) {
  ScEnv E;
  float* f = static_cast<float*>(base);
  E.pose = f; f += sc_align4(nl * 12);
  E.link_c = reinterpret_cast<float4*>(f); f += nl * 4;
  E.shape_c = reinterpret_cast<float4*>(f); f += (ns + 2) * 4;
  E.force = f; f += sc_align4(nb * 3);
  E.count = reinterpret_cast<int*>(f); f += 4;
  E.hits = reinterpret_cast<unsigned short*>(f);
  return E;
}
struct ScTab {  // the staged tables
  const unsigned* pair;
  const float* lsph;
  const unsigned short* sp;
  const float* shape;
  const int* meta;
  const float* sample;
};
__device__ __forceinline__ bool sc_spheres_overlap(float4 a, float4 b) {
  const float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z, rs = a.w + b.w;
  return dx * dx + dy * dy + dz * dz < rs * rs;
}
__device__ __forceinline__ void sc_pose(const float* pose, int l, M3& R, V3& t) {
  const float4* q = reinterpret_cast<const float4*>(pose + 12 * l);
  const float4 a = q[0], b = q[1], c = q[2];
  R = M3{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x}};
  t = v3(c.y, c.z, c.w);
}
// sample sphere k (of shape sa) against shape sb
__device__ __forceinline__ void sc_item(const ScTab& T, const SimParams& p, const ScEnv& W, int sa, int sb, int k) {
  const int ma = T.meta[2 * sa], mb = T.meta[2 * sb];
  const float4 smp = *reinterpret_cast<const float4*>(T.sample + 4 * k);
  M3 Ra, Rb;
  V3 pa, pb;
  sc_pose(W.pose, ma & 0xff, Ra, pa);
  const V3 c = mul(Ra, v3(smp.x, smp.y, smp.z)) + pa;
  const float rho = smp.w;
  const float4 sc = W.shape_c[sb];
  const V3 dc = c - v3(sc.x, sc.y, sc.z);
  const float reach = rho + sc.w;
  if (dot(dc, dc) >= reach * reach) return;
  sc_pose(W.pose, mb & 0xff, Rb, pb);
  const V3 cl = mulT(Rb, c - pb);  // in link lb's frame
  const float* S = T.shape + 16 * sb;
  const M3 Rs = ld_m3_f(S + 3);
  V3 g;
  const float d = sc_sdf((mb >> 16) & 0xff, ld3_f(S + 12), mulT(Rs, cl - ld3_f(S)), g);
  const float depth = rho - d;
  if (depth > 0.f) {
    const V3 f = fminf(p.pen_k * depth, p.pen_fmax) * mul(Rb, mul(Rs, g));  // pushes the sample's body out
    const int ba = (ma >> 8) & 0xff, bb = (mb >> 8) & 0xff;
    atomicAdd(&W.force[3 * ba], f.x); atomicAdd(&W.force[3 * ba + 1], f.y); atomicAdd(&W.force[3 * ba + 2], f.z);
    atomicAdd(&W.force[3 * bb], -f.x); atomicAdd(&W.force[3 * bb + 1], -f.y); atomicAdd(&W.force[3 * bb + 2], -f.z);
    W.count[1] = 1;
  }
}
// World frame (columns = axes) and half extents of shape s's oriented bounding box.
__device__ __forceinline__ void sc_obb(const ScTab& T, const ScEnv& W, int s, M3& R, V3& half) {
  const float* S = T.shape + 16 * s;
  const int ms = T.meta[2 * s];
  M3 Rl;
  V3 pl;
  sc_pose(W.pose, ms & 0xff, Rl, pl);
  R = mul(Rl, ld_m3_f(S + 3));
  const int kind = (ms >> 16) & 0xff;  // box: its half extents; cylinder r x r x h; capsule r x r x (h + r)
  half = kind == 0 ? ld3_f(S + 12) : v3(S[12], S[12], kind == 2 ? S[13] + S[12] : S[13]);
}
// true when one of the 6 face normals separates the two boxes (with a margin for rounding): certainly no contact
__device__ __forceinline__ bool sc_obb_separated(const ScTab& T, const ScEnv& W, int sa, int sb) {
  M3 A, B;
  V3 ha, hb;
  sc_obb(T, W, sa, A, ha);
  sc_obb(T, W, sb, B, hb);
  const float4 ca = W.shape_c[sa], cb = W.shape_c[sb];
  const V3 t = mulT(A, v3(cb.x - ca.x, cb.y - ca.y, cb.z - ca.z));  // in A's frame
  const M3 C = mulAtB(A, B);                                        // B's axes in A's frame
  const float eps = 1e-5f;
  float c[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) c[i] = fabsf(C.a[i]) + 1e-6f;
  const float ta[3] = {t.x, t.y, t.z}, hA[3] = {ha.x, ha.y, ha.z}, hB[3] = {hb.x, hb.y, hb.z};
  bool sep = false;
#pragma unroll
  for (int i = 0; i < 3; ++i) sep |= fabsf(ta[i]) > hA[i] + c[3 * i] * hB[0] + c[3 * i + 1] * hB[1] + c[3 * i + 2] * hB[2] + eps;
#pragma unroll
  for (int j = 0; j < 3; ++j)
    sep |= fabsf(ta[0] * C.a[j] + ta[1] * C.a[3 + j] + ta[2] * C.a[6 + j]) > hB[j] + c[j] * hA[0] + c[3 + j] * hA[1] + c[6 + j] * hA[2] + eps;
  return sep;
}
__global__ void __launch_bounds__(kScEnvs * 32, 2) k_self_collision(DevModel m, SimParams p, DyrosSimBuffers b) {
  extern __shared__ float4 sc_smem[];
  int* tab = reinterpret_cast<int*>(sc_smem);
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < m.sc_hot_words / 4; i += blockDim.x)  // (constant tables: before the wait)
    reinterpret_cast<int4*>(tab)[i] = reinterpret_cast<const int4*>(m.sc_hot)[i];
  pdl_wait();
  const int lane = threadIdx.x & 31, slot = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  const int e = blockIdx.x * kScEnvs + slot;
  const bool live = e < p.N;
  const ScEnv W = sc_env_views(reinterpret_cast<char*>(tab + m.sc_hot_words) + (size_t)slot * sc_env_bytes(m.nl, m.sc_ns, m.nb),
                               m.nl, m.sc_ns, m.nb);
  if (live) {
    const float* pose = b.link_pose + (size_t)e * m.nl * 12;
    for (int i = lane; i < m.nl * 3; i += 32)  // (12 floats per link: the env's block is 16-byte aligned)
      reinterpret_cast<float4*>(W.pose)[i] = reinterpret_cast<const float4*>(pose)[i];
    for (int i = lane; i < m.nb * 3; i += 32) W.force[i] = 0.f;
    if (lane < 2) W.count[lane] = 0;
  }
  __syncthreads();
  if (!live) return;
  ScTab T;
  T.pair = reinterpret_cast<const unsigned*>(tab + m.sc_o_pair);
  T.lsph = reinterpret_cast<const float*>(tab + m.sc_o_lsph);
  T.sp = reinterpret_cast<const unsigned short*>(tab + m.sc_o_sp);
  T.shape = reinterpret_cast<const float*>(tab + m.sc_o_shape);
  T.meta = tab + m.sc_o_meta;
  T.sample = reinterpret_cast<const float*>(tab + m.sc_o_sample);
  for (int l = lane; l < m.nl; l += 32) {
    const float4 ls = *reinterpret_cast<const float4*>(T.lsph + 4 * l);
    M3 R;
    V3 t;
    sc_pose(W.pose, l, R, t);
    const V3 c = mul(R, v3(ls.x, ls.y, ls.z)) + t;
    W.link_c[l] = make_float4(c.x, c.y, c.z, ls.w);
  }
  for (int s = lane; s < m.sc_ns; s += 32) {
    const float4 s0 = *reinterpret_cast<const float4*>(T.shape + 16 * s);
    M3 R;
    V3 t;
    sc_pose(W.pose, T.meta[2 * s] & 0xff, R, t);
    const V3 c = mul(R, v3(s0.x, s0.y, s0.z)) + t;
    W.shape_c[s] = make_float4(c.x, c.y, c.z, T.shape[16 * s + 15]);
  }
  if (lane < 2) W.shape_c[m.sc_ns + lane] = make_float4(lane ? -1e18f : 1e18f, 0.f, 0.f, 0.f);
  __syncwarp();
  // 1a. link spheres: which chunks of the shape-pair list hold pairs of links that are near each other at all
  unsigned active = 0;
  {
    const char* lcs = reinterpret_cast<const char*>(W.link_c);
    for (int base = lane; base < m.sc_np; base += 128) {
      unsigned pt[4], mk = 0;
#pragma unroll
      for (int u = 0; u < 4; ++u) pt[u] = base + 32 * u < m.sc_np ? T.pair[base + 32 * u] : 0u;  // (0: link 0 against itself, no chunk)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float4 a = *reinterpret_cast<const float4*>(lcs + ((pt[u] & 0xffu) << 4));
        const float4 c = *reinterpret_cast<const float4*>(lcs + ((pt[u] >> 4) & 0xff0u));
        if (sc_spheres_overlap(a, c)) mk |= pt[u] >> 16;
      }
      active |= __reduce_or_sync(kFull, mk);
    }
  }
  // 1b. bounding spheres of the candidate shape pairs in the active chunks (the list is padded to whole chunks with a
  //     far-apart dummy pair)
  const char* centres = reinterpret_cast<const char*>(W.shape_c);
  for (int c0 = 0; c0 < m.sc_nq_padded; c0 += m.sc_chunk, active >>= 1) {
    if (!(active & 1u)) continue;
    for (int base = c0 + lane; base < c0 + m.sc_chunk; base += SC_SWEEP_BATCH) {
      unsigned sp[4];
      float4 ca[4], cb[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) sp[u] = T.sp[base + 32 * u];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        ca[u] = *reinterpret_cast<const float4*>(centres + ((sp[u] & 0xffu) << 4));
        cb[u] = *reinterpret_cast<const float4*>(centres + ((sp[u] >> 4) & 0xff0u));
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (sc_spheres_overlap(ca[u], cb[u])) {
          const int at = atomicAdd(&W.count[0], 1);
          if (at < p.sc_hits_cap) W.hits[at] = (unsigned short)sp[u];
        }
      }
    }
  }
  __syncwarp();
  if (W.count[0] > p.sc_hits_cap) {
    // more overlapping spheres than the list holds (a badly contorted robot): sweep again, plainly, and let every lane
    // run the narrow phase of its own hits (both ways, all samples); the list is not used
#pragma unroll 1
    for (int q = lane; q < m.sc_nq; q += 32) {
      const int sp = T.sp[q], sa = sp & 0xff, sb = sp >> 8;
      if (!sc_spheres_overlap(W.shape_c[sa], W.shape_c[sb])) continue;
      const int xa = T.meta[2 * sa + 1], xb = T.meta[2 * sb + 1];
#pragma unroll 1
      for (int k = 0; k < (xa >> 16) + (xb >> 16); ++k) {
        const bool fwd = k < (xa >> 16);
        sc_item(T, p, W, fwd ? sa : sb, fwd ? sb : sa, fwd ? (xa & 0xffff) + k : (xb & 0xffff) + k - (xa >> 16));
      }
    }
    __syncwarp();
    if (lane == 0) W.count[0] = 0;
  }
  __syncwarp();
  const int n2 = min(W.count[0], p.sc_hits_cap);
  int nh = 0;  // 2. oriented boxes; the survivors are compacted in place
  for (int base = 0; base < n2; base += 32) {
    const int h = base + lane;
    int sp = 0;
    bool keep = false;
    if (h < n2) {
      sp = W.hits[h];
      keep = !sc_obb_separated(T, W, sp & 0xff, sp >> 8);
    }
    const unsigned bal = __ballot_sync(kFull, keep);  // (also orders this round's reads before its writes)
    if (keep) W.hits[nh + __popc(bal & lt)] = (unsigned short)sp;
    nh += __popc(bal);
  }
  __syncwarp();
  for (int h = lane >> 4; h < nh; h += 2) {  // 3. samples against exact shapes, 16 lanes per shape pair
    const int sp = W.hits[h], sa = sp & 0xff, sb = sp >> 8;
    const int xa = T.meta[2 * sa + 1], xb = T.meta[2 * sb + 1];
    const int na = xa >> 16, nb = xb >> 16;
    const int t = lane & 15;
    if (t < na) sc_item(T, p, W, sa, sb, (xa & 0xffff) + t);
    else if (t - na < nb) sc_item(T, p, W, sb, sa, (xb & 0xffff) + t - na);
  }
  __syncwarp();
  const bool any_hit = W.count[1] != 0;
  float* out = b.self_contact_force + (size_t)e * m.nb * 3;
  float* net = b.net_contact_force + (size_t)e * m.nb * 3;
  for (int i = lane; i < m.nb * 3; i += 32) {
    const float f = any_hit ? W.force[i] : 0.f;
    out[i] = f;
    if (any_hit) net[i] += f;
  }
}
static size_t sc_smem_bytes(const Sim* sim) {
  return (size_t)sim->m.sc_hot_words * 4 + (size_t)kScEnvs * sc_env_bytes(sim->m.nl, sim->m.sc_ns, sim->m.nb);
}
int launch_self_collision(Sim* sim, cudaStream_t s, bool pdl) {
  if (!has_self_collision(sim)) return 0;
  if (sim->p.sc_hits_cap == 0) {
    // DYROS_SC_TEST_CAPS=<hits>: shrinks the hit list so that tests reach the overflow path on ordinary poses
    int h = kScHits;
    if (const char* v = getenv("DYROS_SC_TEST_CAPS")) sscanf(v, "%d", &h);
    sim->p.sc_hits_cap = std::max(1, std::min(h, kScHits));
    DY_CUDA(cudaFuncSetAttribute(k_self_collision, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc_smem_bytes(sim)));
  }
  // (launched WITHOUT the programmatic-serialisation attribute whatever `pdl` says: as a programmatic dependent of the
  // physics kernel, whose CTAs own whole SMs, this kernel measured ~50 us slower per step; profiles/r2_carveout.md)
  (void)pdl;
  DY_CUDA(launch_kernel(k_self_collision, dim3((sim->p.N + kScEnvs - 1) / kScEnvs), dim3(kScEnvs * 32), sc_smem_bytes(sim), s, false,
                        sim->m, sim->p, sim->b));
  return 0;
}

// gym.refresh_dof_force_tensor (tensors.rst.txt "DOF force tensor", used by tasks/humanoid.py:85,245): the generalised force
// at every DOF = applied actuation (clamped to the ctrlrange when clamp_effort is set) plus the joint's passive spring and
// damper, evaluated on the current state. One thread per DOF.
__global__ void __launch_bounds__(256) k_dof_force(DevModel m, SimParams p, DyrosSimBuffers b, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.N * m.nd) return;
  const int d = i % m.nd;
  float tq = b.dof_actuation_force[i];
  if (p.clamp_effort) {
    const float lim = m.dof_effort[d];
    tq = tq > lim ? lim : (tq < -lim ? -lim : tq);
  }
  out[i] = tq - b.dof_damping[i] * b.dof_state[2 * i + 1] - m.dof_stiffness[d] * b.dof_state[2 * i];
}
int launch_refresh_dof_force(Sim* sim, float* out, cudaStream_t s) {
  const int n = sim->p.N * sim->m.nd;
  k_dof_force<<<(n + 255) / 256, 256, 0, s>>>(sim->m, sim->p, sim->b, out);
  DY_LAUNCH_CHECK();
  return 0;
}

// gym.refresh_force_sensor_tensor (tasks/humanoid.py:80,243; create_asset_force_sensor :167-168): per sensor the net contact
// force on its body over the last sub-step, expressed in the sensor frame (body rotation x sensor rotation), as
// [force 3, torque 3]. The contact model keeps one net force per body (net_contact_force), not its line of action: the
// torque entries are zero. Needs rigid_body_state to be current (the caller refreshes it first). One thread per sensor.
__global__ void __launch_bounds__(128) k_force_sensors(DevModel m, SimParams p, DyrosSimBuffers b, const int32_t* __restrict__ sensor_body,
                                                       const float* __restrict__ sensor_pose, int ns, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.N * ns) return;
  const int e = i / ns, s = i - e * ns, body = sensor_body[s];
  const float* rb = b.rigid_body_state + ((size_t)e * m.nb + body) * 13;
  const M3 Rb = quat_to_mat(rb[3], rb[4], rb[5], rb[6]);
  const float* sp = sensor_pose + 7 * s;
  const M3 Rs = quat_to_mat(sp[3], sp[4], sp[5], sp[6]);
  const V3 F = ld3_f(b.net_contact_force + ((size_t)e * m.nb + body) * 3);
  const V3 f = mulT(Rs, mulT(Rb, F));
  float* o = out + (size_t)i * 6;
  o[0] = f.x; o[1] = f.y; o[2] = f.z; o[3] = 0.f; o[4] = 0.f; o[5] = 0.f;
}
int launch_refresh_force_sensors(Sim* sim, const int32_t* sensor_body, const float* sensor_pose, int ns, float* out, cudaStream_t s) {
  const int n = sim->p.N * ns;
  k_force_sensors<<<(n + 127) / 128, 128, 0, s>>>(sim->m, sim->p, sim->b, sensor_body, sensor_pose, ns, out);
  DY_LAUNCH_CHECK();
  return 0;
}

int launch_refresh_rigid_body_state(Sim* sim, cudaStream_t s) {
  k_rigid_body_state<<<(sim->p.N + 63) / 64, 64, 0, s>>>(sim->m, sim->p, sim->b);
  DY_LAUNCH_CHECK();
  return 0;
}

__global__ void __launch_bounds__(256) k_fill(uint4* __restrict__ p, size_t n16, unsigned v) {
  const uint4 x = make_uint4(v, v, v, v);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) p[i] = x;
}
int launch_fill(void* buf, size_t bytes, int value, cudaStream_t s) {
  static bool once = false;
  if (!once) {
    DY_CUDA(prefer_max_smem_carveout(k_fill));
    once = true;
  }
  k_fill<<<148 * 8, 256, 0, s>>>(static_cast<uint4*>(buf), bytes / 16, 0x01010101u * (unsigned)(value & 0xff));
  DY_LAUNCH_CHECK();
  return 0;
}
int configure_physics_aux_kernels() {  // (k_simulate / k_step_physics already take all of the shared memory)
  DY_CUDA(prefer_max_smem_carveout(k_rigid_body_state)); DY_CUDA(prefer_max_smem_carveout(k_self_collision));
  DY_CUDA(prefer_max_smem_carveout(k_dof_force)); DY_CUDA(prefer_max_smem_carveout(k_force_sensors));
  return 0;
}

}  // namespace dyros
