// One sub-step of gym.simulate as the program of ONE ROLE acting on ONE env with LPE = 8 LANES.
//
// Replaces the body of `gym.simulate` (reference call site tasks/dyros_dynamic_walk.py:525; the reference's
// implementation is closed-source PhysX). Same model and same formulas as the single-lane role program it supersedes
// (physics_roles.cuh, kept as the CPU-tested statement of the algorithm; dense fp64 restatement in
// oracle/physics_oracle.py; DESIGN.md section 4): articulated-body forward dynamics in world axes about the link
// origins, implicit joint damping / rotor inertia, penalty ground contact for every primitive except the sole corners,
// fixed-sweep projected Gauss-Seidel on the sole corners with the exact articulated inverse inertia.
//
// What changed is the mapping to the machine. The single-lane program ran one env per lane and one warp per role, so
// a 4096-env shard put 4 busy warps on an SM and its time was the dependent-issue latency of one instruction stream.
// Here 8 lanes share an env (4 envs per warp, 7 warps per role and SM at 28 envs per SM):
//   * the 6x6 articulated inertias live DISTRIBUTED: lane c holds column c (= row c, they are symmetric) and component c
//     of the bias force, so the rank-1 downdate, the shift to the parent and the products with spatial vectors cost 6
//     FMA per lane instead of 36, exchanged with width-8 shuffles;
//   * the per-link terms that depend on no other link (joint transform, rigid inertia in world axes, velocity-product
//     force, external wrench, velocity-product acceleration) run with LANE = LINK, 8 links of the role at a time;
//   * 3-vectors and the chained kinematic passes are REPLICATED in the 8 lanes (same instruction count as one lane,
//     no shuffles), read from shared memory with 128-bit broadcast loads.
// Roles, per-link scratch blocks in shared memory and release/acquire stage flags are as before, the flags now per
// group of 4 envs (one warp per role), not per CTA.
// The same source compiles for the host with every `real` emulated as 8 lanes (tests/native/hostemu_lanes.cu).
#pragma once
#include "internal.h"
#include "lanes.cuh"

#if defined(__CUDACC__) && !defined(DYROS_LANE_EMU)
#define HDL __device__ __forceinline__
#else
#define HDL inline
#endif

namespace dyros {
namespace ln {

// ---- per-link scratch block of one env (floats); every 3-vector sits on a 16-byte boundary
constexpr int LB = 48;
constexpr int B_S = 0;    // 3  joint axis s, world axes          (base: impulse response dv, 6 words from here)
constexpr int B_Q = 3;    // 1  joint angle
constexpr int B_R = 4;    // 3  offset from the parent's origin r, world axes
constexpr int B_QD = 7;   // 1  joint velocity qd -> qd* (predicted) -> new qd
constexpr int B_SC = 8;   // 4  [tau -> u, damping -> 1/D, armature -> S^T dp, free]   (base: dt w x u)
constexpr int B_U = 12;   // 8  U = IA S (6) + 2 zero words                           (base: predicted velocity v0*)
constexpr int B_A = 20;   // 28 phase-dependent, see A_*
// relative to B_A
constexpr int A_W = 0, A_V = 4, A_POSE = 8;            // pass 1: angular velocity, velocity of the origin, world pose (R 9, p 3);
                                                       //         before that A_POSE holds the joint rotation E of pass 1a
constexpr int A_HM = 0, A_I = 4, A_P = 12, A_C = 20;   // own terms: m c (3) + mass, inertia about the origin (6+2),
                                                       //         bias force p - f_ext (6+2 zeros), velocity-product acceleration (6+2)
constexpr int A_CIA = 0, A_CPA = 21;                   // pass 2: contribution to a parent that is not the next link: IA (21, packed), pA (6)
constexpr int A_ACC = 0, A_DV = 8;                     // pass 3 / down pass, links with children in other roles: a' (6), dv (6)
constexpr int A_ROWS = 0;                              // leg-chain links: 2 contact rows of 8 words (response 6, 1/(J.cv), free)
constexpr int A_YT = 16;                               // leg-chain link k: row k of Y = Om_lca G (6+2), see feet part 2
constexpr int A_OM0 = 6;                               // base: a0 at A_ACC, inverse inertia (21, packed) from here
constexpr int ROWS_PER_LINK = 2;
// per-env extra scratch
constexpr int X_FOOTPOSE = 0;                          // MAX_FEET * 12
constexpr int X_Z = X_FOOTPOSE + MAX_FEET * 12;        // 2 (sweep parity) * MAX_FEET * 8: base velocity change of a sweep
constexpr int X_PD = X_Z + 2 * MAX_FEET * 8;           // MAX_FEET * 8  impulse arriving at the common ancestor from a foot
constexpr int X_ROOT = X_PD + MAX_FEET * 8;            // 16 (13 used): root state in, root state out
constexpr int X_PUSH = X_ROOT + 16;                    // 4  world force at the base body's COM for this sub-step
constexpr int X_OML = X_PUSH + 4;                      // 24 (21 used): inverse inertia at the feet's common ancestor
constexpr int PT_WORDS = 8;                            // active sole point: candidate (int), bias, lam (3), location xa (3)
constexpr int X_PTS = X_OML + 24;                      // MAX_FEET * MAX_ACTIVE_PTS * PT_WORDS
constexpr int X_MU = X_PTS + MAX_FEET * MAX_ACTIVE_PTS * PT_WORDS;  // 4 (1 used): friction coefficient of this env
constexpr int X_CV = X_MU + 4;                         // MAX_CSLOTS * 8: velocity-product acceleration of the links whose block
                                                       // receives their contribution to the parent (A_CPA overlaps A_C)
constexpr int X_MASS = X_CV + MAX_CSLOTS * 8;          // nb per-body mass scales (last: sized by the model)
// the words of the scratch block that the kernels' slab copies fill and read back (physics_cta.cuh)
struct LanesScratch {
  static constexpr int link = LB, q = B_Q, qd = B_QD, tau = B_SC, damping = B_SC + 1, armature = B_SC + 2;
  static constexpr int mu = X_MU, mass = X_MASS, root = X_ROOT, push = X_PUSH;
};

HD int env_scratch_floats(int nl, int nb) {
  int n = nl * LB + X_MASS + nb;
  n = (n + 3) & ~3;
  // stride = 8 mod 32 words: the 4 envs of a warp (8 lanes each) touch 4 disjoint groups of 8 banks for any field
  while ((n & 31) != 8) n += 4;
  return n;
}

// flags of one group of envs (ints): stage reached by each link, plus the hand-shakes of the contact stage
constexpr int F_LINK = 0;                      // [DYROS_MAX_LINKS]
constexpr int F_Z = DYROS_MAX_LINKS;           // [MAX_FEET] sweeps published
constexpr int F_PD = F_Z + MAX_FEET;           // [MAX_FEET] base impulse published
constexpr int F_OML = F_PD + MAX_FEET;         // [1] inverse inertia at the LCA published
constexpr int QF_COUNT = (F_OML + 1 + 3) & ~3;
// CTA-wide flags published by the I/O warps of the fused step
constexpr int F_IO_PRE = 0;                    // push staged, contact forces zeroed
constexpr int F_IO_TAU = 1;                    // torque, damping and armature staged
constexpr int F_IO_DONE = 2;                   // the I/O group no longer reads the joint angles
constexpr int IOF_COUNT = 4;
constexpr int ST_PASS1 = 1, ST_PASS2 = 2, ST_PASS3 = 3, ST_DOWN = 4, ST_STRIDE = 8;

#define LREC(idx) (hot + m.o_prog + (idx) * REC_WORDS)
#define LRI(R, field) (reinterpret_cast<const int*>(R)[field])
#define LBLK(link) (sm + (link) * LB)

// global-memory views of one env (device pointers on the GPU, host pointers in the emulation)
struct EnvIO {
  float* contact;          // nb*3 net contact force of this sub-step (zeroed before the sub-step)
  const float* rb_force;   // nb*3 or NULL
  const float* rb_torque;  // nb*3 or NULL
  float* link_pose;        // nl*12 or NULL: world pose of every link as pass 1 finds it (for the self-collision pass)
  bool push;               // X_PUSH holds a force for the base body
  bool live;               // false: padding lanes, no global writes
};
HDL void export_pose(const EnvIO& io, int link, const M3& Rw, V3 pw) {
  if (!io.link_pose || !io.live) return;
  float* o = io.link_pose + 12 * link;
  for (int c = 0; c < 9; ++c) st(o + c, Rw.a[c]);
  st(o + 9, pw.x); st(o + 10, pw.y); st(o + 11, pw.z);
}

HDL V3 ldv3(const float* p) { return V3{ld(p), ld(p + 1), ld(p + 2)}; }
HDL void stv3(float* p, V3 a) { st(p, a.x); st(p + 1, a.y); st(p + 2, a.z); }
HDL V3 ldv3q(const float* p) {  // 3-vector on a 16-byte boundary (the fourth word is ignored)
  real a, b, c, d;
  ld4(p, a, b, c, d);
  return V3{a, b, c};
}
HDL V3 ldv3l(const float* p, li i) { return V3{ldl(p, i), ldl(p, i + 1), ldl(p, i + 2)}; }
HDL V3 sel3(lb m, V3 a, V3 b) { return V3{sel(m, a.x, b.x), sel(m, a.y, b.y), sel(m, a.z, b.z)}; }
HDL M3 ld_pose_rot(const float* p, real& px, real& py, real& pz) {  // 12 words on a 16-byte boundary: R row-major, p
  M3 R;
  ld4(p, R.a[0], R.a[1], R.a[2], R.a[3]);
  ld4(p + 4, R.a[4], R.a[5], R.a[6], R.a[7]);
  ld4(p + 8, R.a[8], px, py, pz);
  return R;
}
HDL void st_pose(float* p, const M3& R, V3 t) {
  st4(p, R.a[0], R.a[1], R.a[2], R.a[3]);
  st4(p + 4, R.a[4], R.a[5], R.a[6], R.a[7]);
  st4(p + 8, R.a[8], t.x, t.y, t.z);
}
HDL SV ld_sv8(const float* p) {  // 6 words on a 16-byte boundary (8-word slot)
  real a, b, c, d, e, f, g, h;
  ld4(p, a, b, c, d);
  ld4(p + 4, e, f, g, h);
  return SV{V3{a, b, c}, V3{d, e, f}};
}
HDL void st_sv8(float* p, SV a) {
  st4(p, a.w.x, a.w.y, a.w.z, a.v.x);
  st4(p + 4, a.v.y, a.v.z, real(0), real(0));
}
HDL ABI ld_abi_packed(const float* p) {  // st_abi layout (phys_math.cuh): I (6), H (9 row-major), M (6)
  ABI a;
  a.I = S3{ld(p), ld(p + 1), ld(p + 2), ld(p + 3), ld(p + 4), ld(p + 5)};
  for (int i = 0; i < 9; ++i) a.H.a[i] = ld(p + 6 + i);
  a.M = S3{ld(p + 15), ld(p + 16), ld(p + 17), ld(p + 18), ld(p + 19), ld(p + 20)};
  return a;
}
HDL void st_abi_packed(float* p, const ABI& a) {
  st(p, a.I.xx); st(p + 1, a.I.yy); st(p + 2, a.I.zz); st(p + 3, a.I.xy); st(p + 4, a.I.xz); st(p + 5, a.I.yz);
  for (int i = 0; i < 9; ++i) st(p + 6 + i, a.H.a[i]);
  st(p + 15, a.M.xx); st(p + 16, a.M.yy); st(p + 17, a.M.zz); st(p + 18, a.M.xy); st(p + 19, a.M.xz); st(p + 20, a.M.yz);
}
// index of entry (a, b) of a symmetric 3x3 in S3 order xx yy zz xy xz yz
HDL li sym3(li a, li b) { return seli(a == b, a, a + b + li(2)); }

// Lane constants of a group: what lane c needs to pick "its" column out of replicated data.
struct LaneConst {
  li c, cm;          // lane index, c mod 3
  lb ang, lin, act;  // c < 3, 3 <= c < 6, c < 6
  real e0, e1, e2;   // unit vector of axis cm (zero in the idle lanes 6, 7)
  li ix0, ix1, ix2;  // S3 indices of column cm of a symmetric 3x3
  li s1, s2;         // lanes holding the linear columns (cm+1)%3 and (cm+2)%3
};
HDL LaneConst make_lane_const(const Ln& g) {
  LaneConst k;
  k.c = lane_index(g);
  k.cm = k.c % li(3);
  k.ang = k.c < li(3);
  k.act = k.c < li(6);
  k.lin = k.act && !k.ang;
  k.e0 = sel(k.act && (k.cm == li(0)), real(1), real(0));
  k.e1 = sel(k.act && (k.cm == li(1)), real(1), real(0));
  k.e2 = sel(k.act && (k.cm == li(2)), real(1), real(0));
  k.ix0 = sym3(li(0), k.cm);
  k.ix1 = sym3(li(1), k.cm);
  k.ix2 = sym3(li(2), k.cm);
  k.s1 = li(3) + (k.cm + li(1)) % li(3);
  k.s2 = li(3) + (k.cm + li(2)) % li(3);
  return k;
}
// packed (st_abi) index of entry (r, c) of a symmetric 6x6 for the lane's own column c; idle lanes get a valid index
HDL li packed_index(const LaneConst& k, int r) {
  if (r < 3) return seli(k.ang, sym3(li(r), k.cm), li(6 + 3 * r) + k.cm);
  return seli(k.ang, li(6 + (r - 3)) + k.cm * li(3), li(15) + sym3(li(r - 3), k.cm));
}
// component c of a replicated spatial vector (zero in the idle lanes)
HDL real pick6(const LaneConst& k, SV a) {
  real w = k.e0 * a.w.x + k.e1 * a.w.y + k.e2 * a.w.z;
  real v = k.e0 * a.v.x + k.e1 * a.v.y + k.e2 * a.v.z;
  return sel(k.ang, w, v);
}
// replicate a distributed spatial vector
HDL SV gather6(const Ln& g, real x) { return SV{V3{bc(g, x, 0), bc(g, x, 1), bc(g, x, 2)}, V3{bc(g, x, 3), bc(g, x, 4), bc(g, x, 5)}}; }
// [[I,H],[H^T,M]] column c times nothing: product of a distributed symmetric 6x6 (col = the lane's column) with a
// replicated spatial vector; the result is distributed (component c in lane c)
HDL real col_dot(const real* col, SV a) {
  return col[0] * a.w.x + col[1] * a.w.y + col[2] * a.w.z + col[3] * a.v.x + col[4] * a.v.y + col[5] * a.v.z;
}

// ---- penalty ground contact of one location on a link, lane = link, masked by `on`
//      (oracle: PhysicsOracle._external_wrench.add_point); xw = the location relative to the link origin, world axes
HDL void penalty_point(const SimParams& p, real mu, SV v, V3 xw, real depth, float* contact, li body, lb on, bool live, SV& fext) {
  on = on && (depth > real(0));
  if (!any(on)) return;
  V3 vel_w = v.v + cross(v.w, xw);
  real fn = real(p.pen_k) * depth - real(p.pen_c) * vel_w.z;
  fn = sel(fn < real(0), real(0), sel(fn > real(p.pen_fmax), real(p.pen_fmax), fn));
  real speed = sqrt_r(vel_w.x * vel_w.x + vel_w.y * vel_w.y);
  real lim = mu * fn / sel(speed > real(1e-6), speed, real(1e-6));
  real coef = sel(real(p.pen_c) < lim, real(p.pen_c), lim);
  V3 Fw = v3(-coef * vel_w.x, -coef * vel_w.y, fn);
  if (live) {  // bodies belong to exactly one link, links to exactly one lane: no two lanes touch the same words
    li o = seli(on, body * li(3), li(0));
    stl(contact, o, ldl(contact, o) + Fw.x, on);
    stl(contact, o + li(1), ldl(contact, o + li(1)) + Fw.y, on);
    stl(contact, o + li(2), ldl(contact, o + li(2)) + Fw.z, on);
  }
  V3 z3 = v3(0, 0, 0);
  fext.w = fext.w + sel3(on, cross(xw, Fw), z3);
  fext.v = fext.v + sel3(on, Fw, z3);
}

// One sub-step for role `role` of one env. `qflags`: the stage flags of the env's group; `ioflags`: the CTA-wide flags
// of the fused step's I/O warps (used with io_async only); `epoch`: sub-steps done so far in this launch (the flags
// are monotonic). The env's inputs must have been staged into `sm` and made visible.
template <class Sync>
HDL void env_substep_lanes(const EnvIO& io, float* sm, int* qflags, const int* ioflags, int epoch, const float* hot,
                           const DevModel& m, const SimParams& p, int role, Sync& sync, const Ln& g, bool io_async) {
  const int nl = m.nl;
  float* X = sm + nl * LB;
  const int* hoti = reinterpret_cast<const int*>(hot);
  const real dt = real(p.dt);
  const int base = epoch * ST_STRIDE;
  const int len = m.role_len[role];
  const bool base_role = role == m.base_role;
  const int rec0 = m.prog_start[role];
  int* fl = qflags + F_LINK;
  const LaneConst lc = make_lane_const(g);
  const V3 zero3 = v3(0, 0, 0);

  sync.mark(0);
  // ---- pass 1a, LANE = LINK: joint rotations E(q) of the role's links (no dependencies)
  for (int j0 = 0; j0 < len; j0 += LPE) {
    const li j = lc.c + li(j0);
    const lb on = j < li(len);
    if (any(on)) {
      const li ro = seli(on, j + li(rec0), li(rec0)) * li(REC_WORDS) + li(m.o_prog);
      const li bo = ldli(hoti, ro + li(R_LINK)) * li(LB);
      real sq, cq;
      sincos_r(ldl(sm, bo + li(B_Q)), &sq, &cq);
      M3 E0;
      for (int i = 0; i < 9; ++i) E0.a[i] = ldl(hot, ro + li(R_E + i));
      const M3 E = mul(axis_rot_T(ldv3l(hot, ro + li(R_AXIS)), sq, cq), E0);
      for (int i = 0; i < 9; ++i) stl(sm, bo + li(B_A + A_POSE + i), E.a[i], on);
    }
  }
  lane_fence();
  sync.mark(16);
  // ---- pass 1b, replicated chain root -> leaves: world pose, axis and offset in world axes, velocity. Along a chain
  //      the parent's results are carried in registers; the scratch block is only read for the first link of a chain.
  int prev = -1;
  SV v_prev = sv_zero();
  M3 Rw_prev;
  V3 pw_prev = zero3;
  if (base_role) {
    float* A = LBLK(0) + B_A;
    const float* rs = X + X_ROOT;
    real r0, r1, r2, r3, r4, r5, r6, r7, r8, r9, r10, r11, r12, r13, r14, r15;
    ld4(rs, r0, r1, r2, r3);
    ld4(rs + 4, r4, r5, r6, r7);
    ld4(rs + 8, r8, r9, r10, r11);
    ld4(rs + 12, r12, r13, r14, r15);
    const V3 pw = v3(r0, r1, r2);
    const M3 R0 = quat_to_mat(r3, r4, r5, r6);
    const SV v0{v3(r10, r11, r12), v3(r7, r8, r9)};  // root state: world angular velocity, world velocity of the base origin
    st4(A + A_W, v0.w.x, v0.w.y, v0.w.z, real(0));
    st4(A + A_V, v0.v.x, v0.v.y, v0.v.z, real(0));
    st_pose(A + A_POSE, R0, pw);
    export_pose(io, 0, R0, pw);
    sync.signal(fl + 0, base + ST_PASS1);
    prev = 0;
    v_prev = v0;
    Rw_prev = R0;
    pw_prev = pw;
  }
  for (int k = 0; k < len; ++k) {
    const float* R = LREC(rec0 + k);
    const int i = LRI(R, R_LINK), par = LRI(R, R_PARENT), flg = LRI(R, R_FLAGS);
    float* L = LBLK(i);
    float* A = L + B_A;
    if (par != prev) {
      if (flg & RF_PARENT_FOREIGN) sync.wait(fl + par, base + ST_PASS1);
      const float* Ap = LBLK(par) + B_A;
      v_prev = SV{ldv3q(Ap + A_W), ldv3q(Ap + A_V)};
      real px, py, pz;
      Rw_prev = ld_pose_rot(Ap + A_POSE, px, py, pz);
      pw_prev = v3(px, py, pz);
    }
    real e9, e10, e11;
    const M3 E = ld_pose_rot(A + A_POSE, e9, e10, e11);
    const V3 rw = mul(Rw_prev, ldv3q(R + R_R));  // offset of this link's origin from its parent's, world axes
    Rw_prev = mulABt(Rw_prev, E);
    const V3 sw = mul(Rw_prev, ldv3q(R + R_AXIS));  // joint axis, world axes
    const real qd = ld(L + B_QD);
    pw_prev = pw_prev + rw;
    v_prev = SV{v_prev.w + qd * sw, v_prev.v + cross(v_prev.w, rw)};
    prev = i;
    stv3(L + B_S, sw);
    st4(L + B_R, rw.x, rw.y, rw.z, qd);
    st4(A + A_W, v_prev.w.x, v_prev.w.y, v_prev.w.z, real(0));
    st4(A + A_V, v_prev.v.x, v_prev.v.y, v_prev.v.z, real(0));
    st_pose(A + A_POSE, Rw_prev, pw_prev);
    export_pose(io, i, Rw_prev, pw_prev);
    // published only where another role reads it: by foreign children (pose, velocity), or by the foreign parent,
    // which must not overwrite its pose before this link has used it
    if (flg & (RF_PUBLISH | RF_PARENT_FOREIGN)) sync.signal(fl + i, base + ST_PASS1);
  }
  sync.mark(17);
  sync.mark(1);
  // The own-terms phase overwrites the pose of a link: every child of this role's links that lives in another role must
  // have read its parent's pose first.
  for (int k = 0; k < m.n_xchild[role]; ++k) sync.wait(fl + m.xchild[role][k], base + ST_PASS1);
  if (base_role) {  // ... and so must the children of the base (the base is on no role's list)
    const float* R0 = LREC(0);
    for (int j = 0; j < LRI(R0, R_NCHILD); ++j)
      if (LRI(R0, R_CHILD0 + j) & REC_FOREIGN) sync.wait(fl + (LRI(R0, R_CHILD0 + j) & ~REC_FOREIGN), base + ST_PASS1);
  }
  if (io_async) sync.wait_io(ioflags + F_IO_PRE, epoch + 1);
  lane_fence();
  sync.mark(2);
  // ---- pass 1c, LANE = LINK: everything of pass 2 that depends on the link alone: rigid inertia about the origin in
  //      world axes, velocity-product force minus external wrench (applied wrenches, penalty ground contact),
  //      velocity-product acceleration of the joint. The base role's list ends with the base itself (record 0).
  {
    const int nitems = len + (base_role ? 1 : 0);
    const real mu = ld(X + X_MU);
    for (int j0 = 0; j0 < nitems; j0 += LPE) {
      const li j = lc.c + li(j0);
      const lb on = j < li(nitems);
      if (!any(on)) continue;
      const lb joint = on && (j < li(len));
      const li ro = seli(joint, j + li(rec0), li(0)) * li(REC_WORDS) + li(m.o_prog);
      const li link = ldli(hoti, ro + li(R_LINK));
      const li bo = link * li(LB);
      const li ao = bo + li(B_A);
      M3 Rw;
      for (int i = 0; i < 9; ++i) Rw.a[i] = ldl(sm, ao + li(A_POSE + i));
      const V3 pw = ldv3l(sm, ao + li(A_POSE + 9));
      const SV v{ldv3l(sm, ao + li(A_W)), ldv3l(sm, ao + li(A_V))};
      const li nbody = ldli(hoti, ro + li(R_NBODY));
      // rigid inertia of the link's bodies (link coordinates), scaled per body
      real par[10];
      for (int q = 0; q < 10; ++q) par[q] = real(0);
      SV fext = sv_zero();
      const bool wrench = io.rb_force != nullptr;
      for (int jb = 0; jb < MAX_LINK_BODIES; ++jb) {
        const lb bon = on && (li(jb) < nbody);
        if (!any(bon)) continue;
        const li b = seli(bon, ldli(hoti, ro + li(R_BODY0 + jb)), li(0));
        const real sc = sel(bon, ldl(X, li(X_MASS) + b), real(0));
        real ib[10];
        for (int q = 0; q < 10; ++q) {
          ib[q] = sc * ldl(hot, li(m.o_body_inertia) + b * li(10) + li(q));
          par[q] = par[q] + ib[q];
        }
        // applied world wrenches at the bodies' COMs (tensors.rst.txt:322-335); the push acts on body 0
        const lb pushed = bon && (b == li(0)) && io.push;
        if (wrench || any(pushed)) {
          V3 F = sel3(pushed, ldv3q(X + X_PUSH), zero3), T = zero3;
          if (wrench) {
            F = F + sel3(bon, ldv3l(io.rb_force, b * li(3)), zero3);
            T = sel3(bon, ldv3l(io.rb_torque, b * li(3)), zero3);
          }
          const real inv = rcp_r(sel(ib[0] > real(1e-30), ib[0], real(1e-30)));
          const V3 com = mul(Rw, v3(ib[1] * inv, ib[2] * inv, ib[3] * inv));
          fext.w = fext.w + cross(com, F) + T;
          fext.v = fext.v + F;
        }
      }
      const V3 h = mul(Rw, v3(par[1], par[2], par[3]));  // m c, world axes
      const S3 Iw = rot_sym(Rw, S3{par[4], par[5], par[6], par[7], par[8], par[9]});
      // penalty ground contact: nothing of the link can reach z = 0 unless its origin is within its reach
      const lb near = on && (pw.z < ldl(hot, ro + li(R_REACH)));
      if (any(near)) {
        const V3 nrm = v3(Rw.a[6], Rw.a[7], Rw.a[8]);  // world z in link coordinates
        li kk = ldli(hoti, ro + li(R_PT0));
        const li k1 = ldli(hoti, ro + li(R_PT1));
        while (any(near && (kk < k1))) {
          const lb pon = near && (kk < k1);
          const li ks = seli(pon, kk, li(0));
          const V3 x = ldv3l(m.pt_pos, ks * li(3));
          const real rad = ldl(m.pt_radius, ks);
          const real z = pw.z + dot(nrm, x);
          penalty_point(p, mu, v, mul(Rw, x) - v3(0, 0, rad), rad - z, io.contact, ldli(m.pt_body, ks), pon, io.live, fext);
          kk = kk + li(1);
        }
        li cc = ldli(hoti, ro + li(R_CYL0));
        const li c1 = ldli(hoti, ro + li(R_CYL1));
        while (any(near && (cc < c1))) {
          const lb pon = near && (cc < c1);
          const li ks = seli(pon, cc, li(0));
          const V3 ctr = ldv3l(m.cyl_center, ks * li(3)), a = ldv3l(m.cyl_axis, ks * li(3));
          const real rad = ldl(m.cyl_size, ks * li(2)), hh = ldl(m.cyl_size, ks * li(2) + li(1));
          const real az = dot(nrm, a);
          const real s = sel(az >= real(0), real(-1), real(1));
          const V3 d = neg(nrm - az * a);
          const real dn = sqrt_r(dot(d, d));
          V3 rim = ctr + (s * hh) * a;
          rim = rim + sel(dn > real(1e-6), rad / sel(dn > real(1e-6), dn, real(1)), real(0)) * d;
          const real z = pw.z + dot(nrm, rim);
          penalty_point(p, mu, v, mul(Rw, rim), -z, io.contact, ldli(m.cyl_body, ks), pon, io.live, fext);
          cc = cc + li(1);
        }
      }
      const SV pA = SV{cross(v.w, mul(Iw, v.w)), cross(v.w, cross(v.w, h))} - fext;
      // classical velocity-product acceleration of the joint: [w_p x s qd; w_p x (w_p x r)], w_p = w - s qd
      const V3 sw = ldv3l(sm, bo + li(B_S)), rw = ldv3l(sm, bo + li(B_R));
      const real qd = sel(joint, ldl(sm, bo + li(B_QD)), real(0));
      const V3 wp = v.w - qd * sw;
      const SV cv{sel3(joint, cross(wp, qd * sw), zero3), sel3(joint, cross(wp, cross(wp, rw)), zero3)};
      // the foot pose is needed after this block has been overwritten
      const li f = ldli(hoti, ro + li(R_FOOT));
      const lb fon = on && (f >= li(0));
      if (any(fon)) {
        const li fo = li(nl * LB + X_FOOTPOSE) + seli(fon, f, li(0)) * li(12);
        for (int i = 0; i < 9; ++i) stl(sm, fo + li(i), Rw.a[i], fon);
        stl(sm, fo + li(9), pw.x, fon);
        stl(sm, fo + li(10), pw.y, fon);
        stl(sm, fo + li(11), pw.z, fon);
      }
      const real z = real(0);
      const real own[28] = {h.x, h.y, h.z, par[0], Iw.xx, Iw.yy, Iw.zz, Iw.xy, Iw.xz, Iw.yz, z, z,
                            pA.w.x, pA.w.y, pA.w.z, pA.v.x, pA.v.y, pA.v.z, z, z,
                            cv.w.x, cv.w.y, cv.w.z, cv.v.x, cv.v.y, cv.v.z, z, z};
      for (int i = 0; i < 28; ++i) stl(sm, ao + li(i), own[i], on);
    }
  }
  if (io_async) sync.wait_io(ioflags + F_IO_TAU, epoch + 1);
  lane_fence();
  sync.mark(18);
  // ---- pass 2, leaves -> root, DISTRIBUTED: lane c holds column c of the articulated inertia and component c of the
  //      bias force; the base role ends with the base itself (k = -1, record 0): inverse articulated inertia, base
  //      acceleration, predicted base velocity
  {
    real colp[6], pp = real(0);  // contribution of the link handled just before, to its parent
    for (int r = 0; r < 6; ++r) colp[r] = real(0);
    prev = -1;
    for (int k = len - 1; k >= (base_role ? -1 : 0); --k) {
      const float* R = k < 0 ? LREC(0) : LREC(rec0 + k);
      const int i = LRI(R, R_LINK);
      float* L = LBLK(i);
      float* A = L + B_A;
      real col[6], pc;
      {  // the link's own column: [[Ibar, h~], [h~^T, m 1]]
        real hx, hy, hz, mass;
        ld4(A + A_HM, hx, hy, hz, mass);
        const V3 Xc = cross(v3(hx, hy, hz), v3(lc.e0, lc.e1, lc.e2));  // h x e
        col[0] = sel(lc.ang, ldl(A + A_I, lc.ix0), Xc.x);
        col[1] = sel(lc.ang, ldl(A + A_I, lc.ix1), Xc.y);
        col[2] = sel(lc.ang, ldl(A + A_I, lc.ix2), Xc.z);
        col[3] = sel(lc.ang, -Xc.x, mass * lc.e0);
        col[4] = sel(lc.ang, -Xc.y, mass * lc.e1);
        col[5] = sel(lc.ang, -Xc.z, mass * lc.e2);
        pc = ldl(A + A_P, lc.c);
      }
      for (int j = 0; j < LRI(R, R_NCHILD); ++j) {
        const int cf = LRI(R, R_CHILD0 + j), c = cf & ~REC_FOREIGN;
        if (c == prev) {  // the child handled just before: its contribution is still in registers
          for (int r = 0; r < 6; ++r) col[r] = col[r] + colp[r];
          pc = pc + pp;
        } else {
          if (cf & REC_FOREIGN) sync.wait(fl + c, base + ST_PASS2);
          const float* Ac = LBLK(c) + B_A;
          const real actf = sel(lc.act, real(1), real(0));
          for (int r = 0; r < 6; ++r) col[r] = col[r] + actf * ldl(Ac + A_CIA, packed_index(lc, r));
          pc = pc + actf * ldl(Ac + A_CPA, seli(lc.act, lc.c, li(0)));
        }
      }
      if (k >= 0) {
        real sx, sy, sz, q, rx, ry, rz, qd, tq, damp, arm, free_;
        ld4(L + B_S, sx, sy, sz, q);
        ld4(L + B_R, rx, ry, rz, qd);
        ld4(L + B_SC, tq, damp, arm, free_);
        const V3 sw = v3(sx, sy, sz), rw = v3(rx, ry, rz);
        if (p.clamp_effort) {  // optional clamp of the actuation to the MJCF ctrlrange (SURVEY D2)
          const real lim = ld(R + R_EFF);
          tq = sel(tq > lim, lim, sel(tq < -lim, -lim, tq));
        }
        const real stiff = ld(R + R_STIFF);  // joint spring about q = 0, implicit like the damping
        const real Uc = col[0] * sw.x + col[1] * sw.y + col[2] * sw.z;  // U = IA [s; 0], component c
        const SV U = gather6(g, Uc);
        const real D = dot(sw, U.w) + arm + dt * (damp + dt * stiff);
        const real Dinv = rcp_r(D);
        const V3 pAw = v3(bc(g, pc, 0), bc(g, pc, 1), bc(g, pc, 2));
        const real u = tq - damp * qd - stiff * (q + dt * qd) - dot(sw, pAw);
        const SV cv = ld_sv8(A + A_C);
        // Ia = IA - U U^T / D; pa = pA + Ia c + U u / D
        const real t = Dinv * Uc;
        real ia[6] = {col[0] - t * U.w.x, col[1] - t * U.w.y, col[2] - t * U.w.z,
                      col[3] - t * U.v.x, col[4] - t * U.v.y, col[5] - t * U.v.z};
        real pa = pc + col_dot(ia, cv) + (Dinv * u) * Uc;
        // shift to the parent's origin (r = this origin - parent origin): A' = T^T Ia T, T = [[1, 0], [-r~, 1]]
        // (1) columns: angular column c -= r_(c+2) lin column (c+1) - r_(c+1) lin column (c+2)   (indices mod 3)
        const real ra = sel(lc.ang, lc.e0 * rw.y + lc.e1 * rw.z + lc.e2 * rw.x, real(0));  // r_(cm+1)
        const real rb = sel(lc.ang, lc.e0 * rw.z + lc.e1 * rw.x + lc.e2 * rw.y, real(0));  // r_(cm+2)
        for (int r = 0; r < 6; ++r) ia[r] = ia[r] - rb * sh(g, ia[r], lc.s1) + ra * sh(g, ia[r], lc.s2);
        // (2) rows: top += r x bottom, every column
        {
          const V3 tb = cross(rw, v3(ia[3], ia[4], ia[5]));
          ia[0] = ia[0] + tb.x; ia[1] = ia[1] + tb.y; ia[2] = ia[2] + tb.z;
        }
        {  // bias force: angular part += r x linear part
          const V3 tb = cross(rw, v3(bc(g, pa, 3), bc(g, pa, 4), bc(g, pa, 5)));
          pa = pa + sel(lc.ang, lc.e0 * tb.x + lc.e1 * tb.y + lc.e2 * tb.z, real(0));
        }
        for (int r = 0; r < 6; ++r) colp[r] = ia[r];
        pp = pa;
        prev = i;
        stl(L + B_U, lc.c, Uc, lc.c >= li(0));  // (idle lanes write their zero into the two spare words)
        st4(L + B_SC, u, Dinv, real(0), real(0));
        // the contribution goes through the scratch block unless the parent is the very next link of this role
        // (R_CSLOT >= 0, decided when the model is built)
        const int cslot = LRI(R, R_CSLOT);
        if (cslot >= 0) {
          lane_fence();  // every lane has read the own terms of this block
          st_sv8(X + X_CV + 8 * cslot, cv);  // pass 3 still needs it
          // packed symmetric storage: every entry is written by the lane that holds it with row <= column
          for (int r = 0; r < 6; ++r) {
            const lb le_c = li(r) <= lc.c;
            const lb mine = r < 3 ? (lc.ang && le_c) : (lc.ang || (lc.lin && le_c));
            stl(A + A_CIA, packed_index(lc, r), ia[r], mine);
          }
          stl(A + A_CPA, seli(lc.act, lc.c, li(0)), pa, lc.act);
          if (LRI(R, R_FLAGS) & RF_PARENT_FOREIGN) sync.signal(fl + i, base + ST_PASS2);
          else lane_fence();
        }
        continue;
      }
      sync.mark(3);
      // ---- the base: gather the 6x6, invert, base acceleration, predicted velocity (replicated)
      ABI IA;
      {
        real F[6][6];
        for (int r = 0; r < 6; ++r)
          for (int c = 0; c < 6; ++c) F[r][c] = bc(g, col[r], c);
        IA.I = S3{F[0][0], F[1][1], F[2][2], F[0][1], F[0][2], F[1][2]};
        IA.M = S3{F[3][3], F[4][4], F[5][5], F[3][4], F[3][5], F[4][5]};
        for (int a = 0; a < 3; ++a)
          for (int b = 0; b < 3; ++b) IA.H.a[3 * a + b] = F[a][3 + b];
      }
      const SV pA = gather6(g, pc);
      const ABI Om0 = abi_inverse_spd(IA);
      const SV a0 = real(-1) * mul(Om0, pA);  // [angular acceleration; acceleration of the origin relative to the gravity field]
      // (the base's velocity: its copy in the block was overwritten by the own terms; the root state still holds it)
      const SV v = SV{ldv3(X + X_ROOT + 10), ldv3(X + X_ROOT + 7)};
      lane_fence();  // all lanes have read the base's own terms: the block may be overwritten
      st_sv8(A + A_ACC, a0);  // (the two spare words of the 8-word slot belong to Om0: written next)
      st_abi_packed(A + A_OM0, Om0);
      // Predicted base velocity as the contact stage sees it. The model (oracle/physics_oracle.py) advances the base
      // twist by its BODY-frame components, i.e. it holds the body frame fixed over the step: in world axes that is the
      // classical update minus dt w x u; the term is given back when the base is integrated.
      const V3 rot = dt * cross(v.w, v.v);
      const SV vs{v.w + dt * a0.w, v.v + dt * (a0.v + v3(p.g[0], p.g[1], p.g[2])) - rot};
      st_sv8(L + B_U, vs);
      st4(L + B_SC, rot.x, rot.y, rot.z, real(0));
      sync.signal(fl + 0, base + ST_PASS2);
      // inverse inertia at the feet's common ancestor: Om_j = X Om_parent X^T + S D^-1 S^T down the shared links
      ABI Oml = Om0;
      for (int k2 = 0; k2 < m.shared_len; ++k2) {
        const float* Ls = LBLK(LRI(LREC(m.shared_rec[k2]), R_LINK));
        const V3 ss = ldv3q(Ls + B_S), rs = ldv3q(Ls + B_R);
        const real Dinv = ld(Ls + B_SC + 1);
        const SV w = Dinv * shift_force_T(rs, ld_sv8(Ls + B_U));
        const SV y = mul(Oml, w);
        Oml = inv_joint_update(inv_shift_to_child(rs, Oml), ss, shift_motion(rs, y), dot(w, y) + Dinv);
      }
      st_abi_packed(X + X_OML, Oml);
      sync.signal(qflags + F_OML, epoch + 1);
    }
  }
  if (!base_role) sync.mark(3);
  sync.mark(4);
  // ---- feet, part 1 (needs pass 2 of the own leg chain only), DISTRIBUTED: up the chain, lane c carries column c of
  //      G = map foot force -> force on the current link, and column c of Om = sum_j g_j g_j^T / D_j, g_j = S_j^T G_j
  int foot = -1;
  for (int f = 0; f < m.num_feet; ++f)
    if (m.foot_role[f] == role) foot = f;
  real Gc[6], Om[6];
  for (int r = 0; r < 6; ++r) {
    Gc[r] = real(0);
    Om[r] = real(0);
  }
  if (foot >= 0) {
    Gc[0] = sel(lc.ang, lc.e0, real(0)); Gc[1] = sel(lc.ang, lc.e1, real(0)); Gc[2] = sel(lc.ang, lc.e2, real(0));
    Gc[3] = sel(lc.lin, lc.e0, real(0)); Gc[4] = sel(lc.lin, lc.e1, real(0)); Gc[5] = sel(lc.lin, lc.e2, real(0));
    for (int k = m.chain_len[foot] - 1; k >= 0; --k) {
      const float* L = LBLK(LRI(LREC(m.chain_rec[foot][k]), R_LINK));
      const V3 sw = ldv3q(L + B_S), rw = ldv3q(L + B_R);
      const real Dinv = ld(L + B_SC + 1);
      const SV U = ld_sv8(L + B_U);
      const real gc = sw.x * Gc[0] + sw.y * Gc[1] + sw.z * Gc[2];
      const SV gg = gather6(g, gc);
      const real t = Dinv * gc;
      Om[0] = Om[0] + t * gg.w.x; Om[1] = Om[1] + t * gg.w.y; Om[2] = Om[2] + t * gg.w.z;
      Om[3] = Om[3] + t * gg.v.x; Om[4] = Om[4] + t * gg.v.y; Om[5] = Om[5] + t * gg.v.z;
      // G_c <- shift_force_T(r, G_c - U g_c / D)
      Gc[0] = Gc[0] - t * U.w.x; Gc[1] = Gc[1] - t * U.w.y; Gc[2] = Gc[2] - t * U.w.z;
      Gc[3] = Gc[3] - t * U.v.x; Gc[4] = Gc[4] - t * U.v.y; Gc[5] = Gc[5] - t * U.v.z;
      const V3 tb = cross(rw, v3(Gc[3], Gc[4], Gc[5]));
      Gc[0] = Gc[0] + tb.x; Gc[1] = Gc[1] + tb.y; Gc[2] = Gc[2] + tb.z;
    }
  }
  // active sole points of this foot (needs the foot pose of pass 1 only), LANE = CANDIDATE: candidates below the contact
  // offset, at most MAX_ACTIVE_PTS in candidate order, with their location relative to the foot origin and the velocity
  // bias of the non-penetration row; kept in the env's scratch (X_PTS)
  int nact = 0;
  const real inv_dt = rcp_r(dt);
  float* const pts = X + X_PTS + (foot >= 0 ? foot : 0) * MAX_ACTIVE_PTS * PT_WORDS;
  if (foot >= 0) {
    real px, py, pz;
    const M3 Rwf = ld_pose_rot(X + X_FOOTPOSE + 12 * foot, px, py, pz);
    const V3 nrm = v3(Rwf.a[6], Rwf.a[7], Rwf.a[8]);
    for (int j0 = 0; j0 < m.foot_npts[foot]; j0 += LPE) {
      const li kc = lc.c + li(j0);
      const lb valid = kc < li(m.foot_npts[foot]);
      const li fo = li(m.o_foot_pts) + (li(foot * MAX_SOLVER_PTS) + seli(valid, kc, li(0))) * li(4);
      const V3 x = ldv3l(hot, fo);
      const real rad = ldl(hot, fo + li(3));
      const real phi = pz + dot(nrm, x) - rad;
      const lb hit = valid && (phi < real(p.contact_offset));
      const li slot = grank(g, hit) + li(nact);
      const lb keep = hit && (slot < li(MAX_ACTIVE_PTS));
      const li po = seli(keep, slot, li(0)) * li(PT_WORDS);
      const V3 xa = mul(Rwf, x) - v3(0, 0, rad);  // the sphere's lowest point, relative to the foot origin, world axes
      const real bias = sel(phi >= real(0), -phi * inv_dt, fmin_r(-real(p.erp) * phi * inv_dt, real(p.max_depen_vel)));
      stl(pts, po, int_bits_as_real(kc), keep);
      stl(pts, po + li(1), bias, keep);
      stl(pts, po + li(2), real(0), keep);
      stl(pts, po + li(3), real(0), keep);
      stl(pts, po + li(4), real(0), keep);
      stl(pts, po + li(5), xa.x, keep);
      stl(pts, po + li(6), xa.y, keep);
      stl(pts, po + li(7), xa.z, keep);
      nact += gcount(g, hit);
    }
    nact = nact < MAX_ACTIVE_PTS ? nact : MAX_ACTIVE_PTS;
    lane_fence();
  }
  sync.mark(5);
  // ---- pass 3, replicated chain root -> leaves: joint accelerations, predicted joint velocities
  prev = -1;
  SV a_prev = sv_zero();
  for (int k = 0; k < len; ++k) {
    const float* R = LREC(rec0 + k);
    const int i = LRI(R, R_LINK), par = LRI(R, R_PARENT), flg = LRI(R, R_FLAGS);
    if (flg & RF_PARENT_BASE) {
      if (!base_role) sync.wait(fl + 0, base + ST_PASS2);
    } else if (flg & RF_PARENT_FOREIGN) {
      sync.wait(fl + par, base + ST_PASS3);
    }
    float* L = LBLK(i);
    if (par != prev) a_prev = ld_sv8(LBLK(par) + B_A + A_ACC);
    real sx, sy, sz, q, rx, ry, rz, qd, u, Dinv, x2, x3;
    ld4(L + B_S, sx, sy, sz, q);
    ld4(L + B_R, rx, ry, rz, qd);
    ld4(L + B_SC, u, Dinv, x2, x3);
    const V3 sw = v3(sx, sy, sz), rw = v3(rx, ry, rz);
    const int cslot = LRI(R, R_CSLOT);
    SV a = shift_motion(rw, a_prev) + (cslot >= 0 ? ld_sv8(X + X_CV + 8 * cslot) : ld_sv8(L + B_A + A_C));
    const real qdd = Dinv * (u - dot(ld_sv8(L + B_U), a));
    a.w = a.w + qdd * sw;
    a_prev = a;
    prev = i;
    st(L + B_QD, qd + dt * qdd);
    if (flg & (RF_PUBLISH | RF_KEEP)) {  // read by children that are not the next link of this role
      st_sv8(L + B_A + A_ACC, a);
      if (flg & RF_PUBLISH) sync.signal(fl + i, base + ST_PASS3);
      else lane_fence();
    }
  }
  sync.mark(6);
  // ---- feet, part 2: predicted foot velocity, Om += G^T Om_lca G, rows of the active points, the sweeps
  if (foot >= 0) {
    const int gf = foot;
    const int clen = m.chain_len[gf];
    SV V = ld_sv8(LBLK(0) + B_U);  // base role published v0* with ST_PASS2 (waited for in pass 3)
    SV P = sv_zero();              // accumulated contact impulse on the foot (world axes, about the foot origin)
    if (m.shared_len > 0) {  // predicted velocity of the common ancestor (needs pass 3 of the shared links)
      sync.wait(fl + m.lca, base + ST_PASS3);
      for (int k = 0; k < m.shared_len; ++k) {
        const float* Ls = LBLK(LRI(LREC(m.shared_rec[k]), R_LINK));
        V = shift_motion(ldv3q(Ls + B_R), V);
        V.w = V.w + ld(Ls + B_QD) * ldv3q(Ls + B_S);
      }
    }
    for (int k = 0; k < clen; ++k) {
      const float* L = LBLK(LRI(LREC(m.chain_rec[gf][k]), R_LINK));
      real rx, ry, rz, qd;
      ld4(L + B_R, rx, ry, rz, qd);
      V = shift_motion(v3(rx, ry, rz), V);
      V.w = V.w + qd * ldv3q(L + B_S);
    }
    real Yc[6];  // column c of Y = Om_lca G
    {
      sync.wait(qflags + F_OML, epoch + 1);
      const ABI Om0 = ld_abi_packed(X + X_OML);  // inverse inertia at the common ancestor (= the base's for TOCABI)
      const SV y = mul(Om0, SV{v3(Gc[0], Gc[1], Gc[2]), v3(Gc[3], Gc[4], Gc[5])});
      Yc[0] = y.w.x; Yc[1] = y.w.y; Yc[2] = y.w.z; Yc[3] = y.v.x; Yc[4] = y.v.y; Yc[5] = y.v.z;
      // Om column c += G^T Y_c: entry a = G_a . Y_c
      for (int a = 0; a < 6; ++a) {
        real s = real(0);
        for (int r = 0; r < 6; ++r) s = s + bc(g, Gc[r], a) * Yc[r];
        Om[a] = Om[a] + s;
      }
      // rows of Y for the feet's coupling (z = Y dP needs row r in lane r): transposed through the chain links' blocks
      for (int r = 0; r < 6; ++r) stl(LBLK(m.chain[gf][r]) + B_A + A_YT, lc.c, Yc[r], lc.c >= li(0));
      lane_fence();
    }
    real Yr[6];  // row c of Y in lane c (row r sits in the block of chain link r); zero in the idle lanes
    for (int a = 0; a < 6; ++a) {
      real acc = real(0);
      for (int r = 0; r < 6; ++r) acc = sel(lc.c == li(r), ld(LBLK(m.chain[gf][r]) + B_A + A_YT + a), acc);
      Yr[a] = acc;
    }
    // rows of the active points, DISTRIBUTED: response cv = Om J (component c in lane c) and 1 / (J . cv) per direction
    // (world z, x, y), parked in the blocks of the first chain links (ROWS_PER_LINK per link)
    for (int a = 0; a < nact; ++a) {
      const V3 xa = ldv3(pts + a * PT_WORDS + 5);
      for (int d = 0; d < 3; ++d) {
        const V3 dir = d == 0 ? v3(0, 0, 1) : (d == 1 ? v3(1, 0, 0) : v3(0, 1, 0));
        const SV J{cross(xa, dir), dir};
        const real cvc = col_dot(Om, J);
        const SV cv = gather6(g, cvc);
        const int row = a * 3 + d;
        float* rw = LBLK(m.chain[gf][row / ROWS_PER_LINK]) + B_A + A_ROWS + (row % ROWS_PER_LINK) * 8;
        st_sv8(rw, cv);
        st(rw + 6, rcp_r(dot(J, cv)));
      }
    }
    sync.mark(7);
    // fixed number of sweeps, replicated; Gauss-Seidel inside a foot, Jacobi between the feet (coupled through the base)
    const real mu = ld(X + X_MU);
    for (int s = 0; s < p.sweeps; ++s) {
      SV dP = sv_zero();
      for (int a = 0; a < nact; ++a) {
        float* pt = pts + a * PT_WORDS;
        real kf, bias, l0, l1, l2, xx, xy, xz;
        ld4(pt, kf, bias, l0, l1);
        ld4(pt + 4, l2, xx, xy, xz);
        const V3 xa = v3(xx, xy, xz);
        real lam[3] = {l0, l1, l2};
        for (int d = 0; d < 3; ++d) {
          const V3 dir = d == 0 ? v3(0, 0, 1) : (d == 1 ? v3(1, 0, 0) : v3(0, 1, 0));
          const SV J{cross(xa, dir), dir};
          const int row = a * 3 + d;
          const float* rw = LBLK(m.chain[gf][row / ROWS_PER_LINK]) + B_A + A_ROWS + (row % ROWS_PER_LINK) * 8;
          real c0, c1, c2, c3, c4, c5, winv, c7;
          ld4(rw, c0, c1, c2, c3);
          ld4(rw + 4, c4, c5, winv, c7);
          const real vrel = dot(J, V);
          real nw;
          if (d == 0) {
            nw = lam[0] + (bias - vrel) * winv;
            nw = sel(nw > real(0), nw, real(0));
          } else {
            const real lim = mu * lam[0];
            nw = lam[d] - vrel * winv;
            nw = sel(nw > lim, lim, sel(nw < -lim, -lim, nw));
          }
          const real delta = nw - lam[d];
          lam[d] = nw;
          V = V + delta * SV{v3(c0, c1, c2), v3(c3, c4, c5)};
          dP = dP + delta * J;
        }
        st(pt + 2, lam[0]);
        st(pt + 3, lam[1]);
        st(pt + 4, lam[2]);
      }
      P = P + dP;
      if (m.num_feet == 2) {
        // base velocity change caused by this sweep's impulses: z = Om_lca G dP = Y dP, row c in lane c
        // (double-buffered by sweep parity)
        const int seq = epoch * 64 + s + 1;
        const real zc = Yr[0] * dP.w.x + Yr[1] * dP.w.y + Yr[2] * dP.w.z + Yr[3] * dP.v.x + Yr[4] * dP.v.y + Yr[5] * dP.v.z;
        stl(X + X_Z + ((s & 1) * MAX_FEET + gf) * 8, lc.c, zc, lc.c >= li(0));
        sync.signal(qflags + F_Z + gf, seq);
        sync.wait(qflags + F_Z + (1 - gf), seq);
        const SV z = ld_sv8(X + X_Z + ((s & 1) * MAX_FEET + (1 - gf)) * 8);
        // response of this foot: G^T z, component c = G_c . z
        const real rc = Gc[0] * z.w.x + Gc[1] * z.w.y + Gc[2] * z.w.z + Gc[3] * z.v.x + Gc[4] * z.v.y + Gc[5] * z.v.z;
        V = V + gather6(g, rc);
      }
    }
    sync.mark(8);
    // contact impulse -> joint space: the foot impulse P travels up the chain as a force f_j = G_j P;
    // S^T dp of link j is -s_j . f_j, what arrives at the common ancestor is -f
    {
      SV f = P;
      for (int k = clen - 1; k >= 0; --k) {
        float* L = LBLK(LRI(LREC(m.chain_rec[gf][k]), R_LINK));
        const V3 sw = ldv3q(L + B_S), rw = ldv3q(L + B_R);
        const real sd = dot(sw, f.w);
        st(L + B_SC + 2, -sd);
        f = shift_force_T(rw, f - (ld(L + B_SC + 1) * sd) * ld_sv8(L + B_U));
      }
      st_sv8(X + X_PD + 8 * gf, real(-1) * f);
    }
    sync.signal(qflags + F_PD + gf, epoch + 1);
    if (io.live) {
      const int* fbody = hoti + m.o_foot_body + gf * MAX_SOLVER_PTS;
      for (int a = 0; a < nact; ++a) {  // world force over this sub-step: rows (n, t1, t2) = world (z, x, y)
        const float* pt = pts + a * PT_WORDS;
        const li kc = real_bits_as_int(ld(pt));
        const li o = ldli(fbody, kc) * li(3);
        const lb first = lc.c == li(0);  // one lane does the read-modify-write
        stl(io.contact, o, ldl(io.contact, o) + ld(pt + 3) * inv_dt, first);
        stl(io.contact, o + li(1), ldl(io.contact, o + li(1)) + ld(pt + 4) * inv_dt, first);
        stl(io.contact, o + li(2), ldl(io.contact, o + li(2)) + ld(pt + 2) * inv_dt, first);
      }
    }
  }
  sync.mark(9);
  // ---- base response to the contact impulses (base role, replicated)
  if (base_role) {
    SV pd = sv_zero();
    for (int f = 0; f < m.num_feet; ++f) {
      sync.wait(qflags + F_PD + f, epoch + 1);
      pd = pd + ld_sv8(X + X_PD + 8 * f);  // impulse arriving at the common ancestor
    }
    for (int k = m.shared_len - 1; k >= 0; --k) {  // ... and from there up the shared links to the base
      float* Ls = LBLK(LRI(LREC(m.shared_rec[k]), R_LINK));
      const real sd = dot(ldv3q(Ls + B_S), pd.w);
      st(Ls + B_SC + 2, sd);
      pd = shift_force_T(ldv3q(Ls + B_R), pd - (ld(Ls + B_SC + 1) * sd) * ld_sv8(Ls + B_U));
    }
    st_sv8(LBLK(0) + B_S, real(-1) * mul(ld_abi_packed(LBLK(0) + B_A + A_OM0), pd));
    sync.signal(fl + 0, base + ST_DOWN);
  }
  sync.mark(10);
  // ---- down the tree, replicated: joint velocity changes, speed cap, integration, limit projection
  if (io_async) sync.wait_io(ioflags + F_IO_DONE, epoch + 1);
  prev = -1;
  for (int k = 0; k < len; ++k) {
    const float* R = LREC(rec0 + k);
    const int i = LRI(R, R_LINK), par = LRI(R, R_PARENT), flg = LRI(R, R_FLAGS);
    if (flg & RF_PARENT_BASE) {
      if (!base_role) sync.wait(fl + 0, base + ST_DOWN);
    } else if (flg & RF_PARENT_FOREIGN) {
      sync.wait(fl + par, base + ST_DOWN);
    }
    float* L = LBLK(i);
    if (par != prev) a_prev = par == 0 ? ld_sv8(LBLK(0) + B_S) : ld_sv8(LBLK(par) + B_A + A_DV);
    real sx, sy, sz, q, rx, ry, rz, qds, u, Dinv, dp, x3;
    ld4(L + B_S, sx, sy, sz, q);
    ld4(L + B_R, rx, ry, rz, qds);
    ld4(L + B_SC, u, Dinv, dp, x3);
    const V3 sw = v3(sx, sy, sz);
    SV dv = shift_motion(v3(rx, ry, rz), a_prev);
    const real dqd = -Dinv * (dot(ld_sv8(L + B_U), dv) + dp);
    dv.w = dv.w + dqd * sw;
    a_prev = dv;
    prev = i;
    if (flg & (RF_PUBLISH | RF_KEEP)) {
      st_sv8(L + B_A + A_DV, dv);
      if (flg & RF_PUBLISH) sync.signal(fl + i, base + ST_DOWN);
      else lane_fence();
    }
    // joint velocity cap (dof_prop['velocity'], T:372), explicit Euler on the angle, limit projection
    const real vl = ld(R + R_VLIM);
    real qdn = qds + dqd;
    qdn = sel(qdn > vl, vl, sel(qdn < -vl, -vl, qdn));
    real qn = q + dt * qdn;
    const real lo = ld(R + R_LO), up = ld(R + R_UP);
    const lb over = qn > up, under = qn < lo;
    qdn = sel(over, sel(qdn < real(0), qdn, real(0)), sel(under, sel(qdn > real(0), qdn, real(0)), qdn));
    qn = sel(over, up, sel(under, lo, qn));
    st(L + B_Q, qn);  // new joint state; the slab copy writes it to dof_state
    st(L + B_QD, qdn);
  }
  sync.mark(11);
  // ---- base integration (base role, replicated): the base velocity is already in world axes
  if (base_role) {
    const float* L = LBLK(0);
    const SV vb = ld_sv8(L + B_U) + ld_sv8(L + B_S);
    V3 ww = vb.w;
    const V3 vw = vb.v + ldv3q(L + B_SC);
    const real wn = sqrt_r(dot(ww, ww));
    ww = sel(wn > real(p.max_ang_vel), real(p.max_ang_vel) / sel(wn > real(p.max_ang_vel), wn, real(1)), real(1)) * ww;
    float* rs = X + X_ROOT;
    real r0, r1, r2, qx, qy, qz, qw, r7;
    ld4(rs, r0, r1, r2, qx);
    ld4(rs + 4, qy, qz, qw, r7);
    const real h = real(0.5) * dt;
    const real nx = qx + h * (ww.x * qw + ww.y * qz - ww.z * qy);
    const real ny = qy + h * (-ww.x * qz + ww.y * qw + ww.z * qx);
    const real nz = qz + h * (ww.x * qy - ww.y * qx + ww.z * qw);
    const real nw = qw + h * (-ww.x * qx - ww.y * qy - ww.z * qz);
    const real inv = rcp_r(sqrt_r(nx * nx + ny * ny + nz * nz + nw * nw));
    lane_fence();
    st4(rs, r0 + dt * vw.x, r1 + dt * vw.y, r2 + dt * vw.z, nx * inv);
    st4(rs + 4, ny * inv, nz * inv, nw * inv, vw.x);
    st4(rs + 8, vw.y, vw.z, ww.x, ww.y);
    st(rs + 12, ww.z);
  }
  sync.mark(12);
}

}  // namespace ln
}  // namespace dyros
