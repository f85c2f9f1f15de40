// One sub-step of gym.simulate, written as the program of ONE ROLE acting on ONE env.
//
// Replaces the body of `gym.simulate` (reference call site tasks/dyros_dynamic_walk.py:525; the reference's
// implementation is closed-source PhysX) for a floating-base tree of revolute joints: articulated-body
// forward dynamics (Featherstone ABA) with implicit joint damping and rotor inertia, penalty ground contact for all
// collision primitives except the sole corners, and a fixed-sweep projected Gauss-Seidel solve of the sole-corner
// contacts in the 6-D space of each foot link using the exact articulated inverse inertia (O(n) recursion up the
// leg chains). The model and every formula are stated independently (dense, fp64) in oracle/physics_oracle.py;
// see DESIGN.md section 4.
//
// Coordinates: every spatial quantity of a link is expressed in WORLD axes with the link's origin as reference point,
// and accelerations are classical (d/dt of the origin's velocity), as in most production articulation solvers. The
// transforms between a link and its parent are then pure translations (no 3x3 rotations inside the recursions); the
// price is one rotation of the link's rigid inertia per sub-step and the classical velocity-product terms
// c = [w_p x s qd; w_p x (w_p x r)], p = [w x I w; w x (w x h)].
//
// Parallel decomposition (GPU): the link tree is cut into DYROS_LANES "roles" (model/tables.py::role_programs: torso
// + left arm, head + right arm (+ base), left leg, right leg for TOCABI). A CTA holds one warp per role; lane = env,
// so a warp runs the same link operation on up to 32 envs (no divergence, warp-uniform table reads). Roles exchange
// per-link results through the env's scratch block in shared memory and order themselves with per-link stage flags
// (release/acquire on shared memory): a role only ever waits for what it actually consumes, so the legs run their
// three tree passes and the whole contact stage while the arm roles are still in theirs.
// The same source is compiled for the host by tests/native/hostemu.cu (one thread per role, atomics for the flags).
#pragma once
#include "internal.h"
#include "phys_math.cuh"

namespace dyros {

// per-link scratch block (floats) of one env
constexpr int LS_E = 0;    // 9  pass 1a: parent->link rotation; from pass 1b on: joint axis s (3) and offset from the
                           //    parent's origin r (3), both in world axes (LS_S, LS_R)
constexpr int LS_V = 9;    // 6  link velocity [w; u], later the impulse response dv
constexpr int LS_A = 15;   // 27 pass1: world pose(12) at +6 | pass2: contribution to parent IA(21) pA(6) |
                           //    pass3: a'(6); leg-chain links then also hold contact rows (14) and g = S^T G (6);
                           //    the first chain link keeps g in X_G0 (the base may still be reading its A block)
constexpr int LS_U = 42;   // 6  U = IA S (base: predicted velocity v0*)
constexpr int LS_SC = 48;  // 4  [qd -> qd*, tau -> u, damping -> 1/D, armature -> S^T dp]
constexpr int LS_Q = 52;   // 1  joint angle
constexpr int LS = 53;
constexpr int LS_S = LS_E, LS_R = LS_E + 3;
constexpr int LS_WP = LS_E + 6;  // 3  from pass 1b on: the parent's angular velocity (pass 3 of a link whose parent is
                                 //    not the role's previous link: the parent's LS_V may hold dv by then)
constexpr int A_POSE = 6, A_CIA = 0, A_CPA = 21, A_ACC = 0, A_OM0 = 6, A_ROWS = 6, A_G = 21;
constexpr int ROWS_PER_LINK = 2;  // contact rows (7 floats each) parked in one leg-chain link's block
// per-env extra scratch
constexpr int X_FOOTPOSE = 0;                        // MAX_FEET * 12
constexpr int X_Z = X_FOOTPOSE + MAX_FEET * 12;      // 2 (double buffer) * MAX_FEET * 6: base velocity change of a sweep
constexpr int X_PD = X_Z + 2 * MAX_FEET * 6;         // MAX_FEET * 6  impulse arriving at the base from a foot
constexpr int X_G0 = X_PD + MAX_FEET * 6;            // MAX_FEET * 6  g = S^T G of the first leg-chain link (see A_G)
constexpr int X_ROOT = X_G0 + MAX_FEET * 6;          // 13 (+3 pad): root state in, root state out
constexpr int X_PUSH = X_ROOT + 13;                  // 3  world force at the base body's COM for this sub-step
constexpr int X_OML = X_ROOT + 16;                   // 21: inverse inertia at the feet's common ancestor (LCA)
constexpr int PT_WORDS = 5;                          // active sole point: candidate index (int), bias, impulse lam(3)
constexpr int X_PTS = X_OML + 21;                    // MAX_FEET * MAX_ACTIVE_PTS * PT_WORDS
constexpr int X_MU = X_PTS + MAX_FEET * MAX_ACTIVE_PTS * PT_WORDS;    // 1  friction coefficient of this env's ground contacts
constexpr int X_MASS = X_MU + 1;                     // nb per-body mass scales (last: sized by the model)
// the words of the scratch block that the kernels' slab copies fill and read back (physics_cta.cuh)
struct RolesScratch {
  static constexpr int link = LS, q = LS_Q, qd = LS_SC, tau = LS_SC + 1, damping = LS_SC + 2, armature = LS_SC + 3;
  static constexpr int mu = X_MU, mass = X_MASS, root = X_ROOT, push = X_PUSH;
};

HD int env_scratch_floats(int nl, int nb) {
  int n = nl * LS + X_MASS + nb;
  return n | 1;  // odd stride: the 32 envs of a warp touch 32 different banks for any field
}

// CTA-wide flags (ints): stage reached by each link, plus the hand-shakes of the contact stage
constexpr int F_LINK = 0;                         // [DYROS_MAX_LINKS]
constexpr int F_Z = DYROS_MAX_LINKS;              // [MAX_FEET] sweeps published
constexpr int F_PD = F_Z + MAX_FEET;              // [MAX_FEET] base impulse published
constexpr int F_OML = F_PD + MAX_FEET;            // [1] inverse inertia at the LCA published
constexpr int F_IO_PRE = F_OML + 1;               // [1] fused step: push staged, contact forces zeroed (I/O warp)
constexpr int F_IO_TAU = F_IO_PRE + 1;            // [1] fused step: torque, damping and armature staged (I/O warp)
constexpr int F_IO_DONE = F_IO_TAU + 1;           // [1] fused step: the I/O group no longer reads the joint angles
constexpr int F_COUNT = F_IO_DONE + 1;
constexpr int ST_PASS1 = 1, ST_PASS2 = 2, ST_PASS3 = 3, ST_DOWN = 4, ST_STRIDE = 8;

// The hot model tables are read from the staged copy `hot` (shared memory on the GPU) through word offsets.
#define HI(field, idx) (reinterpret_cast<const int*>(hot)[m.o_##field + (idx)])
#define HF(field, idx) (hot[m.o_##field + (idx)])
#define HF3(field, idx) ld3_f(hot + m.o_##field + 3 * (idx))
#define BLK(link) (sm + (link) * LS)
// record of a link in the flattened role programs (one base address, constant offsets: no dependent table walks)
#define REC(idx) (hot + m.o_prog + (idx) * REC_WORDS)
#define RI(R, field) (reinterpret_cast<const int*>(R)[field])

// global-memory views of one env (all device pointers on the GPU, host pointers in the emulation)
struct EnvIO {
  float* root;             // 13
  float* dof_state;        // nd*2
  const float* tau;        // nd
  const float* damping;    // nd
  const float* armature;   // nd
  const float* mass_scale; // nb
  const float* friction;   // 1 or NULL (SimParams.mu)
  float* contact;          // nb*3
  const float* push;       // 3 or NULL
  const float* rb_force;   // nb*3 or NULL
  const float* rb_torque;  // nb*3 or NULL
  float* link_pose;        // nl*12 or NULL: world pose of every link as pass 1 finds it (for the self-collision pass)
  bool live;               // false: padding lane, no global writes
};
HD void export_pose(const EnvIO& io, int link, const M3& Rw, V3 pw) {
  if (!io.link_pose || !io.live) return;
  float* o = io.link_pose + 12 * link;
  for (int c = 0; c < 9; ++c) o[c] = (float)Rw.a[c];
  o[9] = (float)pw.x; o[10] = (float)pw.y; o[11] = (float)pw.z;
}

// ---- the ground (DESIGN.md section 4), a compile-time parameter of the role program: the plane z = 0 with normal +z,
//      or a heightfield. Vertex (i, j) of the field sits at (ox + i dx, oy + j dy, oz + dz s[i, j]); each cell is split
//      along its diagonal (i, j)-(i+1, j+1); outside the field's x-y rectangle there is no ground.
// (PlaneGround, FieldGround: internal.h)

HD real field_sample(const int16_t* s) {
#ifdef __CUDA_ARCH__
  return (real)__ldg(s);  // read-only path: the samples are shared by every env and stay in L2
#else
  return (real)*s;
#endif
}

// Height h and unit upward normal n of the heightfield at (x, y); false outside the field. Grid coordinates
// u = (x - ox) / dx, v = (y - oy) / dy; the cell is (floor u, floor v), except that the last row / column of vertices
// belongs to the cell before it. Inside the cell (fu, fv), a point with fu >= fv (on the diagonal or on the +x side of
// it) takes the triangle (i, j), (i+1, j), (i+1, j+1); any other the triangle (i, j), (i, j+1), (i+1, j+1).
HD bool field_query(const FieldGround& g, real x, real y, real& h, V3& n) {
  const real u = (x - g.ox) / g.dx, v = (y - g.oy) / g.dy;
  if (!(u >= 0 && v >= 0 && u <= (real)(g.nr - 1) && v <= (real)(g.nc - 1))) return false;
  int i = (int)u, j = (int)v;
  i = i < g.nr - 2 ? i : g.nr - 2;
  j = j < g.nc - 2 ? j : g.nc - 2;
  const real fu = u - (real)i, fv = v - (real)j;
  const int16_t* c = g.s + (size_t)i * g.nc + j;
  const real h00 = g.dz * field_sample(c), h11 = g.dz * field_sample(c + g.nc + 1);
  real gu, gv;  // height change per grid step along u and along v on the chosen triangle
  if (fu >= fv) {
    const real h10 = g.dz * field_sample(c + g.nc);
    gu = h10 - h00;
    gv = h11 - h10;
  } else {
    const real h01 = g.dz * field_sample(c + 1);
    gu = h11 - h01;
    gv = h01 - h00;
  }
  h = g.oz + h00 + fu * gu + fv * gv;
  const real sx = gu / g.dx, sy = gv / g.dy;
  const real inv = 1 / sqrt(1 + sx * sx + sy * sy);
  n = v3(-sx * inv, -sy * inv, inv);
  return true;
}

// Tangent directions of a contact with ground normal n: t1 = normalize(n_z, 0, -n_x), t2 = n x t1 (world x and y for
// n = +z).
HD void field_tangents(V3 n, V3& t1, V3& t2) {
  const real inv = 1 / sqrt(n.z * n.z + n.x * n.x);
  t1 = v3(n.z * inv, 0, -n.x * inv);
  t2 = cross(n, t1);
}

// Heightfield: the active sole points of foot g (X_PTS, at most MAX_ACTIVE_PTS) from the start-of-step foot pose
// (X_FOOTPOSE); returns their number and the foot's world rotation. Gap phi = (z_c - h) n_z - r of a candidate sphere
// (centre c, radius r); active when phi < contact_offset. The ground normal of active point a is kept in LS_WP of the
// a-th link of the foot's chain (>= 6 links, all in the foot's role): so this runs after the role's pass 3, the last
// reader of LS_WP, and the env scratch block needs no extra words (the CTA still holds 28 TOCABI envs).
HD int field_select(const FieldGround& gnd, const DevModel& m, const SimParams& p, real* sm, real* X, int g, real inv_dt,
                    M3& Rwf) {
  Rwf = ld_m3(X + X_FOOTPOSE + 12 * g);
  const V3 pf = ld3(X + X_FOOTPOSE + 12 * g + 9);
  real* const pts = X + X_PTS + g * MAX_ACTIVE_PTS * PT_WORDS;
  int nact = 0;
  real h;
  V3 n;
#pragma unroll 1
  for (int k = 0; k < m.foot_npts[g]; ++k) {
    const V3 c = pf + mul(Rwf, v3(m.foot_pt_pos[g][k][0], m.foot_pt_pos[g][k][1], m.foot_pt_pos[g][k][2]));
    if (!field_query(gnd, c.x, c.y, h, n)) continue;
    real phi = (c.z - h) * n.z - m.foot_pt_radius[g][k];
    if (phi < p.contact_offset && nact < MAX_ACTIVE_PTS) {
      real* pt = pts + nact * PT_WORDS;
      reinterpret_cast<int*>(pt)[0] = k;
      pt[1] = phi >= 0 ? -phi * inv_dt : fmin_r(-p.erp * phi * inv_dt, p.max_depen_vel);
      pt[2] = pt[3] = pt[4] = 0;
      st3(BLK(m.chain[g][nact]) + LS_WP, n);
      ++nact;
    }
  }
  return nact;
}

// Heightfield: active sole point `a` of foot g -> its contact location relative to the foot origin, world axes (the
// sphere's point along -n), and its row directions n, t1, t2.
HD void field_sole_point(const DevModel& m, const real* sm, const real* X, const M3& Rwf, int g, int a, V3& xa, V3* dirs) {
  const int k = reinterpret_cast<const int*>(X + X_PTS + (g * MAX_ACTIVE_PTS + a) * PT_WORDS)[0];
  dirs[0] = ld3(BLK(m.chain[g][a]) + LS_WP);
  field_tangents(dirs[0], dirs[1], dirs[2]);
  xa = mul(Rwf, v3(m.foot_pt_pos[g][k][0], m.foot_pt_pos[g][k][1], m.foot_pt_pos[g][k][2])) - m.foot_pt_radius[g][k] * dirs[0];
}

// ---- penalty ground contact of one location on a link (oracle: PhysicsOracle._external_wrench.add_point);
//      xw = the location relative to the link origin, world axes; v = [w; u] of the link
HD void penalty_point(const SimParams& p, real mu, SV v, V3 xw, real depth, float* cf, bool live, SV& fext) {
  if (!(depth > 0)) return;
  V3 vel_w = v.v + cross(v.w, xw);
  real fn = p.pen_k * depth - p.pen_c * vel_w.z;
  fn = fn < 0 ? 0 : (fn > p.pen_fmax ? p.pen_fmax : fn);
  real speed = sqrt(vel_w.x * vel_w.x + vel_w.y * vel_w.y);
  real lim = mu * fn / (speed > (real)1e-6 ? speed : (real)1e-6);
  real coef = p.pen_c < lim ? p.pen_c : lim;
  V3 Fw = v3(-coef * vel_w.x, -coef * vel_w.y, fn);
  if (live) {
    cf[0] += (float)Fw.x;
    cf[1] += (float)Fw.y;
    cf[2] += (float)Fw.z;
  }
  fext.w = fext.w + cross(xw, Fw);
  fext.v = fext.v + Fw;
}
// the same against a ground of unit normal n at the contact location: normal force along n damped by v.n, friction on
// the tangential part of the velocity (= penalty_point for n = +z)
HD void penalty_point_n(const SimParams& p, real mu, SV v, V3 xw, V3 n, real depth, float* cf, bool live, SV& fext) {
  if (!(depth > 0)) return;
  V3 vel_w = v.v + cross(v.w, xw);
  const real vn = dot(vel_w, n);
  real fn = p.pen_k * depth - p.pen_c * vn;
  fn = fn < 0 ? 0 : (fn > p.pen_fmax ? p.pen_fmax : fn);
  const V3 vt = vel_w - vn * n;
  real speed = sqrt(dot(vt, vt));
  real lim = mu * fn / (speed > (real)1e-6 ? speed : (real)1e-6);
  real coef = p.pen_c < lim ? p.pen_c : lim;
  V3 Fw = fn * n - coef * vt;
  if (live) {
    cf[0] += (float)Fw.x;
    cf[1] += (float)Fw.y;
    cf[2] += (float)Fw.z;
  }
  fext.w = fext.w + cross(xw, Fw);
  fext.v = fext.v + Fw;
}

// Rigid inertia of the link of record R about its origin in WORLD axes, from the hot body table (link coordinates),
// the env's per-body mass scales (X_MASS) and the link's world rotation Rw.
HD ABI link_inertia(const real* X, const float* hot, const DevModel& m, const float* R, const M3& Rw) {
  real par[10];
  {  // first body (most links have exactly one): straight-line code; massless links (extra hinges of a body) have none
    const bool any = RI(R, R_NBODY) > 0;
    int b = any ? RI(R, R_BODY0) : 0;
    real sc = any ? X[X_MASS + b] : (real)0;
#pragma unroll
    for (int k = 0; k < 10; ++k) par[k] = sc * HF(body_inertia, b * 10 + k);
  }
#pragma unroll 1
  for (int j = 1; j < RI(R, R_NBODY); ++j) {
    int b = RI(R, R_BODY0 + j);
    real sc = X[X_MASS + b];
#pragma unroll
    for (int k = 0; k < 10; ++k) par[k] += sc * HF(body_inertia, b * 10 + k);
  }
  return abi_rigid(par[0], mul(Rw, v3(par[1], par[2], par[3])), rot_sym(Rw, S3{par[4], par[5], par[6], par[7], par[8], par[9]}));
}

// External wrench on the link of record R (world axes, about the link origin): applied body wrenches and penalty
// ground contact.
template <class Ground>
HD SV link_ext_wrench(const EnvIO& io, const real* X, const float* hot, const DevModel& m, const SimParams& p,
                      const float* R, const M3& Rw, V3 pw, SV v, const Ground& gnd) {
  SV fext = sv_zero();
  V3 nrm = v3(Rw.a[6], Rw.a[7], Rw.a[8]);  // world z in link coordinates
  if (io.rb_force || (io.push && RI(R, R_LINK) == 0)) {  // applied world wrenches at the bodies' COMs (tensors.rst.txt:322-335)
#pragma unroll 1
    for (int j = 0; j < RI(R, R_NBODY); ++j) {
      int b = RI(R, R_BODY0 + j);
      V3 F = v3(0, 0, 0), T = v3(0, 0, 0);
      if (io.push && b == 0) F = ld3(X + X_PUSH);
      if (io.rb_force) {
        F = F + ld3_f(io.rb_force + 3 * b);
        T = ld3_f(io.rb_torque + 3 * b);
      }
      real sc = X[X_MASS + b];
      real mb = sc * HF(body_inertia, b * 10);
      real inv = 1 / (mb > (real)1e-30 ? mb : (real)1e-30);
      V3 com = mul(Rw, v3(sc * HF(body_inertia, b * 10 + 1) * inv, sc * HF(body_inertia, b * 10 + 2) * inv,
                          sc * HF(body_inertia, b * 10 + 3) * inv));
      fext.w = fext.w + cross(com, F) + T;
      fext.v = fext.v + F;
    }
  }
  if constexpr (Ground::kField) {
    // Cull: a sphere of radius r <= reach touches where (h - z_c) n_z + r > 0, i.e. z_c < h + r / n_z, and its centre is
    // at most reach - r below the link origin; a cylinder's rim point at most reach below it. So nothing of this link
    // can touch unless pw.z < zmax + reach * cull.
    if (pw.z - gnd.zmax < R[R_REACH] * gnd.cull) {
      const real mu = X[X_MU];
      real h;
      V3 n;
#pragma unroll 1
      for (int k = RI(R, R_PT0); k < RI(R, R_PT1); ++k) {
        const V3 xw = mul(Rw, ld3_f(m.pt_pos + 3 * k));
        const real rad = m.pt_radius[k];
        const V3 c = pw + xw;
        if (!field_query(gnd, c.x, c.y, h, n)) continue;
        penalty_point_n(p, mu, v, xw - rad * n, n, (h - c.z) * n.z + rad, io.contact + 3 * m.pt_body[k], io.live, fext);
      }
#pragma unroll 1
      for (int k = RI(R, R_CYL0); k < RI(R, R_CYL1); ++k) {  // the rim point lowest in WORLD z, as for the plane
        V3 c = ld3_f(m.cyl_center + 3 * k), a = ld3_f(m.cyl_axis + 3 * k);
        real rad = m.cyl_size[2 * k], hh = m.cyl_size[2 * k + 1];
        real az = dot(nrm, a);
        real s = az >= 0 ? (real)-1 : (real)1;
        V3 d = neg(nrm - az * a);
        real dn = sqrt(dot(d, d));
        V3 rim = c + (s * hh) * a;
        if (dn > (real)1e-6) rim = rim + (rad / dn) * d;
        const V3 xw = mul(Rw, rim), q = pw + xw;
        if (!field_query(gnd, q.x, q.y, h, n)) continue;
        penalty_point_n(p, mu, v, xw, n, (h - q.z) * n.z, io.contact + 3 * m.cyl_body[k], io.live, fext);
      }
    }
    return fext;
  }
  if (pw.z < R[R_REACH]) {  // nothing of this link can reach z = 0 otherwise
    const real mu = X[X_MU];
#pragma unroll 1
    for (int k = RI(R, R_PT0); k < RI(R, R_PT1); ++k) {
      V3 x = ld3_f(m.pt_pos + 3 * k);
      real rad = m.pt_radius[k];
      real z = pw.z + dot(nrm, x);
      penalty_point(p, mu, v, mul(Rw, x) - v3(0, 0, rad), rad - z, io.contact + 3 * m.pt_body[k], io.live, fext);
    }
#pragma unroll 1
    for (int k = RI(R, R_CYL0); k < RI(R, R_CYL1); ++k) {
      V3 c = ld3_f(m.cyl_center + 3 * k), a = ld3_f(m.cyl_axis + 3 * k);
      real rad = m.cyl_size[2 * k], hh = m.cyl_size[2 * k + 1];
      real az = dot(nrm, a);
      real s = az >= 0 ? (real)-1 : (real)1;
      V3 d = neg(nrm - az * a);
      real dn = sqrt(dot(d, d));
      V3 rim = c + (s * hh) * a;
      if (dn > (real)1e-6) rim = rim + (rad / dn) * d;
      real z = pw.z + dot(nrm, rim);
      penalty_point(p, mu, v, mul(Rw, rim), -z, io.contact + 3 * m.cyl_body[k], io.live, fext);
    }
  }
  return fext;
}

// Inputs of one env -> its scratch block: thread `tid` of `nthreads` cooperating threads (P0).
// (The CUDA kernels do the same with CTA-wide coalesced slab copies, physics_kernels.cu.)
HD void env_stage_inputs(const EnvIO& io, real* sm, const float* hot, const DevModel& m, const SimParams& p, int tid, int nthreads) {
  real* X = sm + m.nl * LS;
  for (int b = tid; b < m.nb; b += nthreads) X[X_MASS + b] = io.mass_scale[b];
  for (int k = tid; k < 13; k += nthreads) X[X_ROOT + k] = io.root[k];
  for (int k = tid; k < 3; k += nthreads) X[X_PUSH + k] = io.push ? io.push[k] : 0.f;
  if (tid == 0) X[X_MU] = io.friction ? io.friction[0] : p.mu;
  if (io.live)
    for (int k = tid; k < 3 * m.nb; k += nthreads) io.contact[k] = 0.f;  // net contact force of THIS sub-step only
  for (int i = 1 + tid; i < m.nl; i += nthreads) {
    int d = HI(dof, i);
    real* L = BLK(i);
    L[LS_Q] = io.dof_state[2 * d];
    L[LS_SC + 0] = io.dof_state[2 * d + 1];
    L[LS_SC + 1] = io.tau[d];
    L[LS_SC + 2] = io.damping[d];
    L[LS_SC + 3] = io.armature[d];
  }
}

// Results of one env: scratch -> global (after the sub-step, all roles done).
HD void env_store_outputs(const EnvIO& io, const real* sm, const float* hot, const DevModel& m, int tid, int nthreads) {
  if (!io.live) return;
  const real* X = sm + m.nl * LS;
  for (int k = tid; k < 13; k += nthreads) io.root[k] = (float)X[X_ROOT + k];
  for (int i = 1 + tid; i < m.nl; i += nthreads) {
    int d = HI(dof, i);
    io.dof_state[2 * d] = (float)BLK(i)[LS_Q];
    io.dof_state[2 * d + 1] = (float)BLK(i)[LS_SC];
  }
}

// One sub-step for role `role` of one env. `flags`: the CTA-wide stage flags; `epoch`: sub-steps done so far in this
// launch (the flags are monotonic). The env's inputs must have been staged (env_stage_inputs) and made visible;
// with `io_async` the per-sub-step inputs are staged concurrently by another warp, which publishes F_IO_PRE (push,
// zeroed contact forces: needed by the force loop), F_IO_TAU (torque, damping, armature: needed by pass 2) and
// F_IO_DONE (it has finished reading the joint angles, which the last pass overwrites).
// `gnd`: the ground (PlaneGround or FieldGround).
template <class Sync, class Ground = PlaneGround>
HD void env_substep_role(const EnvIO& io, real* sm, int* flags, int epoch, const float* hot, const DevModel& m,
                         const SimParams& p, int role, Sync& sync, bool io_async = false, const Ground& gnd = Ground()) {
  const int nl = m.nl;
  real* X = sm + nl * LS;
  const real dt = p.dt;
  const int base = epoch * ST_STRIDE;
  const int len = m.role_len[role];
  const bool base_role = role == m.base_role;
  int* fl = flags + F_LINK;

  sync.mark(0);
  const int rec0 = m.prog_start[role];
  // ---- pass 1, root -> leaves: world poses, joint axes / offsets in world axes, velocities
  // Along a chain the parent is the link handled just before: its results are carried in registers (`prev`), the
  // scratch block is only read for the first link of a chain. The same holds for the other tree passes.
  int prev = -1;
  SV v_prev = sv_zero();
  M3 Rw_prev;
  V3 pw_prev = v3(0, 0, 0);
  if (base_role) {
    real* L = BLK(0);
    const real* rs = X + X_ROOT;
    V3 pw = ld3(rs);
    M3 R0 = quat_to_mat(rs[3], rs[4], rs[5], rs[6]);
    SV v0{ld3(rs + 10), ld3(rs + 7)};  // root state: world angular velocity, world velocity of the base origin
    st6(L + LS_V, v0);
    st_m3(L + LS_A + A_POSE, R0);
    st3(L + LS_A + A_POSE + 9, pw);
    export_pose(io, 0, R0, pw);
    sync.signal(fl + 0, base + ST_PASS1);
    prev = 0;
    v_prev = v0;
    Rw_prev = R0;
    pw_prev = pw;
  }
  // (a) joint transforms: local to each link, no dependencies
  for (int k = 0; k < len; ++k) {
    const float* R = REC(rec0 + k);
    real* L = BLK(RI(R, R_LINK));
    real sq, cq;
    sincos_r(L[LS_Q], &sq, &cq);
    st_m3(L + LS_E, mul(axis_rot_T(ld3_f(R + R_AXIS), sq, cq), ld_m3_f(R + R_E)));
  }
  sync.mark(16);
  // (b) propagation root -> leaves: world pose, axis and offset in world axes, velocity; this is the only chained
  //     part and what the children in other roles wait for
  for (int k = 0; k < len; ++k) {
    const float* R = REC(rec0 + k);
    const int i = RI(R, R_LINK), par = RI(R, R_PARENT);
    real* L = BLK(i);
    if (par != prev) {
      if (RI(R, R_FLAGS) & RF_PARENT_FOREIGN) sync.wait(fl + par, base + ST_PASS1);
      const real* Lp = BLK(par);
      v_prev = ld6(Lp + LS_V);
      Rw_prev = ld_m3(Lp + LS_A + A_POSE);
      pw_prev = ld3(Lp + LS_A + A_POSE + 9);
    }
    M3 E = ld_m3(L + LS_E);
    if (k == 0 || par != prev) st3(L + LS_WP, v_prev.w);  // (pass 3 starts its chains where this pass does, and at k = 0)
    const V3 rw = mul(Rw_prev, ld3_f(R + R_R));  // offset of this link's origin from its parent's, world axes
    Rw_prev = mulABt(Rw_prev, E);
    const V3 sw = mul(Rw_prev, ld3_f(R + R_AXIS));  // joint axis, world axes
    pw_prev = pw_prev + rw;
    v_prev = SV{v_prev.w + L[LS_SC] * sw, v_prev.v + cross(v_prev.w, rw)};
    prev = i;
    st3(L + LS_S, sw);
    st3(L + LS_R, rw);
    st6(L + LS_V, v_prev);
    st_m3(L + LS_A + A_POSE, Rw_prev);
    st3(L + LS_A + A_POSE + 9, pw_prev);
    export_pose(io, i, Rw_prev, pw_prev);
    // published only where another role reads it: by foreign children (pose, velocity), or by the foreign parent,
    // which must not overwrite its pose before this link has used it
    if (RI(R, R_FLAGS) & (RF_PUBLISH | RF_PARENT_FOREIGN)) sync.signal(fl + i, base + ST_PASS1);
  }
  sync.mark(17);
  sync.mark(1);
  // Pass 2 overwrites A (pose) of a link with its contribution to the parent: every child of this role's links that
  // lives in another role must have read its parent's pose first.
  for (int k = 0; k < m.n_xchild[role]; ++k) sync.wait(fl + m.xchild[role][k], base + ST_PASS1);
  if (io_async) {
    sync.wait_io(flags + F_IO_PRE, epoch + 1);
    sync.wait_io(flags + F_IO_TAU, epoch + 1);
  }
  sync.mark(2);
  // ---- pass 2, leaves -> root: articulated inertias and bias forces; the base role ends with the base itself
  //      (k = -1, record 0): inverse articulated inertia, base acceleration, predicted base velocity
  prev = -1;
  ABI cia_prev;
  SV cpa_prev = sv_zero();
  for (int k = len - 1; k >= (base_role ? -1 : 0); --k) {
    const float* R = k < 0 ? REC(0) : REC(rec0 + k);
    const int i = RI(R, R_LINK);
    real* L = BLK(i);
    real* A = L + LS_A;
    // rigid inertia (rotated to world axes), velocity-product force and external wrench of the link itself (its world
    // pose is still in A: read it before the block is overwritten with the contribution to the parent)
    const SV v = ld6(L + LS_V);
    ABI IA;
    SV pA;
    {
      M3 Rw = ld_m3(A + A_POSE);
      V3 pw = ld3(A + A_POSE + 9);
      const int f = RI(R, R_FOOT);
      if (f >= 0) {
        st_m3(X + X_FOOTPOSE + 12 * f, Rw);
        st3(X + X_FOOTPOSE + 12 * f + 9, pw);
      }
      IA = link_inertia(X, hot, m, R, Rw);
      const V3 h = v3(IA.H.a[7], IA.H.a[2], IA.H.a[3]);  // m c, world axes
      pA = SV{cross(v.w, mul(IA.I, v.w)), cross(v.w, cross(v.w, h))} - link_ext_wrench(io, X, hot, m, p, R, Rw, pw, v, gnd);
    }
    for (int j = 0; j < RI(R, R_NCHILD); ++j) {
      const int cf = RI(R, R_CHILD0 + j), c = cf & ~REC_FOREIGN;
      if (c == prev) {  // the child handled just before: its contribution is still in registers
        IA = IA + cia_prev;
        pA = pA + cpa_prev;
      } else {
        if (cf & REC_FOREIGN) sync.wait(fl + c, base + ST_PASS2);
        const real* Ac = BLK(c) + LS_A;
        IA = IA + ld_abi(Ac + A_CIA);
        pA = pA + ld6(Ac + A_CPA);
      }
    }
    if (k >= 0) {
      const V3 sw = ld3(L + LS_S), rw = ld3(L + LS_R);
      real qd = L[LS_SC], tq = L[LS_SC + 1], damp = L[LS_SC + 2], arm = L[LS_SC + 3];
      if (p.clamp_effort) {  // optional clamp of the actuation to the MJCF ctrlrange (SURVEY D2)
        real lim = R[R_EFF];
        tq = tq > lim ? lim : (tq < -lim ? -lim : tq);
      }
      const real stiff = R[R_STIFF];  // joint spring about q = 0, implicit like the damping
      SV U{mul(IA.I, sw), mulT(IA.H, sw)};
      real D = dot(sw, U.w) + arm + dt * (damp + dt * stiff);
      real Dinv = 1 / D;
      real u = tq - damp * qd - stiff * (L[LS_Q] + dt * qd) - dot(sw, pA.w);
      // classical velocity-product acceleration of the joint: [w_p x s qd; w_p x (w_p x r)], w_p = w - s qd
      const V3 wp = v.w - qd * sw;
      SV c{cross(wp, qd * sw), cross(wp, cross(wp, rw))};
      ABI Ia = rank1_sub(IA, U, Dinv);
      SV pa = pA + mul(Ia, c) + (Dinv * u) * U;
      cia_prev = abi_shift_to_parent(rw, Ia);
      cpa_prev = shift_force_T(rw, pa);
      prev = i;
      st_abi(A + A_CIA, cia_prev);
      st6(A + A_CPA, cpa_prev);
      st6(L + LS_U, U);
      L[LS_SC + 1] = u;
      L[LS_SC + 2] = Dinv;
      L[LS_SC + 3] = 0;
      if (RI(R, R_FLAGS) & RF_PARENT_FOREIGN) sync.signal(fl + i, base + ST_PASS2);
      continue;
    }
    sync.mark(3);
    ABI Om0 = abi_inverse_spd(IA);
    SV a0 = (real)-1 * mul(Om0, pA);  // [angular acceleration; acceleration of the origin relative to the gravity field]
    st6(A + A_ACC, a0);
    st_abi(A + A_OM0, Om0);
    // Predicted base velocity as the contact stage sees it. The model (oracle/physics_oracle.py) advances the base
    // twist by its BODY-frame components, i.e. it holds the body frame fixed over the step: in world axes that is the
    // classical update minus dt w x u; the term is given back when the base is integrated.
    const V3 rot = dt * cross(v.w, v.v);
    SV vs{v.w + dt * a0.w, v.v + dt * (a0.v + v3(p.g[0], p.g[1], p.g[2])) - rot};
    st6(L + LS_U, vs);
    st3(L + LS_SC, rot);
    sync.signal(fl + 0, base + ST_PASS2);
    // inverse inertia at the feet's common ancestor: Om_j = X Om_parent X^T + S D^-1 S^T down the shared links
    ABI Oml = Om0;
#pragma unroll 1
    for (int k2 = 0; k2 < m.shared_len; ++k2) {
      const float* Rs = REC(m.shared_rec[k2]);
      const real* Ls = BLK(RI(Rs, R_LINK));
      const V3 ss = ld3(Ls + LS_S), rs = ld3(Ls + LS_R);
      real Dinv = Ls[LS_SC + 2];
      SV w = Dinv * shift_force_T(rs, ld6(Ls + LS_U));
      SV y = mul(Oml, w);
      Oml = inv_joint_update(inv_shift_to_child(rs, Oml), ss, shift_motion(rs, y), dot(w, y) + Dinv);
    }
    st_abi(X + X_OML, Oml);
    sync.signal(flags + F_OML, epoch + 1);
  }
  if (!base_role) sync.mark(3);
  sync.mark(4);
  // ---- feet, part 1 (needs pass 2 of the own leg chain only): up the chain, G = map foot force -> force on the
  //      current link; Om = sum_j g_j g_j^T / D_j with g_j = S_j^T G_j (kept per chain link for the impulse pass)
  int foot = -1;
  for (int f = 0; f < m.num_feet; ++f)
    if (m.foot_role[f] == role) foot = f;
  SV G[6];              // columns: force arriving at the base per unit foot force
  ABI Om;               // inverse inertia seen at the foot link
  if (foot >= 0) {
#pragma unroll
    for (int c = 0; c < 6; ++c) G[c] = sv_zero();
    G[0].w.x = 1; G[1].w.y = 1; G[2].w.z = 1; G[3].v.x = 1; G[4].v.y = 1; G[5].v.z = 1;
    Om.I = S3{0, 0, 0, 0, 0, 0};
    Om.M = S3{0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int c = 0; c < 9; ++c) Om.H.a[c] = 0;
    for (int k = m.chain_len[foot] - 1; k >= 0; --k) {
      const float* R = REC(m.chain_rec[foot][k]);
      real* L = BLK(RI(R, R_LINK));
      const V3 sw = ld3(L + LS_S), rw = ld3(L + LS_R);
      real Dinv = L[LS_SC + 2];
      SV U = ld6(L + LS_U);
      real gj[6];
#pragma unroll
      for (int c = 0; c < 6; ++c) gj[c] = dot(sw, G[c].w);
#pragma unroll
      for (int c = 0; c < 6; ++c) (k == 0 ? X + X_G0 + foot * 6 : L + LS_A + A_G)[c] = gj[c];
      Om.I.xx += Dinv * gj[0] * gj[0]; Om.I.yy += Dinv * gj[1] * gj[1]; Om.I.zz += Dinv * gj[2] * gj[2];
      Om.I.xy += Dinv * gj[0] * gj[1]; Om.I.xz += Dinv * gj[0] * gj[2]; Om.I.yz += Dinv * gj[1] * gj[2];
      Om.M.xx += Dinv * gj[3] * gj[3]; Om.M.yy += Dinv * gj[4] * gj[4]; Om.M.zz += Dinv * gj[5] * gj[5];
      Om.M.xy += Dinv * gj[3] * gj[4]; Om.M.xz += Dinv * gj[3] * gj[5]; Om.M.yz += Dinv * gj[4] * gj[5];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) Om.H.a[3 * a + b] += Dinv * gj[a] * gj[3 + b];
#pragma unroll
      for (int c = 0; c < 6; ++c) G[c] = shift_force_T(rw, G[c] - (Dinv * gj[c]) * U);
    }
  }
  // active sole points of this foot (needs the foot pose of pass 1 only): candidates below the contact offset, at
  // most MAX_ACTIVE_PTS, with their offsets from the foot origin and the velocity bias of the non-penetration row;
  // kept in the env's scratch (X_PTS) so that the per-point loops below stay rolled (small instruction footprint)
  M3 Rwf;
  // contact location of candidate k of foot g relative to the foot origin (world axes): the sphere's lowest point
  auto sole_point = [&](int g, int k) {
    return mul(Rwf, v3(m.foot_pt_pos[g][k][0], m.foot_pt_pos[g][k][1], m.foot_pt_pos[g][k][2])) - v3(0, 0, m.foot_pt_radius[g][k]);
  };
  int nact = 0;
  const real inv_dt = 1 / dt;
  real* const pts = X + X_PTS + (foot >= 0 ? foot : 0) * MAX_ACTIVE_PTS * PT_WORDS;
  if constexpr (Ground::kField) {
    // (heightfield: selected after pass 3, field_select)
  } else if (foot >= 0) {
    const int g = foot;
    Rwf = ld_m3(X + X_FOOTPOSE + 12 * g);
    const real pz = X[X_FOOTPOSE + 12 * g + 11];
    const V3 nrm = v3(Rwf.a[6], Rwf.a[7], Rwf.a[8]);
#pragma unroll 1
    for (int k = 0; k < m.foot_npts[g]; ++k) {
      V3 x = v3(m.foot_pt_pos[g][k][0], m.foot_pt_pos[g][k][1], m.foot_pt_pos[g][k][2]);
      real rad = m.foot_pt_radius[g][k];
      real phi = pz + dot(nrm, x) - rad;
      if (phi < p.contact_offset && nact < MAX_ACTIVE_PTS) {
        real* pt = pts + nact * PT_WORDS;
        reinterpret_cast<int*>(pt)[0] = k;
        pt[1] = phi >= 0 ? -phi * inv_dt : fmin_r(-p.erp * phi * inv_dt, p.max_depen_vel);
        pt[2] = pt[3] = pt[4] = 0;
        ++nact;
      }
    }
  }
  sync.mark(5);
  // ---- pass 3, root -> leaves: joint accelerations, predicted joint velocities
  prev = -1;
  SV a_prev = sv_zero();
  V3 w_prev = v3(0, 0, 0);  // angular velocity of the parent (start-of-step velocities: for the velocity-product term)
  for (int k = 0; k < len; ++k) {
    const float* R = REC(rec0 + k);
    const int i = RI(R, R_LINK), par = RI(R, R_PARENT), flg = RI(R, R_FLAGS);
    if (flg & RF_PARENT_BASE) {
      if (!base_role) sync.wait(fl + 0, base + ST_PASS2);
    } else if (flg & RF_PARENT_FOREIGN) {
      sync.wait(fl + par, base + ST_PASS3);
    }
    real* L = BLK(i);
    if (par != prev) {
      a_prev = ld6(BLK(par) + LS_A + A_ACC);
      w_prev = ld3(L + LS_WP);
    }
    const V3 sw = ld3(L + LS_S), rw = ld3(L + LS_R);
    real qd = L[LS_SC];
    SV a = shift_motion(rw, a_prev) + SV{cross(w_prev, qd * sw), cross(w_prev, cross(w_prev, rw))};
    real qdd = L[LS_SC + 2] * (L[LS_SC + 1] - dot(ld6(L + LS_U), a));
    a.w = a.w + qdd * sw;
    a_prev = a;
    w_prev = w_prev + qd * sw;
    prev = i;
    st6(L + LS_A + A_ACC, a);
    L[LS_SC] = qd + dt * qdd;
    if (flg & RF_PUBLISH) sync.signal(fl + i, base + ST_PASS3);
  }
  sync.mark(6);
  // ---- feet, part 2: predicted foot velocity, Om += G^T Om0 G, active sole points and their rows, the sweeps
  if (foot >= 0) {
    const int g = foot;
    const int clen = m.chain_len[g];
    if constexpr (Ground::kField) nact = field_select(gnd, m, p, sm, X, g, inv_dt, Rwf);
    SV Y[6];              // Om_lca G
    SV V = ld6(BLK(0) + LS_U);  // base role published v0* with ST_PASS2 (waited for in pass 3)
    SV P = sv_zero();     // accumulated contact impulse on the foot (world axes, about the foot origin)
    if (m.shared_len > 0) {  // predicted velocity of the common ancestor (needs pass 3 of the shared links)
      sync.wait(fl + m.lca, base + ST_PASS3);
#pragma unroll 1
      for (int k = 0; k < m.shared_len; ++k) {
        const real* Ls = BLK(RI(REC(m.shared_rec[k]), R_LINK));
        V = shift_motion(ld3(Ls + LS_R), V);
        V.w = V.w + Ls[LS_SC] * ld3(Ls + LS_S);
      }
    }
    for (int k = 0; k < clen; ++k) {
      const real* L = BLK(RI(REC(m.chain_rec[g][k]), R_LINK));
      V = shift_motion(ld3(L + LS_R), V);
      V.w = V.w + L[LS_SC] * ld3(L + LS_S);
    }
    {
      sync.wait(flags + F_OML, epoch + 1);
      ABI Om0 = ld_abi(X + X_OML);  // inverse inertia at the common ancestor (= the base's for TOCABI)
#pragma unroll
      for (int c = 0; c < 6; ++c) Y[c] = mul(Om0, G[c]);
      real w[6][6];
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = a; b < 6; ++b) w[a][b] = dot(G[a], Y[b]);
      Om.I.xx += w[0][0]; Om.I.yy += w[1][1]; Om.I.zz += w[2][2]; Om.I.xy += w[0][1]; Om.I.xz += w[0][2]; Om.I.yz += w[1][2];
      Om.M.xx += w[3][3]; Om.M.yy += w[4][4]; Om.M.zz += w[5][5]; Om.M.xy += w[3][4]; Om.M.xz += w[3][5]; Om.M.yz += w[4][5];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) Om.H.a[3 * a + b] += w[a][3 + b];
    }
    // rows of the active points: response cv = Om J and 1 / (J . cv) per direction (world z, x, y), parked in the
    // blocks of the first chain links (ROWS_PER_LINK per link)
    // (heightfield: rows n, t1, t2 of the point's ground normal)
    if constexpr (Ground::kField) {
#pragma unroll 1
      for (int a = 0; a < nact; ++a) {
        V3 xa, dirs[3];
        field_sole_point(m, sm, X, Rwf, g, a, xa, dirs);
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          SV J{cross(xa, dirs[d]), dirs[d]};
          SV cv = mul(Om, J);
          const int row = a * 3 + d;
          real* rw = BLK(m.chain[g][row / ROWS_PER_LINK]) + LS_A + A_ROWS + (row % ROWS_PER_LINK) * 7;
          st6(rw, cv);
          rw[6] = 1 / dot(J, cv);
        }
      }
    } else {
#pragma unroll 1
    for (int a = 0; a < nact; ++a) {
      const V3 xa = sole_point(g, reinterpret_cast<const int*>(pts + a * PT_WORDS)[0]);
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const V3 dir = d == 0 ? v3(0, 0, 1) : (d == 1 ? v3(1, 0, 0) : v3(0, 1, 0));
        SV J{cross(xa, dir), dir};
        SV cv = mul(Om, J);
        const int row = a * 3 + d;
        real* rw = BLK(m.chain[g][row / ROWS_PER_LINK]) + LS_A + A_ROWS + (row % ROWS_PER_LINK) * 7;
        st6(rw, cv);
        rw[6] = 1 / dot(J, cv);
      }
    }
    }
    sync.mark(7);
    // fixed number of sweeps; Gauss-Seidel inside a foot, Jacobi between the feet (coupled through the base)
    const real mu = X[X_MU];
    for (int s = 0; s < p.sweeps; ++s) {
      SV dP = sv_zero();
      if constexpr (Ground::kField) {
#pragma unroll 1
        for (int a = 0; a < nact; ++a) {
          real* pt = pts + a * PT_WORDS;
          V3 xa, dirs[3];
          field_sole_point(m, sm, X, Rwf, g, a, xa, dirs);
          const real bias = pt[1];
          real lam[3] = {pt[2], pt[3], pt[4]};
#pragma unroll
          for (int d = 0; d < 3; ++d) {
            SV J{cross(xa, dirs[d]), dirs[d]};
            const int row = a * 3 + d;
            const real* rw = BLK(m.chain[g][row / ROWS_PER_LINK]) + LS_A + A_ROWS + (row % ROWS_PER_LINK) * 7;
            real vrel = dot(J, V);
            real nw;
            if (d == 0) {
              nw = lam[0] + (bias - vrel) * rw[6];
              nw = nw > 0 ? nw : 0;
            } else {
              real lim = mu * lam[0];
              nw = lam[d] - vrel * rw[6];
              nw = nw > lim ? lim : (nw < -lim ? -lim : nw);
            }
            real delta = nw - lam[d];
            lam[d] = nw;
            V = V + delta * ld6(rw);
            dP = dP + delta * J;
          }
          pt[2] = lam[0];
          pt[3] = lam[1];
          pt[4] = lam[2];
        }
      } else {
#pragma unroll 1
      for (int a = 0; a < nact; ++a) {
        real* pt = pts + a * PT_WORDS;
        const V3 xa = sole_point(g, reinterpret_cast<const int*>(pt)[0]);
        const real bias = pt[1];
        real lam[3] = {pt[2], pt[3], pt[4]};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const V3 dir = d == 0 ? v3(0, 0, 1) : (d == 1 ? v3(1, 0, 0) : v3(0, 1, 0));
          SV J{cross(xa, dir), dir};
          const int row = a * 3 + d;
          const real* rw = BLK(m.chain[g][row / ROWS_PER_LINK]) + LS_A + A_ROWS + (row % ROWS_PER_LINK) * 7;
          real vrel = dot(J, V);
          real nw;
          if (d == 0) {
            nw = lam[0] + (bias - vrel) * rw[6];
            nw = nw > 0 ? nw : 0;
          } else {
            real lim = mu * lam[0];
            nw = lam[d] - vrel * rw[6];
            nw = nw > lim ? lim : (nw < -lim ? -lim : nw);
          }
          real delta = nw - lam[d];
          lam[d] = nw;
          V = V + delta * ld6(rw);
          dP = dP + delta * J;
        }
        pt[2] = lam[0];
        pt[3] = lam[1];
        pt[4] = lam[2];
      }
      }
      P = P + dP;
      if (m.num_feet == 2) {
        // base velocity change caused by this sweep's impulses: Om0 G dP = sum_c dP_c Y_c (double-buffered by sweep parity)
        const int seq = epoch * 64 + s + 1;
        st6(X + X_Z + ((s & 1) * MAX_FEET + g) * 6,
            dP.w.x * Y[0] + dP.w.y * Y[1] + dP.w.z * Y[2] + dP.v.x * Y[3] + dP.v.y * Y[4] + dP.v.z * Y[5]);
        sync.signal(flags + F_Z + g, seq);
        sync.wait(flags + F_Z + (1 - g), seq);
        SV z = ld6(X + X_Z + ((s & 1) * MAX_FEET + (1 - g)) * 6);  // response of this foot: G^T z
        V = V + SV{v3(dot(G[0], z), dot(G[1], z), dot(G[2], z)), v3(dot(G[3], z), dot(G[4], z), dot(G[5], z))};
      }
    }
    sync.mark(8);
    // contact impulse -> joint space: S^T dp on the leg chain, impulse arriving at the base
    for (int k = 0; k < clen; ++k) {
      real* L = BLK(m.chain[g][k]);
      const real* gj = k == 0 ? X + X_G0 + g * 6 : L + LS_A + A_G;
      L[LS_SC + 3] = -(gj[0] * P.w.x + gj[1] * P.w.y + gj[2] * P.w.z + gj[3] * P.v.x + gj[4] * P.v.y + gj[5] * P.v.z);
    }
    st6(X + X_PD + 6 * g, (real)-1 * (P.w.x * G[0] + P.w.y * G[1] + P.w.z * G[2] + P.v.x * G[3] + P.v.y * G[4] + P.v.z * G[5]));
    sync.signal(flags + F_PD + g, epoch + 1);
    if (io.live) {
#pragma unroll 1
      for (int a = 0; a < nact; ++a) {  // world force over this sub-step: rows (n, t1, t2) = world (z, x, y)
        const real* pt = pts + a * PT_WORDS;
        float* cf = io.contact + 3 * m.foot_pt_body[g][reinterpret_cast<const int*>(pt)[0]];
        if constexpr (Ground::kField) {  // (lam_n n + lam_1 t1 + lam_2 t2) / dt
          V3 xa, dirs[3];
          field_sole_point(m, sm, X, Rwf, g, a, xa, dirs);
          const V3 F = (pt[2] * inv_dt) * dirs[0] + (pt[3] * inv_dt) * dirs[1] + (pt[4] * inv_dt) * dirs[2];
          cf[0] += (float)F.x;
          cf[1] += (float)F.y;
          cf[2] += (float)F.z;
          continue;
        }
        cf[0] += (float)(pt[3] * inv_dt);
        cf[1] += (float)(pt[4] * inv_dt);
        cf[2] += (float)(pt[2] * inv_dt);
      }
    }
  }
  sync.mark(9);
  // ---- base response to the contact impulses (base role)
  if (base_role) {
    SV pd = sv_zero();
    for (int f = 0; f < m.num_feet; ++f) {
      sync.wait(flags + F_PD + f, epoch + 1);
      pd = pd + ld6(X + X_PD + 6 * f);  // impulse arriving at the common ancestor
    }
#pragma unroll 1
    for (int k = m.shared_len - 1; k >= 0; --k) {  // ... and from there up the shared links to the base
      real* Ls = BLK(RI(REC(m.shared_rec[k]), R_LINK));
      real sd = dot(ld3(Ls + LS_S), pd.w);
      Ls[LS_SC + 3] = sd;
      pd = shift_force_T(ld3(Ls + LS_R), pd - (Ls[LS_SC + 2] * sd) * ld6(Ls + LS_U));
    }
    st6(BLK(0) + LS_V, (real)-1 * mul(ld_abi(BLK(0) + LS_A + A_OM0), pd));
    sync.signal(fl + 0, base + ST_DOWN);
  }
  sync.mark(10);
  // ---- down the tree: joint velocity changes, speed cap, integration, limit projection
  if (io_async) sync.wait_io(flags + F_IO_DONE, epoch + 1);
  prev = -1;
  for (int k = 0; k < len; ++k) {
    const float* R = REC(rec0 + k);
    const int i = RI(R, R_LINK), par = RI(R, R_PARENT), flg = RI(R, R_FLAGS);
    if (flg & RF_PARENT_BASE) {
      if (!base_role) sync.wait(fl + 0, base + ST_DOWN);
    } else if (flg & RF_PARENT_FOREIGN) {
      sync.wait(fl + par, base + ST_DOWN);
    }
    real* L = BLK(i);
    if (par != prev) a_prev = ld6(BLK(par) + LS_V);  // (re-used register set: the parent's velocity change)
    const V3 sw = ld3(L + LS_S);
    SV dv = shift_motion(ld3(L + LS_R), a_prev);
    real dqd = -L[LS_SC + 2] * (dot(ld6(L + LS_U), dv) + L[LS_SC + 3]);
    dv.w = dv.w + dqd * sw;
    a_prev = dv;
    prev = i;
    st6(L + LS_V, dv);
    if (flg & RF_PUBLISH) sync.signal(fl + i, base + ST_DOWN);
    // joint velocity cap (dof_prop['velocity'], T:372), explicit Euler on the angle, limit projection
    real vl = R[R_VLIM];
    real qdn = L[LS_SC] + dqd;
    qdn = qdn > vl ? vl : (qdn < -vl ? -vl : qdn);
    real qn = L[LS_Q] + dt * qdn;
    real lo = R[R_LO], up = R[R_UP];
    if (qn > up) {
      qn = up;
      qdn = qdn < 0 ? qdn : 0;
    } else if (qn < lo) {
      qn = lo;
      qdn = qdn > 0 ? qdn : 0;
    }
    L[LS_Q] = qn;      // new joint state; env_store_outputs / the slab copy writes it to dof_state
    L[LS_SC] = qdn;
  }
  sync.mark(11);
  // ---- base integration (base role): the base velocity is already in world axes
  if (base_role) {
    const real* L = BLK(0);
    SV vb = ld6(L + LS_U) + ld6(L + LS_V);
    V3 ww = vb.w, vw = vb.v + ld3(L + LS_SC);
    real wn = sqrt(dot(ww, ww));
    if (wn > p.max_ang_vel) ww = (p.max_ang_vel / wn) * ww;
    {
      real* rs = X + X_ROOT;
      real qx = rs[3], qy = rs[4], qz = rs[5], qw = rs[6];
      real h = (real)0.5 * dt;
      real nx = qx + h * (ww.x * qw + ww.y * qz - ww.z * qy);
      real ny = qy + h * (-ww.x * qz + ww.y * qw + ww.z * qx);
      real nz = qz + h * (ww.x * qy - ww.y * qx + ww.z * qw);
      real nw = qw + h * (-ww.x * qx - ww.y * qy - ww.z * qz);
      real inv = 1 / sqrt(nx * nx + ny * ny + nz * nz + nw * nw);
      rs[0] = rs[0] + dt * vw.x;
      rs[1] = rs[1] + dt * vw.y;
      rs[2] = rs[2] + dt * vw.z;
      rs[3] = nx * inv;
      rs[4] = ny * inv;
      rs[5] = nz * inv;
      rs[6] = nw * inv;
      rs[7] = vw.x; rs[8] = vw.y; rs[9] = vw.z;
      rs[10] = ww.x; rs[11] = ww.y; rs[12] = ww.z;
    }
  }
  sync.mark(12);
}

}  // namespace dyros
