// TEST INFRASTRUCTURE ONLY. CPU build of the triangle-mesh ground's narrow phase: the grid of dyros_sim_set_triangle_mesh
// (isaacgymdyros_b200/csrc/mesh_grid.h) and the kernel's mesh_query (physics_roles.cuh), compiled for the host, so that
// tests can compare both with a brute-force fp64 restatement. Never linked into the product.
#include "hostemu.cu"
#include "mesh_grid.h"

// Builds the grid for query margin `margin`, then queries n spheres (centres c (n, 3), radii r (n)) with the bucket
// height cull at `contact_offset`: s (n), normal (n, 3), hit (n) 0 / 1. info: kept triangles, dropped triangles, grid
// cells, list entries. Returns 0, or 1 with the builder's message in err.
extern "C" int dyros_hostemu_mesh_query(const DyrosTriangleMesh* mesh, float margin, float contact_offset, const float* c,
                                        const float* r, int n, float* s, float* nrm, int* hit, long long* info, char* err,
                                        int errlen) {
  MeshGrid mg;
  const std::string e = build_mesh_grid(mesh, margin, mg);
  if (!e.empty()) {
    snprintf(err, errlen, "%s", e.c_str());
    return 1;
  }
  MeshGround g = mg.g;
  g.tri = mg.tri.data();
  g.cell = mg.cell.data();
  g.list = mg.list.data();
  info[0] = mg.kept;
  info[1] = mg.dropped;
  info[2] = (long long)mg.cell.size();
  info[3] = (long long)mg.list.size();
  for (int k = 0; k < n; ++k) {
    real sk = 0;
    V3 nk = v3(0, 0, 0);
    hit[k] = mesh_query(g, v3(c[3 * k], c[3 * k + 1], c[3 * k + 2]), r[k], contact_offset, sk, nk) ? 1 : 0;
    s[k] = sk;
    nrm[3 * k] = nk.x;
    nrm[3 * k + 1] = nk.y;
    nrm[3 * k + 2] = nk.z;
  }
  return 0;
}

// dyros_hostemu_simulate (hostemu.cu) on a triangle mesh: the kernel's role program with Ground = MeshGround, one
// thread per role, on the grid dyros_sim_set_triangle_mesh builds (margin from the model as there). cull = 0 switches the
// bucket and per-link height culls off.
extern "C" int dyros_hostemu_simulate_mesh(const DyrosSimDesc* d, const DyrosModelDesc* md, const DyrosTriangleMesh* mesh,
                                           float* root, float* dof_state, const float* tau, const float* damping,
                                           const float* armature, const float* mass_scale, float* contact,
                                           const float* push, const float* friction, int cull, char* err, int errlen) {
  Blob bl;
  DevModel m;
  ModelOffsets off;
  std::string e = build_model_tables(md, bl, m, off);
  if (!e.empty()) {
    snprintf(err, errlen, "%s", e.c_str());
    return 1;
  }
  resolve_model(m, off, bl.host.data());
  SimParams p;
  fill_sim_params(d, p);
  float max_radius = 0;
  for (int i = 0; i < md->num_points; ++i) max_radius = std::max(max_radius, (float)md->pt_radius[i]);
  MeshGrid mg;
  e = build_mesh_grid(mesh, (double)p.contact_offset + max_radius + kMeshDepthAllowance, mg);
  if (!e.empty()) {
    snprintf(err, errlen, "%s", e.c_str());
    return 1;
  }
  MeshGround g = mg.g;
  g.tri = mg.tri.data();
  g.cell = mg.cell.data();
  g.list = mg.list.data();
  if (!cull) {  // every height bound +inf: each point scans its bucket, each link its candidates
    const float inf = INFINITY;
    for (int4& c : mg.cell) {
      memcpy(&c.z, &inf, 4);
      memcpy(&c.w, &inf, 4);
    }
    g.zmax = g.ztop = INFINITY;
  }
  p.mu = mesh->dynamic_friction;
  const float* hot = reinterpret_cast<const float*>(bl.host.data());
  std::vector<real> scratch(env_scratch_floats(m.nl, m.nb));
  for (int env = 0; env < p.N; ++env) {
    EnvIO io;
    io.root = root + (size_t)env * 13;
    io.dof_state = dof_state + (size_t)env * m.nd * 2;
    io.tau = tau + (size_t)env * m.nd;
    io.damping = damping + (size_t)env * m.nd;
    io.armature = armature + (size_t)env * m.nd;
    io.mass_scale = mass_scale + (size_t)env * m.nb;
    io.contact = contact + (size_t)env * m.nb * 3;
    io.push = push ? push + (size_t)env * 3 : nullptr;
    io.rb_force = nullptr;
    io.rb_torque = nullptr;
    io.friction = friction ? friction + env : nullptr;
    io.link_pose = nullptr;
    io.live = true;
    std::vector<int> flags(F_COUNT, 0);
    std::barrier<> bar(DYROS_LANES);
    std::vector<std::thread> th;
    for (int role = 0; role < DYROS_LANES; ++role)
      th.emplace_back([&, role]() {
        EnvIO mine = io;
        HostRoleSync sync{role};
        for (int s = 0; s < p.substeps; ++s) {
          env_stage_inputs(mine, scratch.data(), hot, m, p, role, DYROS_LANES);
          bar.arrive_and_wait();
          env_substep_role(mine, scratch.data(), flags.data(), s, hot, m, p, role, sync, false, g);
          bar.arrive_and_wait();
          env_store_outputs(mine, scratch.data(), hot, m, role, DYROS_LANES);
          bar.arrive_and_wait();
        }
      });
    for (auto& t : th) t.join();
  }
  return 0;
}
