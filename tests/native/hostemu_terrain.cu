// TEST INFRASTRUCTURE ONLY. CPU emulation of the heightfield instantiation of the physics kernel's role program
// (isaacgymdyros_b200/csrc/physics_roles.cuh with Ground = FieldGround), on the harness of hostemu.cu: one thread per
// role, atomic stage flags. Also exports the kernel's height / normal query itself. Never linked into the product.
#include "hostemu.cu"

static FieldGround make_field(const int16_t* samples, int nr, int nc, const float* scale, const float* origin) {
  FieldGround g{};
  g.s = samples;
  g.nr = nr;
  g.nc = nc;
  g.dx = scale[0];
  g.dy = scale[1];
  g.dz = scale[2];
  g.ox = origin[0];
  g.oy = origin[1];
  g.oz = origin[2];
  g.zmax = 1e30f;  // the per-link cull is checked on the GPU build; here every link tests its candidates
  g.cull = 1.f;
  return g;
}

// field_query at n points (x, y): h (n), normal (n, 3), inside (n) 0 / 1
extern "C" void dyros_hostemu_field_query(const int16_t* samples, int nr, int nc, const float* scale, const float* origin,
                                          const float* xy, int n, float* h, float* nrm, int* inside) {
  const FieldGround g = make_field(samples, nr, nc, scale, origin);
  for (int k = 0; k < n; ++k) {
    real hk = 0;
    V3 nk = v3(0, 0, 0);
    inside[k] = field_query(g, xy[2 * k], xy[2 * k + 1], hk, nk) ? 1 : 0;
    h[k] = hk;
    nrm[3 * k] = nk.x;
    nrm[3 * k + 1] = nk.y;
    nrm[3 * k + 2] = nk.z;
  }
}

// dyros_hostemu_simulate on a heightfield; `cull` (may be NULL): zmax and 1 / min n_z as dyros_sim_set_heightfield
// derives them, so that the per-link reach cull of the GPU build runs too
extern "C" int dyros_hostemu_simulate_terrain(const DyrosSimDesc* d, const DyrosModelDesc* md, const int16_t* samples, int nr,
                                              int nc, const float* scale, const float* origin, const float* cull, float* root,
                                              float* dof_state, const float* tau, const float* damping, const float* armature,
                                              const float* mass_scale, float* contact, const float* push,
                                              const float* friction, char* err, int errlen) {
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
  FieldGround g = make_field(samples, nr, nc, scale, origin);
  if (cull) {
    g.zmax = cull[0];
    g.cull = cull[1];
  }
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

