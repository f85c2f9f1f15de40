// TEST INFRASTRUCTURE ONLY. CPU emulation of the CUDA physics kernel's role programs: the very same source
// (isaacgymdyros_b200/csrc/physics_roles.cuh) compiled for the host, one thread per role with atomic stage flags
// where the GPU uses release/acquire on shared memory. Lets the CPU test suite compare the kernel's O(n) recursions
// and its dataflow synchronisation with the dense fp64 oracle (oracle/physics_oracle.py) without a GPU.
// Never linked into the product.
#include <barrier>
#include <chrono>
#include <thread>
#include <vector>

#include "host_model.h"
#include "physics_roles.cuh"

namespace dyros {
void set_error(const char*, ...) {}
}  // namespace dyros
using namespace dyros;

// One role held back at one stage marker (sync.mark) of every sub-step: the result must not depend on how far the
// other roles get meanwhile, i.e. on anything but the stage flags.
static int g_hold_role = -1, g_hold_mark = -1, g_hold_us = 0;
extern "C" void dyros_hostemu_hold_role(int role, int mark, int microseconds) {
  g_hold_role = role;
  g_hold_mark = mark;
  g_hold_us = microseconds;
}

struct HostRoleSync {
  int role;
  void mark(int id) const {
    if (role == g_hold_role && id == g_hold_mark) std::this_thread::sleep_for(std::chrono::microseconds(g_hold_us));
  }
  void signal(int* f, int v) const { __atomic_store_n(f, v, __ATOMIC_RELEASE); }
  void wait(const int* f, int v) const {
    while (__atomic_load_n(f, __ATOMIC_ACQUIRE) < v) std::this_thread::yield();
  }
  void wait_io(const int* f, int v) const { wait(f, v); }
};

extern "C" int dyros_hostemu_simulate(const DyrosSimDesc* d, const DyrosModelDesc* md, float* root, float* dof_state,
                                      const float* tau, const float* damping, const float* armature,
                                      const float* mass_scale, float* contact, const float* push, const float* rb_force,
                                      const float* rb_torque, const float* friction, char* err, int errlen) {
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
    io.rb_force = rb_force ? rb_force + (size_t)env * m.nb * 3 : nullptr;
    io.rb_torque = rb_torque ? rb_torque + (size_t)env * m.nb * 3 : nullptr;
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
          env_substep_role(mine, scratch.data(), flags.data(), s, hot, m, p, role, sync);
          bar.arrive_and_wait();
          env_store_outputs(mine, scratch.data(), hot, m, role, DYROS_LANES);
          bar.arrive_and_wait();  // (applied wrenches act over the whole simulate() call: all of its sub-steps)
        }
      });
    for (auto& t : th) t.join();
  }
  return 0;
}

extern "C" int dyros_hostemu_layout(const DyrosModelDesc* md, int* hot_bytes, int* env_scratch_bytes) {
  Blob bl;
  DevModel m;
  ModelOffsets off;
  if (!build_model_tables(md, bl, m, off).empty()) return 1;
  *hot_bytes = m.hot_bytes;
  *env_scratch_bytes = env_scratch_floats(m.nl, m.nb) * (int)sizeof(real);
  return 0;
}

// Dynamic shared memory of a physics CTA holding `epb` envs (mirrors phys_smem_bytes in physics_kernels.cu).
extern "C" long dyros_hostemu_cta_smem_bytes(const DyrosModelDesc* md, int epb) {
  Blob bl;
  DevModel m;
  ModelOffsets off;
  if (!build_model_tables(md, bl, m, off).empty()) return -1;
  return (long)m.hot_bytes + (((F_COUNT + 3) & ~3) + (long)epb * env_scratch_floats(m.nl, m.nb)) * (long)sizeof(float);
}
