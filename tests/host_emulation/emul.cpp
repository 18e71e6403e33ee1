// Host emulation of the warp-per-env engine (earl_benchmark_b200/csrc/mj_engine.cuh compiled with NL = 1).
// TEST INFRASTRUCTURE: lets the CPU suite check the exact kernel source against the fp64 checker without a GPU.
// The product library never links or loads this file.
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../earl_benchmark_b200/csrc/mj_engine.cuh"
#include "../../earl_benchmark_b200/csrc/mj_model_host.hpp"
#include "../../earl_benchmark_b200/csrc/mj_step.cuh"
#include "phases.hpp"

using namespace earl::mj;

struct Emu {
  HostModel hm;
  Work w;
};

extern "C" {

void* emu_create(const void* blob, long long nbytes, const TaskSpec* task, char* err, int errlen) {
  Emu* e = new Emu();
  std::string msg;
  if (!build_model(blob, (size_t)nbytes, *task, &e->hm, &msg)) {
    strncpy(err, msg.c_str(), errlen - 1);
    delete e;
    return nullptr;
  }
  memset(&e->w, 0, sizeof(Work));
  return e;
}
void emu_destroy(void* h) { delete static_cast<Emu*>(h); }

void emu_set_state(void* h, const double* qpos, const double* qvel, const double* warm, const double* mocap_pos,
                   const double* mocap_quat, const double* ctrl) {
  Emu* e = static_cast<Emu*>(h);
  load_state(e->hm.m, e->w, qpos, qvel, warm, mocap_pos, mocap_quat, ctrl);  // also: the cached broad-phase candidates are stale
}
void emu_get_state(void* h, double* qpos, double* qvel, double* warm, double* mocap_pos) {
  Emu* e = static_cast<Emu*>(h);
  const Model& m = e->hm.m;
  for (int k = 0; k < m.nq; ++k) qpos[k] = e->w.qpos[k];
  for (int k = 0; k < m.nv; ++k) { qvel[k] = e->w.qvel[k]; warm[k] = e->w.warm[k]; }
  for (int k = 0; k < 3; ++k) mocap_pos[k] = e->w.mocap_pos[k];
}
void emu_substeps(void* h, int n) {
  Emu* e = static_cast<Emu*>(h);
  for (int k = 0; k < n; ++k) substep<1>(e->hm.m, e->hm.hull_vert.data(), e->w, 0);
}
void emu_env_step(void* h, const float* action, float* obs7) {
  Emu* e = static_cast<Emu*>(h);
  env_step<1>(e->hm.m, e->hm.hull_vert.data(), e->w, action, 0);
  observe(e->hm.m, e->w, obs7);
}
// position-dependent pieces, for unit checks
void emu_forward_parts(void* h, double* M, double* bias, double* xpos) {
  Emu* e = static_cast<Emu*>(h);
  const Model& m = e->hm.m;
  kinematics<1>(m, e->w, 0);
  mass_matrix<1>(m, e->w, 0);
  bias_forces<1>(m, e->w, 0);
  for (int i = 0; i < m.nv; ++i) {
    bias[i] = e->w.bias[i];
    for (int j = 0; j < m.nv; ++j) M[i * m.nv + j] = e->w.M[i][j];
  }
  for (int b = 0; b < m.nbody; ++b)
    for (int k = 0; k < 3; ++k) xpos[3 * b + k] = e->w.xpos[b][k];
}
int emu_info(void* h, int what) {
  Emu* e = static_cast<Emu*>(h);
  switch (what) {
    case 0: return e->w.nefc;
    case 1: return e->w.ncon;
    case 2: return e->w.solver_iter;
    case 3: return e->w.bad;
    case 4: return e->hm.m.npair;
    case 5: return e->w.nhit;
  }
  return -1;
}
}
extern "C" int emu_hits(void* h, int* pairs) {
  Emu* e = static_cast<Emu*>(h);
  for (int k = 0; k < e->w.nhit; ++k) {
    pairs[2 * k] = e->hm.m.pair_g1[e->w.hit_list[k]];
    pairs[2 * k + 1] = e->hm.m.pair_g2[e->w.hit_list[k]];
  }
  return e->w.nhit;
}
#if defined(MJ_DEBUG)
extern "C" void emu_mpr_stats(long* out) { out[0] = earl::mj::g_support_calls; out[1] = earl::mj::g_mpr_calls; out[2] = earl::mj::g_mpr_hits; }
#endif
// direct entry point for the geometry unit tests: the kernel's box-box routine on caller-supplied boxes
extern "C" int emu_box_box(const float* p1, const float* R1, const float* s1, const float* p2, const float* R2, const float* s2,
                           float margin, float* out /* [8][7] */) {
  static NarrowScratch S;
  const int n = box_box(p1, R1, s1, p2, R2, s2, margin, S.rc, &S);
  for (int c = 0; c < n; ++c) {
    for (int k = 0; k < 3; ++k) { out[7 * c + k] = S.rc[c].pos[k]; out[7 * c + 3 + k] = S.rc[c].normal[k]; }
    out[7 * c + 6] = S.rc[c].dist;
  }
  return n;
}
extern "C" int emu_mpr(int t1, const float* size1, const float* p1, const float* R1, int t2, const float* size2, const float* p2,
                       const float* R2, float margin, float* out /* depth, dir[3], pos[3] */) {
  static NarrowScratch S;
  S.o1 = CObj{t1, 0, 0.5f * margin, p1, R1, size1, nullptr};
  S.o2 = CObj{t2, 0, 0.5f * margin, p2, R2, size2, nullptr};
  return mpr_penetration<1>(S.o1, S.o2, out, out + 1, out + 4, &S, 0);
}

// the phases of one substep (tests/host_emulation/phases.hpp) and readers of what they leave behind; the signatures are
// those of the device harness (devemul.cu), where `i` picks one of a batch of states -- here there is one state, i = 0
extern "C" {
void ph_caps(int* out) { read_caps(out); }
void emu_run(void* h, int stage, int nsub) {
  Emu* e = static_cast<Emu*>(h);
  run_stage<1>(e->hm.m, e->hm.hull_vert.data(), e->w, stage, nsub, 0);
}
int ph_state(void* h, int i, double* qpos, double* qvel, double* warm) {
  if (i != 0) return -1;
  read_state(static_cast<Emu*>(h)->hm.m, static_cast<Emu*>(h)->w, qpos, qvel, warm);
  return 0;
}
int ph_info(void* h, int i, int* out) {
  if (i != 0) return -1;
  read_info(static_cast<Emu*>(h)->w, out);
  return 0;
}
int ph_forward(void* h, int i, double* xpos, double* xmat, double* M, double* bias) {
  if (i != 0) return -1;
  read_forward(static_cast<Emu*>(h)->hm.m, static_cast<Emu*>(h)->w, xpos, xmat, M, bias);
  return 0;
}
int ph_hits(void* h, int i, int* pairs) { return i != 0 ? -1 : read_hits(static_cast<Emu*>(h)->hm.m, static_cast<Emu*>(h)->w, pairs); }
int ph_contacts(void* h, int i, double* dist, double* pos, double* frame, int* geoms) {
  return i != 0 ? -1 : read_contacts(static_cast<Emu*>(h)->w, dist, pos, frame, geoms);
}
int ph_rows(void* h, int i, int* type, double* J, double* pos, double* R, double* D, double* aref, int* con, double* mu, double* fri) {
  return i != 0 ? -1 : read_rows(static_cast<Emu*>(h)->hm.m, static_cast<Emu*>(h)->w, type, J, pos, R, D, aref, con, mu, fri);
}
int ph_solve(void* h, int i, double* acc, double* fcon, double* smooth, double* force) {
  if (i != 0) return -1;
  read_solve(static_cast<Emu*>(h)->hm.m, static_cast<Emu*>(h)->w, acc, fcon, smooth, force);
  return 0;
}
// spd_solve<1> (chol_factor + chol_solve) on one caller matrix in the LDM-padded layout A [MAXV][LDM], x [MAXV]
int emu_spd_solve(int n, float* A, float* x) {
  if (n < 1 || n > MAXV) return -1;
  return spd_solve<1>(reinterpret_cast<real(*)[LDM]>(A), n, x, 0);
}
}
