// Device twin of emul.cpp: the engine source (earl_benchmark_b200/csrc/mj_*.cuh) compiled for sm_100a with NL = 32, as
// the product runs it, with entry points that stop after one phase of a substep and hand its workspace back.
// TEST INFRASTRUCTURE: the product library never links or loads this file.
//
// One 32-thread block per state, its `Work` in global memory (B states per launch); the model and the hull vertices in
// global memory, as the kitchen unit keeps them.  MJ_BARRIER_DOMAINS stays undefined: with one warp per block the
// block-wide phase barrier is a __syncthreads over that warp.  Every size is checked on the host before a launch.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../earl_benchmark_b200/csrc/mj_model_host.hpp"
#include "phases.hpp"

using namespace earl::mj;

#define DEV_API extern "C" __attribute__((visibility("default")))

namespace {

constexpr int kMaxItems = 1 << 16;  // unit entry points: items / directions / vertices / cases per call

struct Dev {
  HostModel hm;
  Model* d_model = nullptr;
  real* d_hull = nullptr;
  Work* d_work = nullptr;
  int cap = 0, n = 0;
  std::vector<Work> h_work;
};

int report(cudaError_t e, char* err, int errlen) {
  if (e == cudaSuccess) return 0;
  if (err && errlen > 0) snprintf(err, errlen, "%s", cudaGetErrorString(e));
  return 1;
}
// launch result + completion of the work of this call
int finish(char* err, int errlen) {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  return report(e, err, errlen);
}
int fail(const char* msg, char* err, int errlen) {
  if (err && errlen > 0) snprintf(err, errlen, "%s", msg);
  return 1;
}

__global__ void __launch_bounds__(32) stage_kernel(const Model* __restrict__ gm, const real* __restrict__ hull, Work* works, int stage, int nsub) {
  run_stage<32>(*gm, hull, works[blockIdx.x], stage, nsub, threadIdx.x);
}

__global__ void __launch_bounds__(32) spd_kernel(const int* ns, real (*A)[MAXV][LDM], real (*x)[MAXV], int* ok) {
  const int b = blockIdx.x;
  const int r = spd_solve<32>(A[b], ns[b], x[b], threadIdx.x);
  if (threadIdx.x == 0) ok[b] = r;
}

// the broad phase's lane-strided passes over `nitems` items, each appending the flagged ones (collide())
__global__ void __launch_bounds__(32) append_kernel(Work* works, int which, int nitems, const int* flags) {
  Work& w = works[blockIdx.x];
  const int lane = threadIdx.x;
  const int* f = flags + (size_t)blockIdx.x * nitems;
  for (int p0 = 0; p0 < nitems; p0 += 32) {
    const int p = p0 + lane;
    const int flag = p < nitems ? f[p] : 0;
    if (which == 0) compact_append<32>(w, p, flag, lane);
    else cand_append<32>(w, p, flag, lane);
  }
}

// support point of a mesh geom at the origin in world axes (no margin) in direction dirs[blockIdx.x]
__global__ void __launch_bounds__(32) support_kernel(const real* hull, int nvert, const double* dirs, double* out) {
  const real R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, pos[3] = {0, 0, 0};
  CObj o{GEOM_MESH, nvert, 0.0f, pos, R, pos, hull};
  double res[3];
  support_geom<32>(o, dirs + 3 * blockIdx.x, res, threadIdx.x);
  if (threadIdx.x == 0)
    for (int k = 0; k < 3; ++k) out[3 * blockIdx.x + k] = res[k];
}

template <class T>
int dalloc(T** p, size_t count, char* err, int errlen) {
  return report(cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)), err, errlen);
}
template <class T>
int upload(T* dst, const T* src, size_t count, char* err, int errlen) {
  return report(cudaMemcpy(dst, src, count * sizeof(T), cudaMemcpyHostToDevice), err, errlen);
}
template <class T>
int download(T* dst, const T* src, size_t count, char* err, int errlen) {
  return report(cudaMemcpy(dst, src, count * sizeof(T), cudaMemcpyDeviceToHost), err, errlen);
}

}  // namespace

DEV_API void ph_caps(int* out) { read_caps(out); }

DEV_API void dev_destroy(void* h) {
  Dev* d = static_cast<Dev*>(h);
  if (!d) return;
  cudaFree(d->d_model);
  cudaFree(d->d_hull);
  cudaFree(d->d_work);
  delete d;
}

DEV_API void* dev_create(const void* blob, long long nbytes, const TaskSpec* task, int cap, char* err, int errlen) {
  if (cap < 1 || cap > kMaxItems) { fail("dev_create: batch capacity out of range", err, errlen); return nullptr; }
  Dev* d = new Dev();
  std::string msg;
  if (!build_model(blob, (size_t)nbytes, *task, &d->hm, &msg)) {
    fail(msg.c_str(), err, errlen);
    delete d;
    return nullptr;
  }
  d->cap = cap;
  d->h_work.resize(cap);
  memset(d->h_work.data(), 0, sizeof(Work) * cap);
  const size_t nh = d->hm.hull_vert.size() > 0 ? d->hm.hull_vert.size() : 1;
  if (dalloc(&d->d_model, 1, err, errlen) || dalloc(&d->d_hull, nh, err, errlen) || dalloc(&d->d_work, cap, err, errlen) ||
      upload(d->d_model, &d->hm.m, 1, err, errlen) ||
      (d->hm.hull_vert.size() && upload(d->d_hull, d->hm.hull_vert.data(), d->hm.hull_vert.size(), err, errlen))) {
    dev_destroy(d);
    return nullptr;
  }
  return d;
}

// n states: qpos [n][nq], qvel / warm [n][nv], mocap_pos [n][3], mocap_quat [n][4], ctrl [n][nu]
DEV_API int dev_set_states(void* h, int n, const double* qpos, const double* qvel, const double* warm, const double* mocap_pos,
                           const double* mocap_quat, const double* ctrl, char* err, int errlen) {
  Dev* d = static_cast<Dev*>(h);
  if (n < 1 || n > d->cap) return fail("dev_set_states: state count out of range", err, errlen);
  const Model& m = d->hm.m;
  for (int i = 0; i < n; ++i)
    load_state(m, d->h_work[i], qpos + (size_t)i * m.nq, qvel + (size_t)i * m.nv, warm + (size_t)i * m.nv, mocap_pos + 3 * (size_t)i,
               mocap_quat + 4 * (size_t)i, ctrl + (size_t)i * m.nu);
  d->n = n;
  return upload(d->d_work, d->h_work.data(), n, err, errlen);
}

// one launch over the n states of the last dev_set_states; the workspaces are then read back for the ph_* readers
DEV_API int dev_run(void* h, int stage, int nsub, char* err, int errlen) {
  Dev* d = static_cast<Dev*>(h);
  if (d->n < 1) return fail("dev_run: no states", err, errlen);
  if (stage < STAGE_FORWARD || stage > STAGE_SUBSTEPS) return fail("dev_run: unknown stage", err, errlen);
  if (nsub < 0 || nsub > 10000) return fail("dev_run: substep count out of range", err, errlen);
  stage_kernel<<<d->n, 32>>>(d->d_model, d->d_hull, d->d_work, stage, nsub);
  if (finish(err, errlen)) return 1;
  return download(d->h_work.data(), d->d_work, d->n, err, errlen);
}

// readers of state i after dev_run (same signatures as emul.cpp's, where i is always 0)
#define DEV_STATE(i)                                                              \
  Dev* d = static_cast<Dev*>(h);                                                  \
  if ((i) < 0 || (i) >= d->n) return -1;                                          \
  const Model& m = d->hm.m;                                                       \
  const Work& w = d->h_work[i];                                                   \
  (void)m;

DEV_API int ph_state(void* h, int i, double* qpos, double* qvel, double* warm) { DEV_STATE(i) read_state(m, w, qpos, qvel, warm); return 0; }
DEV_API int ph_info(void* h, int i, int* out) { DEV_STATE(i) read_info(w, out); return 0; }
DEV_API int ph_forward(void* h, int i, double* xpos, double* xmat, double* M, double* bias) {
  DEV_STATE(i) read_forward(m, w, xpos, xmat, M, bias);
  return 0;
}
DEV_API int ph_hits(void* h, int i, int* pairs) { DEV_STATE(i) return read_hits(m, w, pairs); }
DEV_API int ph_contacts(void* h, int i, double* dist, double* pos, double* frame, int* geoms) {
  DEV_STATE(i) return read_contacts(w, dist, pos, frame, geoms);
}
DEV_API int ph_rows(void* h, int i, int* type, double* J, double* pos, double* R, double* D, double* aref, int* con, double* mu, double* fri) {
  DEV_STATE(i) return read_rows(m, w, type, J, pos, R, D, aref, con, mu, fri);
}
DEV_API int ph_solve(void* h, int i, double* acc, double* fcon, double* smooth, double* force) {
  DEV_STATE(i) read_solve(m, w, acc, fcon, smooth, force);
  return 0;
}

// ------------------------------------------------------------------------------------------------ unit entry points
// spd_solve<32> on `count` caller matrices A [count][MAXV][LDM] (lower triangle read, overwritten by the factor) and
// right-hand sides x [count][MAXV], sizes n [count]; ok [count] is spd_solve's return value
DEV_API int dev_spd_solve(int count, const int* n, float* A, float* x, int* ok, char* err, int errlen) {
  if (count < 1 || count > kMaxItems) return fail("dev_spd_solve: case count out of range", err, errlen);
  for (int b = 0; b < count; ++b)
    if (n[b] < 1 || n[b] > MAXV) return fail("dev_spd_solve: matrix size out of range", err, errlen);
  int* dn = nullptr; int* dok = nullptr;
  real (*dA)[MAXV][LDM] = nullptr;
  real (*dx)[MAXV] = nullptr;
  int rc = dalloc(&dn, count, err, errlen) || dalloc(&dok, count, err, errlen) ||
           dalloc(reinterpret_cast<real**>(&dA), (size_t)count * MAXV * LDM, err, errlen) ||
           dalloc(reinterpret_cast<real**>(&dx), (size_t)count * MAXV, err, errlen) || upload(dn, n, count, err, errlen) ||
           upload(&dA[0][0][0], A, (size_t)count * MAXV * LDM, err, errlen) || upload(&dx[0][0], x, (size_t)count * MAXV, err, errlen);
  if (!rc) {
    spd_kernel<<<count, 32>>>(dn, dA, dx, dok);
    rc = finish(err, errlen) || download(A, &dA[0][0][0], (size_t)count * MAXV * LDM, err, errlen) ||
         download(x, &dx[0][0], (size_t)count * MAXV, err, errlen) || download(ok, dok, count, err, errlen);
  }
  cudaFree(dn); cudaFree(dok); cudaFree(dA); cudaFree(dx);
  return rc;
}

// compact_append<32> (which 0: hit list, MAXHIT) or cand_append<32> (which 1: candidate list, MAXCAND) over `nitems`
// items per case, flags [count][nitems], starting from empty lists (cand: a valid cache) filled with 0xffff.  Out: both
// whole list arrays, hit [count][MAXHIT] and cand [count][MAXCAND] (adjacent in the workspace: a write past the end of
// one lands in the other), info [count][2] = (nhit, bad) or (ncand, broad_valid)
DEV_API int dev_append(int which, int count, int nitems, const int* flags, int* hit, int* cand, int* info, char* err, int errlen) {
  if (which != 0 && which != 1) return fail("dev_append: which must be 0 or 1", err, errlen);
  if (count < 1 || count > 1024 || nitems < 1 || nitems > kMaxItems) return fail("dev_append: size out of range", err, errlen);
  std::vector<Work> hw(count);
  memset(hw.data(), 0, sizeof(Work) * count);
  for (auto& w : hw) {
    memset(w.hit_list, 0xff, sizeof(w.hit_list));
    memset(w.cand_list, 0xff, sizeof(w.cand_list));
    w.broad_valid = 1;
  }
  Work* dw = nullptr;
  int* df = nullptr;
  int rc = dalloc(&dw, count, err, errlen) || dalloc(&df, (size_t)count * nitems, err, errlen) || upload(dw, hw.data(), count, err, errlen) ||
           upload(df, flags, (size_t)count * nitems, err, errlen);
  if (!rc) {
    append_kernel<<<count, 32>>>(dw, which, nitems, df);
    rc = finish(err, errlen) || download(hw.data(), dw, count, err, errlen);
  }
  cudaFree(dw); cudaFree(df);
  if (rc) return rc;
  for (int b = 0; b < count; ++b) {
    const Work& w = hw[b];
    for (int k = 0; k < MAXHIT; ++k) hit[(size_t)b * MAXHIT + k] = w.hit_list[k];
    for (int k = 0; k < MAXCAND; ++k) cand[(size_t)b * MAXCAND + k] = w.cand_list[k];
    info[2 * b] = which == 0 ? w.nhit : w.ncand;
    info[2 * b + 1] = which == 0 ? w.bad : w.broad_valid;
  }
  return 0;
}

// support_geom<32> of a mesh with vertices hull [nvert][3] in directions dirs [ndir][3]: out [ndir][3]
DEV_API int dev_support(int nvert, const float* hull, int ndir, const double* dirs, double* out, char* err, int errlen) {
  if (nvert < 1 || nvert > kMaxItems || ndir < 1 || ndir > kMaxItems) return fail("dev_support: size out of range", err, errlen);
  real* dh = nullptr;
  double* dd = nullptr;
  double* dout = nullptr;
  int rc = dalloc(&dh, (size_t)3 * nvert, err, errlen) || dalloc(&dd, (size_t)3 * ndir, err, errlen) || dalloc(&dout, (size_t)3 * ndir, err, errlen) ||
           upload(dh, hull, (size_t)3 * nvert, err, errlen) || upload(dd, dirs, (size_t)3 * ndir, err, errlen);
  if (!rc) {
    support_kernel<<<ndir, 32>>>(dh, nvert, dd, dout);
    rc = finish(err, errlen) || download(out, dout, (size_t)3 * ndir, err, errlen);
  }
  cudaFree(dh); cudaFree(dd); cudaFree(dout);
  return rc;
}
