// earl_tt3.cu -- three-object tabletop task (include/earl_tt3_b200.h): kernels + C ABI.
//
// Replaces earl_benchmark/envs/tabletop_manipulation_3obj.py (cited below as 3OBJ:line) under
// earl_benchmark/wrappers/persistent_state_wrapper.py (PSW:line).  One thread per environment; the task is
// HBM-bound integer/fp64 bookkeeping (no tensor cores):
//   * state: four double2 planes [4][N] (fist, object A, B, C) + one uint2 {flags, steps_since_reset} per env,
//     read and written with fully coalesced 16 / 8-byte accesses;
//   * actions [N,3] f32 and observations [N,20] f32 are row-major at the boundary: a block moves its 256-env
//     tile through shared memory so the global accesses are contiguous float4 (3 KB in, 20 KB out per block);
//   * algorithmic bytes per env-step: read 12 + 64 + 8 = 84, write fist 16 + meta 8 + obs 80 + 4 + 1 + 1 = 110  (194 B;
//     + 16 for the envs that drag an object: only that plane is written back).
// Compiled with --fmad=false: every fp64 / fp32 operation below rounds exactly where numpy rounds; the one
// fused operation numpy's BLAS performs (the 2-element fp64 dot) is written as an explicit fma.
// There is no CPU fallback in this file.
#include "../../include/earl_tt3_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include <cuda_runtime.h>

#include "tt3_env.cuh"

namespace earl {
int set_error(int code, const char* msg);  // earl_b200.cu
}

namespace {

constexpr int kBlock = 256;
constexpr int kObs = 20, kAct = 3;

struct T3Params {
  double2* q[4];          // [N] each: fist, object A, B, C
  uint2* meta;            // [N] {flags, steps_since_reset}
  long long* interventions;  // [N]
  const float* goal_f32;  // [G,10] fp32 casts of the goal table (what _get_obs emits)
  const double* goal_f64; // [G,10]
  const float* actions;   // [N,3]
  float* obs;             // [N,20]
  float* reward;          // [N]
  uint8_t* done;          // [N]
  uint8_t* success;       // [N] or null
  int n;
  int first;              // launch covers envs [first, first+count), first % 256 == 0
  int count;
  int dense;
  unsigned long long horizon;
  double act_lo, act_span, threshold, clip, success_radius;
  double init_qpos[8];
};

__device__ __forceinline__ void pdl_wait_prior_grid() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

using earl::tt3::EnvConst;
using earl::tt3::EnvState;
using earl::tt3::marker;

// stage one env's observation row (20 floats = 5 float4) in the block's tile: slot 5*t + j is conflict-free
// for 16-byte shared-memory accesses (5 is odd)
__device__ __forceinline__ void stage_obs(float4* tile, int t, const float (&o)[8], float m, const float* g) {
  tile[5 * t + 0] = make_float4(o[0], o[1], o[2], o[3]);
  tile[5 * t + 1] = make_float4(o[4], o[5], o[6], o[7]);
  tile[5 * t + 2] = make_float4(m, m, g[0], g[1]);
  tile[5 * t + 3] = make_float4(g[2], g[3], g[4], g[5]);
  tile[5 * t + 4] = make_float4(g[6], g[7], g[8], g[9]);
}

// contiguous float4 copy of the block's observation tile to global memory
__device__ __forceinline__ void flush_obs(const float4* tile, float* obs, int base, int n) {
  const int rows = min(kBlock, n - base);
  float4* dst = reinterpret_cast<float4*>(obs + (size_t)base * kObs);
  for (int k = threadIdx.x; k < rows * 5; k += kBlock) dst[k] = tile[k];
}

__global__ void __launch_bounds__(kBlock) tt3_step_kernel(const __grid_constant__ T3Params p) {
  __shared__ float4 s_obs[kBlock * 5];
  __shared__ float4 s_act4[kBlock * kAct / 4];
  float* s_act = reinterpret_cast<float*>(s_act4);
  const int end = p.first + p.count;
  const int base = p.first + blockIdx.x * kBlock;
  const int t = threadIdx.x;
  const int i = base + t;
  const int rows = min(kBlock, end - base);
  pdl_wait_prior_grid();  // nothing is read before the previous grid in the stream (the previous step, or the
                          // caller's action producer) has completed and flushed
  {  // actions of the tile: contiguous 16-byte loads when the tile starts on a 16-byte boundary (always, unless the
     // caller's buffer or a ring slot of a batch that is not a multiple of 4 envs is only 4-byte aligned)
    const float* asrc = p.actions + (size_t)base * kAct;
    if ((reinterpret_cast<uintptr_t>(asrc) & 15u) == 0) {
      const float4* src = reinterpret_cast<const float4*>(asrc);
      const int full = rows * kAct / 4;
      if (t < full) s_act4[t] = __ldcs(src + t);
      const int rem = rows * kAct - full * 4;
      if (t < rem) s_act[full * 4 + t] = asrc[full * 4 + t];
    } else {
      for (int k = t; k < rows * kAct; k += kBlock) s_act[k] = asrc[k];
    }
  }
  __syncthreads();
  if (i < end) {
    const double2 f = p.q[0][i], oa = p.q[1][i], ob = p.q[2][i], oc = p.q[3][i];
    const uint2 m = p.meta[i];
    const uint32_t row = (m.x >> 8) & 0xffu;
    EnvState st{f.x, f.y, {oa.x, ob.x, oc.x}, {oa.y, ob.y, oc.y}, m.x & 3u};
    const EnvConst ec{p.act_lo, p.act_span, p.threshold, p.clip, p.success_radius};
    earl::tt3::move(ec, st, s_act[kAct * t], s_act[kAct * t + 1], s_act[kAct * t + 2]);  // 3OBJ:86-144
    const uint32_t att = st.att;
    p.q[0][i] = make_double2(st.fx, st.fy);
#pragma unroll
    for (int k = 0; k < 3; ++k)  // only the dragged object's plane is written back
      if (att == (uint32_t)(k + 1)) p.q[1 + k][i] = make_double2(st.ox[k], st.oy[k]);
    float o[8];
    earl::tt3::observe8(st, o);  // 3OBJ:49-54
    float g[10];
    {
      const float2* gr = reinterpret_cast<const float2*>(p.goal_f32 + row * 10);
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const float2 v = __ldg(gr + k);
        g[2 * k] = v.x;
        g[2 * k + 1] = v.y;
      }
    }
    stage_obs(s_obs, t, o, marker(att), g);
    const bool succ = earl::tt3::success(o, g, p.success_radius);
    const float rew = p.dense ? (float)earl::tt3::dense(o, g) : (succ ? 1.0f : 0.0f);  // 3OBJ:146-159
    // PSW:22-31
    const uint32_t steps = m.y == 0xffffffffu ? m.y : m.y + 1u;
    p.meta[i] = make_uint2((m.x & ~3u) | att, steps);
    __stcs(p.reward + i, rew);
    p.done[i] = (unsigned long long)steps >= p.horizon ? 1 : 0;
    if (p.success) p.success[i] = succ ? 1 : 0;
  }
  __syncthreads();
  flush_obs(s_obs, p.obs, base, end);
}

// PSW:17-20 + 3OBJ:67-84 for the masked envs; also serves reset_goal (state untouched) and _get_obs
// mode 0: reset, 1: set goal only, 2: observation only
__global__ void __launch_bounds__(kBlock) tt3_reset_kernel(const __grid_constant__ T3Params p, const uint8_t* mask,
                                                           const int32_t* goal_idx, const double* init_qpos, int mode,
                                                           int num_goals) {
  const int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= p.n) return;
  const bool on = !mask || mask[i];
  uint2 m = p.meta[i];
  if (on && mode <= 1) {
    int row = goal_idx ? goal_idx[i] : 0;
    row = row < 0 ? 0 : (row >= num_goals ? num_goals - 1 : row);
    m.x = (m.x & ~0xff00u) | ((uint32_t)row << 8);
    if (mode == 0) {
      m.x &= ~3u;
      m.y = 0;
      p.interventions[i] += 1;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        p.q[k][i] = init_qpos ? make_double2(init_qpos[(size_t)i * 8 + 2 * k], init_qpos[(size_t)i * 8 + 2 * k + 1])
                              : make_double2(p.init_qpos[2 * k], p.init_qpos[2 * k + 1]);
    }
    p.meta[i] = m;
  }
  if (p.obs && on) {
    float* o = p.obs + (size_t)i * kObs;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double2 v = p.q[k][i];
      o[2 * k] = (float)v.x;
      o[2 * k + 1] = (float)v.y;
    }
    o[8] = o[9] = marker(m.x & 3u);
    const float* g = p.goal_f32 + ((m.x >> 8) & 0xffu) * 10;
#pragma unroll
    for (int k = 0; k < 10; ++k) o[10 + k] = g[k];
  }
}

// compute_reward / is_successful on caller observations (3OBJ:146-165)
__global__ void __launch_bounds__(kBlock) tt3_reward_kernel(const float* obs, long long num, float* reward, uint8_t* success,
                                                            int dense, double radius) {
  const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= num) return;
  const float* r = obs + i * kObs;
  float o[8], g[10];
#pragma unroll
  for (int k = 0; k < 8; ++k) o[k] = r[k];
#pragma unroll
  for (int k = 0; k < 10; ++k) g[k] = r[10 + k];
  const bool succ = earl::tt3::success(o, g, radius);
  if (reward) reward[i] = dense ? (float)earl::tt3::dense(o, g) : (succ ? 1.0f : 0.0f);
  if (success) success[i] = succ ? 1 : 0;
}

__global__ void __launch_bounds__(kBlock) tt3_state_kernel(const __grid_constant__ T3Params p, double* qpos_out, int32_t* att_out,
                                                           const double* qpos_in, const int32_t* att_in) {
  const int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= p.n) return;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (qpos_in) p.q[k][i] = make_double2(qpos_in[(size_t)i * 8 + 2 * k], qpos_in[(size_t)i * 8 + 2 * k + 1]);
    if (qpos_out) {
      const double2 v = p.q[k][i];
      qpos_out[(size_t)i * 8 + 2 * k] = v.x;
      qpos_out[(size_t)i * 8 + 2 * k + 1] = v.y;
    }
  }
  if (att_in) {
    uint2 m = p.meta[i];
    const int a = att_in[i];
    m.x = (m.x & ~3u) | (uint32_t)(a < 0 ? 0 : (a > 3 ? 3 : a));
    p.meta[i] = m;
  }
  if (att_out) att_out[i] = (int32_t)(p.meta[i].x & 3u);
}

__global__ void __launch_bounds__(kBlock) tt3_counters_kernel(const __grid_constant__ T3Params p, long long* interventions,
                                                              uint32_t* steps) {
  const int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= p.n) return;
  if (interventions) interventions[i] = p.interventions[i];
  if (steps) steps[i] = p.meta[i].y;
}

thread_local char g_msg[512];

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_msg, sizeof(g_msg), fmt, ap);
  va_end(ap);
  return earl::set_error(code, g_msg);
}

#define CU(call)                                                                  \
  do {                                                                            \
    cudaError_t e_ = (call);                                                      \
    if (e_ != cudaSuccess) return fail(EARL_ERR_CUDA, "%s (earl_tt3.cu:%d)", cudaGetErrorString(e_), __LINE__); \
  } while (0)

}  // namespace

struct earl_tt3_handle {
  earl_tt3_config cfg{};
  T3Params p{};
  int64_t total_steps = 0;
  int64_t launches = 0;
  std::vector<void*> owned;
  float* d_act = nullptr;
  float* d_obs = nullptr;
  float* d_rew = nullptr;
  uint8_t* d_done = nullptr;
  uint8_t* d_succ = nullptr;
  cudaStream_t in_stream = nullptr, out_stream = nullptr;
  static constexpr int kMaxChunks = 8;
  cudaEvent_t chunk_ev[kMaxChunks] = {};

  template <typename T>
  int alloc(T** ptr, size_t count, bool zero = true) {
    void* q = nullptr;
    if (cudaMalloc(&q, count * sizeof(T) + 16) != cudaSuccess) {
      cudaGetLastError();
      return fail(EARL_ERR_NOMEM, "cudaMalloc of %zu bytes failed", count * sizeof(T));
    }
    owned.push_back(q);
    if (zero && cudaMemset(q, 0, count * sizeof(T)) != cudaSuccess) return fail(EARL_ERR_CUDA, "cudaMemset failed");
    *ptr = static_cast<T*>(q);
    return 0;
  }
};

namespace {

int check(const earl_tt3_handle* h) {
  if (!h) return fail(EARL_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->cfg.device));
  return 0;
}

int grid_for(long long n) { return (int)((n + kBlock - 1) / kBlock); }

int launch_step(earl_tt3_handle* h, int first, int count, const float* actions, float* obs, float* reward, uint8_t* done,
                uint8_t* success, cudaStream_t s) {
  T3Params p = h->p;
  p.first = first;
  p.count = count;
  p.actions = actions;
  p.obs = obs;
  p.reward = reward;
  p.done = done;
  p.success = success;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid_for(count));
  cfg.blockDim = dim3(kBlock);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  CU(cudaLaunchKernelEx(&cfg, tt3_step_kernel, p));
  h->launches += 1;
  return 0;
}

bool aligned16(const void* q) { return ((uintptr_t)q & 15u) == 0; }

}  // namespace

extern "C" {

int earl_tt3_create(const earl_tt3_config* cfg, size_t cfg_nbytes, earl_tt3_handle** out) {
  if (!cfg || !out) return fail(EARL_ERR_INVALID, "null argument");
  if (cfg_nbytes != sizeof(earl_tt3_config)) return fail(EARL_ERR_INVALID, "earl_tt3_config size mismatch (%zu)", cfg_nbytes);
  if (cfg->num_envs < 1) return fail(EARL_ERR_INVALID, "num_envs must be >= 1");
  if (cfg->num_goals < 1 || cfg->num_goals > EARL_TT3_MAX_GOALS) return fail(EARL_ERR_INVALID, "num_goals out of range");
  if (cfg->flags & ~(uint32_t)EARL_FLAG_DENSE_REWARD) return fail(EARL_ERR_UNSUPPORTED, "unsupported flag for the three-object tabletop");
  if (cfg->episode_horizon < 1) return fail(EARL_ERR_INVALID, "episode_horizon must be >= 1");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) {
    cudaGetLastError();
    return fail(EARL_ERR_CUDA, "no usable CUDA device (requested %d); there is no CPU fallback", cfg->device);
  }
  CU(cudaSetDevice(cfg->device));
  earl_tt3_handle* h = new (std::nothrow) earl_tt3_handle();
  if (!h) return fail(EARL_ERR_NOMEM, "out of host memory");
  h->cfg = *cfg;
  const size_t n = (size_t)cfg->num_envs;
  T3Params& p = h->p;
  int rc = 0;
  for (int k = 0; k < 4 && !rc; ++k) rc = h->alloc(&p.q[k], n);
  if (!rc) rc = h->alloc(&p.meta, n);
  if (!rc) rc = h->alloc(&p.interventions, n);
  float* gf = nullptr;
  double* gd = nullptr;
  if (!rc) rc = h->alloc(&gf, (size_t)EARL_TT3_MAX_GOALS * 10);
  if (!rc) rc = h->alloc(&gd, (size_t)EARL_TT3_MAX_GOALS * 10);
  if (rc) {
    earl_tt3_destroy(h);
    return rc;
  }
  float g32[EARL_TT3_MAX_GOALS][10];
  for (int r = 0; r < EARL_TT3_MAX_GOALS; ++r)
    for (int k = 0; k < 10; ++k) g32[r][k] = (float)cfg->goal_table[r][k];
  if (cudaMemcpy(gf, g32, sizeof(g32), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(gd, cfg->goal_table, sizeof(cfg->goal_table), cudaMemcpyHostToDevice) != cudaSuccess) {
    earl_tt3_destroy(h);
    return fail(EARL_ERR_CUDA, "goal table upload failed");
  }
  p.goal_f32 = gf;
  p.goal_f64 = gd;
  p.n = cfg->num_envs;
  p.first = 0;
  p.count = cfg->num_envs;
  p.dense = (cfg->flags & EARL_FLAG_DENSE_REWARD) ? 1 : 0;
  p.horizon = (unsigned long long)cfg->episode_horizon;
  p.act_lo = -cfg->move_distance;
  p.act_span = cfg->move_distance - (-cfg->move_distance);
  p.threshold = cfg->threshold;
  p.clip = cfg->clip;
  p.success_radius = cfg->success_radius;
  for (int k = 0; k < 8; ++k) p.init_qpos[k] = cfg->initial_state[k];
  *out = h;
  return 0;
}

int earl_tt3_destroy(earl_tt3_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (void* q : h->owned) cudaFree(q);
  if (h->in_stream) cudaStreamDestroy(h->in_stream);
  if (h->out_stream) cudaStreamDestroy(h->out_stream);
  for (auto& ev : h->chunk_ev)
    if (ev) cudaEventDestroy(ev);
  delete h;
  return 0;
}

int earl_tt3_reset(earl_tt3_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev, const double* init_qpos_dev,
                   float* obs_out_dev, void* stream) {
  if (int rc = check(h)) return rc;
  T3Params p = h->p;
  p.obs = obs_out_dev;
  tt3_reset_kernel<<<grid_for(p.n), kBlock, 0, (cudaStream_t)stream>>>(p, mask_dev, goal_idx_dev, init_qpos_dev, 0, h->cfg.num_goals);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_tt3_set_goal(earl_tt3_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev, void* stream) {
  if (int rc = check(h)) return rc;
  T3Params p = h->p;
  p.obs = nullptr;
  tt3_reset_kernel<<<grid_for(p.n), kBlock, 0, (cudaStream_t)stream>>>(p, mask_dev, goal_idx_dev, nullptr, 1, h->cfg.num_goals);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_tt3_step(earl_tt3_handle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
                  uint8_t* success_dev, void* stream) {
  if (int rc = check(h)) return rc;
  if (!actions_dev || !obs_dev || !reward_dev || !done_dev) return fail(EARL_ERR_INVALID, "null device buffer");
  if (!aligned16(obs_dev)) return fail(EARL_ERR_INVALID, "obs must be 16-byte aligned");
  if (int rc = launch_step(h, 0, h->p.n, actions_dev, obs_dev, reward_dev, done_dev, success_dev, (cudaStream_t)stream)) return rc;
  h->total_steps += 1;
  return 0;
}

int earl_tt3_rollout(earl_tt3_handle* h, const float* actions_dev, int32_t action_ring, int32_t num_steps, float* obs_dev,
                     float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, int32_t out_ring, void* stream) {
  if (int rc = check(h)) return rc;
  if (!actions_dev || !obs_dev || !reward_dev || !done_dev || action_ring < 1 || out_ring < 1 || num_steps < 0)
    return fail(EARL_ERR_INVALID, "bad rollout argument");
  const size_t n = (size_t)h->p.n;
  if (!aligned16(obs_dev)) return fail(EARL_ERR_INVALID, "obs must be 16-byte aligned");
  for (int t = 0; t < num_steps; ++t) {
    const size_t a = (size_t)(t % action_ring), o = (size_t)(t % out_ring);
    if (int rc = launch_step(h, 0, (int)n, actions_dev + a * n * kAct, obs_dev + o * n * kObs, reward_dev + o * n, done_dev + o * n,
                             success_dev ? success_dev + o * n : nullptr, (cudaStream_t)stream))
      return rc;
    h->total_steps += 1;
  }
  return 0;
}

int earl_tt3_step_host(earl_tt3_handle* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host,
                       uint8_t* success_host) {
  if (int rc = check(h)) return rc;
  if (!actions_host || !obs_host || !reward_host || !done_host) return fail(EARL_ERR_INVALID, "null host buffer");
  const size_t n = (size_t)h->p.n;
  if (!h->d_act) {
    int rc = h->alloc(&h->d_act, n * kAct, false);
    if (!rc) rc = h->alloc(&h->d_obs, n * kObs, false);
    if (!rc) rc = h->alloc(&h->d_rew, n, false);
    if (!rc) rc = h->alloc(&h->d_done, n, false);
    if (!rc) rc = h->alloc(&h->d_succ, n, false);
    if (rc) return rc;
    CU(cudaStreamCreateWithFlags(&h->in_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->out_stream, cudaStreamNonBlocking));
    for (auto& ev : h->chunk_ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
  // chunked pipeline over the full-duplex PCIe link: the upload of chunk c+1 overlaps the kernel and the
  // downloads of chunk c
  CU(cudaDeviceSynchronize());  // order after whatever the caller enqueued on its own streams
  int chunks = (int)(n / (256 * 1024));
  chunks = chunks < 1 ? 1 : (chunks > earl_tt3_handle::kMaxChunks ? earl_tt3_handle::kMaxChunks : chunks);
  const size_t per = (((n + chunks - 1) / chunks + 255) / 256) * 256;  // ceil: never more than `chunks` iterations
  cudaStream_t si = h->in_stream, so = h->out_stream;
  int c = 0;
  for (size_t off = 0; off < n && c < earl_tt3_handle::kMaxChunks; off += per, ++c) {
    const size_t cnt = off + per <= n ? per : n - off;
    CU(cudaMemcpyAsync(h->d_act + off * kAct, actions_host + off * kAct, cnt * kAct * sizeof(float), cudaMemcpyHostToDevice, si));
    CU(cudaEventRecord(h->chunk_ev[c], si));
    CU(cudaStreamWaitEvent(so, h->chunk_ev[c], 0));
    if (int rc = launch_step(h, (int)off, (int)cnt, h->d_act, h->d_obs, h->d_rew, h->d_done, success_host ? h->d_succ : nullptr, so))
      return rc;
    CU(cudaMemcpyAsync(obs_host + off * kObs, h->d_obs + off * kObs, cnt * kObs * sizeof(float), cudaMemcpyDeviceToHost, so));
  }
  // the small outputs (6 B per env) go back in one copy each after the last chunk: fewer, larger copies (profiles/r01/e2e_sweep_r01.txt)
  CU(cudaMemcpyAsync(reward_host, h->d_rew, n * sizeof(float), cudaMemcpyDeviceToHost, so));
  CU(cudaMemcpyAsync(done_host, h->d_done, n, cudaMemcpyDeviceToHost, so));
  if (success_host) CU(cudaMemcpyAsync(success_host, h->d_succ, n, cudaMemcpyDeviceToHost, so));
  h->total_steps += 1;
  CU(cudaStreamSynchronize(so));
  return 0;
}

int earl_tt3_get_obs(earl_tt3_handle* h, float* obs_dev, void* stream) {
  if (int rc = check(h)) return rc;
  if (!obs_dev) return fail(EARL_ERR_INVALID, "null obs");
  T3Params p = h->p;
  p.obs = obs_dev;
  tt3_reset_kernel<<<grid_for(p.n), kBlock, 0, (cudaStream_t)stream>>>(p, nullptr, nullptr, nullptr, 2, h->cfg.num_goals);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_tt3_compute_reward(earl_tt3_handle* h, const float* obs_dev, int64_t num_obs, float* reward_dev, uint8_t* success_dev,
                            void* stream) {
  if (int rc = check(h)) return rc;
  if (!obs_dev || num_obs < 0) return fail(EARL_ERR_INVALID, "bad observation buffer");
  if (num_obs == 0) return 0;
  tt3_reward_kernel<<<grid_for(num_obs), kBlock, 0, (cudaStream_t)stream>>>(obs_dev, (long long)num_obs, reward_dev, success_dev,
                                                                           h->p.dense, h->p.success_radius);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_tt3_counters(earl_tt3_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev, uint32_t* steps_since_reset_dev,
                      void* stream) {
  if (int rc = check(h)) return rc;
  if (total_steps_host) *total_steps_host = h->total_steps;
  if (num_interventions_dev || steps_since_reset_dev) {
    tt3_counters_kernel<<<grid_for(h->p.n), kBlock, 0, (cudaStream_t)stream>>>(h->p, (long long*)num_interventions_dev,
                                                                              steps_since_reset_dev);
    CU(cudaGetLastError());
    h->launches += 1;
  }
  return 0;
}

int earl_tt3_get_state(earl_tt3_handle* h, double* qpos_dev, int32_t* attached_dev, void* stream) {
  if (int rc = check(h)) return rc;
  tt3_state_kernel<<<grid_for(h->p.n), kBlock, 0, (cudaStream_t)stream>>>(h->p, qpos_dev, attached_dev, nullptr, nullptr);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_tt3_set_state(earl_tt3_handle* h, const double* qpos_dev, const int32_t* attached_dev, void* stream) {
  if (int rc = check(h)) return rc;
  tt3_state_kernel<<<grid_for(h->p.n), kBlock, 0, (cudaStream_t)stream>>>(h->p, nullptr, nullptr, qpos_dev, attached_dev);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int64_t earl_tt3_launch_count(const earl_tt3_handle* h) { return h ? h->launches : 0; }

}  // extern "C"
