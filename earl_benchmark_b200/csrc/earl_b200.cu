// earl_b200.cu -- C-ABI implementation (include/earl_b200.h) of the batched EARL environment step.
// Host side: handle, device allocations, launch configuration, host-buffer path, snapshots, RNG streams.
// Device side: tabletop_kernels.cuh.  There is no CPU fallback anywhere in this file.
#include "../../include/earl_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include <cuda_runtime.h>

#include "mt19937.hpp"
#include "tabletop_kernels.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(EARL_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

}  // namespace

namespace earl {
// shared with earl_mj.cu: sets the thread-local message behind earl_last_error() and returns `code`
int set_error(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}
}  // namespace earl

namespace {

struct SnapshotHeader {
  uint32_t magic;  // 'ESNP'
  int32_t env_kind;
  int32_t num_envs;
  uint32_t flags;
  int64_t total_steps;
};
constexpr uint32_t kSnapMagic = 0x45534e50u;

}  // namespace

struct earl_handle {
  earl_config cfg{};
  earl_tabletop_model model{};
  earl::TabletopParams p{};
  int device = 0;
  int sm_count = 0;
  int step_grid = 0;
  bool tile_step = false;  // the one-tile-per-CTA kernel runs the step instead of the persistent LSU kernel (see earl_create)
  int host_zerocopy = 1;   // EARL_TT_HOST_ZEROCOPY=0: staged copy pipeline instead of the step kernel reading / writing the pinned host buffers itself
  int64_t total_steps = 0;
  int64_t launches = 0;
  // owned device memory
  std::vector<void*> owned;
  // host-path staging
  float* d_act = nullptr;
  float* d_obs = nullptr;
  float* d_rew = nullptr;
  uint8_t* d_done = nullptr;
  uint8_t* d_succ = nullptr;
  cudaStream_t host_stream = nullptr;
  cudaStream_t in_stream = nullptr;
  static constexpr int kMaxChunks = 16;
  cudaEvent_t chunk_ev[kMaxChunks] = {};
  // recorded on the caller's stream after every state-mutating launch (reset / set_goal / step / rollout); the
  // host-buffer step, which runs on the handle's private streams, waits on it (ADVICE r1: it could race a reset)
  cudaEvent_t order_ev = nullptr;
  bool order_pending = false;
  double* d_stats = nullptr;
  float* final_obs = nullptr;  // EARL_FLAG_FINAL_OBS: the caller's [N,12] buffer (earl_set_final_obs)

  template <typename T>
  int alloc(T** ptr, size_t count, bool zero = true) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
    if (e != cudaSuccess) return fail(EARL_ERR_NOMEM, "cudaMalloc(%zu B) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    if (zero) {
      e = cudaMemset(q, 0, count * sizeof(T));
      if (e != cudaSuccess) return fail(EARL_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    }
    owned.push_back(q);
    *ptr = static_cast<T*>(q);
    return 0;
  }
};

namespace {

bool f64(const earl_handle* h) { return h->cfg.flags & EARL_FLAG_STATE_F64; }

bool per_env_goals(const earl_handle* h) { return h->cfg.flags & EARL_FLAG_PER_ENV_GOALS; }

bool has_final_obs(const earl_handle* h) { return h->cfg.flags & EARL_FLAG_FINAL_OBS; }

bool fast_path(const earl_handle* h) {
  return !(h->cfg.flags & (EARL_FLAG_DENSE_REWARD | EARL_FLAG_LIFELONG | EARL_FLAG_AUTO_RESET | EARL_FLAG_EVAL_STATS |
                           EARL_FLAG_PER_ENV_GOALS));
}

int check_handle(const earl_handle* h) {
  if (!h) return fail(EARL_ERR_INVALID, "null handle");
  cudaError_t e = cudaSetDevice(h->device);
  if (e != cudaSuccess) return fail(EARL_ERR_CUDA, "cudaSetDevice(%d) failed: %s", h->device, cudaGetErrorString(e));
  return 0;
}

int upload_goal_tables(earl_handle* h) {
  // fp32 rows padded to 8 floats (two float4 per row) + fp64 rows
  std::vector<float> g32(256 * 8, 0.f);
  for (int r = 0; r < 256; ++r)
    for (int c = 0; c < 6; ++c) g32[r * 8 + c] = (float)h->model.goal_table[r][c];
  CU(cudaMemcpy(const_cast<float4*>(h->p.goal32), g32.data(), g32.size() * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(const_cast<double*>(h->p.goal64), &h->model.goal_table[0][0], 256 * 6 * sizeof(double),
                cudaMemcpyHostToDevice));
  return 0;
}

// Launch a step kernel with the programmatic-stream-serialization attribute (PDL): it may start while the previous
// grid in the stream drains, and waits for it in griddepcontrol.wait.
cudaError_t launch_pdl(void (*kernel)(const earl::TabletopParams), int grid, cudaStream_t s, const earl::TabletopParams& p) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)earl::kTTBlock);
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, p);
}

template <typename K>
int occupancy_grid(K kernel, int sm_count, int* grid) {
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, earl::kTTBlock, 0));
  if (per_sm < 1) per_sm = 1;
  *grid = sm_count * per_sm;
  return 0;
}

// One step of envs [first, first+count) (whole batch: first=0, count=N).  IO pointers are those of env 0.
// zero_copy: the outputs are pinned host memory (step_host_zerocopy); the tile kernel writes reward / done / success as
// 16-byte vectors.  Only for handles on the FAST fp32 path.
int launch_step_range(earl_handle* h, int first, int count, const float* actions, float* obs, float* reward,
                      uint8_t* done, uint8_t* success, cudaStream_t s, bool zero_copy = false) {
  earl::TabletopParams p = h->p;
  p.n_total = h->p.n;
  p.n = first + count;
  p.actions = actions;
  p.obs = obs;
  p.reward = reward;
  p.done = done;
  p.success = success;
  const bool fast = fast_path(h);
  p.first = first;
  const int tiles = (p.n - p.first + earl::kTTBlock - 1) / earl::kTTBlock;
  if (zero_copy || h->tile_step) {  // one 256-env tile per CTA (obs rows are 48 B: every tile starts 16-byte aligned)
    CU(launch_pdl(zero_copy ? earl::tabletop_step_tile_kernel<true> : earl::tabletop_step_tile_kernel<false>, tiles, s, p));
    h->launches += 1;
    return 0;
  }
  const int grid = tiles < h->step_grid ? tiles : h->step_grid;
  if (has_final_obs(h)) {
    if (f64(h) && per_env_goals(h)) earl::tabletop_step_kernel<true, false, 1, true, true><<<grid, earl::kTTBlock, 0, s>>>(p, h->final_obs);
    else if (f64(h)) earl::tabletop_step_kernel<true, false, 1, false, true><<<grid, earl::kTTBlock, 0, s>>>(p, h->final_obs);
    else if (per_env_goals(h)) earl::tabletop_step_kernel<false, false, 1, true, true><<<grid, earl::kTTBlock, 0, s>>>(p, h->final_obs);
    else earl::tabletop_step_kernel<false, false, 1, false, true><<<grid, earl::kTTBlock, 0, s>>>(p, h->final_obs);
  } else if (f64(h)) {
    if (fast) earl::tabletop_step_kernel<true, true><<<grid, earl::kTTBlock, 0, s>>>(p);
    else if (per_env_goals(h)) earl::tabletop_step_kernel<true, false, 1, true><<<grid, earl::kTTBlock, 0, s>>>(p);
    else earl::tabletop_step_kernel<true, false><<<grid, earl::kTTBlock, 0, s>>>(p);
  } else {
    if (fast) CU(launch_pdl(earl::tabletop_step_kernel<false, true>, grid, s, p));
    else if (per_env_goals(h)) earl::tabletop_step_kernel<false, false, 1, true><<<grid, earl::kTTBlock, 0, s>>>(p);
    else earl::tabletop_step_kernel<false, false><<<grid, earl::kTTBlock, 0, s>>>(p);
  }
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int launch_step(earl_handle* h, const float* actions, float* obs, float* reward, uint8_t* done, uint8_t* success,
                cudaStream_t s) {
  if (int rc = launch_step_range(h, 0, h->p.n, actions, obs, reward, done, success, s)) return rc;
  h->total_steps += 1;
  return 0;
}

// remember that `s` carries work the private host-path streams must wait for
int note_stream(earl_handle* h, cudaStream_t s) {
  if (!h->order_ev) CU(cudaEventCreateWithFlags(&h->order_ev, cudaEventDisableTiming));
  CU(cudaEventRecord(h->order_ev, s));
  h->order_pending = true;
  return 0;
}

// a final-observation handle steps only once its buffer is registered, like an auto-reset handle with a stream
int check_final_obs(const earl_handle* h) {
  if (has_final_obs(h) && !h->final_obs) return fail(EARL_ERR_INVALID, "EARL_FLAG_FINAL_OBS handles need earl_set_final_obs before the first step");
  return 0;
}

int check_io(const void* a, const void* o, const void* r, const void* d) {
  if (!a || !o || !r || !d) return fail(EARL_ERR_INVALID, "actions, obs, reward and done must be non-null");
  if (((uintptr_t)o & 15u) || ((uintptr_t)a & 3u)) return fail(EARL_ERR_INVALID, "obs must be 16-byte aligned, actions 4-byte aligned");
  return 0;
}

}  // namespace

extern "C" {

int earl_abi_version(void) { return EARL_ABI_VERSION; }

const char* earl_last_error(void) { return g_err; }

void earl_tabletop_thresholds(double threshold, double success_radius, double* attach_sq, float* success_sq) {
  // smallest double x with sqrt(x) >= threshold  =>  (sqrt(s) < threshold) == (s < x) for every s
  double x = threshold * threshold;
  while (std::sqrt(x) >= threshold && x > 0.0) x = std::nextafter(x, 0.0);
  while (std::sqrt(x) < threshold) x = std::nextafter(x, INFINITY);
  *attach_sq = x;
  // largest float y with (double)sqrtf(y) <= radius  =>  ((double)sqrtf(s) <= radius) == (s <= y)
  float y = (float)(success_radius * success_radius);
  while ((double)std::sqrt(y) <= success_radius) y = std::nextafterf(y, INFINITY);
  while ((double)std::sqrt(y) > success_radius && y > 0.f) y = std::nextafterf(y, 0.f);
  *success_sq = y;
}

int earl_create(const earl_config* cfg, const void* model_blob, size_t model_nbytes, earl_handle** out) {
  if (!cfg || !out) return fail(EARL_ERR_INVALID, "null cfg/out");
  *out = nullptr;
  if (cfg->env_kind != EARL_ENV_TABLETOP)
    return fail(EARL_ERR_UNSUPPORTED, "env_kind %d is not built yet (only tabletop_manipulation)", cfg->env_kind);
  if (cfg->num_envs < 1) return fail(EARL_ERR_INVALID, "num_envs must be >= 1");
  if (cfg->episode_horizon < 1) return fail(EARL_ERR_INVALID, "episode_horizon must be >= 1");
  if ((cfg->flags & EARL_FLAG_LIFELONG) && cfg->goal_change_frequency < 1)
    return fail(EARL_ERR_INVALID, "lifelong handles need goal_change_frequency >= 1");
  if ((cfg->flags & EARL_FLAG_FINAL_OBS) && !(cfg->flags & EARL_FLAG_AUTO_RESET))
    return fail(EARL_ERR_INVALID, "EARL_FLAG_FINAL_OBS needs EARL_FLAG_AUTO_RESET");
  if (!model_blob || model_nbytes != sizeof(earl_tabletop_model))
    return fail(EARL_ERR_INVALID, "model blob must be an earl_tabletop_model (%zu B), got %zu B", sizeof(earl_tabletop_model), model_nbytes);
  const earl_tabletop_model* m = static_cast<const earl_tabletop_model*>(model_blob);
  if (m->magic != EARL_TABLETOP_MAGIC || m->num_goals < 1 || m->num_goals > 256)
    return fail(EARL_ERR_INVALID, "bad tabletop model blob (magic %08x, %d goals)", m->magic, m->num_goals);

  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(EARL_ERR_INVALID, "device %d out of range (%d visible)", cfg->device, ndev);
  CU(cudaSetDevice(cfg->device));

  earl_handle* h = new (std::nothrow) earl_handle();
  if (!h) return fail(EARL_ERR_NOMEM, "host allocation failed");
  h->cfg = *cfg;
  h->model = *m;
  h->device = cfg->device;
  if (h->cfg.goal_stream_rows < 1) h->cfg.goal_stream_rows = 1;
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, cfg->device);
  if (e != cudaSuccess) { delete h; return fail(EARL_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)); }
  h->sm_count = prop.multiProcessorCount;

  const size_t n = (size_t)cfg->num_envs;
  earl::TabletopParams& p = h->p;
  int rc = 0;
  float4* g32 = nullptr;
  double* g64 = nullptr;
  uint8_t* stream_rows = nullptr;
  if (f64(h)) { double* q = nullptr; rc = h->alloc(&q, n * 4); p.qpos = q; }
  else { float4* q = nullptr; rc = h->alloc(&q, n); p.qpos = q; }
  if (!rc) rc = h->alloc(&p.meta, n);
  if (!rc) rc = h->alloc(&p.interventions, n);
  if (!rc) rc = h->alloc(&p.goal_cursor, n);
  if (!rc) rc = h->alloc(&stream_rows, n * (size_t)h->cfg.goal_stream_rows);
  if (!rc) rc = h->alloc(&g32, 512);
  if (!rc) rc = h->alloc(&g64, 256 * 6);
  if (!rc && (cfg->flags & EARL_FLAG_LIFELONG)) { rc = h->alloc(&p.ll_steps, n); if (!rc) rc = h->alloc(&p.ll_return, n); }
  if (!rc && (cfg->flags & EARL_FLAG_EVAL_STATS)) rc = h->alloc(&p.ep_return, n);
  if (!rc && per_env_goals(h)) rc = h->alloc(&p.env_goal, n * 2);
  if (!rc) rc = h->alloc(&h->d_stats, 4);
  if (rc) { earl_destroy(h); return rc; }
  p.goal_stream = stream_rows;
  p.goal32 = g32;
  p.goal64 = g64;
  p.n = cfg->num_envs;
  p.n_total = cfg->num_envs;
  p.goal_stream_rows = h->cfg.goal_stream_rows;
  p.features = cfg->flags;
  p.horizon = (unsigned long long)cfg->episode_horizon;
  p.goal_change_frequency = (unsigned long long)(cfg->goal_change_frequency > 0 ? cfg->goal_change_frequency : 1);
  p.act_lo = -m->move_distance;
  p.act_span = m->move_distance - (-m->move_distance);  // (ub - lb), tabletop_manipulation.py:131-132
  p.threshold = m->threshold;
  p.clip = m->clip;
  p.success_radius = m->success_radius;
  earl_tabletop_thresholds(m->threshold, m->success_radius, &p.attach_sq, &p.success_sq);
  for (int k = 0; k < 4; ++k) p.init_qpos[k] = m->initial_state[k];
  rc = upload_goal_tables(h);
  if (!rc && per_env_goals(h)) {
    // every env starts on the goal of its (zeroed) meta row, row 0, as a handle without per-env goals does
    earl::TabletopGoalArgs a{p.goal32, 0, 0, nullptr, nullptr};
    earl::tabletop_set_goals_kernel<false><<<(p.n + 255) / 256, 256>>>(p, a);
    cudaError_t le = cudaGetLastError();
    if (le == cudaSuccess) le = cudaDeviceSynchronize();
    if (le != cudaSuccess) rc = fail(EARL_ERR_CUDA, "per-env goal initialisation: %s", cudaGetErrorString(le));
    h->launches += 1;
  }
  if (rc) { earl_destroy(h); return rc; }

  const bool fast = fast_path(h);
  if (has_final_obs(h))
    rc = f64(h) ? (per_env_goals(h) ? occupancy_grid(earl::tabletop_step_kernel<true, false, 1, true, true>, h->sm_count, &h->step_grid)
                                    : occupancy_grid(earl::tabletop_step_kernel<true, false, 1, false, true>, h->sm_count, &h->step_grid))
                : (per_env_goals(h) ? occupancy_grid(earl::tabletop_step_kernel<false, false, 1, true, true>, h->sm_count, &h->step_grid)
                                    : occupancy_grid(earl::tabletop_step_kernel<false, false, 1, false, true>, h->sm_count, &h->step_grid));
  else if (f64(h)) rc = fast ? occupancy_grid(earl::tabletop_step_kernel<true, true>, h->sm_count, &h->step_grid)
                 : per_env_goals(h) ? occupancy_grid(earl::tabletop_step_kernel<true, false, 1, true>, h->sm_count, &h->step_grid)
                        : occupancy_grid(earl::tabletop_step_kernel<true, false>, h->sm_count, &h->step_grid);
  else rc = fast ? occupancy_grid(earl::tabletop_step_kernel<false, true>, h->sm_count, &h->step_grid)
                 : per_env_goals(h) ? occupancy_grid(earl::tabletop_step_kernel<false, false, 1, true>, h->sm_count, &h->step_grid)
                 : occupancy_grid(earl::tabletop_step_kernel<false, false>, h->sm_count, &h->step_grid);
  if (rc) { earl_destroy(h); return rc; }
  // measured on B200 (DESIGN.md section 4): while the 24 B/env state fits in L2 next to the streams the persistent LSU
  // kernel wins (more resident warps hide L2 latency); once everything streams from HBM (above ~3M envs) the
  // one-tile-per-CTA kernel does.  It only implements the FAST fp32 step.
  h->tile_step = fast && !f64(h) && cfg->num_envs > 3 * 1024 * 1024;
  if (const char* v = getenv("EARL_TT_HOST_ZEROCOPY")) h->host_zerocopy = atoi(v);
  e = cudaStreamCreateWithFlags(&h->host_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { earl_destroy(h); return fail(EARL_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
  *out = h;
  return 0;
}

int earl_destroy(earl_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  for (void* q : h->owned) cudaFree(q);
  if (h->host_stream) cudaStreamDestroy(h->host_stream);
  if (h->in_stream) cudaStreamDestroy(h->in_stream);
  for (auto& ev : h->chunk_ev) if (ev) cudaEventDestroy(ev);
  if (h->order_ev) cudaEventDestroy(h->order_ev);
  delete h;
  return 0;
}

int earl_num_envs(const earl_handle* h) { return h ? h->cfg.num_envs : 0; }
int earl_obs_dim(const earl_handle* h) { return h ? earl::kTTObs : 0; }
int earl_action_dim(const earl_handle* h) { return h ? earl::kTTAct : 0; }
int64_t earl_launch_count(const earl_handle* h) { return h ? h->launches : 0; }

int earl_set_goal_stream(earl_handle* h, const uint8_t* rows_host, int32_t num_rows) {
  if (int rc = check_handle(h)) return rc;
  if (!rows_host || num_rows != h->cfg.goal_stream_rows)
    return fail(EARL_ERR_INVALID, "goal stream must have exactly goal_stream_rows=%d rows (got %d)", h->cfg.goal_stream_rows, num_rows);
  const size_t nb = (size_t)num_rows * h->cfg.num_envs;
  for (size_t k = 0; k < nb; ++k)
    if (rows_host[k] >= h->model.num_goals) return fail(EARL_ERR_INVALID, "goal stream entry %zu = %u >= num_goals %d", k, rows_host[k], h->model.num_goals);
  CU(cudaMemcpy(const_cast<uint8_t*>(h->p.goal_stream), rows_host, nb, cudaMemcpyHostToDevice));
  return 0;
}

int earl_set_goal_table(earl_handle* h, const double* rows_host, int32_t first_row, int32_t count) {
  if (int rc = check_handle(h)) return rc;
  if (!rows_host || first_row < 0 || count < 1 || first_row + count > 256) return fail(EARL_ERR_INVALID, "goal table rows out of range");
  memcpy(&h->model.goal_table[first_row][0], rows_host, (size_t)count * 6 * sizeof(double));
  if (first_row + count > h->model.num_goals) h->model.num_goals = first_row + count;
  CU(cudaDeviceSynchronize());
  return upload_goal_tables(h);
}

static int reset_impl(earl_handle* h, const uint8_t* mask, const int32_t* goal_idx, const double* init_qpos,
                      float* obs_out, int goal_only, void* stream) {
  if (int rc = check_handle(h)) return rc;
  earl::TabletopResetArgs a{mask, goal_idx, init_qpos, obs_out, goal_only};
  const int grid = (h->p.n + 255) / 256;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (f64(h)) earl::tabletop_reset_kernel<true><<<grid, 256, 0, s>>>(h->p, a);
  else earl::tabletop_reset_kernel<false><<<grid, 256, 0, s>>>(h->p, a);
  CU(cudaGetLastError());
  h->launches += 1;
  return note_stream(h, s);
}

int earl_reset(earl_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev, const double* init_qpos_dev,
               float* obs_out_dev, void* stream) {
  return reset_impl(h, mask_dev, goal_idx_dev, init_qpos_dev, obs_out_dev, 0, stream);
}

int earl_set_goal(earl_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev, void* stream) {
  return reset_impl(h, mask_dev, goal_idx_dev, nullptr, nullptr, 1, stream);
}

int earl_set_goals(earl_handle* h, const void* goals_dev, int32_t goal_dtype, const uint8_t* mask_dev, float* obs_out_dev,
                   void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!per_env_goals(h)) return fail(EARL_ERR_INVALID, "earl_set_goals needs a handle created with EARL_FLAG_PER_ENV_GOALS");
  if (!goals_dev) return fail(EARL_ERR_INVALID, "null goals");
  if (goal_dtype != EARL_GOAL_F32 && goal_dtype != EARL_GOAL_F64) return fail(EARL_ERR_INVALID, "goal_dtype must be EARL_GOAL_F32 or EARL_GOAL_F64");
  if ((uintptr_t)obs_out_dev & 15u) return fail(EARL_ERR_INVALID, "obs_out must be 16-byte aligned");
  earl::TabletopGoalArgs a{goals_dev, goal_dtype == EARL_GOAL_F64, 6, mask_dev, obs_out_dev};
  const int grid = (h->p.n + 255) / 256;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (f64(h)) earl::tabletop_set_goals_kernel<true><<<grid, 256, 0, s>>>(h->p, a);
  else earl::tabletop_set_goals_kernel<false><<<grid, 256, 0, s>>>(h->p, a);
  CU(cudaGetLastError());
  h->launches += 1;
  return note_stream(h, s);
}

int earl_get_goals(earl_handle* h, float* goals_out_dev, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!per_env_goals(h)) return fail(EARL_ERR_INVALID, "earl_get_goals needs a handle created with EARL_FLAG_PER_ENV_GOALS");
  if (!goals_out_dev) return fail(EARL_ERR_INVALID, "null goals_out");
  // the first 6 of the 8 floats of every env's slot
  CU(cudaMemcpy2DAsync(goals_out_dev, 6 * sizeof(float), h->p.env_goal, 2 * sizeof(float4), 6 * sizeof(float), (size_t)h->p.n,
                       cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

int earl_set_final_obs(earl_handle* h, float* final_obs_dev) {
  if (int rc = check_handle(h)) return rc;
  if (!has_final_obs(h)) return fail(EARL_ERR_INVALID, "earl_set_final_obs needs a handle created with EARL_FLAG_FINAL_OBS");
  if (!final_obs_dev || ((uintptr_t)final_obs_dev & 15u)) return fail(EARL_ERR_INVALID, "final_obs must be non-null and 16-byte aligned");
  h->final_obs = final_obs_dev;
  return 0;
}

int earl_step(earl_handle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
              uint8_t* success_dev, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_io(actions_dev, obs_dev, reward_dev, done_dev)) return rc;
  if (int rc = check_final_obs(h)) return rc;
  if (int rc = launch_step(h, actions_dev, obs_dev, reward_dev, done_dev, success_dev, static_cast<cudaStream_t>(stream))) return rc;
  return note_stream(h, static_cast<cudaStream_t>(stream));
}

int earl_rollout(earl_handle* h, const float* actions_dev, int32_t action_ring, int32_t num_steps, float* obs_dev,
                 float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, int32_t out_ring, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (int rc = check_io(actions_dev, obs_dev, reward_dev, done_dev)) return rc;
  if (action_ring < 1 || out_ring < 1 || num_steps < 0) return fail(EARL_ERR_INVALID, "rings must be >= 1 and num_steps >= 0");
  if (has_final_obs(h)) return fail(EARL_ERR_INVALID, "earl_rollout does not take EARL_FLAG_FINAL_OBS handles (one final-observation buffer per step)");
  const size_t n = (size_t)h->p.n;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int32_t t = 0; t < num_steps; ++t) {
    const size_t ia = (size_t)(t % action_ring), io = (size_t)(t % out_ring);
    int rc = launch_step(h, actions_dev + ia * n * earl::kTTAct, obs_dev + io * n * earl::kTTObs, reward_dev + io * n,
                         done_dev + io * n, success_dev ? success_dev + io * n : nullptr, s);
    if (rc) return rc;
  }
  return note_stream(h, s);
}

}  // extern "C"
namespace {
// device alias of a pinned, mapped host buffer (cudaHostAlloc / cudaHostRegister under unified addressing); null otherwise
template <class T>
T* mapped_alias(T* host) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return at.type == cudaMemoryTypeHost ? static_cast<T*>(at.devicePointer) : nullptr;
}

// Zero-copy host step: the one-tile-per-CTA kernel reads the actions from, and writes observations / reward / done / success
// to, the caller's pinned host buffers directly -- full-line coalesced float4 traffic over PCIe in both directions at once,
// no staging copies, no chunk pipeline, one launch.  Only for the FAST configuration and mapped, 16-byte aligned buffers.
bool step_host_zerocopy(earl_handle* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host,
                        uint8_t* success_host, int* rc_out) {
  if (!h->host_zerocopy || !fast_path(h) || f64(h)) return false;
  const float* a = mapped_alias(actions_host);
  float* o = mapped_alias(obs_host);
  float* r = mapped_alias(reward_host);
  uint8_t* d = mapped_alias(done_host);
  uint8_t* su = success_host ? mapped_alias(success_host) : nullptr;
  if (!a || !o || !r || !d || (success_host && !su) || ((uintptr_t)o & 15u) || ((uintptr_t)a & 15u)) return false;
  if (!h->host_stream) return false;
  cudaStream_t so = h->host_stream;
  auto run = [&]() -> int {
    if (h->order_pending) {
      CU(cudaStreamWaitEvent(so, h->order_ev, 0));
      if (h->in_stream) CU(cudaStreamWaitEvent(h->in_stream, h->order_ev, 0));
      h->order_pending = false;
    }
    if (int rc = launch_step_range(h, 0, h->p.n, a, o, r, d, su, so, /*zero_copy=*/true)) return rc;
    h->total_steps += 1;
    CU(cudaStreamSynchronize(so));
    return 0;
  };
  *rc_out = run();
  return true;
}
}  // namespace
extern "C" {

int earl_step_host(earl_handle* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host,
                   uint8_t* success_host) {
  if (int rc = check_handle(h)) return rc;
  if (!actions_host || !obs_host || !reward_host || !done_host) return fail(EARL_ERR_INVALID, "null host buffer");
  if (int rc = check_final_obs(h)) return rc;
  {
    int rc = 0;
    if (step_host_zerocopy(h, actions_host, obs_host, reward_host, done_host, success_host, &rc)) return rc;
  }
  const size_t n = (size_t)h->p.n;
  if (!h->d_act) {
    int rc = h->alloc(&h->d_act, n * earl::kTTAct, false);
    if (!rc) rc = h->alloc(&h->d_obs, n * earl::kTTObs, false);
    if (!rc) rc = h->alloc(&h->d_rew, n, false);
    if (!rc) rc = h->alloc(&h->d_done, n, false);
    if (!rc) rc = h->alloc(&h->d_succ, n, false);
    if (rc) return rc;
    CU(cudaStreamCreateWithFlags(&h->in_stream, cudaStreamNonBlocking));
    for (auto& ev : h->chunk_ev) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
  // Chunked software pipeline over the PCIe link: the host->device copy of chunk c+1 (in_stream) overlaps the
  // kernel and the device->host copies of chunk c (host_stream); the link is full duplex.
  constexpr int kMaxChunks = earl_handle::kMaxChunks;
  int chunks = (int)(n / (256 * 1024));
  chunks = chunks < 1 ? 1 : (chunks > kMaxChunks ? kMaxChunks : chunks);
  // the three small outputs (6 B per env) go back in one copy each after the last chunk instead of one per chunk:
  // fewer, larger device->host copies per step: their fixed costs are what separates this path from the link rate
  // (1M envs, env-steps/s: 8 chunks, all outputs per chunk 7.8e8; 8 chunks + tail 8.4e8; 4 chunks + tail 8.8e8; 2 chunks
  // + tail 8.7e8; 16 chunks + tail 7.9e8; one chunk 8.2e8 -- profiles/r01/e2e_sweep_r01.txt)
  const bool tail = chunks > 1;
  // ceil(n / chunks) rounded up to whole 256-env tiles: at most `chunks` iterations (floor could give chunks + 1 and
  // index chunk_ev out of bounds, ADVICE r1); chunk boundaries stay tile- and 16-byte aligned
  const size_t per = (((n + chunks - 1) / chunks + 255) / 256) * 256;
  cudaStream_t si = h->in_stream, so = h->host_stream;
  if (h->order_pending) {  // resets / device steps queued on the caller's stream come first
    CU(cudaStreamWaitEvent(si, h->order_ev, 0));
    CU(cudaStreamWaitEvent(so, h->order_ev, 0));
    h->order_pending = false;
  }
  uint8_t* d_succ = success_host ? h->d_succ : nullptr;
  int c = 0;
  for (size_t off = 0; off < n && c < kMaxChunks; off += per, ++c) {
    const size_t cnt = (off + per <= n && c + 1 < kMaxChunks) ? per : n - off;
    CU(cudaMemcpyAsync(h->d_act + off * earl::kTTAct, actions_host + off * earl::kTTAct, cnt * earl::kTTAct * sizeof(float),
                       cudaMemcpyHostToDevice, si));
    CU(cudaEventRecord(h->chunk_ev[c], si));
    CU(cudaStreamWaitEvent(so, h->chunk_ev[c], 0));
    if (int rc = launch_step_range(h, (int)off, (int)cnt, h->d_act, h->d_obs, h->d_rew, h->d_done, d_succ, so)) return rc;
    CU(cudaMemcpyAsync(obs_host + off * earl::kTTObs, h->d_obs + off * earl::kTTObs, cnt * earl::kTTObs * sizeof(float),
                       cudaMemcpyDeviceToHost, so));
    if (tail) continue;
    CU(cudaMemcpyAsync(reward_host + off, h->d_rew + off, cnt * sizeof(float), cudaMemcpyDeviceToHost, so));
    CU(cudaMemcpyAsync(done_host + off, h->d_done + off, cnt, cudaMemcpyDeviceToHost, so));
    if (success_host) CU(cudaMemcpyAsync(success_host + off, h->d_succ + off, cnt, cudaMemcpyDeviceToHost, so));
  }
  if (tail) {
    CU(cudaMemcpyAsync(reward_host, h->d_rew, n * sizeof(float), cudaMemcpyDeviceToHost, so));
    CU(cudaMemcpyAsync(done_host, h->d_done, n, cudaMemcpyDeviceToHost, so));
    if (success_host) CU(cudaMemcpyAsync(success_host, h->d_succ, n, cudaMemcpyDeviceToHost, so));
  }
  h->total_steps += 1;
  CU(cudaStreamSynchronize(so));
  return 0;
}

int earl_set_host_zerocopy(earl_handle* h, int32_t enable) {
  if (int rc = check_handle(h)) return rc;
  h->host_zerocopy = enable ? 1 : 0;
  return 0;
}

int earl_get_obs(earl_handle* h, float* obs_dev, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!obs_dev || ((uintptr_t)obs_dev & 15u)) return fail(EARL_ERR_INVALID, "obs must be non-null and 16-byte aligned");
  const int grid = (h->p.n + 255) / 256;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (f64(h)) earl::tabletop_get_obs_kernel<true><<<grid, 256, 0, s>>>(h->p, obs_dev);
  else earl::tabletop_get_obs_kernel<false><<<grid, 256, 0, s>>>(h->p, obs_dev);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_compute_reward(earl_handle* h, const float* obs_dev, int64_t num_obs, float* reward_dev, uint8_t* success_dev,
                        void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!obs_dev || num_obs < 0 || ((uintptr_t)obs_dev & 15u)) return fail(EARL_ERR_INVALID, "bad obs buffer");
  if (num_obs == 0) return 0;
  const unsigned grid = (unsigned)((num_obs + 255) / 256);
  earl::tabletop_reward_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      obs_dev, num_obs, h->cfg.flags, h->p.success_sq, reward_dev, success_dev);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int earl_counters(earl_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev, uint32_t* steps_since_reset_dev,
                  double* lifelong_return_dev, void* stream) {
  if (int rc = check_handle(h)) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t n = (size_t)h->p.n;
  if (total_steps_host) *total_steps_host = h->total_steps;
  if (num_interventions_dev)
    CU(cudaMemcpyAsync(num_interventions_dev, h->p.interventions, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
  if (steps_since_reset_dev)  // strided copy of meta.y
    CU(cudaMemcpy2DAsync(steps_since_reset_dev, sizeof(uint32_t), reinterpret_cast<const uint32_t*>(h->p.meta) + 1,
                         sizeof(uint2), sizeof(uint32_t), n, cudaMemcpyDeviceToDevice, s));
  if (lifelong_return_dev) {
    if (!h->p.ll_return) return fail(EARL_ERR_INVALID, "lifelong_return needs EARL_FLAG_LIFELONG");
    CU(cudaMemcpyAsync(lifelong_return_dev, h->p.ll_return, n * sizeof(double), cudaMemcpyDeviceToDevice, s));
  }
  return 0;
}

int earl_eval_stats(earl_handle* h, double* out4_dev, void* stream) {
  if (int rc = check_handle(h)) return rc;
  if (!out4_dev) return fail(EARL_ERR_INVALID, "null out4");
  if (!h->p.ep_return) return fail(EARL_ERR_INVALID, "eval stats need EARL_FLAG_EVAL_STATS");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CU(cudaMemsetAsync(out4_dev, 0, 4 * sizeof(double), s));
  int grid = (h->p.n + 255) / 256;
  if (grid > h->sm_count * 4) grid = h->sm_count * 4;
  earl::tabletop_eval_stats_kernel<<<grid, 256, 0, s>>>(h->p, out4_dev);
  CU(cudaGetLastError());
  h->launches += 1;
  return 0;
}

// snapshot layout: SnapshotHeader | qpos f64[N,4] | flags u32[N] | steps_since_reset u32[N] |
//                  num_interventions i64[N] | goal_cursor u32[N] | ll_steps u32[N] | ll_return f64[N] | ep_return f64[N]
size_t earl_state_nbytes(const earl_handle* h) {
  if (!h) return 0;
  const size_t n = (size_t)h->cfg.num_envs;
  return sizeof(SnapshotHeader) + n * (32 + 4 + 4 + 8 + 4 + 4 + 8 + 8);
}

int earl_get_state(earl_handle* h, void* dst_host, size_t nbytes) {
  if (int rc = check_handle(h)) return rc;
  if (!dst_host || nbytes != earl_state_nbytes(h)) return fail(EARL_ERR_INVALID, "snapshot buffer must be %zu B", earl_state_nbytes(h));
  CU(cudaDeviceSynchronize());
  const size_t n = (size_t)h->p.n;
  uint8_t* w = static_cast<uint8_t*>(dst_host);
  SnapshotHeader hd{kSnapMagic, h->cfg.env_kind, h->cfg.num_envs, h->cfg.flags, h->total_steps};
  memcpy(w, &hd, sizeof(hd));
  w += sizeof(hd);
  double* q = reinterpret_cast<double*>(w);
  if (f64(h)) {
    CU(cudaMemcpy(q, h->p.qpos, n * 32, cudaMemcpyDeviceToHost));
  } else {
    std::vector<float> tmp(n * 4);
    CU(cudaMemcpy(tmp.data(), h->p.qpos, n * 16, cudaMemcpyDeviceToHost));
    for (size_t k = 0; k < n * 4; ++k) q[k] = (double)tmp[k];
  }
  w += n * 32;
  std::vector<uint2> meta(n);
  CU(cudaMemcpy(meta.data(), h->p.meta, n * sizeof(uint2), cudaMemcpyDeviceToHost));
  uint32_t* fl = reinterpret_cast<uint32_t*>(w);
  uint32_t* st = fl + n;
  for (size_t k = 0; k < n; ++k) { fl[k] = meta[k].x; st[k] = meta[k].y; }
  w += n * 8;
  CU(cudaMemcpy(w, h->p.interventions, n * 8, cudaMemcpyDeviceToHost));
  w += n * 8;
  CU(cudaMemcpy(w, h->p.goal_cursor, n * 4, cudaMemcpyDeviceToHost));
  w += n * 4;
  if (h->p.ll_steps) CU(cudaMemcpy(w, h->p.ll_steps, n * 4, cudaMemcpyDeviceToHost)); else memset(w, 0, n * 4);
  w += n * 4;
  if (h->p.ll_return) CU(cudaMemcpy(w, h->p.ll_return, n * 8, cudaMemcpyDeviceToHost)); else memset(w, 0, n * 8);
  w += n * 8;
  if (h->p.ep_return) CU(cudaMemcpy(w, h->p.ep_return, n * 8, cudaMemcpyDeviceToHost)); else memset(w, 0, n * 8);
  return 0;
}

int earl_set_state(earl_handle* h, const void* src_host, size_t nbytes) {
  if (int rc = check_handle(h)) return rc;
  if (!src_host || nbytes != earl_state_nbytes(h)) return fail(EARL_ERR_INVALID, "snapshot buffer must be %zu B", earl_state_nbytes(h));
  const uint8_t* r = static_cast<const uint8_t*>(src_host);
  SnapshotHeader hd;
  memcpy(&hd, r, sizeof(hd));
  if (hd.magic != kSnapMagic || hd.env_kind != h->cfg.env_kind || hd.num_envs != h->cfg.num_envs)
    return fail(EARL_ERR_INVALID, "snapshot does not match this handle (kind %d, N %d)", hd.env_kind, hd.num_envs);
  CU(cudaDeviceSynchronize());
  h->total_steps = hd.total_steps;
  r += sizeof(hd);
  const size_t n = (size_t)h->p.n;
  const double* q = reinterpret_cast<const double*>(r);
  if (f64(h)) {
    CU(cudaMemcpy(h->p.qpos, q, n * 32, cudaMemcpyHostToDevice));
  } else {
    std::vector<float> tmp(n * 4);
    for (size_t k = 0; k < n * 4; ++k) tmp[k] = (float)q[k];
    CU(cudaMemcpy(h->p.qpos, tmp.data(), n * 16, cudaMemcpyHostToDevice));
  }
  r += n * 32;
  const uint32_t* fl = reinterpret_cast<const uint32_t*>(r);
  const uint32_t* st = fl + n;
  std::vector<uint2> meta(n);
  for (size_t k = 0; k < n; ++k) {
    if (((fl[k] & earl::kGoalMask) >> earl::kGoalShift) >= (uint32_t)h->model.num_goals)
      return fail(EARL_ERR_INVALID, "snapshot env %zu has goal row out of range", k);
    meta[k] = make_uint2(fl[k], st[k]);
  }
  CU(cudaMemcpy(h->p.meta, meta.data(), n * sizeof(uint2), cudaMemcpyHostToDevice));
  r += n * 8;
  CU(cudaMemcpy(h->p.interventions, r, n * 8, cudaMemcpyHostToDevice));
  r += n * 8;
  CU(cudaMemcpy(h->p.goal_cursor, r, n * 4, cudaMemcpyHostToDevice));
  r += n * 4;
  if (h->p.ll_steps) CU(cudaMemcpy(h->p.ll_steps, r, n * 4, cudaMemcpyHostToDevice));
  r += n * 4;
  if (h->p.ll_return) CU(cudaMemcpy(h->p.ll_return, r, n * 8, cudaMemcpyHostToDevice));
  r += n * 8;
  if (h->p.ep_return) CU(cudaMemcpy(h->p.ep_return, r, n * 8, cudaMemcpyHostToDevice));
  return 0;
}

// ------------------------------------------------------------------------------------------ host RNG streams

struct earl_rng {
  earl::MT19937 mt;
};

earl_rng* earl_rng_create(int32_t kind, const uint32_t* seed_limbs, int32_t num_limbs) {
  if (!seed_limbs || num_limbs < 1 || (kind != 0 && kind != 1)) { fail(EARL_ERR_INVALID, "bad rng arguments"); return nullptr; }
  earl_rng* r = new (std::nothrow) earl_rng();
  if (!r) return nullptr;
  if (kind == 0) r->mt.init_by_array(seed_limbs, num_limbs);
  else r->mt.init_genrand(seed_limbs[0]);
  return r;
}

void earl_rng_destroy(earl_rng* r) { delete r; }

uint32_t earl_rng_next_u32(earl_rng* r) { return r->mt.next(); }

void earl_rng_py_randbelow(earl_rng* r, uint32_t n, int64_t count, int32_t* out) {
  for (int64_t k = 0; k < count; ++k) out[k] = (int32_t)r->mt.py_randbelow(n);
}

void earl_rng_tabletop_goal_rows(earl_rng* r, const uint8_t* task_to_row, uint32_t num_tasks, int64_t count, uint8_t* out) {
  for (int64_t k = 0; k < count; ++k) out[k] = task_to_row[r->mt.py_randbelow(num_tasks)];
}

void earl_rng_np_randint(earl_rng* r, uint32_t n, int64_t count, int32_t* out) {
  for (int64_t k = 0; k < count; ++k) out[k] = (int32_t)r->mt.np_randint(n);
}

void earl_rng_np_uniform(earl_rng* r, double low, double high, int64_t count, double* out) {
  for (int64_t k = 0; k < count; ++k) out[k] = low + (high - low) * r->mt.np_double();
}

// Replays envs/sawyer_peg.py SawyerPegV2._draw_one (reference sawyer_peg.py:144-152,192-229) with the same double operations
// in the same order, so the results are bit-identical with the numpy arithmetic there.
void earl_rng_peg_reset_draws(earl_rng* r, int32_t wide_init, int32_t reset_at_goal, int64_t count, int32_t* rows_out, double* pos_out) {
  // _random_reset_space = (obj_low, goal_low) .. (obj_high, goal_high), sawyer_peg.py:64-69,102-105
  static const double lo[6] = {0.0, 0.5, 0.02, -0.35, 0.4, -0.001}, hi[6] = {0.2, 0.7, 0.02, -0.25, 0.7, 0.001};
  // wide_initial_states (sawyer_peg.py:50-58)
  static const double wide[22][3] = {{-0.3, 0.8, 0.02}, {-0.4, 0.8, 0.02}, {-0.3, 0.9, 0.02}, {-0.4, 0.9, 0.02}, {-0.2, 0.8, 0.02},
                                     {-0.2, 0.75, 0.02}, {-0.2, 0.9, 0.02}, {-0.1, 0.77, 0.02}, {0.0, 0.9, 0.02}, {0.1, 0.8, 0.02},
                                     {0.15, 0.75, 0.02}, {-0.3, 0.4, 0.02}, {-0.4, 0.4, 0.02}, {-0.3, 0.45, 0.02}, {-0.4, 0.45, 0.02},
                                     {-0.2, 0.4, 0.02}, {-0.2, 0.45, 0.02}, {-0.2, 0.38, 0.02}, {-0.1, 0.42, 0.02}, {0.0, 0.45, 0.02},
                                     {0.1, 0.36, 0.02}, {0.15, 0.44, 0.02}};
  const double goal[3] = {-0.3 + 0.03, 0.6, 0.0 + 0.13};                   // goal_states[0][4:] (sawyer_peg.py:46)
  const double box[2] = {goal[0] - 0.03, goal[1] - 0.0};                    // pos_box[:2] = goal[4:] - (0.03, 0, 0.13)
  earl::MT19937& mt = r->mt;
  auto uniform = [&](double l, double h) { return l + (h - l) * mt.np_double(); };
  auto sample_peg = [&](double* p) {  // _get_state_rand_vec()[:3], redrawn while ||p[:2] - box|| < 0.1
    for (;;) {
      double u[6];
      for (int k = 0; k < 6; ++k) u[k] = uniform(0.0, 1.0);
      for (int k = 0; k < 3; ++k) p[k] = lo[k] + (hi[k] - lo[k]) * u[k];
      const double dx = p[0] - box[0], dy = p[1] - box[1];
      if (!(std::sqrt(dx * dx + dy * dy) < 0.1)) return;
    }
  };
  for (int64_t i = 0; i < count; ++i) {
    double* p = pos_out + 3 * i;
    int row = 0;
    if (!reset_at_goal) {
      mt.np_randint(1);  // get_next_goal() over one goal: consumes nothing
      if (wide_init) {
        if (uniform(0.0, 1.0) < 0.5) {
          sample_peg(p);
        } else {
          const uint32_t k = mt.np_randint(22);
          const double base[3] = {wide[k][0] - -0.1, wide[k][1] - 0.0, wide[k][2] - 0.0};
          for (int c = 0; c < 3; ++c) p[c] = base[c] + uniform(-0.02, 0.02);
        }
      } else {
        sample_peg(p);  // random_init
      }
    } else {
      row = 1 + (int)mt.np_randint(15);
      const double base[3] = {goal[0] - -0.1, goal[1] - 0.0, goal[2] - 0.0};
      for (int c = 0; c < 3; ++c) p[c] = base[c] + uniform(-0.02, 0.02);
    }
    rows_out[i] = row;
  }
}

}  // extern "C"
