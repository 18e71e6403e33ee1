// tabletop_kernels.cuh -- sm_100a kernels for the batched tabletop_manipulation step.
//
// What is computed (reference, paths relative to the reference root):
//   envs/tabletop_manipulation.py:128-174  step + move         (action rescale, attach, drag, clip)
//   envs/tabletop_manipulation.py:55-60    _get_obs
//   envs/tabletop_manipulation.py:176-204  compute_reward / is_successful
//   wrappers/persistent_state_wrapper.py:22-31  counters + reset-free horizon `done`
//   wrappers/lifelong_wrapper.py:30-44     lifelong return + periodic goal swap
//
// Shape of the work: ~40 flops and 113 B of HBM traffic per env-step, no reuse, no cross-env coupling
// => a pure HBM-streaming kernel.  One thread per environment instance, state in structure-of-arrays
// form so every warp-level access is one or a few full 128-B lines:
//     qpos   float4[N]  (or 2x double2[N] with EARL_FLAG_STATE_F64)   16 B r + 16 B w
//     meta   uint2[N]   {flags: bit0 attached, bit1 success-any, bit2 success-last, bits 8..15 goal row;
//                        steps_since_reset (saturating u32)}           8 B r +  8 B w
//     action float[N,3] read once (streaming, no L1 allocate)         12 B r
//     obs    float[N,12] written once; rows are staged through shared memory so each warp issues three
//                        fully coalesced 512-B st.global.cs.v4        48 B w
//     reward float[N], done u8[N] (streaming stores)                    5 B w
// Arithmetic follows the reference bit for bit: the position update is evaluated in fp64 with explicit
// round-to-nearest intrinsics (no FMA contraction) and rounded ONCE to fp32 for the observation; the
// success norm is evaluated in fp32 on that observation and compared with 0.2 in fp64.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "eval_stats.cuh"

namespace earl {

constexpr int kTTBlock = 256;            // threads per CTA (8 warps)
constexpr int kTTObs = 12;
constexpr int kTTAct = 3;

// meta.x bit layout
constexpr uint32_t kAttached = 1u;
constexpr uint32_t kSuccessAny = 2u;
constexpr uint32_t kSuccessLast = 4u;
constexpr uint32_t kGoalShift = 8u;
constexpr uint32_t kGoalMask = 0xffu << kGoalShift;

// feature bits (mirror EARL_FLAG_*)
constexpr uint32_t kDense = 0x01u, kWide = 0x02u, kF64 = 0x04u, kLifelong = 0x08u, kAutoReset = 0x10u,
                   kResetAtGoal = 0x20u, kEvalStats = 0x40u, kPerEnvGoals = 0x80u;

struct TabletopParams {
  // hot state
  void* qpos;        // float4[N] | double[N][4]
  uint2* meta;       // {flags, steps_since_reset}
  // optional hot state
  uint32_t* ll_steps;   // steps_since_goal_change   (lifelong)
  double* ll_return;    // lifelong_return           (lifelong)
  double* ep_return;    // episode return            (eval stats)
  // cold state
  long long* interventions;    // num_interventions
  uint32_t* goal_cursor;       // goal-stream draws taken so far
  const uint8_t* goal_stream;  // [R,N] pre-drawn goal rows
  const float4* goal32;        // [256][2] goal rows as fp32, padded to 8 floats
  const double* goal64;        // [256][6]
  // io of this launch
  const float* actions;  // [N,3]
  float* obs;            // [N,12]
  float* reward;         // [N]
  uint8_t* done;         // [N]
  uint8_t* success;      // [N] or null
  int n;        // one past the last env this launch touches (chunked host path: first + count)
  int n_total;  // envs of the handle = row stride of goal_stream[R,N]; never changes with the chunk (ADVICE r1: a chunked
                // launch used `n` as the stride and read other envs' draws)
  int first;  // first env this launch touches (chunked host path); multiple of 32
              // the launch covers envs [first, n)
  int goal_stream_rows;
  uint32_t features;
  unsigned long long horizon;
  unsigned long long goal_change_frequency;
  // constants of the task (earl_tabletop_model)
  double act_lo, act_span;  // -move_distance, move_distance - (-move_distance)
  double threshold, clip, success_radius;
  // sqrt-free forms of the two radius tests, exact by monotonicity of correctly rounded sqrt (computed on
  // the host by earl_tabletop_thresholds): sqrt(s) < threshold <=> s < attach_sq;
  // (double)sqrtf(s) <= success_radius <=> s <= success_sq
  double attach_sq;
  float success_sq;
  double init_qpos[4];
  // EARL_FLAG_PER_ENV_GOALS: the goal each env pursues, [N][2] float4 (goal[0:4], goal[4:6] + 2 pad), null otherwise.
  // Every assignment of a goal row (reset, reset_goal, lifelong swap, auto-reset) also copies that row here.
  float4* env_goal;
};

// Programmatic dependent launch: step t+1 may be scheduled while step t drains; nothing of the state is
// touched before the previous grid has completed and flushed (griddepcontrol.wait).  Both are no-ops
// for launches without the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_wait_prior_grid() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

__device__ __forceinline__ double clipd(double x, double lo, double hi) {
  // np.clip: NaN propagates (both comparisons false)
  return x < lo ? lo : (x > hi ? hi : x);
}

// np.linalg.norm on fp32 data: fp32 products and sums in index order, fp32 sqrt, nothing fused
__device__ __forceinline__ float norm2_f32(float a, float b) {
  return __fsqrt_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)));
}

// is_successful on an fp32 observation (tabletop_manipulation.py:197-204): fp32 products summed in index
// order in fp64 and rounded to fp32 (what np.linalg.norm does), nothing fused; `success_sq` is the exact sqrt-free threshold (see TabletopParams)
__device__ __forceinline__ bool tt_success(const float4& pos, const float4& g0, bool wide, float success_sq) {
  // pos = obs[0:4]; g0 = obs[6:10] = goal[0:4]
  const float dz = __fsub_rn(pos.z, g0.z), dw = __fsub_rn(pos.w, g0.w);
  float s;
  if (wide) {
    s = __fadd_rn(__fmul_rn(dz, dz), __fmul_rn(dw, dw));
  } else {
    // numpy's fp32 dot accumulates the fp32 products in fp64 and rounds once (OpenBLAS sdot; DESIGN.md section 10):
    // with two terms that equals the fp32 sum above, with four it does not
    const float dx = __fsub_rn(pos.x, g0.x), dy = __fsub_rn(pos.y, g0.y);
    double acc = __dadd_rn((double)__fmul_rn(dx, dx), (double)__fmul_rn(dy, dy));
    acc = __dadd_rn(acc, (double)__fmul_rn(dz, dz));
    acc = __dadd_rn(acc, (double)__fmul_rn(dw, dw));
    s = (float)acc;
  }
  return s <= success_sq;
}

// dense reward (tabletop_manipulation.py:179-189), fp64 after the fp32 norms as numpy 1.22 evaluates it
__device__ __forceinline__ double tt_dense_reward(const float4& pos, const float4& g0) {
  float n1 = norm2_f32(__fsub_rn(pos.z, g0.z), __fsub_rn(pos.w, g0.w));
  double r = (double)(-n1);
  r += 2.0 * exp(-((double)n1 * (double)n1) / 0.01);
  double g = 0.5 * (double)norm2_f32(__fsub_rn(pos.x, pos.z), __fsub_rn(pos.y, pos.w));
  r += -g;
  r += 0.5 * exp(-(g * g) / 0.01);
  return r;
}

struct TTState {
  double fx, fy, mx, my;
  uint32_t flags;
};

// step() + move(): tabletop_manipulation.py:128-174.  Updates s in place.
__device__ __forceinline__ void tt_move(TTState& s, float a0f, float a1f, float a2f, const TabletopParams& p) {
  const double a0 = __dadd_rn(p.act_lo, __dmul_rn(__dmul_rn(__dadd_rn(clipd((double)a0f, -1.0, 1.0), 1.0), 0.5), p.act_span));
  const double a1 = __dadd_rn(p.act_lo, __dmul_rn(__dmul_rn(__dadd_rn(clipd((double)a1f, -1.0, 1.0), 1.0), 0.5), p.act_span));
  const double a2 = __dadd_rn(p.act_lo, __dmul_rn(__dmul_rn(__dadd_rn(clipd((double)a2f, -1.0, 1.0), 1.0), 0.5), p.act_span));
  bool attached = s.flags & kAttached;
  if (a2 > 0.0) {
    if (!attached) {
      // dist = np.linalg.norm(fist - mug) < threshold, on the PRE-move positions (:144-152)
      const double dx = __dsub_rn(s.fx, s.mx), dy = __dsub_rn(s.fy, s.my);
      attached = __fma_rn(dy, dy, __dmul_rn(dx, dx)) < p.attach_sq;  // == sqrt(.) < threshold, exactly
    }
  } else {
    attached = false;
  }
  const double nfx = clipd(__dadd_rn(s.fx, a0), -p.clip, p.clip);
  const double nfy = clipd(__dadd_rn(s.fy, a1), -p.clip, p.clip);
  if (attached) {  // the mug moves by the CLIPPED fist delta (:158-163)
    s.mx = clipd(__dadd_rn(s.mx, __dsub_rn(nfx, s.fx)), -p.clip, p.clip);
    s.my = clipd(__dadd_rn(s.my, __dsub_rn(nfy, s.fy)), -p.clip, p.clip);
  }
  s.fx = nfx;
  s.fy = nfy;
  s.flags = (s.flags & ~kAttached) | (attached ? kAttached : 0u);
}

template <bool F64>
__device__ __forceinline__ void tt_load_state(const TabletopParams& p, int i, TTState& s, uint32_t& steps) {
  if (F64) {
    const double2* q = reinterpret_cast<const double2*>(p.qpos) + 2 * (size_t)i;
    double2 f = q[0], m = q[1];
    s.fx = f.x; s.fy = f.y; s.mx = m.x; s.my = m.y;
  } else {
    float4 q = reinterpret_cast<const float4*>(p.qpos)[i];
    s.fx = q.x; s.fy = q.y; s.mx = q.z; s.my = q.w;
  }
  uint2 m = p.meta[i];
  s.flags = m.x;
  steps = m.y;
}

template <bool F64>
__device__ __forceinline__ void tt_store_state(const TabletopParams& p, int i, const TTState& s, const float4& pos32,
                                               uint32_t steps) {
  if (F64) {
    double2* q = reinterpret_cast<double2*>(p.qpos) + 2 * (size_t)i;
    q[0] = make_double2(s.fx, s.fy);
    q[1] = make_double2(s.mx, s.my);
  } else {
    reinterpret_cast<float4*>(p.qpos)[i] = pos32;  // the fp32 state IS the observation
  }
  p.meta[i] = make_uint2(s.flags, steps);
}

// Warp-cooperative store of 32 observation rows (48 B each) staged in shared memory:
// three st.global.cs.v4 per lane, each covering 512 contiguous bytes per warp.
__device__ __forceinline__ void tt_store_obs_tile(float* __restrict__ obs, const float* tile, int warp_base, int n,
                                                  int lane) {
  const int cnt = min(32, n - warp_base);  // envs of this warp that exist
  float4* dst = reinterpret_cast<float4*>(obs + (size_t)warp_base * kTTObs);
  const float4* src = reinterpret_cast<const float4*>(tile);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int idx = lane + 32 * k;
    if (idx < cnt * 3) __stcs(dst + idx, src[idx]);
  }
}

// The hot kernel.  FAST = sparse reward, no lifelong / auto-reset / eval-stats (the headline config);
// the general instantiation handles every feature with warp-uniform runtime branches.  GOALS (general kernel only) =
// EARL_FLAG_PER_ENV_GOALS: each env's goal is streamed from p.env_goal (+32 B read per env step) instead of being
// looked up in the goal table through the row in meta.
template <bool F64, bool FAST, int MINB = 1, bool GOALS = false>
__global__ void __launch_bounds__(kTTBlock, MINB) tabletop_step_kernel(const TabletopParams p) {
  constexpr bool FINAL = false;
  float* const final_obs = nullptr;
#include "tabletop_step_body.inc"
}

// EARL_FLAG_FINAL_OBS handles (general kernel, FINAL = true): the fused auto-reset first stores the env's pre-reset
// observation row to final_obs [N,12].  An overload with one more template parameter and the buffer as a second argument,
// sharing the body above textually: the kernels of every other handle keep their symbol names, parameter layout and code
// (moving the body into an inlined device function reorders their registers).
template <bool F64, bool FAST, int MINB, bool GOALS, bool FINAL>
__global__ void __launch_bounds__(kTTBlock, MINB) tabletop_step_kernel(const TabletopParams p, float* final_obs) {
#include "tabletop_step_body.inc"
}

// ------------------------------------------------------------------------------------------ tile kernel
// The same FAST step (sparse reward, fp32 state, no lifelong / auto-reset / eval-stats) as ONE 256-env TILE PER CTA:
// not persistent, so the grid is N / 256 independent blocks that the hardware scheduler spreads over the 148 SMs as
// they finish (no tail imbalance, 8 CTAs resident per SM).  State (float4 qpos, uint2 meta) moves as fully coalesced 16 /
// 8-byte accesses; the tile's 3 KB of row-major actions and 12 KB of row-major observations are staged through shared
// memory so every global access is a contiguous float4 (observation slot 3*t + j: conflict-free for 16-byte accesses,
// gcd(3, 8) = 1).  This is the design that reached 0.98 of the HBM copy peak on the three-object task (csrc/earl_tt3.cu);
// it replaces the cp.async.bulk pipeline (0.93-0.95) and the persistent LSU kernel (0.87-0.88) above ~3M envs, where
// nothing is L2-resident (VERDICT r1, item 5).
// VEC: reward / done / success are staged through shared memory and leave as 16-byte vectors (the zero-copy host step, whose
// outputs are pinned host memory behind a PCIe link); the device-resident step writes them per env (0.7 % faster on HBM).
template <bool VEC>
__global__ void __launch_bounds__(kTTBlock, 8) tabletop_step_tile_kernel(const __grid_constant__ TabletopParams p) {
  __shared__ float4 s_obs[kTTBlock * 3];
  __shared__ float4 s_act4[kTTBlock * kTTAct / 4];
  __shared__ float4 s_rew4[kTTBlock / 4];
  __shared__ uint4 s_done16[kTTBlock / 16], s_succ16[kTTBlock / 16];
  float* s_act = reinterpret_cast<float*>(s_act4);
  float* s_rew = reinterpret_cast<float*>(s_rew4);
  uint8_t* s_done = reinterpret_cast<uint8_t*>(s_done16);
  uint8_t* s_succ = reinterpret_cast<uint8_t*>(s_succ16);
  const int t = threadIdx.x;
  const int base = p.first + blockIdx.x * kTTBlock;
  const int i = base + t;
  const int rows = min(kTTBlock, p.n - base);
  const bool wide = p.features & kWide;
  pdl_wait_prior_grid();
  {
    const float* asrc = p.actions + (size_t)base * kTTAct;
    if ((reinterpret_cast<uintptr_t>(asrc) & 15u) == 0) {
      const float4* src = reinterpret_cast<const float4*>(asrc);
      const int full = rows * kTTAct / 4;
      if (t < full) s_act4[t] = __ldcs(src + t);
      const int rem = rows * kTTAct - full * 4;
      if (t < rem) s_act[full * 4 + t] = asrc[full * 4 + t];
    } else {
      for (int k = t; k < rows * kTTAct; k += kTTBlock) s_act[k] = asrc[k];
    }
  }
  __syncthreads();
  if (i < p.n) {
    TTState s;
    uint32_t steps;
    tt_load_state<false>(p, i, s, steps);
    const uint32_t gi = (s.flags & kGoalMask) >> kGoalShift;
    const float4 g0 = __ldg(p.goal32 + 2 * gi), g1 = __ldg(p.goal32 + 2 * gi + 1);
    tt_move(s, s_act[kTTAct * t], s_act[kTTAct * t + 1], s_act[kTTAct * t + 2], p);
    const float4 pos32 = make_float4(__double2float_rn(s.fx), __double2float_rn(s.fy), __double2float_rn(s.mx),
                                     __double2float_rn(s.my));
    const bool succ = tt_success(pos32, g0, wide, p.success_sq);
    steps = steps == 0xffffffffu ? steps : steps + 1u;   // PersistentStateWrapper.step (persistent_state_wrapper.py:25-29)
    tt_store_state<false>(p, i, s, pos32, steps);
    if (VEC) {
      s_rew[t] = succ ? 1.f : 0.f;
      s_done[t] = (unsigned long long)steps >= p.horizon ? 1 : 0;
      s_succ[t] = succ ? 1 : 0;
    } else {
      __stcs(p.reward + i, succ ? 1.f : 0.f);
      p.done[i] = (unsigned long long)steps >= p.horizon ? 1 : 0;
      if (p.success) p.success[i] = succ ? 1 : 0;
    }
    const float att = (s.flags & kAttached) ? 0.f : -1.f;
    s_obs[3 * t] = pos32;                                  // tabletop_manipulation.py:55-60
    s_obs[3 * t + 1] = make_float4(att, att, g0.x, g0.y);
    s_obs[3 * t + 2] = make_float4(g0.z, g0.w, g1.x, g1.y);
  }
  __syncthreads();
  float4* dst = reinterpret_cast<float4*>(p.obs + (size_t)base * kTTObs);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int idx = t + kTTBlock * k;
    if (idx < rows * 3) __stcs(dst + idx, s_obs[idx]);
  }
  // reward (4 B), done and success (1 B per env) leave as 16-byte vectors too: a whole tile is 1 KB + 256 B + 256 B of
  // contiguous full lines instead of 32-byte warp stores -- what a PCIe link wants when the outputs are pinned host memory
  // (earl_step_host, zero-copy path), and fewer store instructions on HBM.  Ragged tile or unaligned buffers: one env each.
  if (!VEC) return;
  const bool vec = rows == kTTBlock &&
                   !((reinterpret_cast<uintptr_t>(p.reward) | reinterpret_cast<uintptr_t>(p.done) | reinterpret_cast<uintptr_t>(p.success)) & 15u);
  if (vec) {
    if (t < kTTBlock / 4) __stcs(reinterpret_cast<float4*>(p.reward + base) + t, s_rew4[t]);
    else if (t < kTTBlock / 4 + kTTBlock / 16) __stcs(reinterpret_cast<uint4*>(p.done + base) + (t - kTTBlock / 4), s_done16[t - kTTBlock / 4]);
    else if (t < kTTBlock / 4 + kTTBlock / 8 && p.success)
      __stcs(reinterpret_cast<uint4*>(p.success + base) + (t - kTTBlock / 4 - kTTBlock / 16), s_succ16[t - kTTBlock / 4 - kTTBlock / 16]);
  } else if (i < p.n) {
    __stcs(p.reward + i, s_rew[t]);
    p.done[i] = s_done[t];
    if (p.success) p.success[i] = s_succ[t];
  }
}

// ------------------------------------------------------------------------------------------ cold kernels

struct TabletopResetArgs {
  const uint8_t* mask;       // [N] or null
  const int32_t* goal_idx;   // [N] or null -> goal stream
  const double* init_qpos;   // [N,4] or null
  float* obs_out;            // [N,12] or null
  int set_goal_only;         // reset_goal(): only the goal changes
};

template <bool F64>
__global__ void tabletop_reset_kernel(const TabletopParams p, const TabletopResetArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  if (a.mask && !a.mask[i]) return;
  TTState s;
  uint32_t steps;
  tt_load_state<F64>(p, i, s, steps);
  uint32_t gi;
  if (a.goal_idx) {
    gi = (uint32_t)a.goal_idx[i] & 0xffu;
  } else {
    const uint32_t c = p.goal_cursor[i];
    gi = p.goal_stream[(size_t)(c % (uint32_t)p.goal_stream_rows) * p.n_total + i];
    p.goal_cursor[i] = c + 1u;
  }
  if (p.env_goal) {  // the assigned row replaces any goal set with earl_set_goals
    p.env_goal[2 * (size_t)i] = p.goal32[2 * gi];
    p.env_goal[2 * (size_t)i + 1] = p.goal32[2 * gi + 1];
  }
  if (a.set_goal_only) {
    s.flags = (s.flags & ~kGoalMask) | (gi << kGoalShift);
  } else {
    s.flags = gi << kGoalShift;  // attached_object = (-1,-1), success bits cleared
    steps = 0u;
    p.interventions[i] += 1;
    if (a.init_qpos) {
      const double* q = a.init_qpos + 4 * (size_t)i;
      s.fx = q[0]; s.fy = q[1]; s.mx = q[2]; s.my = q[3];
    } else if (p.features & kResetAtGoal) {
      const double* g = p.goal64 + 6 * gi;
      s.fx = g[0]; s.fy = g[1]; s.mx = g[2]; s.my = g[3];
    } else {
      s.fx = p.init_qpos[0]; s.fy = p.init_qpos[1]; s.mx = p.init_qpos[2]; s.my = p.init_qpos[3];
    }
    if (p.features & kLifelong) p.ll_steps[i] = 0u;
    if (p.features & kEvalStats) p.ep_return[i] = 0.0;
  }
  const float4 pos32 = make_float4(__double2float_rn(s.fx), __double2float_rn(s.fy), __double2float_rn(s.mx),
                                   __double2float_rn(s.my));
  tt_store_state<F64>(p, i, s, pos32, steps);
  if (a.obs_out) {
    const float4 g0 = p.goal32[2 * gi], g1 = p.goal32[2 * gi + 1];
    const float att = (s.flags & kAttached) ? 0.f : -1.f;
    float4* row = reinterpret_cast<float4*>(a.obs_out + (size_t)i * kTTObs);
    row[0] = pos32;
    row[1] = make_float4(att, att, g0.x, g0.y);
    row[2] = make_float4(g0.z, g0.w, g1.x, g1.y);
  }
}

template <bool F64>
__global__ void tabletop_get_obs_kernel(const TabletopParams p, float* __restrict__ obs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  TTState s;
  uint32_t steps;
  tt_load_state<F64>(p, i, s, steps);
  const uint32_t gi = (s.flags & kGoalMask) >> kGoalShift;
  const float4* g = p.env_goal ? p.env_goal + 2 * (size_t)i : p.goal32 + 2 * gi;
  const float4 g0 = g[0], g1 = g[1];
  const float att = (s.flags & kAttached) ? 0.f : -1.f;
  float4* row = reinterpret_cast<float4*>(obs + (size_t)i * kTTObs);
  row[0] = make_float4(__double2float_rn(s.fx), __double2float_rn(s.fy), __double2float_rn(s.mx),
                       __double2float_rn(s.my));
  row[1] = make_float4(att, att, g0.x, g0.y);
  row[2] = make_float4(g0.z, g0.w, g1.x, g1.y);
}

// earl_set_goals: env i (mask[i] != 0, or every env when mask is null) pursues goals[i * goal_stride .. + 6] from now on,
// fp64 input rounded to fp32 as the goal-table upload rounds it; then the observation row of EVERY env (the current one
// for envs outside the mask) goes to obs_out when it is non-null.  The goal row in meta is left alone: it is what the
// snapshot records, and the next row assignment overrides the custom goal.
struct TabletopGoalArgs {
  const void* goals;   // f32 or f64 [N][goal_stride]
  int goal_f64;
  int goal_stride;     // 6, or 0 = the same goal for every env
  const uint8_t* mask;
  float* obs_out;
};

template <bool F64>
__global__ void tabletop_set_goals_kernel(const TabletopParams p, const TabletopGoalArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  float4 g0, g1;
  if (!a.mask || a.mask[i]) {
    float v[6];
    const size_t at = (size_t)a.goal_stride * i;
#pragma unroll
    for (int k = 0; k < 6; ++k)
      v[k] = a.goal_f64 ? __double2float_rn(static_cast<const double*>(a.goals)[at + k]) : static_cast<const float*>(a.goals)[at + k];
    g0 = make_float4(v[0], v[1], v[2], v[3]);
    g1 = make_float4(v[4], v[5], 0.f, 0.f);
    p.env_goal[2 * (size_t)i] = g0;
    p.env_goal[2 * (size_t)i + 1] = g1;
  } else {
    if (!a.obs_out) return;
    g0 = p.env_goal[2 * (size_t)i];
    g1 = p.env_goal[2 * (size_t)i + 1];
  }
  if (!a.obs_out) return;
  TTState s;
  uint32_t steps;
  tt_load_state<F64>(p, i, s, steps);
  const float att = (s.flags & kAttached) ? 0.f : -1.f;
  float4* row = reinterpret_cast<float4*>(a.obs_out + (size_t)i * kTTObs);
  row[0] = make_float4(__double2float_rn(s.fx), __double2float_rn(s.fy), __double2float_rn(s.mx), __double2float_rn(s.my));
  row[1] = make_float4(att, att, g0.x, g0.y);
  row[2] = make_float4(g0.z, g0.w, g1.x, g1.y);
}

// compute_reward(obs) / is_successful(obs) on caller-supplied observations
__global__ void tabletop_reward_kernel(const float* __restrict__ obs, long long m, uint32_t features, float success_sq,
                                       float* __restrict__ reward, uint8_t* __restrict__ success) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const float4* row = reinterpret_cast<const float4*>(obs + i * kTTObs);
  const float4 pos = row[0], r1 = row[1], r2 = row[2];
  const float4 g0 = make_float4(r1.z, r1.w, r2.x, r2.y);
  const bool succ = tt_success(pos, g0, features & kWide, success_sq);
  if (reward) reward[i] = (features & kDense) ? (float)tt_dense_reward(pos, g0) : (succ ? 1.f : 0.f);
  if (success) success[i] = succ ? 1 : 0;
}

// (sum episode return, #success at last step, #success at any step, N) -> out4 (pre-zeroed)
__global__ void tabletop_eval_stats_kernel(const TabletopParams p, double* __restrict__ out4) {
  double ret = 0.0, last = 0.0, any = 0.0, cnt = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += gridDim.x * blockDim.x) {
    const uint32_t f = p.meta[i].x;
    ret += p.ep_return[i];
    last += (f & kSuccessLast) ? 1.0 : 0.0;
    any += (f & kSuccessAny) ? 1.0 : 0.0;
    cnt += 1.0;
  }
  block_add_eval_stats(ret, last, any, cnt, out4);
}

}  // namespace earl
