// earl_mj_kitchen.cu -- the kitchen capacity set of the articulated-body engine (24 dofs, 128 geoms, 112 rows, 24
// contacts; joint-equality / friction-loss / pyramidal rows, capsule geoms) and its ENGINE-LEVEL entry points
// (include/earl_mj_kitchen_b200.h).  One warp per environment; the 27.1 KB workspace of an environment lives in shared
// memory (8 environments in flight per SM), the 37 KB model stays in global memory (L1 / L2 resident: every block reads
// the same tables).  No CPU fallback.
//
// Compiled a second time as earl_mj_kitchen_xl.cu (MJK_XL: 544 rows, 48 contacts, 2 environments per block) for the
// REDO PASS: an env step in which some substep outgrew the 112 rows / 24 contacts (~0.1 % of them) is not stored by the
// step kernel but listed, and re-stepped from its untouched state by the extra-large instantiation, which runs
// CONCURRENTLY on four SMs the step kernel leaves free (programmatic dependent launch; it polls the list and the step
// kernel's exit counter).
#define MJ_CAPSET_KITCHEN 1
#ifdef MJK_XL
#define MJ_CAPSET_KITCHEN_XL 1
#define mj mjkx  // engine namespace of this translation unit: no symbol is shared with any other capacity set
#else
#define mj mjk
// the 8 warps of a block keep in phase in two groups of 4 (two named barriers): less waiting for the slowest warp, and the
// kitchen's phases still fit the instruction caches twice (measured 1.54e5 -> 1.60e5 env-steps/s; the door / peg sets lose
// 19 % with the same split: their 16 warps per SM want one phase resident)
#ifndef MJ_BARRIER_DOMAINS
#define MJ_BARRIER_DOMAINS 2
#endif
#endif
#include "../../include/earl_mj_kitchen_b200.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "mj_model_host.hpp"
#include "mj_step.cuh"

namespace earl {
int set_error(int code, const char* msg);  // earl_b200.cu
}

namespace {

using namespace earl::mj;

int failf(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return earl::set_error(code, buf);
}
#define CU(call)                                                                                                 \
  do {                                                                                                           \
    cudaError_t e_ = (call);                                                                                     \
    if (e_ != cudaSuccess)                                                                                       \
      return failf(EARL_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);    \
  } while (0)

#ifndef MJK_WPB
#ifdef MJK_XL
#define MJK_WPB 2
#else
#define MJK_WPB 8
#endif
#endif
#ifndef MJK_BPS
#define MJK_BPS 1
#endif
constexpr int kWPB = MJK_WPB;  // warps (= environments in flight) per block
constexpr int kBPS = MJK_BPS;  // resident blocks per SM (each block is one phase-barrier domain)
constexpr size_t kWorkStride = (sizeof(Work) + 15) & ~size_t(15);
constexpr size_t kSmemBytes = kWPB * kWorkStride;
static_assert(kBPS * (kSmemBytes + 1024) <= 228 * 1024, "workspaces exceed the shared memory of an SM");
#if defined(MJ_BARRIER_DOMAINS)
static_assert(kWPB % MJ_BARRIER_DOMAINS == 0, "barrier domains must divide the warps of a block");
#endif

// All warps of a block walk the same number of environments and substeps (the engine's phase barriers are block-wide);
// a warp without an environment of its own shadows the last one and stores nothing.  Primary set: environments whose
// substeps outgrow the capacities keep their input state and are flagged in info[:, 3]; the extra-large instantiation
// (only_flagged 1) then walks the flagged ones.  only_flagged 2: primary set, everything stored (EARL_MJ_REDO=0).
__global__ void __launch_bounds__(kWPB * 32, 1)
mjk_substeps_kernel(const Model* __restrict__ gm, const real* __restrict__ hull, int n, int nsub, float* qpos, float* qvel, float* warm,
                    const double* mocap_pos, float4 mocap_quat, const float* ctrl, int* info, int only_flagged) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Work& w = *reinterpret_cast<Work*>(smem + warp * kWorkStride);
  const Model& m = *gm;
  const int nq = m.nq, nv = m.nv;
  for (int base = blockIdx.x * kWPB; base < n; base += gridDim.x * kWPB) {
    bool own = base + warp < n;
    const int env = own ? base + warp : n - 1;
    if (only_flagged == 1) {
      own = own && (info[4 * env + 3] & 14);
      if (!__syncthreads_or(own)) continue;
    }
    for (int k = lane; k < nq; k += 32) w.qpos[k] = qpos[(size_t)env * nq + k];
    for (int k = lane; k < nv; k += 32) { w.qvel[k] = qvel[(size_t)env * nv + k]; w.warm[k] = warm[(size_t)env * nv + k]; }
    if (lane == 0) {
      for (int k = 0; k < 3; ++k) w.mocap_pos[k] = mocap_pos[(size_t)env * 3 + k];
      w.mocap_quat[0] = mocap_quat.x; w.mocap_quat[1] = mocap_quat.y; w.mocap_quat[2] = mocap_quat.z; w.mocap_quat[3] = mocap_quat.w;
      for (int k = 0; k < m.nu; ++k) w.ctrl[k] = ctrl[(size_t)env * m.nu + k];
      w.bad = 0; w.acc_iter = w.acc_rows = w.acc_con = w.acc_mpr = w.acc_sup = 0; w.broad_valid = 0; w.acc_rebuild = 0; w.peak_efc = w.peak_con = w.peak_hit = 0;
    }
    __syncwarp();
    for (int s = 0; s < nsub; ++s) substep<32>(m, hull, w, lane);
    __syncwarp();
    if (own) {
      if (only_flagged != 0 || !(w.bad & 14)) {
        for (int k = lane; k < nq; k += 32) qpos[(size_t)env * nq + k] = w.qpos[k];
        for (int k = lane; k < nv; k += 32) { qvel[(size_t)env * nv + k] = w.qvel[k]; warm[(size_t)env * nv + k] = w.warm[k]; }
      }
      if (lane == 0) {
        info[4 * env] = w.nefc; info[4 * env + 1] = w.ncon; info[4 * env + 2] = w.acc_iter; info[4 * env + 3] = w.bad | (only_flagged == 1 ? 16 : 0);
      }
    }
    __syncthreads();
  }
}


// ------------------------------------------------------------------------------------------------ task layer
constexpr int kNQ = 23, kRobot = 9, kObj = 14, kObs = 46, kAct = 9, kSites = 8;

struct TaskArgs {
  int n, frame_skip;
  unsigned flags;
  long long horizon, goal_change_frequency;
  double goal[kNQ], init_qpos[kNQ], pos_noise_amp[kNQ], pos_bound[kRobot][2], vel_bound[kRobot][2];
  double midpoint[3], mocap_low[3], mocap_high[3], noise_ratio;
  int site[kSites];
  // per-env state (device)
  float *qpos, *qvel, *warm;        // [N,23]
  double* mocap;                    // [N,3]
  double* last_qp;                  // [N,9]   Robot_VelAct observation cache (last NOISY robot qpos)
  double* sites;                    // [N,8,3] site positions of the last forward pass
  unsigned long long* rng;          // [N,4]   PCG64 state hi, lo, inc hi, lo
  unsigned* steps_since_reset;
  unsigned* steps_since_goal_change;
  long long* num_interventions;
  double* lifelong_return;
  unsigned long long* work;         // 12 counters
  int* cost;                        // [N] estimated cost of the last env step (visiting order of the next one)
  float4 mocap_quat;
  // redo pass (null redo_list: disabled, overflowing steps are stored as they are and only counted)
  long long* redo_list;             // [N] entries (step tag << 32 | env): the tag tells a fresh entry from an older step's
  unsigned* sched;                  // [kRedoCount] listed, [kRedoNext] claimed, [kMainDone] step-kernel blocks finished, [kNextChunk]
  unsigned redo_tag, main_blocks;
  // an env whose last step outgrew the step kernel's capacities (prim_*) is "heavy": the step kernel hands it to the redo
  // kernel at the START of its next step (heavy envs lead the visiting order), so that its latency overlaps the step kernel
  unsigned char* heavy;             // [N]
  int prim_efc, prim_con, prim_hit;
  // pre-drawn reset stream (EARL_FLAG_AUTO_RESET): draw e of env i is configuration ring_config[e * n + i], a row of
  // ring_table [K,14] (object qpos), e = ring_cursor[i] mod ring_rows
  const unsigned char* ring_config;
  const double* ring_table;
  unsigned* ring_cursor;
  int ring_rows;
};
enum { kRedoCount = 0, kRedoNext = 1, kMainDone = 2, kNextChunk = 3, kSchedWords = 4 };

// numpy's PCG64 (pcg64.h: pcg_setseq_128_step_r + pcg_output_xsl_rr_128_64) and Generator.uniform(-1, 1)
struct Pcg { unsigned __int128 state, inc; };
__device__ __forceinline__ double pcg_uniform_pm1(Pcg& g) {
  const unsigned __int128 mult = ((unsigned __int128)0x2360ED051FC65DA4ULL << 64) | 0x4385DF649FCCF645ULL;
  g.state = g.state * mult + g.inc;
  const unsigned long long hi = (unsigned long long)(g.state >> 64), lo = (unsigned long long)g.state;
  const unsigned long long x = hi ^ lo;
  const unsigned rot = (unsigned)(hi >> 58);
  const unsigned long long out = (x >> rot) | (x << ((64 - rot) & 63));
  const double r = (double)(out >> 11) * (1.0 / 9007199254740992.0);
  return -1.0 + 2.0 * r;  // random_uniform(low, high - low): low + range * next_double
}

// Robot.get_obs (franka_robot.py:137-168): four draws per observation -- robot qpos (9), robot qvel (9, discarded), object
// qpos (14), object qvel (14, discarded); obs46 = [noisy robot qpos, noisy object qpos, goal] when non-null
__device__ void kitchen_observe(const TaskArgs& a, const Work& w, Pcg& g, double ratio, double* last_qp, double* obs46) {
  double qp[kRobot];
  // __dmul_rn / __dadd_rn: never contracted into a fused multiply-add, so the sums round exactly like numpy's
  for (int i = 0; i < kRobot; ++i) qp[i] = __dadd_rn((double)w.qpos[i], __dmul_rn(__dmul_rn(ratio, a.pos_noise_amp[i]), pcg_uniform_pm1(g)));
  for (int i = 0; i < kRobot; ++i) pcg_uniform_pm1(g);
  for (int i = 0; i < kRobot; ++i) { last_qp[i] = qp[i]; if (obs46) obs46[i] = qp[i]; }
  for (int i = 0; i < kObj; ++i) {
    const double o = __dadd_rn((double)w.qpos[kRobot + i], __dmul_rn(__dmul_rn(ratio, a.pos_noise_amp[kRobot + i]), pcg_uniform_pm1(g)));
    if (obs46) obs46[kRobot + i] = o;
  }
  for (int i = 0; i < kObj; ++i) pcg_uniform_pm1(g);
  if (obs46) for (int i = 0; i < kNQ; ++i) obs46[kNQ + i] = a.goal[i];
}

// KitchenV0.step :91-105 + Robot_VelAct.ctrl_velocity_limits / ctrl_position_limits (franka_robot.py:172-174,255-264):
// mocap update and the nu = 2 controls do_simulation writes (mujoco_env.py:148-153)
__device__ void kitchen_control(const TaskArgs& a, const float* act9, const double* last_qp, double* mocap, real* ctrl2) {
  double sc[kRobot];
  for (int i = 0; i < kRobot; ++i) {
    double x = act9 ? (double)act9[i] : 0.0;
    x = x < -1.0 ? -1.0 : (x > 1.0 ? 1.0 : x);
    sc[i] = 0.0 + x * 2.0;  // act_mid + a * act_amp
  }
  if (act9)
    for (int k = 0; k < 3; ++k) {
      const double p = __dadd_rn(mocap[k], __dmul_rn(sc[k], 0.01));
      mocap[k] = p < a.mocap_low[k] ? a.mocap_low[k] : (p > a.mocap_high[k] ? a.mocap_high[k] : p);
    }
  const double dur = (double)a.frame_skip * 0.002;  // skip * model.opt.timestep
  for (int i = 0; i < 2; ++i) {
    double v = sc[i] < a.vel_bound[i][0] ? a.vel_bound[i][0] : (sc[i] > a.vel_bound[i][1] ? a.vel_bound[i][1] : sc[i]);
    double p = __dadd_rn(last_qp[i], __dmul_rn(v, dur));
    p = p < a.pos_bound[i][0] ? a.pos_bound[i][0] : (p > a.pos_bound[i][1] ? a.pos_bound[i][1] : p);
    ctrl2[i] = (real)p;
  }
}

// Kitchen._get_reward_n_score / is_successful (ENV/kitchen.py:141-183) on the noisy observation
__device__ double kitchen_reward(const double* obs, const double* mocap, const double* sites, bool* success) {
  double s = 0;
  for (int i = 9; i < 23; ++i) { const double d = obs[i] - obs[i + 23]; s += d * d; }
  const double dist = sqrt(s);
  double r = -10 * dist;
  *success = dist <= 0.3;
  // component_to_state_idx (:15-25) in dict order: burner0..3, light_switch, slide_cabinet, hinge_cabinet, microwave
  const int first[8] = {9, 11, 13, 15, 17, 19, 20, 22}, count[8] = {2, 2, 2, 2, 2, 1, 2, 1};
  bool reaching = false;
  for (int c = 0; c < 8; ++c) {
    double q = 0;
    for (int k = 0; k < count[c]; ++k) { const double d = obs[first[c] + k] - obs[first[c] + k + 23]; q += d * d; }
    if (sqrt(q) < count[c] * 0.01) r += 1;
    else if (!reaching) {
      reaching = true;
      double t = 0;
      for (int k = 0; k < 3; ++k) { const double d = mocap[k] - sites[3 * c + k]; t += d * d; }
      r += -0.5 * sqrt(t);
    }
  }
  return r;
}

__device__ __forceinline__ void task_load(const TaskArgs& a, Work& w, int env, int lane) {
  for (int k = lane; k < kNQ; k += 32) { w.qpos[k] = a.qpos[(size_t)env * kNQ + k]; w.qvel[k] = a.qvel[(size_t)env * kNQ + k]; w.warm[k] = a.warm[(size_t)env * kNQ + k]; }
  if (lane == 0) {
    for (int k = 0; k < 3; ++k) w.mocap_pos[k] = a.mocap[(size_t)env * 3 + k];
    w.mocap_quat[0] = a.mocap_quat.x; w.mocap_quat[1] = a.mocap_quat.y; w.mocap_quat[2] = a.mocap_quat.z; w.mocap_quat[3] = a.mocap_quat.w;
    w.bad = 0; w.acc_iter = w.acc_rows = w.acc_con = w.acc_mpr = w.acc_sup = 0; w.broad_valid = 0; w.acc_rebuild = 0; w.peak_efc = w.peak_con = w.peak_hit = 0;
  }
  __syncwarp();
}
__device__ __forceinline__ void task_store(const TaskArgs& a, const Model& m, const Work& w, int env, int lane) {
  for (int k = lane; k < kNQ; k += 32) { a.qpos[(size_t)env * kNQ + k] = w.qpos[k]; a.qvel[(size_t)env * kNQ + k] = w.qvel[k]; a.warm[(size_t)env * kNQ + k] = w.warm[k]; }
  if (lane < kSites) {  // site positions of the LAST forward pass (one substep stale, as sim.data.site_xpos after sim.step())
    real p[3];
    site_xpos(m, w, a.site[lane], p);
    for (int k = 0; k < 3; ++k) a.sites[((size_t)env * kSites + lane) * 3 + k] = (double)p[k];
  }
  if (lane == 0) for (int k = 0; k < 3; ++k) a.mocap[(size_t)env * 3 + k] = w.mocap_pos[k];
  __syncwarp();
}

struct TaskCounters { unsigned long long it = 0, rows = 0, con = 0, bad = 0, over = 0, env = 0, ov_hit = 0, ov_con = 0, ov_row = 0, redone = 0; };
struct TaskIo {
  const float* actions; const double* object_qpos; double* obs_out; double* reward_out; unsigned char* done_out; unsigned char* success_out;
};

// One environment of the task kernels, all lanes of its warp.  mode 0: env step, mode 1: reset (slot = row of object_qpos /
// obs_out; object_qpos null: the env's next draw of the reset stream), mode 2: env step of the redo pass, mode 3: reset
// from the reset stream after a step (obs row = env).  `own` false: the warp only keeps its block's phase barriers company.
// Returns false when the step overflowed the capacities and was handed to the redo pass (nothing stored).
__device__ __forceinline__ bool task_env(const Model& m, const real* hull, const TaskArgs& a, const TaskIo& io, Work& w, int mode, int env,
                                         int slot, bool own, int lane, TaskCounters& c) {
  Pcg g;
  double last_qp[kRobot];
  const bool stepping = mode == 0 || mode == 2;
  const bool ring = mode == 3 || (mode == 1 && !io.object_qpos);
  if (!stepping) {  // Kitchen.reset_model: robot.reset (sim.reset, qpos write, forward, 5 cached observations at ratio 1)
    const double* obj = ring ? a.ring_table + (size_t)kObj * a.ring_config[(size_t)(a.ring_cursor[env] % (unsigned)a.ring_rows) * a.n + env]
                             : io.object_qpos + (size_t)slot * kObj;
    for (int k = lane; k < kNQ; k += 32) {
      const double q = k < kRobot ? a.init_qpos[k] : obj[k - kRobot];
      w.qpos[k] = (real)q; w.qvel[k] = 0; w.warm[k] = 0;
    }
    if (lane == 0) {
      for (int k = 0; k < 3; ++k) w.mocap_pos[k] = a.midpoint[k];
      w.mocap_quat[0] = a.mocap_quat.x; w.mocap_quat[1] = a.mocap_quat.y; w.mocap_quat[2] = a.mocap_quat.z; w.mocap_quat[3] = a.mocap_quat.w;
      w.bad = 0; w.acc_iter = w.acc_rows = w.acc_con = w.acc_mpr = w.acc_sup = 0; w.broad_valid = 0; w.acc_rebuild = 0; w.peak_efc = w.peak_con = w.peak_hit = 0;
    }
    __syncwarp();
  } else {
    task_load(a, w, env, lane);
  }
  if (lane == 0) {
    const unsigned long long* r = a.rng + (size_t)env * 4;
    g.state = ((unsigned __int128)r[0] << 64) | r[1];
    g.inc = ((unsigned __int128)r[2] << 64) | r[3];
    if (!stepping) {
      for (int k = 0; k < 5; ++k) kitchen_observe(a, w, g, 1.0, last_qp, nullptr);  // _observation_cache_refresh: default ratio 1
      kitchen_control(a, nullptr, last_qp, w.mocap_pos, w.ctrl);
    } else {
      for (int k = 0; k < kRobot; ++k) last_qp[k] = a.last_qp[(size_t)env * kRobot + k];
      kitchen_control(a, io.actions + (size_t)env * kAct, last_qp, w.mocap_pos, w.ctrl);
    }
  }
  __syncwarp();
  const int nsub = stepping ? a.frame_skip : 10 * a.frame_skip;
  // Capacity overflow (step kernel): nothing is stored, the env is listed for the redo pass AT THE SUBSTEP IT HAPPENS IN, so
  // that its re-step starts while this chunk is still running; the warp then only keeps the phase barriers company.
  const bool watch = mode == 0 && a.redo_list != nullptr;
  int s = 0;
  for (; s < nsub; ++s) {
    substep<32>(m, hull, w, lane);  // ends with a warp barrier: w.bad (lane 0, collision / row phases) is visible to all lanes
    if (watch && (w.bad & 14)) break;
  }
  __syncwarp();
  if (s < nsub) {
    if (own && lane == 0) {
      const unsigned at = atomicAdd(&a.sched[kRedoCount], 1u);
      *reinterpret_cast<volatile long long*>(a.redo_list + at) = ((long long)a.redo_tag << 32) | (long long)(unsigned)env;
      __threadfence();
    }
    for (++s; s < nsub; ++s) substep_idle<32>();
    return false;
  }
  // A step that left a non-finite state (or whose factorisation broke down) is NOT stored: the environment stays at its
  // last good state, the step returns that state's (noisy) observation with reward 0 and is counted in work[5]
  // (SURVEY 5; the reference only prints MuJoCo's warning, ADEPT/simulation/module.py:123-126, and carries NaNs on).
  bool fin = true;
  for (int k = lane; k < kNQ; k += 32) fin = fin && isfinite(w.qpos[k]) && isfinite(w.qvel[k]);
  const bool failed = stepping && (!__all_sync(0xffffffffu, fin) || (w.bad & 1));
  if (failed) {
    const unsigned bad_k = w.bad | 1u;
    __syncwarp();
    task_load(a, w, env, lane);
    kinematics<32>(m, w, lane);
    if (lane == 0) w.bad = bad_k;
    __syncwarp();
  }
  if (!own) return true;
  task_store(a, m, w, env, lane);
  if (lane == 0) {
    double obs[kObs];
    kitchen_observe(a, w, g, a.noise_ratio, last_qp, obs);
    for (int k = 0; k < kRobot; ++k) a.last_qp[(size_t)env * kRobot + k] = last_qp[k];
    unsigned long long* r = a.rng + (size_t)env * 4;
    r[0] = (unsigned long long)(g.state >> 64); r[1] = (unsigned long long)g.state;
    double* orow = io.obs_out ? io.obs_out + (size_t)(mode == 1 ? slot : env) * kObs : nullptr;
    // estimated warp instructions above the contact-free baseline: loose broad-phase passes (~9k each), extra Newton
    // iterations (~6k), contacts (~1.5k per contact and substep), portal-refinement support calls (~0.3k)
    a.cost[env] = 9000 * w.acc_rebuild + 6000 * (w.acc_iter - a.frame_skip) + 1500 * w.acc_con + 300 * w.acc_sup;
    if (mode == 2) {
      const bool heavy = w.peak_efc > a.prim_efc || w.peak_con > a.prim_con || w.peak_hit > a.prim_hit;
      a.heavy[env] = heavy ? 1 : 0;
      if (heavy) a.cost[env] = 1 << 30;  // top bucket: visited (and listed) first
    }
    if (orow) for (int k = 0; k < kObs; ++k) orow[k] = obs[k];
    if (stepping) {
      bool ok;
      double rew = kitchen_reward(obs, w.mocap_pos, a.sites + (size_t)env * kSites * 3, &ok);
      if (failed) { rew = 0.0; ok = false; }
      io.reward_out[env] = rew;
      if (io.success_out) io.success_out[env] = ok;
      const unsigned st = a.steps_since_reset[env] + 1;  // PersistentStateWrapper.step (persistent_state_wrapper.py:22-31)
      a.steps_since_reset[env] = st;
      io.done_out[env] = (long long)st >= a.horizon;
      if (a.flags & EARL_FLAG_LIFELONG) {              // LifelongWrapper.step (lifelong_wrapper.py:30-44)
        a.lifelong_return[env] += rew;
        const unsigned sg = a.steps_since_goal_change[env] + 1;
        if (a.goal_change_frequency > 0 && (long long)sg >= a.goal_change_frequency) {
          // reset_goal() (a single goal: nothing changes) and env._get_obs(): a second noisy observation, returned
          // instead of the first and cached for the next control; the reward stays the one already computed
          a.steps_since_goal_change[env] = 0;
          kitchen_observe(a, w, g, a.noise_ratio, last_qp, obs);
          for (int k = 0; k < kRobot; ++k) a.last_qp[(size_t)env * kRobot + k] = last_qp[k];
          r[0] = (unsigned long long)(g.state >> 64); r[1] = (unsigned long long)g.state;
          if (orow) for (int k = 0; k < kObs; ++k) orow[k] = obs[k];
        } else {
          a.steps_since_goal_change[env] = sg;
        }
      }
    } else {
      a.steps_since_reset[env] = 0;                     // PersistentStateWrapper.reset (:17-20)
      a.steps_since_goal_change[env] = 0;               // LifelongWrapper.reset (:25-28)
      a.num_interventions[env] += 1;
      a.heavy[env] = 0;
      if (ring) a.ring_cursor[env] += 1;
    }
    c.it += w.acc_iter; c.rows += w.acc_rows; c.con += w.acc_con; c.bad += (w.bad & 1) ? 1 : 0; c.over += (w.bad & 14) ? 1 : 0; c.env += 1;
    c.ov_hit += (w.bad & 2) ? 1 : 0; c.ov_con += (w.bad & 4) ? 1 : 0; c.ov_row += (w.bad & 8) ? 1 : 0;
    c.redone += mode == 2 ? 1 : 0;
  }
  return true;
}

__device__ __forceinline__ void task_flush(const TaskArgs& a, const TaskCounters& c, int mode, int lane) {
  if (lane == 0 && c.env) {
    const bool resetting = mode == 1 || mode == 3;
    atomicAdd(&a.work[0], resetting ? 0ULL : c.env);
    atomicAdd(&a.work[1], c.env * (unsigned long long)(resetting ? 10 * a.frame_skip : a.frame_skip));
    atomicAdd(&a.work[2], c.it); atomicAdd(&a.work[3], c.rows); atomicAdd(&a.work[4], c.con);
    atomicAdd(&a.work[5], c.bad); atomicAdd(&a.work[6], c.over); atomicAdd(&a.work[7], c.redone);
    atomicAdd(&a.work[8], c.ov_hit); atomicAdd(&a.work[9], c.ov_con); atomicAdd(&a.work[10], c.ov_row);
  }
}

#ifndef MJK_XL
// mode 0: one env step of every environment.  mode 1: reset of the environments in env_ids.  mode 3: reset of every
// environment whose io.done_out (read here: the done array of the step just taken) is set, from the reset stream.
__global__ void __launch_bounds__(kWPB * 32, kBPS)
mjk_task_kernel(const Model* __restrict__ gm, const real* __restrict__ hull, const TaskArgs a, int mode, const int* env_ids, int count,
                const TaskIo io) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Work& w = *reinterpret_cast<Work*>(smem + warp * kWorkStride);
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // lets the concurrent redo kernel start (no-op otherwise)
  TaskCounters c;
  if (mode == 3) {
    // static stride over chunks of kWPB consecutive envs; a chunk without a done env is left at once, in one with some the
    // other warps shadow a reset they do not store (the phase barriers are block-wide)
    for (int base = blockIdx.x * kWPB; base < count; base += gridDim.x * kWPB) {
      const bool in = base + warp < count;
      const int env = in ? base + warp : count - 1;
      const bool own = in && io.done_out[env];
      if (!__syncthreads_or(own)) continue;
      task_env(*gm, hull, a, io, w, 3, env, env, own, lane, c);
      __syncthreads();
    }
    task_flush(a, c, 3, lane);
    return;
  }
  // Step: chunks of kWPB consecutive entries of the cost-sorted order are handed out dynamically (a block that draws expensive
  // chunks takes fewer of them).  Reset: static stride.
  __shared__ int s_chunk;
  const bool dynamic = mode == 0;
  for (int it = 0;; ++it) {
    if (dynamic) {
      if (threadIdx.x == 0) s_chunk = (int)atomicAdd(&a.sched[kNextChunk], 1u);
      __syncthreads();
    }
    const int base = (dynamic ? s_chunk : blockIdx.x + it * (int)gridDim.x) * kWPB;
    if (base >= count) break;
    const bool own = base + warp < count;
    const int slot = own ? base + warp : count - 1;
    const int env = env_ids ? env_ids[slot] : slot;
    bool heavy = false;
    if (mode == 0 && a.redo_list) {
      heavy = own && a.heavy[env];
      if (heavy && lane == 0) {
        const unsigned at = atomicAdd(&a.sched[kRedoCount], 1u);
        *reinterpret_cast<volatile long long*>(a.redo_list + at) = ((long long)a.redo_tag << 32) | (long long)(unsigned)env;
        __threadfence();
      }
      if (__syncthreads_and(heavy || !own)) continue;  // a chunk of heavy envs only: nothing to step here
    }
    task_env(*gm, hull, a, io, w, mode, env, slot, own && !heavy, lane, c);
    __syncthreads();
  }
  task_flush(a, c, mode, lane);
  if (mode == 0 && a.redo_list) {
    __syncthreads();
    if (threadIdx.x == 0) { __threadfence(); atomicAdd(&a.sched[kMainDone], 1u); }  // the redo kernel polls this
  }
}
#else
// Redo pass: the env steps the step kernel listed, re-stepped from their untouched states with the extra-large capacities.
// Runs while the step kernel does: thread 0 claims up to kWPB listed entries, or waits for one / for the step kernel's end.
__global__ void __launch_bounds__(kWPB * 32, 1)
mjk_redo_kernel(const Model* __restrict__ gm, const real* __restrict__ hull, const TaskArgs a, const TaskIo io) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int s_base, s_take;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Work& w = *reinterpret_cast<Work*>(smem + warp * kWorkStride);
  TaskCounters c;
  volatile unsigned* sched = a.sched;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) {
      int base = 0, take = 0;
      for (;;) {
        const unsigned cnt = sched[kRedoCount], nx = sched[kRedoNext];
        if (nx < cnt) {
          const unsigned t = cnt - nx < (unsigned)kWPB ? cnt - nx : (unsigned)kWPB;
          if (atomicCAS(&a.sched[kRedoNext], nx, nx + t) == nx) { base = (int)nx; take = (int)t; break; }
          continue;
        }
        if (sched[kMainDone] >= a.main_blocks) {
          __threadfence();
          if (sched[kRedoNext] >= sched[kRedoCount]) break;  // step kernel over, list consumed
          continue;
        }
        __nanosleep(1000);
      }
      s_base = base;
      s_take = take;
    }
    __syncthreads();
    const int base = s_base, take = s_take;
    if (take == 0) break;
    const bool own = warp < take;
    long long entry;  // the slot was counted before it was written: wait for this step's tag
    do {
      entry = *reinterpret_cast<volatile long long*>(a.redo_list + base + (own ? warp : 0));
    } while ((unsigned)(entry >> 32) != a.redo_tag);
    const int env = (int)(unsigned)(entry & 0xffffffffll);
    task_env(*gm, hull, a, io, w, 2, env, env, own, lane, c);
  }
  task_flush(a, c, 2, lane);
}
#endif


#ifdef MJK_XL
}  // namespace

// Launches the redo kernel behind the step kernel (the previous launch in `stream`) as its programmatic dependent: it may
// start while the step kernel still runs, on the SMs that one leaves free, and never calls griddepcontrol.wait -- it polls
// the step kernel's list and exit counter.  TaskArgs / TaskIo / Model have the same layout in both instantiations (only
// the workspace capacities differ); the sizes are checked.
extern "C" int earl_mjkx_redo_pass(const void* d_model, size_t model_bytes, const void* d_hull, const void* task_args, size_t args_bytes,
                                   const void* task_io, size_t io_bytes, int blocks, void* stream) {
  if (!d_model || !task_args || !task_io || model_bytes != sizeof(Model) || args_bytes != sizeof(TaskArgs) || io_bytes != sizeof(TaskIo))
    return failf(EARL_ERR_INVALID, "kitchen redo pass: argument layout mismatch (%zu / %zu / %zu vs %zu / %zu / %zu)", model_bytes, args_bytes,
                 io_bytes, sizeof(Model), sizeof(TaskArgs), sizeof(TaskIo));
  static bool configured[64] = {};
  int dev = 0;
  CU(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    CU(cudaFuncSetAttribute(mjk_redo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    configured[dev] = true;
  }
  TaskArgs a;
  TaskIo io;
  memcpy(&a, task_args, sizeof(a));
  memcpy(&io, task_io, sizeof(io));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(blocks > 0 ? blocks : 1));
  cfg.blockDim = dim3((unsigned)(kWPB * 32));
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  CU(cudaLaunchKernelEx(&cfg, mjk_redo_kernel, static_cast<const Model*>(d_model), static_cast<const real*>(d_hull), a, io));
  return 0;
}

// Second pass of earl_mjk_engine_substeps: the environments the primary set flagged (info[:, 3] & 14), from their untouched
// input states, with the extra-large capacities; info[:, 3] gets bit 4 (and again bits 1-3 if even this set overflowed).
extern "C" int earl_mjkx_substeps_flagged(const void* d_model, size_t model_bytes, const void* d_hull, int n, int nsub, float* qpos, float* qvel,
                                          float* warm, const double* mocap_pos, const float* mocap_quat4, const float* ctrl, int* info,
                                          int sm_count, void* stream) {
  if (!d_model || model_bytes != sizeof(Model)) return failf(EARL_ERR_INVALID, "kitchen substeps: model layout mismatch");
  static bool configured[64] = {};
  int dev = 0;
  CU(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !configured[dev]) {
    CU(cudaFuncSetAttribute(mjk_substeps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    configured[dev] = true;
  }
  const int blocks = (n + kWPB - 1) / kWPB;
  const int grid = blocks < 4 * sm_count ? blocks : 4 * sm_count;
  mjk_substeps_kernel<<<grid, kWPB * 32, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const Model*>(d_model), static_cast<const real*>(d_hull), n, nsub, qpos, qvel, warm, mocap_pos,
      make_float4(mocap_quat4[0], mocap_quat4[1], mocap_quat4[2], mocap_quat4[3]), ctrl, info, 1);
  CU(cudaGetLastError());
  return 0;
}
#else  // !MJK_XL: the rest of the file is the primary instantiation's host side

extern "C" int earl_mjkx_substeps_flagged(const void* d_model, size_t model_bytes, const void* d_hull, int n, int nsub, float* qpos, float* qvel,
                                          float* warm, const double* mocap_pos, const float* mocap_quat4, const float* ctrl, int* info,
                                          int sm_count, void* stream);  // earl_mj_kitchen_xl.cu

extern "C" int earl_mjkx_redo_pass(const void* d_model, size_t model_bytes, const void* d_hull, const void* task_args, size_t args_bytes,
                                   const void* task_io, size_t io_bytes, int blocks, void* stream);  // earl_mj_kitchen_xl.cu

// Visiting order of the next env step: environments bucketed by the estimated cost of the step they just took, most
// expensive bucket first, so the warps of a block (which meet at block-wide phase barriers) carry similar work.
constexpr int kBuckets = 32;
__global__ void mjk_bucket_kernel(const int* cost, int n, int width, unsigned char* bucket, int* rank, unsigned* counts) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  int b = cost[env] <= 0 ? 0 : 1 + cost[env] / width;
  b = b > kBuckets - 1 ? kBuckets - 1 : b;
  bucket[env] = (unsigned char)b;
  rank[env] = (int)atomicAdd(&counts[b], 1u);
}
__global__ void mjk_order_kernel(const unsigned char* bucket, const int* rank, int n, unsigned* counts, int* order) {
  __shared__ unsigned base[kBuckets];
  if (threadIdx.x == 0) {
    unsigned acc = 0;
    for (int b = kBuckets - 1; b >= 0; --b) { base[b] = acc; acc += counts[b]; }
  }
  __syncthreads();
  for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < n; env += gridDim.x * blockDim.x) order[base[bucket[env]] + rank[env]] = env;
}
__global__ void mjk_iota_kernel(int* order, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) order[i] = i;
}

}  // namespace

struct earl_mjk_engine {
  HostModel hm;
  int device = 0, sm_count = 0;
  float mocap_quat[4] = {1, 0, 0, 0};  // the model's mocap orientation (the task never moves it)
  Model* d_model = nullptr;
  real* d_hull = nullptr;
};

extern "C" {

int earl_mjk_engine_create(const void* model_blob, size_t model_nbytes, int32_t device, earl_mjk_engine** out) {
  if (!model_blob || !out) return failf(EARL_ERR_INVALID, "null argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return failf(EARL_ERR_CUDA, "no CUDA device: the kitchen engine has no CPU path");
  if (device < 0 || device >= ndev) return failf(EARL_ERR_INVALID, "device %d out of range", device);
  earl_mjk_engine* e = new (std::nothrow) earl_mjk_engine();
  if (!e) return failf(EARL_ERR_NOMEM, "out of host memory");
  TaskSpec t;
  memset(&t, 0, sizeof(t));
  t.frame_skip = 40;
  t.obj_geom = -1;
  std::string msg;
  if (!build_model(model_blob, model_nbytes, t, &e->hm, &msg)) {
    delete e;
    return failf(EARL_ERR_INVALID, "%s", msg.c_str());
  }
  e->device = device;
  for (int k = 0; k < 4; ++k) e->mocap_quat[k] = (float)e->hm.mocap_quat0[k];
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  e->sm_count = prop.multiProcessorCount;
  CU(cudaMalloc(&e->d_model, sizeof(Model)));
  CU(cudaMemcpy(e->d_model, &e->hm.m, sizeof(Model), cudaMemcpyHostToDevice));
  const size_t hb = (e->hm.hull_vert.size() + 4) * sizeof(real);
  CU(cudaMalloc(&e->d_hull, hb));
  CU(cudaMemcpy(e->d_hull, e->hm.hull_vert.data(), e->hm.hull_vert.size() * sizeof(real), cudaMemcpyHostToDevice));
  CU(cudaFuncSetAttribute(mjk_substeps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  *out = e;
  return 0;
}

int earl_mjk_engine_destroy(earl_mjk_engine* e) {
  if (!e) return 0;
  cudaSetDevice(e->device);
  cudaFree(e->d_model);
  cudaFree(e->d_hull);
  delete e;
  return 0;
}

int earl_mjk_engine_nv(const earl_mjk_engine* e) { return e ? e->hm.m.nv : 0; }

int earl_mjk_engine_substeps(earl_mjk_engine* e, int32_t num_envs, int32_t nsub, float* qpos_dev, float* qvel_dev, float* warm_dev,
                             const double* mocap_pos_dev, const float* mocap_quat_host, const float* ctrl_dev, int32_t* info_dev,
                             void* stream) {
  if (!e) return failf(EARL_ERR_INVALID, "null engine");
  if (num_envs <= 0 || nsub < 0 || !qpos_dev || !qvel_dev || !warm_dev || !mocap_pos_dev || !mocap_quat_host || !ctrl_dev || !info_dev)
    return failf(EARL_ERR_INVALID, "bad arguments");
  CU(cudaSetDevice(e->device));
  const int blocks = (num_envs + kWPB - 1) / kWPB;
  const int grid = blocks < e->sm_count ? blocks : e->sm_count;
  const float4 mq = make_float4(mocap_quat_host[0], mocap_quat_host[1], mocap_quat_host[2], mocap_quat_host[3]);
  const bool redo = !(getenv("EARL_MJ_REDO") && atoi(getenv("EARL_MJ_REDO")) == 0);
  mjk_substeps_kernel<<<grid, kWPB * 32, kSmemBytes, static_cast<cudaStream_t>(stream)>>>(
      e->d_model, e->d_hull, num_envs, nsub, qpos_dev, qvel_dev, warm_dev, mocap_pos_dev, mq, ctrl_dev, info_dev, redo ? 0 : 2);
  CU(cudaGetLastError());
  if (redo)
    return earl_mjkx_substeps_flagged(e->d_model, sizeof(Model), e->d_hull, num_envs, nsub, qpos_dev, qvel_dev, warm_dev, mocap_pos_dev,
                                      mocap_quat_host, ctrl_dev, info_dev, e->sm_count, stream);
  return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ task-level ABI
static_assert(sizeof(earl_mjk_config) == 984, "earl_mjk_config layout (mirrored by envs/kitchen.py::MjkConfig)");
struct earl_mjk_handle {
  earl_mjk_engine* eng = nullptr;
  TaskArgs a{};
  int64_t total_steps = 0;
  bool seeded = false;
  int* d_order = nullptr;           // visiting order of the next step (cost-sorted)
  unsigned char* d_bucket = nullptr;
  int* d_rank = nullptr;
  unsigned* d_counts = nullptr;
  int bucket_width = 60000;  // flat between 40k and 160k (measured); EARL_MJK_BUCKET_WIDTH overrides
  bool redo_sms_fixed = false;      // EARL_MJ_REDO_SMS given: no adaptation
  unsigned* h_redo_seen = nullptr;  // pinned: redo-list length of a recent step (async copy, read without waiting)
  int ring_configs = 0;             // rows of the reset stream's configuration table
  int redo_sms = 4;          // SMs the step kernel leaves to the concurrent redo kernel (EARL_MJ_REDO_SMS; measured 2: 1.49e5, 4: 1.54e5, 6: 1.53e5)
  std::vector<void*> owned;
  template <typename T>
  int alloc(T** ptr, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
    if (e != cudaSuccess) return failf(EARL_ERR_NOMEM, "cudaMalloc(%zu B) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    e = cudaMemset(q, 0, count * sizeof(T));
    if (e != cudaSuccess) return failf(EARL_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    owned.push_back(q);
    *ptr = static_cast<T*>(q);
    return 0;
  }
};

namespace {
int launch_task(earl_mjk_handle* h, int mode, const int* env_ids, int count, const float* actions, const double* object_qpos,
                double* obs, double* reward, unsigned char* done, unsigned char* success, void* stream) {
  const int blocks = (count + kWPB - 1) / kWPB;
  const int slots = h->eng->sm_count * kBPS;
  int grid = blocks < slots ? blocks : slots;
  TaskArgs a = h->a;
  const TaskIo io{actions, object_qpos, obs, reward, done, success};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (mode != 0) a.redo_list = nullptr;
  if (a.redo_list) {
    // SMs left to the concurrent redo kernel: balanced against the list length L of a recent step -- the step kernel walks
    // (n - L) envs kWPB = 8 per SM, the redo kernel L envs 2 per SM, at about one env step per wave either way:
    // (n - L) / (8 (S - r)) = L / (2 r)  =>  r = S * 4 L / (n + 3 L); at least redo_sms, at most half of the GPU
    int r = h->redo_sms;
    if (!h->redo_sms_fixed && h->h_redo_seen) {
      const double L = (double)*reinterpret_cast<volatile unsigned*>(h->h_redo_seen), S = (double)h->eng->sm_count;
      const int want = (int)(S * 4.0 * L / ((double)count + 3.0 * L) + 0.5);
      r = want > r ? want : r;
      r = r > h->eng->sm_count / 2 ? h->eng->sm_count / 2 : r;
    }
    if (slots >= 2 * r * kBPS && blocks + r * kBPS > slots) grid = grid < slots - r * kBPS ? grid : slots - r * kBPS;
    a.prim_efc = MAXEFC; a.prim_con = MAXCON; a.prim_hit = MAXHIT;
    a.main_blocks = (unsigned)grid;
    a.redo_tag = (unsigned)(h->total_steps & 0x7fffffff);
  }
  if (mode == 0) CU(cudaMemsetAsync(a.sched, 0, kSchedWords * sizeof(unsigned), s));
  mjk_task_kernel<<<grid, kWPB * 32, kSmemBytes, s>>>(h->eng->d_model, h->eng->d_hull, a, mode, env_ids, count, io);
  CU(cudaGetLastError());
  // one redo block per SM: those that find no free SM start as step-kernel blocks retire, so a regime with many overflows
  // (arms deep in the cabinets: 5 % of the env steps) ends with the whole GPU working on the list
  if (a.redo_list)
    if (int rc = earl_mjkx_redo_pass(h->eng->d_model, sizeof(Model), h->eng->d_hull, &a, sizeof(a), &io, sizeof(io), h->eng->sm_count, stream))
      return rc;
  return 0;
}
}  // namespace

extern "C" {

int earl_mjk_create(const earl_mjk_config* cfg, const void* model_blob, size_t model_nbytes, earl_mjk_handle** out) {
  if (!cfg || !model_blob || !out) return failf(EARL_ERR_INVALID, "null argument");
  *out = nullptr;
  if (cfg->num_envs <= 0 || cfg->frame_skip <= 0 || cfg->episode_horizon <= 0) return failf(EARL_ERR_INVALID, "bad kitchen config");
  if (cfg->flags & ~(uint32_t)(EARL_FLAG_LIFELONG | EARL_FLAG_AUTO_RESET)) return failf(EARL_ERR_UNSUPPORTED, "unsupported flags %#x", cfg->flags);
  earl_mjk_engine* eng = nullptr;
  if (int rc = earl_mjk_engine_create(model_blob, model_nbytes, cfg->device, &eng)) return rc;
  earl_mjk_handle* h = new (std::nothrow) earl_mjk_handle();
  if (!h) { earl_mjk_engine_destroy(eng); return failf(EARL_ERR_NOMEM, "out of host memory"); }
  h->eng = eng;
  const Model& m = eng->hm.m;
  if (m.nq != kNQ || m.nv != kNQ || m.nu != 2) { earl_mjk_destroy(h); return failf(EARL_ERR_INVALID, "not the kitchen model (nq %d nv %d nu %d)", m.nq, m.nv, m.nu); }
  for (int k = 0; k < kSites; ++k)
    if (cfg->site[k] < 0 || cfg->site[k] >= m.nsite) { earl_mjk_destroy(h); return failf(EARL_ERR_INVALID, "site index out of range"); }
  TaskArgs& a = h->a;
  a.n = cfg->num_envs; a.frame_skip = cfg->frame_skip; a.flags = cfg->flags; a.horizon = cfg->episode_horizon; a.goal_change_frequency = cfg->goal_change_frequency;
  memcpy(a.goal, cfg->goal, sizeof a.goal); memcpy(a.init_qpos, cfg->init_qpos, sizeof a.init_qpos);
  memcpy(a.pos_noise_amp, cfg->pos_noise_amp, sizeof a.pos_noise_amp);
  memcpy(a.pos_bound, cfg->pos_bound, sizeof a.pos_bound); memcpy(a.vel_bound, cfg->vel_bound, sizeof a.vel_bound);
  memcpy(a.midpoint, cfg->midpoint, sizeof a.midpoint); memcpy(a.mocap_low, cfg->mocap_low, sizeof a.mocap_low);
  memcpy(a.mocap_high, cfg->mocap_high, sizeof a.mocap_high);
  a.noise_ratio = cfg->noise_ratio;
  memcpy(a.site, cfg->site, sizeof a.site);
  const size_t n = (size_t)cfg->num_envs;
  int rc = 0;
  if ((rc = h->alloc(&a.qpos, n * kNQ)) || (rc = h->alloc(&a.qvel, n * kNQ)) || (rc = h->alloc(&a.warm, n * kNQ)) ||
      (rc = h->alloc(&a.mocap, n * 3)) || (rc = h->alloc(&a.last_qp, n * kRobot)) || (rc = h->alloc(&a.sites, n * kSites * 3)) ||
      (rc = h->alloc(&a.rng, n * 4)) || (rc = h->alloc(&a.steps_since_reset, n)) || (rc = h->alloc(&a.steps_since_goal_change, n)) || (rc = h->alloc(&a.num_interventions, n)) ||
      (rc = h->alloc(&a.lifelong_return, n)) || (rc = h->alloc(&a.work, 12)) || (rc = h->alloc(&a.cost, n)) || (rc = h->alloc(&h->d_order, n)) ||
      (rc = h->alloc(&h->d_bucket, n)) || (rc = h->alloc(&h->d_rank, n)) || (rc = h->alloc(&h->d_counts, kBuckets)) ||
      (rc = h->alloc(&a.sched, kSchedWords))) {
    earl_mjk_destroy(h);
    return rc;
  }
  CU(cudaFuncSetAttribute(mjk_task_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  mjk_iota_kernel<<<(cfg->num_envs + 255) / 256, 256>>>(h->d_order, cfg->num_envs);
  CU(cudaGetLastError());
  CU(cudaDeviceSynchronize());  // the first step may be enqueued on any stream
  if (const char* e = getenv("EARL_MJK_BUCKET_WIDTH")) h->bucket_width = atoi(e) > 0 ? atoi(e) : h->bucket_width;
  if (!(getenv("EARL_MJ_REDO") && atoi(getenv("EARL_MJ_REDO")) == 0))
    if ((rc = h->alloc(&a.redo_list, n))) { earl_mjk_destroy(h); return rc; }
  if (const char* e = getenv("EARL_MJ_REDO_SMS")) { const int r = atoi(e); if (r >= 1 && r < eng->sm_count / 8) { h->redo_sms = r; h->redo_sms_fixed = true; } }
  if ((rc = h->alloc(&a.heavy, n))) { earl_mjk_destroy(h); return rc; }
  if (cudaHostAlloc(reinterpret_cast<void**>(&h->h_redo_seen), sizeof(unsigned), cudaHostAllocDefault) == cudaSuccess) *h->h_redo_seen = 0;
  else { h->h_redo_seen = nullptr; cudaGetLastError(); }
  *out = h;
  return 0;
}

int earl_mjk_destroy(earl_mjk_handle* h) {
  if (!h) return 0;
  if (h->eng) cudaSetDevice(h->eng->device);
  for (void* p : h->owned) cudaFree(p);
  if (h->h_redo_seen) cudaFreeHost(h->h_redo_seen);
  earl_mjk_engine_destroy(h->eng);
  delete h;
  return 0;
}

int earl_mjk_seed(earl_mjk_handle* h, const uint64_t* pcg_state_host) {
  if (!h || !pcg_state_host) return failf(EARL_ERR_INVALID, "null argument");
  CU(cudaSetDevice(h->eng->device));
  CU(cudaMemcpy(h->a.rng, pcg_state_host, (size_t)h->a.n * 4 * sizeof(uint64_t), cudaMemcpyHostToDevice));
  h->seeded = true;
  return 0;
}

int earl_mjk_set_reset_stream(earl_mjk_handle* h, const uint8_t* config_host, int32_t rows, const double* table_host, int32_t num_configs) {
  if (!h || !config_host || !table_host) return failf(EARL_ERR_INVALID, "null argument");
  if (!(h->a.flags & EARL_FLAG_AUTO_RESET)) return failf(EARL_ERR_INVALID, "the reset stream belongs to EARL_FLAG_AUTO_RESET handles");
  if (rows < 1 || num_configs < 1 || num_configs > 256) return failf(EARL_ERR_INVALID, "bad reset stream shape (%d rows, %d configurations)", rows, num_configs);
  if (h->a.ring_rows && (h->a.ring_rows != rows || h->ring_configs != num_configs))
    return failf(EARL_ERR_INVALID, "reset stream already has %d rows of %d configurations", h->a.ring_rows, h->ring_configs);
  const size_t n = (size_t)h->a.n, cells = (size_t)rows * n;
  for (size_t k = 0; k < cells; ++k)
    if (config_host[k] >= num_configs) return failf(EARL_ERR_INVALID, "configuration %d out of range", (int)config_host[k]);
  CU(cudaSetDevice(h->eng->device));
  TaskArgs& a = h->a;
  if (!a.ring_rows) {
    int rc = h->alloc(const_cast<unsigned char**>(&a.ring_config), cells);
    if (!rc) rc = h->alloc(const_cast<double**>(&a.ring_table), (size_t)num_configs * kObj);
    if (!rc) rc = h->alloc(&a.ring_cursor, n);
    if (rc) return rc;
    a.ring_rows = rows;
    h->ring_configs = num_configs;
  }
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(const_cast<unsigned char*>(a.ring_config), config_host, cells, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(const_cast<double*>(a.ring_table), table_host, (size_t)num_configs * kObj * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemset(a.ring_cursor, 0, n * sizeof(unsigned)));
  return 0;
}

int earl_mjk_reset(earl_mjk_handle* h, const int32_t* env_ids_dev, int32_t count, const double* object_qpos_dev, double* obs_out_dev,
                   void* stream) {
  if (!h) return failf(EARL_ERR_INVALID, "null argument");
  if (!object_qpos_dev && !h->a.ring_rows)
    return failf(EARL_ERR_INVALID, "object_qpos is required (NULL draws from the reset stream of an auto-reset handle, which has none yet)");
  if (!h->seeded) return failf(EARL_ERR_INVALID, "earl_mjk_seed must be called before the first reset (the observation noise stream)");
  if (!env_ids_dev) count = h->a.n;
  if (count <= 0 || count > h->a.n) return failf(EARL_ERR_INVALID, "bad env count %d", count);
  CU(cudaSetDevice(h->eng->device));
  h->a.mocap_quat = make_float4(h->eng->mocap_quat[0], h->eng->mocap_quat[1], h->eng->mocap_quat[2], h->eng->mocap_quat[3]);
  return launch_task(h, 1, env_ids_dev, count, nullptr, object_qpos_dev, obs_out_dev, nullptr, nullptr, nullptr, stream);
}

int earl_mjk_step(earl_mjk_handle* h, const float* actions_dev, double* obs_dev, double* reward_dev, uint8_t* done_dev, uint8_t* success_dev,
                  void* stream) {
  if (!h || !actions_dev || !obs_dev || !reward_dev || !done_dev) return failf(EARL_ERR_INVALID, "null argument");
  if ((h->a.flags & EARL_FLAG_AUTO_RESET) && !h->a.ring_rows) return failf(EARL_ERR_INVALID, "auto-reset handles need earl_mjk_set_reset_stream before the first step");
  CU(cudaSetDevice(h->eng->device));
  h->a.mocap_quat = make_float4(h->eng->mocap_quat[0], h->eng->mocap_quat[1], h->eng->mocap_quat[2], h->eng->mocap_quat[3]);
  h->total_steps += 1;
  if (int rc = launch_task(h, 0, h->d_order, h->a.n, actions_dev, nullptr, obs_dev, reward_dev, done_dev, success_dev, stream)) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CU(cudaMemsetAsync(h->d_counts, 0, kBuckets * sizeof(unsigned), s));
  mjk_bucket_kernel<<<(h->a.n + 255) / 256, 256, 0, s>>>(h->a.cost, h->a.n, h->bucket_width, h->d_bucket, h->d_rank, h->d_counts);
  mjk_order_kernel<<<64, 256, 0, s>>>(h->d_bucket, h->d_rank, h->a.n, h->d_counts, h->d_order);
  CU(cudaGetLastError());
  if (h->h_redo_seen && h->a.redo_list) CU(cudaMemcpyAsync(h->h_redo_seen, h->a.sched + kRedoCount, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
  // auto reset: the envs whose horizon fired in this step, after the step, redo, bucket and order kernels (plain launch)
  if (h->a.flags & EARL_FLAG_AUTO_RESET)
    if (int rc = launch_task(h, 3, nullptr, h->a.n, nullptr, nullptr, obs_dev, nullptr, done_dev, nullptr, stream)) return rc;
  return 0;
}

int earl_mjk_get_state(earl_mjk_handle* h, double* qpos_host, double* qvel_host, double* warm_host, double* mocap_host, double* last_qp_host,
                       double* sites_host) {
  if (!h) return failf(EARL_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->eng->device));
  CU(cudaDeviceSynchronize());
  const size_t n = (size_t)h->a.n;
  std::vector<float> tmp(n * kNQ);
  const float* src[3] = {h->a.qpos, h->a.qvel, h->a.warm};
  double* dst[3] = {qpos_host, qvel_host, warm_host};
  for (int k = 0; k < 3; ++k) {
    if (!dst[k]) continue;
    CU(cudaMemcpy(tmp.data(), src[k], n * kNQ * sizeof(float), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n * kNQ; ++i) dst[k][i] = tmp[i];
  }
  if (mocap_host) CU(cudaMemcpy(mocap_host, h->a.mocap, n * 3 * sizeof(double), cudaMemcpyDeviceToHost));
  if (last_qp_host) CU(cudaMemcpy(last_qp_host, h->a.last_qp, n * kRobot * sizeof(double), cudaMemcpyDeviceToHost));
  if (sites_host) CU(cudaMemcpy(sites_host, h->a.sites, n * kSites * 3 * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

int earl_mjk_set_state(earl_mjk_handle* h, const double* qpos_host, const double* qvel_host, const double* warm_host,
                       const double* mocap_host, const double* last_qp_host) {
  if (!h) return failf(EARL_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->eng->device));
  CU(cudaDeviceSynchronize());
  const size_t n = (size_t)h->a.n;
  std::vector<float> tmp(n * kNQ);
  float* dst[3] = {h->a.qpos, h->a.qvel, h->a.warm};
  const double* src[3] = {qpos_host, qvel_host, warm_host};
  for (int k = 0; k < 3; ++k) {
    if (!src[k]) continue;
    for (size_t i = 0; i < n * kNQ; ++i) tmp[i] = (float)src[k][i];
    CU(cudaMemcpy(dst[k], tmp.data(), n * kNQ * sizeof(float), cudaMemcpyHostToDevice));
  }
  if (mocap_host) CU(cudaMemcpy(h->a.mocap, mocap_host, n * 3 * sizeof(double), cudaMemcpyHostToDevice));
  if (last_qp_host) CU(cudaMemcpy(h->a.last_qp, last_qp_host, n * kRobot * sizeof(double), cudaMemcpyHostToDevice));
  return 0;
}

int earl_mjk_counters(earl_mjk_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev, uint32_t* steps_since_reset_dev,
                      double* lifelong_return_dev, void* stream) {
  if (!h) return failf(EARL_ERR_INVALID, "null handle");
  CU(cudaSetDevice(h->eng->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t n = (size_t)h->a.n;
  if (total_steps_host) *total_steps_host = h->total_steps;
  if (num_interventions_dev) CU(cudaMemcpyAsync(num_interventions_dev, h->a.num_interventions, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
  if (steps_since_reset_dev) CU(cudaMemcpyAsync(steps_since_reset_dev, h->a.steps_since_reset, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
  if (lifelong_return_dev) CU(cudaMemcpyAsync(lifelong_return_dev, h->a.lifelong_return, n * sizeof(double), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int earl_mjk_work_counters(earl_mjk_handle* h, uint64_t* out7_host) {
  if (!h || !out7_host) return failf(EARL_ERR_INVALID, "null argument");
  CU(cudaSetDevice(h->eng->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(out7_host, h->a.work, 7 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  if (getenv("EARL_MJ_OVERFLOW_DETAIL")) {
    uint64_t d[12];
    CU(cudaMemcpy(d, h->a.work, sizeof(d), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[mjk overflow] env-steps with dropped candidate pairs %llu, dropped contacts %llu, dropped rows %llu\n",
            (unsigned long long)d[8], (unsigned long long)d[9], (unsigned long long)d[10]);
  }
  return 0;
}

int64_t earl_mjk_redo_count(earl_mjk_handle* h) {
  if (!h) return -1;
  unsigned long long v = 0;
  if (cudaSetDevice(h->eng->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
      cudaMemcpy(&v, h->a.work + 7, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess)
    return -1;
  return (int64_t)v;
}

}  // extern "C"
#endif  // MJK_XL
