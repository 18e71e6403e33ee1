/*
 * earl_b200.h -- C ABI of libearl_b200.so: batched, device-resident EARL environment step.
 *
 * The reference (architsharma97/earl_benchmark) has no FFI on this path: its boundary is a Python class
 * surface over mujoco-py.  Every entry point below therefore cites the reference METHOD it replaces
 * (paths relative to the reference root).  The Python package `earl_benchmark_b200` binds these with
 * ctypes and re-exposes the reference surface (EARLEnvs / PersistentStateWrapper / LifelongWrapper /
 * TabletopManipulation), with a leading environment dimension on every array.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; no torch / C++ types cross the boundary;
 *   - one handle per GPU, not thread-safe per handle;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); device-pointer entry
 *     points only ENQUEUE work on it and return; *_host entry points are synchronous;
 *   - the library never frees caller memory and the caller never frees library memory;
 *   - return value 0 = ok, <0 = error (earl_status); earl_last_error() gives a thread-local message.
 *     CUDA errors are sticky and surface at the next call.  There is NO CPU fallback: without a usable
 *     CUDA device every compute entry point fails with EARL_ERR_CUDA.
 *   - "dev" = device pointer, "host" = host pointer, [N,...] = row-major, N = num_envs.
 */
#ifndef EARL_B200_H_
#define EARL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EARL_ABI_VERSION 1

#if defined(EARL_MJ_INTERNAL) && defined(__GNUC__)
/* the library's own per-capacity-set translation units re-declare the entry points under internal names */
#define EARL_API __attribute__((visibility("hidden")))
#elif defined(__GNUC__)
#define EARL_API __attribute__((visibility("default")))
#else
#define EARL_API
#endif

typedef struct earl_handle earl_handle;
typedef struct earl_rng earl_rng;

typedef enum {
  EARL_OK = 0,
  EARL_ERR_INVALID = -1,     /* bad argument / unsupported combination */
  EARL_ERR_CUDA = -2,        /* CUDA runtime error (message has the cudaError string) */
  EARL_ERR_NOMEM = -3,
  EARL_ERR_UNSUPPORTED = -4  /* env kind not built yet */
} earl_status;

/* reference env names, earl_benchmark/__init__.py:112-138 */
typedef enum {
  EARL_ENV_TABLETOP = 0,     /* envs/tabletop_manipulation.py  (3 -> 12) */
  EARL_ENV_SAWYER_DOOR = 1,  /* envs/sawyer_door.py            (4 -> 14) */
  EARL_ENV_SAWYER_PEG = 2,   /* envs/sawyer_peg.py             (4 -> 14) */
  EARL_ENV_KITCHEN = 3       /* envs/kitchen.py                (9 -> 46) */
} earl_env_kind;

/* earl_config.flags */
#define EARL_FLAG_DENSE_REWARD 0x01u  /* reward_type='dense'  (tabletop_manipulation.py:179-189) */
#define EARL_FLAG_WIDE_INIT 0x02u     /* wide_init_distr: success judged on the object only (:201-202) */
#define EARL_FLAG_STATE_F64 0x04u     /* keep qpos in fp64 like the reference (bit-exact long rollouts; +32 B/step) */
#define EARL_FLAG_LIFELONG 0x08u      /* LifelongWrapper on device (wrappers/lifelong_wrapper.py:30-44) */
#define EARL_FLAG_AUTO_RESET 0x10u    /* reset inside the step kernel when the horizon fires (throughput runs) */
#define EARL_FLAG_RESET_AT_GOAL 0x20u /* reset_at_goal=True: resets place the env at its new goal (:109-111) */
#define EARL_FLAG_EVAL_STATS 0x40u    /* accumulate per-env episode return / success for earl_eval_stats */

typedef struct {
  int32_t env_kind;              /* earl_env_kind */
  int32_t num_envs;              /* N >= 1 */
  int32_t device;                /* CUDA device ordinal */
  uint32_t flags;                /* EARL_FLAG_* */
  int64_t episode_horizon;       /* PersistentStateWrapper(episode_horizon), persistent_state_wrapper.py:10-12 */
  int64_t goal_change_frequency; /* LifelongWrapper(goal_change_frequency), lifelong_wrapper.py:19-24; 0 = unused */
  int32_t goal_stream_rows;      /* R: rows of the pre-drawn per-env goal-index stream (see earl_set_goal_stream) */
  int32_t reserved;
} earl_config;

/* Tabletop "model blob": the constants the reference hard-codes (tabletop_manipulation.py:11-16,41-43,
 * 130-132,157,163,202-204).  The task is kinematic, so nothing of the MJCF is needed on the device. */
typedef struct {
  uint32_t magic;          /* EARL_TABLETOP_MAGIC */
  int32_t num_goals;       /* G <= 256 rows in goal_table */
  double threshold;        /* 0.4  attach radius (strict <) */
  double move_distance;    /* 0.2  action scale: a -> -d + (a+1)*0.5*(2d) */
  double clip;             /* 2.8  workspace clip */
  double success_radius;   /* 0.2  sparse success (<=) */
  double initial_state[6]; /* initial_states[0] */
  double goal_table[256][6]; /* candidate goals; rows 0..3 = goal_states, row 4 = initial_states[0] */
} earl_tabletop_model;
#define EARL_TABLETOP_MAGIC 0x54544142u /* 'TTAB' */

/* Pure host helper: the exact sqrt-free forms of the two radius tests the kernels use
 * (tabletop_manipulation.py:149 `dist < self.threshold`, :204 `norm <= 0.2`):
 *   sqrt(s) < threshold  <=>  s < *attach_sq   (fp64);   (double)sqrtf(s) <= success_radius  <=>  s <= *success_sq  (fp32) */
EARL_API void earl_tabletop_thresholds(double threshold, double success_radius, double* attach_sq, float* success_sq);

/* ---------------------------------------------------------------- lifecycle */

EARL_API int earl_abi_version(void);
EARL_API const char* earl_last_error(void);

/* Replaces constructing train/eval env + wrapper: EARLEnvs.get_train_env / get_eval_env,
 * earl_benchmark/__init__.py:112-171.  Allocates all per-env state on `cfg->device`. */
EARL_API int earl_create(const earl_config* cfg, const void* model_blob, size_t model_nbytes, earl_handle** out);
EARL_API int earl_destroy(earl_handle* h);

EARL_API int earl_num_envs(const earl_handle* h);
EARL_API int earl_obs_dim(const earl_handle* h);    /* 12 tabletop */
EARL_API int earl_action_dim(const earl_handle* h); /* 3 tabletop */

/* ---------------------------------------------------------------- goal stream
 * Pre-drawn goal-row indices, u8 [R,N] on the host, copied to the device.  Row e, column i is the goal
 * row env i takes at its e-th goal draw (reset, reset_goal(None) or lifelong goal swap); a per-env
 * cursor advances on every draw and wraps modulo R.  The host fills it from the bit-exact replica of
 * the reference's stream (earl_rng_* below), in the order a Python loop over N reference envs sharing
 * the global `random` module would consume it: draw e of env i = stream[e*N + i].
 * Replaces: random.sample(task_list, 1) in get_next_goal, tabletop_manipulation.py:62-76. */
EARL_API int earl_set_goal_stream(earl_handle* h, const uint8_t* rows_host, int32_t num_rows);

/* ---------------------------------------------------------------- reset / goals
 * PersistentStateWrapper.reset + env.reset (persistent_state_wrapper.py:17-20,
 * tabletop_manipulation.py:105-126) for every env with mask[i] != 0 (mask NULL = all):
 * num_interventions += 1, steps_since_reset = 0, attached cleared, goal <- goal_idx[i] if given else next
 * goal-stream draw, qpos <- init_qpos[i] if given, else the goal (RESET_AT_GOAL) or initial_states[0].
 * Lifelong handles also zero steps_since_goal_change (lifelong_wrapper.py:25-28).
 * Writes the post-reset observation rows of the masked envs to obs_out when non-NULL. */
EARL_API int earl_reset(earl_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev,
               const double* init_qpos_dev /*[N,4]*/, float* obs_out_dev /*[N,O]*/, void* stream);

/* env.reset_goal(goal) (tabletop_manipulation.py:78-81): goal_idx NULL = draw from the goal stream. */
EARL_API int earl_set_goal(earl_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev, void* stream);

/* Replace rows of the goal table (custom goals passed to reset_goal(goal)). */
EARL_API int earl_set_goal_table(earl_handle* h, const double* rows_host /*[count,6]*/, int32_t first_row, int32_t count);

/* ---------------------------------------------------------------- the hot path
 * One PersistentStateWrapper.step (persistent_state_wrapper.py:22-31) of every env, i.e. env.step
 * (tabletop_manipulation.py:128-174) + counters + horizon `done`, and LifelongWrapper.step
 * (lifelong_wrapper.py:30-44) when EARL_FLAG_LIFELONG.  All pointers are device pointers.
 *   actions [N,A] f32 in; obs [N,O] f32 out; reward [N] f32 out; done [N] u8 out;
 *   success [N] u8 out or NULL (is_successful of the new obs; equals reward in sparse mode). */
EARL_API int earl_step(earl_handle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
              uint8_t* success_dev, void* stream);

/* `num_steps` consecutive steps launched back to back without returning to the caller: step t reads
 * actions[t % action_ring] and writes obs/reward/done slot t % out_ring of the rollout buffers
 * ([ring,N,...]).  For open-loop action sequences (random-action throughput runs, demo replay). */
EARL_API int earl_rollout(earl_handle* h, const float* actions_dev, int32_t action_ring, int32_t num_steps, float* obs_dev,
                 float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, int32_t out_ring, void* stream);

/* Same step with HOST buffers, then a synchronise.  This is the call a CPU-side RL loop makes.
 * Pinned (mapped) 16-byte aligned buffers on the sparse fp32-state configuration: ONE launch of the
 * one-tile-per-CTA step kernel that reads the actions from and writes obs/reward/done(/success) to the
 * host buffers itself, full 128-byte lines over PCIe in both directions at once (no staging copies;
 * EARL_TT_HOST_ZEROCOPY=0 turns it off).  Otherwise: chunked pipeline of host->device copy, kernel,
 * device->host copies; pageable memory works there. */
EARL_API int earl_step_host(earl_handle* h, const float* actions_host, float* obs_host, float* reward_host,
                   uint8_t* done_host, uint8_t* success_host);

/* Chooses how earl_step_host moves data when the buffers allow both: 1 = the step kernel reads / writes the pinned host
 * buffers itself (best when this process has the host's PCIe / memory bandwidth to itself: +4 % at 1M envs, +30 % at 64k),
 * 0 = staged copy pipeline (measured better when several ranks share one host: 2 GPUs 0.99 vs 0.96 of the concurrent
 * ceiling).  Default 1 unless EARL_TT_HOST_ZEROCOPY says otherwise; the Python host side sets 0 when the job has more than
 * one rank on the node.  Results are identical either way. */
EARL_API int earl_set_host_zerocopy(earl_handle* h, int32_t enable);

/* env._get_obs() (tabletop_manipulation.py:55-60) for all envs. */
EARL_API int earl_get_obs(earl_handle* h, float* obs_dev, void* stream);

/* env.compute_reward(obs) / env.is_successful(obs) (tabletop_manipulation.py:176-204) on caller-supplied
 * observations [M,O]; either output may be NULL. */
EARL_API int earl_compute_reward(earl_handle* h, const float* obs_dev, int64_t num_obs, float* reward_dev,
                        uint8_t* success_dev, void* stream);

/* ---------------------------------------------------------------- counters / stats / snapshots
 * total_steps (persistent_state_wrapper.py:43-45) is one value for the batch (all envs step together);
 * per-env arrays may be NULL.  num_interventions (:39-41) i64 [N]; steps_since_reset u32 [N] (saturating);
 * lifelong_return (lifelong_wrapper.py:46-48) f64 [N], lifelong handles only. */
EARL_API int earl_counters(earl_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev,
                  uint32_t* steps_since_reset_dev, double* lifelong_return_dev, void* stream);

/* Per-evaluation statistics over the envs of THIS handle (EARL_FLAG_EVAL_STATS), reduced on the device:
 * out4 = { sum of episode returns, number of envs successful at their last step,
 *          number of envs successful at any step since reset, N }.  Multi-GPU callers all-reduce out4
 * (the only collective of the system).  Resetting an env clears its accumulators. */
EARL_API int earl_eval_stats(earl_handle* h, double* out4_dev, void* stream);

/* Snapshot of all per-env state incl. counters (fp64 qpos [N,4], attached, goal index, counters).
 * earl_state_nbytes gives the buffer size; layout is documented in DESIGN.md. Host buffers, synchronous. */
EARL_API size_t earl_state_nbytes(const earl_handle* h);
EARL_API int earl_get_state(earl_handle* h, void* dst_host, size_t nbytes);
EARL_API int earl_set_state(earl_handle* h, const void* src_host, size_t nbytes);

/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
EARL_API int64_t earl_launch_count(const earl_handle* h);

/* ---------------------------------------------------------------- bit-exact host RNG streams
 * MT19937 replicas of the three host generators the reference draws indices and initial states from
 * (SURVEY.md Appendix D).  Pure host code.
 *   kind 0: CPython `random.seed(int)` (init_by_array over the 32-bit limbs of |seed|)
 *   kind 1: legacy numpy `np.random.seed(uint32)` (init_genrand) */
EARL_API earl_rng* earl_rng_create(int32_t kind, const uint32_t* seed_limbs, int32_t num_limbs);
EARL_API void earl_rng_destroy(earl_rng* r);
EARL_API uint32_t earl_rng_next_u32(earl_rng* r);
/* CPython random._randbelow_with_getrandbits(n): used by random.sample(list, 1) -> index */
EARL_API void earl_rng_py_randbelow(earl_rng* r, uint32_t n, int64_t count, int32_t* out);
/* tabletop get_next_goal(): random.sample(task_list.split('-'), 1) mapped to goal-table rows through
 * `task_to_row` (4 entries for 'rc_r-rc_k-rc_g-rc_b' -> rows 0,3,1,2), tabletop_manipulation.py:62-76 */
EARL_API void earl_rng_tabletop_goal_rows(earl_rng* r, const uint8_t* task_to_row, uint32_t num_tasks, int64_t count,
                                 uint8_t* out);
/* legacy numpy randint(0, n): masked rejection on 32-bit draws; n == 1 consumes nothing */
EARL_API void earl_rng_np_randint(earl_rng* r, uint32_t n, int64_t count, int32_t* out);
/* legacy numpy uniform(low, high): 53-bit double from two draws */
EARL_API void earl_rng_np_uniform(earl_rng* r, double low, double high, int64_t count, double* out);
/* SawyerPegV2.reset_model's draws (sawyer_peg.py:192-229) for `count` successive environments on a legacy numpy stream, as
 * the batched env's _draw_one() makes them: the goal row (0, or 1 + randint(15) when reset_at_goal) and the peg position
 * (the 6-uniform _get_state_rand_vec redrawn while within 0.1 of the block, the wide_init mix of that and a jittered
 * wide_initial_states row, or the jittered goal position when reset_at_goal).  rows_out i32 [count], pos_out f64 [count,3]. */
EARL_API void earl_rng_peg_reset_draws(earl_rng* r, int32_t wide_init, int32_t reset_at_goal, int64_t count, int32_t* rows_out,
                                       double* pos_out);

#ifdef __cplusplus
}
#endif
#endif /* EARL_B200_H_ */
