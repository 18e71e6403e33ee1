/*
 * earl_tt3_b200.h -- C ABI of the three-object tabletop task inside libearl_b200.so.
 *
 * Replaces `earl_benchmark/envs/tabletop_manipulation_3obj.py` (class TabletopManipulation, the variant with
 * three draggable objects and closest-object attach) under a PersistentStateWrapper
 * (`earl_benchmark/wrappers/persistent_state_wrapper.py:17-45`).  The reference has no FFI on this path;
 * each entry point cites the Python method it replaces.  Conventions are those of earl_b200.h (plain C,
 * 0 = ok / <0 = earl_status, earl_last_error(), device pointers unless the name ends in _host, work is
 * only ENQUEUED on `stream`, no CPU fallback).
 *
 * Per-env state: qpos[0:8] as fp64 (fist x,y, object A x,y, object B x,y, object C x,y) like the
 * reference keeps it in MuJoCo's qpos, so open-loop rollouts of any length are bit-exact; one u32 of flags
 * (bits 0-1 attached object: 0 none, 1..3 = object_dict entries (0,0) / (0.5,0.5) / (1,1),
 * tabletop_manipulation_3obj.py:31-35; bits 2-3 success at the last / at any step of the episode, kept with
 * EARL_FLAG_EVAL_STATS; bits 8-15 goal row), u32 steps_since_reset, i64 num_interventions, and with
 * EARL_FLAG_EVAL_STATS an f64 episode return.
 * Observation [N,20] f32 = qpos[0:8], attached marker x2, goal[0:10]  (:49-54).
 */
#ifndef EARL_TT3_B200_H_
#define EARL_TT3_B200_H_

#include "earl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct earl_tt3_handle earl_tt3_handle;

#define EARL_TT3_MAX_GOALS 16

typedef struct {
  int32_t num_envs;          /* N >= 1 */
  int32_t device;            /* CUDA device ordinal */
  uint32_t flags;            /* EARL_FLAG_DENSE_REWARD | EARL_FLAG_AUTO_RESET | EARL_FLAG_RESET_AT_GOAL |
                                EARL_FLAG_EVAL_STATS | EARL_FLAG_FINAL_OBS (earl_b200.h; the last only with
                                EARL_FLAG_AUTO_RESET, else EARL_ERR_INVALID); any other flag is EARL_ERR_UNSUPPORTED */
  int32_t num_goals;         /* rows used in goal_table, 1..EARL_TT3_MAX_GOALS (reference: 1, :12-18) */
  int64_t episode_horizon;   /* PersistentStateWrapper(episode_horizon) */
  double threshold;          /* 0.4  attach radius, strict <            (:38, :107) */
  double move_distance;      /* 0.2  action scale                       (:39, :88-89) */
  double clip;               /* 2.8  workspace clip                     (:113, :119) */
  double success_radius;     /* 0.4  sparse success, <=                 (:165) */
  double initial_state[10];  /* initial_states[0]                       (:11) */
  double goal_table[EARL_TT3_MAX_GOALS][10]; /* goal_states             (:12-18) */
} earl_tt3_config;

/* construct env + wrapper (tabletop_manipulation_3obj.py:25-47, persistent_state_wrapper.py:10-15) */
EARL_API int earl_tt3_create(const earl_tt3_config* cfg, size_t cfg_nbytes, earl_tt3_handle** out);
EARL_API int earl_tt3_destroy(earl_tt3_handle* h);

/* PersistentStateWrapper.reset + env.reset (:17-20; tabletop_manipulation_3obj.py:67-84) for envs with
 * mask[i] != 0 (NULL = all): num_interventions += 1, steps_since_reset = 0, attached cleared,
 * goal row <- goal_idx[i] (NULL = row 0), qpos[0:8] <- init_qpos[i] when given (the host computes
 * goal[:8] + uniform(-0.3, 0.3) for reset_at_goal, :72-76).  With init_qpos NULL: on a handle with
 * EARL_FLAG_AUTO_RESET | EARL_FLAG_RESET_AT_GOAL each masked env's next reset-stream row (earl_tt3_set_reset_stream;
 * EARL_ERR_INVALID before one is set), else initial_state[0:8].  Clears the episode statistics (EARL_FLAG_EVAL_STATS).
 * Writes the post-reset observation rows of the masked envs to obs_out when non-NULL. */
EARL_API int earl_tt3_reset(earl_tt3_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev,
                            const double* init_qpos_dev /*[N,8]*/, float* obs_out_dev /*[N,20]*/, void* stream);

/* env.reset_goal(goal) (:61-64): goal row per env (NULL = row 0 for every masked env) */
EARL_API int earl_tt3_set_goal(earl_tt3_handle* h, const uint8_t* mask_dev, const int32_t* goal_idx_dev, void* stream);

/* The hot path: PersistentStateWrapper.step (:22-31) over env.step + move + _get_obs + compute_reward
 * (tabletop_manipulation_3obj.py:86-165).  actions [N,3] f32 in; obs [N,20] f32, reward [N] f32,
 * done [N] u8, success [N] u8 (nullable) out.
 * EARL_FLAG_EVAL_STATS: episode_return += (double)reward, and the success bits are updated, every step.
 * EARL_FLAG_AUTO_RESET: an env whose horizon fired is then reset, in the same kernel, as earl_tt3_reset(mask, goal_idx
 * NULL, init_qpos NULL) resets it: reward, done and success describe the step that ended, its obs row is the post-reset
 * observation. */
EARL_API int earl_tt3_step(earl_tt3_handle* h, const float* actions_dev, float* obs_dev, float* reward_dev,
                           uint8_t* done_dev, uint8_t* success_dev, void* stream);

/* Final observations of an EARL_FLAG_AUTO_RESET | EARL_FLAG_FINAL_OBS handle (EARL_ERR_INVALID on any other handle, and
 * from every step of such a handle before this is called): final_obs [N,20] f32, device, 16-byte aligned, owned by the
 * caller and kept until the handle is destroyed or another buffer is registered.  After a step (earl_tt3_step /
 * earl_tt3_step_host) in which done[i] is set, row i of final_obs is bit for bit the observation row the same handle
 * would have returned from that step without auto-reset (qpos[0:8], attached marker, goal before the reset); the step's
 * obs row i stays the post-reset observation.  Rows of envs that did not finish are not written.  Written by the step
 * kernel inside its fused reset (no extra launch, 80 B per reset env); every other output and all state, statistics and
 * reset-stream cursors are what the handle without the flag computes.  earl_tt3_rollout refuses such a handle. */
EARL_API int earl_tt3_set_final_obs(earl_tt3_handle* h, float* final_obs_dev);

/* `num_steps` steps back to back: step t reads actions[t % action_ring], writes output slot t % out_ring
 * (EARL_ERR_INVALID on an EARL_FLAG_FINAL_OBS handle) */
EARL_API int earl_tt3_rollout(earl_tt3_handle* h, const float* actions_dev, int32_t action_ring, int32_t num_steps,
                              float* obs_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev,
                              int32_t out_ring, void* stream);

/* same step with HOST buffers (copies inside the call, synchronous): the call a CPU-side RL loop makes */
EARL_API int earl_tt3_step_host(earl_tt3_handle* h, const float* actions_host, float* obs_host, float* reward_host,
                                uint8_t* done_host, uint8_t* success_host);

/* Pre-drawn reset stream of an EARL_FLAG_AUTO_RESET | EARL_FLAG_RESET_AT_GOAL handle (EARL_ERR_INVALID on any other):
 * host array f64 [rows, N, 8], row e of env i = the qpos[0:8] of env i's e-th reset (goal[:8] + uniform(-0.3, 0.3),
 * :72-76).  Every reset that is given no init_qpos -- an auto-reset in the step and earl_tt3_reset(init_qpos NULL) --
 * takes the next row of the env's column through a per-env cursor, which wraps modulo `rows`.  Must be set before the
 * first step or reset of such a handle.  Setting it again (same `rows`) replaces the rows and rewinds the cursors.
 * Device memory: 64 * rows + 4 bytes per env.  Synchronous. */
EARL_API int earl_tt3_set_reset_stream(earl_tt3_handle* h, const double* qpos_rows_host, int32_t rows);

/* EARL_FLAG_EVAL_STATS: (sum of episode returns, #envs successful at their last step, #envs successful at any step of
 * the episode, N) -> out4_dev f64 [4], reduced on the device.  A reset clears an env's statistics. */
EARL_API int earl_tt3_eval_stats(earl_tt3_handle* h, double* out4_dev, void* stream);

/* env._get_obs() (:49-54) */
EARL_API int earl_tt3_get_obs(earl_tt3_handle* h, float* obs_dev, void* stream);

/* env.compute_reward(obs) / env.is_successful(obs) (:146-165) on caller observations [M,20] */
EARL_API int earl_tt3_compute_reward(earl_tt3_handle* h, const float* obs_dev, int64_t num_obs, float* reward_dev,
                                     uint8_t* success_dev, void* stream);

/* total_steps / num_interventions / steps_since_reset (persistent_state_wrapper.py:39-45) */
EARL_API int earl_tt3_counters(earl_tt3_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev,
                               uint32_t* steps_since_reset_dev, void* stream);

/* env.sim.data.qpos[:8] and the attached object (0 none, 1..3); either pointer may be NULL */
EARL_API int earl_tt3_get_state(earl_tt3_handle* h, double* qpos_dev /*[N,8]*/, int32_t* attached_dev, void* stream);
EARL_API int earl_tt3_set_state(earl_tt3_handle* h, const double* qpos_dev /*[N,8]*/, const int32_t* attached_dev,
                                void* stream);

EARL_API int64_t earl_tt3_launch_count(const earl_tt3_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* EARL_TT3_B200_H_ */
