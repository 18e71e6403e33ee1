/*
 * earl_mj_kitchen_b200.h -- ENGINE-LEVEL entry points of the kitchen capacity set of libearl_b200.so (round 1).
 *
 * The reference's kitchen step is KitchenV0.step -> Robot.step -> MujocoEnv.do_simulation =
 * 40 x sim.step() (kitchen_assets/adept_envs/adept_envs/franka/kitchen_multitask_v0.py:91-125,
 * adept_envs/mujoco_env.py:148-153) on franka_kitchen_jntpos_act_ab.xml: 23 dofs, 118 colliding geoms, friction loss on
 * every dof, 5 joint equalities, pyramidal friction cones.  What is declared here replaces the `n x sim.step()` part on
 * caller-held state arrays, one warp per environment instance, so that the device engine of this capacity set can be
 * checked against the fp64 checker and measured; the task-level ABI follows below.
 * Same conventions as include/earl_b200.h; all arrays are DEVICE pointers; no CPU fallback.
 */
#ifndef EARL_MJ_KITCHEN_B200_H_
#define EARL_MJ_KITCHEN_B200_H_

#include "earl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct earl_mjk_engine earl_mjk_engine;

/* model_blob: earl_benchmark_b200/models/kitchen.npz serialized by Model.to_blob() (blob version 2).
 * Replaces mujoco_py.load_model_from_path + MjSim (adept_envs/simulation/sim_robot.py:67-69). */
EARL_API int earl_mjk_engine_create(const void* model_blob, size_t model_nbytes, int32_t device, earl_mjk_engine** out);
EARL_API int earl_mjk_engine_destroy(earl_mjk_engine* e);
EARL_API int earl_mjk_engine_nv(const earl_mjk_engine* e);

/* `nsub` x mj_step for every environment (sim.step(), adept_envs/mujoco_env.py:152-153).
 * In / out: qpos, qvel, qacc_warmstart f32 [N, nv].  In: mocap_pos f64 [N,3], mocap_quat f32 [4] (one for all: the task
 * never moves it), ctrl f32 [N,2] (the engine clamps to ctrlrange).  Out: info i32 [N,4] = { rows of the last substep,
 * contacts of the last substep, Newton iterations summed over the substeps, flags (bit 0 non-positive pivot, bits 1-3
 * capacity overflow: candidate pairs / contacts / rows, bit 4: the primary 112-row set overflowed and the environment was
 * re-run from its input state by the 544-row set -- bits 1-3 then refer to that run) }. */
EARL_API int earl_mjk_engine_substeps(earl_mjk_engine* e, int32_t num_envs, int32_t nsub, float* qpos_dev, float* qvel_dev,
                                      float* warm_dev, const double* mocap_pos_dev, const float* mocap_quat_host,
                                      const float* ctrl_dev, int32_t* info_dev, void* stream);

/* ------------------------------------------------------------------------------------------------ task level
 * The reference's Kitchen task (earl_benchmark/envs/kitchen.py over adept_envs KitchenV0 / Robot_VelAct), batched and
 * device resident, with the PersistentStateWrapper / LifelongWrapper bookkeeping fused in like on the other tasks.
 * Observations and rewards are float64 as in the reference (46 x f64); the engine state is float32. */
typedef struct earl_mjk_handle earl_mjk_handle;

typedef struct {
  int32_t num_envs, device;
  uint32_t flags;                 /* EARL_FLAG_LIFELONG | EARL_FLAG_AUTO_RESET | EARL_FLAG_EVAL_STATS | EARL_FLAG_FINAL_OBS
                                     (the last with EARL_FLAG_AUTO_RESET only; any other flag is rejected) */
  int32_t frame_skip;             /* 40 (KitchenV0.__init__, kitchen_multitask_v0.py:38) */
  int64_t episode_horizon;        /* PersistentStateWrapper(episode_horizon) */
  int64_t goal_change_frequency;  /* LifelongWrapper(goal_change_frequency), lifelong_wrapper.py:19-24; 0 = unused */
  double goal[23];                /* ENV/kitchen.py:28-52 */
  double init_qpos[23];           /* kitchen_multitask_v0.py:65-70 */
  double pos_noise_amp[23];       /* franka/robot/franka_config.xml:17-45 */
  double pos_bound[9][2], vel_bound[9][2];
  double midpoint[3], mocap_low[3], mocap_high[3];   /* kitchen_multitask_v0.py:44-48 */
  double noise_ratio;             /* 0.1 (:41) */
  int32_t site[8];                /* site ids in the order burner0..3 (knob1..4_site), light_switch, slide_cabinet,
                                     hinge_cabinet, microwave (ENV/kitchen.py:149-156 via component_to_state_idx :15-25) */
} earl_mjk_config;

EARL_API int earl_mjk_create(const earl_mjk_config* cfg, const void* model_blob, size_t model_nbytes, earl_mjk_handle** out);
EARL_API int earl_mjk_destroy(earl_mjk_handle* h);
/* env.seed(): one PCG64 stream per environment, { state_hi, state_lo, inc_hi, inc_lo } u64 [N,4] on the HOST, taken from
 * numpy's PCG64(SeedSequence(seed)) exactly as gym 0.23.1 seeding.np_random builds env.np_random
 * (adept_envs/mujoco_env.py:113-118). */
EARL_API int earl_mjk_seed(earl_mjk_handle* h, const uint64_t* pcg_state_host);
/* Pre-drawn reset stream of an EARL_FLAG_AUTO_RESET handle: reset_model's np.random.randint(K) (ENV/kitchen.py:122-124)
 * for `rows` successive full resets, config u8 [rows, N] on the HOST, indexing table f64 [num_configs, 14] (HOST, the object
 * qpos of each initial configuration; single-component tasks: one row and an all-zero config).  Every reset of such a handle
 * that is given no object_qpos -- the reset pass after a step whose horizon fired, and earl_mjk_reset(object_qpos NULL) --
 * takes the next entry of each reset env's column through a per-env cursor, which wraps modulo `rows`.  Uploading again
 * (same shape) replaces the stream and rewinds the cursors. */
EARL_API int earl_mjk_set_reset_stream(earl_mjk_handle* h, const uint8_t* config_host, int32_t rows, const double* table_host,
                                       int32_t num_configs);
/* Kitchen.reset_model (ENV/kitchen.py:118-139) for the `count` environments listed in env_ids_dev (NULL = all):
 * qpos <- init_qpos with objects 9.. of object_qpos_dev [count,14] (the drawn initial configuration), zero velocity,
 * robot.reset's five cached observations at noise ratio 1, mocap <- midpoint, 10 x (40 substeps with the control computed
 * from the fifth of them), then the observation (obs_out_dev f64 [count,46], may be NULL).  object_qpos_dev NULL (auto-reset
 * handles only): the configuration is each env's next draw of the reset stream (earl_mjk_set_reset_stream). */
EARL_API int earl_mjk_reset(earl_mjk_handle* h, const int32_t* env_ids_dev, int32_t count, const double* object_qpos_dev,
                            double* obs_out_dev, void* stream);
/* One PersistentStateWrapper.step of every environment: KitchenV0.step (kitchen_multitask_v0.py:91-125: action clip and
 * scale, mocap update, Robot_VelAct control from the LAST NOISY observation, 40 x mj_step), the noisy observation
 * (franka_robot.py:137-168), Kitchen._get_reward_n_score / is_successful (ENV/kitchen.py:141-183), counters and horizon
 * done.  With EARL_FLAG_LIFELONG also LifelongWrapper.step (lifelong_wrapper.py:30-44): lifelong_return += reward and,
 * every goal_change_frequency steps, reset_goal() (one goal: no change) followed by env._get_obs() -- a SECOND noisy
 * observation (46 more draws), which is the one returned and the one the next control is computed from.  With
 * EARL_FLAG_AUTO_RESET every environment whose horizon fired is then reset as earl_mjk_reset(object_qpos NULL) would reset it
 * (one more launch in `stream`, after the step, redo and ordering kernels): reward, done and success describe the step that
 * ended, its obs row is the post-reset observation.  actions f32 [N,9]; obs f64 [N,46]; reward f64 [N]; done u8 [N]; success
 * u8 [N] or NULL. */
EARL_API int earl_mjk_step(earl_mjk_handle* h, const float* actions_dev, double* obs_dev, double* reward_dev, uint8_t* done_dev,
                           uint8_t* success_dev, void* stream);
/* Final observations of an EARL_FLAG_AUTO_RESET | EARL_FLAG_FINAL_OBS handle (EARL_ERR_INVALID on any other handle, and
 * from every step of such a handle before this is called): final_obs f64 [N,46], device, owned by the caller and kept
 * until the handle is destroyed or another buffer is registered.  After an earl_mjk_step in which done[i] is set, row i of
 * final_obs is bit for bit the observation row the same handle would have returned from that step without auto-reset:
 * the noisy observation (the lifelong second draw when the goal swap fell on that step), as the step or redo kernel wrote
 * it; the step's obs row i stays the post-reset observation.  Rows of envs that did not finish are not written.  One more
 * launch per step, in `stream` between the ordering kernels and the reset pass, copying the rows of the reset envs only;
 * every other output and all state, statistics, noise streams and reset-stream cursors are what the handle without the
 * flag computes. */
EARL_API int earl_mjk_set_final_obs(earl_mjk_handle* h, double* final_obs_dev);
/* sim state as host arrays (synchronous): qpos, qvel, qacc_warmstart f64 [N,23], mocap_pos f64 [N,3], last noisy robot
 * qpos f64 [N,9] (the Robot_VelAct observation cache), site positions f64 [N,8,3] of the last forward pass. NULL = skip. */
EARL_API int earl_mjk_get_state(earl_mjk_handle* h, double* qpos_host, double* qvel_host, double* warm_host, double* mocap_host,
                                double* last_qp_host, double* sites_host);
EARL_API int earl_mjk_set_state(earl_mjk_handle* h, const double* qpos_host, const double* qvel_host, const double* warm_host,
                                const double* mocap_host, const double* last_qp_host);
/* total_steps (host), num_interventions i64 [N], steps_since_reset u32 [N], lifelong_return f64 [N] (device, may be NULL) */
EARL_API int earl_mjk_counters(earl_mjk_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev,
                               uint32_t* steps_since_reset_dev, double* lifelong_return_dev, void* stream);
/* EARL_FLAG_EVAL_STATS: out4_dev f64 [4] = { sum over envs of the episode return, #envs successful at their last step,
 * #envs successful at any step, N }.  Every step adds the reward it returns to its env's return and records the success
 * it returns (a failed step adds 0 and is not successful); any reset of an env -- earl_mjk_reset, masked or not, and the
 * auto-reset after a step -- clears its statistics.  Without auto-reset, steps past the horizon keep accumulating.
 * Zeroes out4 and reduces in `stream`, on the device, in one block: the same per-env values give the same bits on every
 * call.  EARL_ERR_INVALID on a handle created without the flag. */
EARL_API int earl_mjk_eval_stats(earl_mjk_handle* h, double* out4_dev, void* stream);
/* { env_steps, substeps, newton_iterations, constraint_rows, contacts, bad_states, overflow_states } since creation */
EARL_API int earl_mjk_work_counters(earl_mjk_handle* h, uint64_t* out7_host);
/* env steps re-stepped by the extra-large capacity set since creation (a substep of theirs outgrew the 112 rows / 24 contacts of the primary set;
 * overflow_states counts what even that set could not hold, or every overflow when EARL_MJ_REDO=0); -1 on error */
EARL_API int64_t earl_mjk_redo_count(earl_mjk_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* EARL_MJ_KITCHEN_B200_H_ */
