/*
 * earl_mj_b200.h -- C ABI of the articulated-body half of libearl_b200.so: batched, device-resident step of the
 * reference's MuJoCo-backed Sawyer tasks (sawyer_door, sawyer_peg), one warp per environment instance.
 *
 * The reference has no FFI on this path: `SawyerDoorV2` / `SawyerPegV2` (earl_benchmark/envs/sawyer_door.py,
 * sawyer_peg.py) inherit metaworld's SawyerXYZEnv.step, which drives MuJoCo 2.1.0 through mujoco-py
 * (frame_skip x sim.step()).  Every entry point cites the reference METHOD it replaces.  Same conventions as
 * include/earl_b200.h: plain C, device pointers unless marked host, `stream` is a cudaStream_t passed as void*,
 * 0 = ok / <0 = earl_status (earl_last_error() has the message), no CPU fallback.
 */
#ifndef EARL_MJ_B200_H_
#define EARL_MJ_B200_H_

#include "earl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct earl_mj_handle earl_mj_handle;

typedef struct {
  int32_t env_kind;         /* EARL_ENV_SAWYER_DOOR or EARL_ENV_SAWYER_PEG */
  int32_t num_envs;
  int32_t device;
  uint32_t flags;           /* EARL_FLAG_EVAL_STATS | EARL_FLAG_LIFELONG | EARL_FLAG_DENSE_REWARD | EARL_FLAG_AUTO_RESET */
  int64_t episode_horizon;  /* PersistentStateWrapper(episode_horizon), persistent_state_wrapper.py:10-12 */
  int64_t goal_change_frequency; /* LifelongWrapper(goal_change_frequency), lifelong_wrapper.py:19-24; 0 = unused */
} earl_mj_config;

/* Task constants that live in the metaworld / EARL Python classes rather than in the MJCF. */
typedef struct {
  int32_t frame_skip;       /* SawyerXYZEnv frame_skip = 5 substeps per env step */
  int32_t hand_site;        /* site index of the 'hand' body frame (get_endeff_pos) */
  int32_t ree_site;         /* 'rightEndEffector' */
  int32_t lee_site;         /* 'leftEndEffector' */
  int32_t obj_geom;         /* door: geom 'handle' (sawyer_door.py:113 get_geom_xpos); -1 when the object is a site */
  int32_t obj_site;         /* peg: site 'pegHead' (sawyer_peg.py:186-187); -1 otherwise */
  int32_t max_newton;       /* cap on Newton iterations per substep (0 = the model's <option iterations>) */
  int32_t obj_qpos_count;   /* leading qpos entries of the object joint written by a reset: 1 door angle, 3 peg xyz (_set_obj_xyz) */
  float mocap_low[3];       /* hand_low */
  float mocap_high[3];      /* hand_high */
  float action_scale;       /* 1/100 (SawyerXYZEnv.action_scale) */
  float success_radius;     /* 0.02 door (sawyer_door.py:177), 0.05 peg (sawyer_peg.py:305) */
  float obj_init_pos[3];    /* dense door reward: self.obj_init_pos (sawyer_door.py:36,150) */
  float hand_init_pos[3];   /* dense door reward: self.hand_init_pos (sawyer_door.py:37-40,156) */
  /* dense peg reward (sawyer_peg.py:231-299); -1 when unused */
  int32_t grasp_site;       /* site 'pegGrasp' */
  int32_t lpad_site;        /* frame of body 'leftpad'  (get_body_com in metaworld's _gripper_caging_reward) */
  int32_t rpad_site;        /* frame of body 'rightpad' */
  int32_t corner_site[4];   /* bottom_right_corner_collision_box_1, top_left_..._1, bottom_right_..._2, top_left_..._2 */
} earl_mj_task;

/* model_blob: the serialized structure-of-arrays model written by earl_benchmark_b200.mjcf.compile.Model.to_blob()
 * (the reference loads the same MJCF through mujoco_py.load_model_from_path, sawyer_door.py:67-70).
 * Replaces constructing SawyerDoorV2 + PersistentStateWrapper, earl_benchmark/__init__.py:119-123,140-141. */
EARL_API int earl_mj_create(const earl_mj_config* cfg, const void* model_blob, size_t model_nbytes, const earl_mj_task* task,
                            earl_mj_handle** out);
EARL_API int earl_mj_destroy(earl_mj_handle* h);
EARL_API int earl_mj_obs_dim(const earl_mj_handle* h);    /* 14 */
EARL_API int earl_mj_action_dim(const earl_mj_handle* h); /* 4 */
EARL_API int earl_mj_nq(const earl_mj_handle* h);
EARL_API int earl_mj_nv(const earl_mj_handle* h);

/* Goal table, f64 [count,7] on the host (goal_states, sawyer_door.py:15-16; reset_goal(goal) for custom goals). */
EARL_API int earl_mj_set_goal_table(earl_mj_handle* h, const double* rows_host, int32_t count);

/* sim.reset() + SawyerXYZEnv._reset_hand(steps): from qpos0, `steps` times { mocap_pos <- hand_init_pos; mocap_quat <-
 * [1,0,1,0]; do_simulation(ctrl, frame_skip) }.  Deterministic, so it is run ONCE on the device and the resulting
 * state is kept as the reset template every later earl_mj_reset copies (sawyer_door.py:111-112). */
EARL_API int earl_mj_build_reset_template(earl_mj_handle* h, const double* hand_init_pos_host, const float* ctrl_host,
                                          int32_t steps);

/* Pre-drawn reset stream of an EARL_FLAG_AUTO_RESET handle: the random draws of reset_model() (sawyer_door.py:114-118,
 * sawyer_peg.py:192-229) for `rows` successive full resets, host arrays obj_qpos f64 [rows, N, obj_qpos_count] and, for
 * tasks whose reset draws the goal (peg reset_at_goal), goal_rows i32 [rows, N] (else NULL).  Every reset of such a handle
 * that is given no obj_qpos -- the reset pass after a step whose horizon fired, and earl_mj_reset(obj_qpos NULL) -- takes
 * the next row of each reset env's column through a per-env cursor, which wraps modulo `rows`.  goal_rows_dev i32 [N] is
 * the caller's array of current goal rows (reset_goal(), sawyer_door.py:100-102): those resets read their goal row from
 * it (and write the drawn one when goal_rows is given); it must stay allocated for the handle's lifetime.  Uploading
 * again (same `rows`) replaces the stream and rewinds the cursors. */
EARL_API int earl_mj_set_reset_stream(earl_mj_handle* h, const double* obj_qpos_host, const int32_t* goal_rows_host, int32_t rows,
                                      int32_t* goal_rows_dev);

/* PersistentStateWrapper.reset + reset_model (persistent_state_wrapper.py:17-20, sawyer_door.py:111-125) for every env
 * with mask[i] != 0 (NULL = all): state <- reset template, object joint <- obj_qpos[i,:] with zero velocity
 * (_set_obj_xyz), goal <- goal_idx[i] (NULL = row 0), num_interventions += 1, steps_since_reset = 0, then a fresh
 * forward-kinematics pass and the observation (obs_out may be NULL).  obj_qpos is f64 [N, obj_qpos_count] (door angle /
 * peg xyz; sawyer_peg.py:192-229): the host draws it from the bit-exact replica of the reference's np.random stream.
 * On an EARL_FLAG_AUTO_RESET handle obj_qpos NULL takes the draws and goal rows from the reset stream instead
 * (earl_mj_set_reset_stream; goal_idx is ignored) and writes the obs rows of the reset envs only. */
EARL_API int earl_mj_reset(earl_mj_handle* h, const uint8_t* mask_dev, const double* obj_qpos_dev, const int32_t* goal_idx_dev,
                           float* obs_out_dev, void* stream);

/* One PersistentStateWrapper.step of every env: SawyerXYZEnv.step (set_xyz_action, do_simulation = frame_skip x
 * mj_step), EARL observation + sparse reward (sawyer_door.py:86-94,168-177), counters and horizon `done`
 * (persistent_state_wrapper.py:22-31).  With EARL_FLAG_LIFELONG also LifelongWrapper.step (lifelong_wrapper.py:30-44):
 * lifelong_return += reward and, every goal_change_frequency steps, reset_goal() -- the observation of that step then
 * carries the new goal while the reward is the pre-swap one.  With EARL_FLAG_AUTO_RESET every env whose horizon fired
 * is then reset as earl_mj_reset(obj_qpos NULL) would reset it (one more launch in `stream`, after the step): reward,
 * done and success describe the step that ended, its obs row is the post-reset observation.  actions [N,4] f32;
 * obs [N,14] f32; reward [N] f32; done [N] u8; success [N] u8 or NULL. */
EARL_API int earl_mj_step(earl_mj_handle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
                          uint8_t* success_dev, void* stream);
/* Same with HOST buffers (copies inside the call, synchronous). */
EARL_API int earl_mj_step_host(earl_mj_handle* h, const float* actions_host, float* obs_host, float* reward_host,
                               uint8_t* done_host, uint8_t* success_host);
/* env._get_obs() from a fresh kinematics pass of the current state. */
EARL_API int earl_mj_get_obs(earl_mj_handle* h, float* obs_dev, void* stream);

/* Physics state of every env as host arrays (synchronous): qpos f64 [N,nq], qvel f64 [N,nv], qacc_warmstart f64 [N,nv],
 * mocap_pos f64 [N,3].  The engine keeps qpos / qvel / warm start in fp32 and mocap_pos in fp64.
 * Replaces sim.get_state() / sim.set_state() (mujoco-py), used by _set_obj_xyz and by state snapshots. */
EARL_API int earl_mj_get_state(earl_mj_handle* h, double* qpos_host, double* qvel_host, double* warm_host, double* mocap_host);
EARL_API int earl_mj_set_state(earl_mj_handle* h, const double* qpos_host, const double* qvel_host, const double* warm_host,
                               const double* mocap_host);

/* total_steps (host scalar), num_interventions i64 [N], steps_since_reset u32 [N], lifelong_return f64 [N]
 * (lifelong_wrapper.py:46-48; EARL_FLAG_LIFELONG handles only); arrays may be NULL. */
EARL_API int earl_mj_counters(earl_mj_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev,
                              uint32_t* steps_since_reset_dev, double* lifelong_return_dev, void* stream);
/* out4 = { sum of episode returns, #envs successful at their last step, #envs successful at any step since reset, N } */
EARL_API int earl_mj_eval_stats(earl_mj_handle* h, double* out4_dev, void* stream);
/* Work counters accumulated by the step kernel since creation (host): { env_steps, substeps, newton_iterations,
 * constraint_rows, contacts, bad_states (env steps with a non-positive Cholesky pivot), overflow_states (env steps in
 * which a fixed capacity -- 24 / 32 candidate pairs, 16 / 24 contacts, 64 / 96 rows for the door / peg capacity set
 * -- dropped work) }. */
EARL_API int earl_mj_work_counters(earl_mj_handle* h, uint64_t* out7_host);
EARL_API int64_t earl_mj_launch_count(const earl_mj_handle* h);
/* env-steps whose substep exceeded the handle's fixed capacities and were therefore re-stepped, from their untouched
 * pre-step record, by the extra-large capacity set (56 contacts / 224 rows) launched after every step kernel; they are
 * NOT counted in overflow_states (that counter now only sees steps that overflow the extra-large set as well).
 * EARL_MJ_REDO=0 at creation restores round 1's drop-and-count behaviour.  -1 on error. */
EARL_API int64_t earl_mj_redo_count(earl_mj_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* EARL_MJ_B200_H_ */
