// entry points and handle type of the "small" capacity set (see earl_mj_impl.inc); internal to the library
#pragma once
#define EARL_MJ_INTERNAL 1
#define earl_mj_handle earl_mjs_handle
#define earl_mj_create earl_mjs_create
#define earl_mj_destroy earl_mjs_destroy
#define earl_mj_obs_dim earl_mjs_obs_dim
#define earl_mj_action_dim earl_mjs_action_dim
#define earl_mj_nq earl_mjs_nq
#define earl_mj_nv earl_mjs_nv
#define earl_mj_set_goal_table earl_mjs_set_goal_table
#define earl_mj_build_reset_template earl_mjs_build_reset_template
#define earl_mj_set_reset_stream earl_mjs_set_reset_stream
#define earl_mj_reset earl_mjs_reset
#define earl_mj_step earl_mjs_step
#define earl_mj_step_host earl_mjs_step_host
#define earl_mj_get_obs earl_mjs_get_obs
#define earl_mj_get_state earl_mjs_get_state
#define earl_mj_set_state earl_mjs_set_state
#define earl_mj_counters earl_mjs_counters
#define earl_mj_eval_stats earl_mjs_eval_stats
#define earl_mj_work_counters earl_mjs_work_counters
#define earl_mj_launch_count earl_mjs_launch_count
#define earl_mj_redo_pass earl_mjs_redo_pass
#define earl_mj_redo_count earl_mjs_redo_count
