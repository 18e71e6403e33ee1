// entry points and handle type of the "extra large" capacity set (see earl_mj_impl.inc); internal to the library
#pragma once
#define EARL_MJ_INTERNAL 1
#define earl_mj_handle earl_mjx_handle
#define earl_mj_create earl_mjx_create
#define earl_mj_destroy earl_mjx_destroy
#define earl_mj_obs_dim earl_mjx_obs_dim
#define earl_mj_action_dim earl_mjx_action_dim
#define earl_mj_nq earl_mjx_nq
#define earl_mj_nv earl_mjx_nv
#define earl_mj_set_goal_table earl_mjx_set_goal_table
#define earl_mj_build_reset_template earl_mjx_build_reset_template
#define earl_mj_set_reset_stream earl_mjx_set_reset_stream
#define earl_mj_reset earl_mjx_reset
#define earl_mj_step earl_mjx_step
#define earl_mj_step_host earl_mjx_step_host
#define earl_mj_get_obs earl_mjx_get_obs
#define earl_mj_get_state earl_mjx_get_state
#define earl_mj_set_state earl_mjx_set_state
#define earl_mj_counters earl_mjx_counters
#define earl_mj_eval_stats earl_mjx_eval_stats
#define earl_mj_work_counters earl_mjx_work_counters
#define earl_mj_launch_count earl_mjx_launch_count
#define earl_mj_redo_pass earl_mjx_redo_pass
#define earl_mj_redo_count earl_mjx_redo_count
