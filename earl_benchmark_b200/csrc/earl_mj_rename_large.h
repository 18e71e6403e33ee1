// entry points and handle type of the "large" capacity set (see earl_mj_impl.inc); internal to the library
#pragma once
#define EARL_MJ_INTERNAL 1
#define earl_mj_handle earl_mjl_handle
#define earl_mj_create earl_mjl_create
#define earl_mj_destroy earl_mjl_destroy
#define earl_mj_obs_dim earl_mjl_obs_dim
#define earl_mj_action_dim earl_mjl_action_dim
#define earl_mj_nq earl_mjl_nq
#define earl_mj_nv earl_mjl_nv
#define earl_mj_set_goal_table earl_mjl_set_goal_table
#define earl_mj_build_reset_template earl_mjl_build_reset_template
#define earl_mj_set_reset_stream earl_mjl_set_reset_stream
#define earl_mj_reset earl_mjl_reset
#define earl_mj_step earl_mjl_step
#define earl_mj_step_host earl_mjl_step_host
#define earl_mj_get_obs earl_mjl_get_obs
#define earl_mj_get_state earl_mjl_get_state
#define earl_mj_set_state earl_mjl_set_state
#define earl_mj_counters earl_mjl_counters
#define earl_mj_eval_stats earl_mjl_eval_stats
#define earl_mj_work_counters earl_mjl_work_counters
#define earl_mj_launch_count earl_mjl_launch_count
#define earl_mj_redo_pass earl_mjl_redo_pass
#define earl_mj_redo_count earl_mjl_redo_count
