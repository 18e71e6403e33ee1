// earl_mj.cu -- the exported entry points of include/earl_mj_b200.h.  The engine is compiled twice from the same sources
// with different fixed capacities (earl_mj_small.cu: 16 contacts / 64 rows, 16 environments in flight per SM;
// earl_mj_large.cu: 24 contacts / 96 rows, 12 per SM); a handle belongs to one of them, chosen by task at creation:
// sawyer_door -> small, sawyer_peg -> large (the peg pushed into the block exceeds 16 contacts in ~1 % of random-action
// steps).  EARL_MJ_CAPSET=small|large overrides the choice (measurements).
#include "../../include/earl_mj_b200.h"

#include <cstdlib>
#include <cstring>
#include <new>

namespace earl {
int set_error(int code, const char* msg);  // earl_b200.cu
}

struct earl_mj_handle {
  int set;     // 0 small, 1 large
  void* impl;  // earl_mjs_handle* / earl_mjl_handle*
};

extern "C" {
// the two capacity sets (hidden visibility; handles passed as void*)
int earl_mjs_create(const earl_mj_config* cfg, const void* model_blob, size_t model_nbytes, const earl_mj_task* task, void** out);
int earl_mjl_create(const earl_mj_config* cfg, const void* model_blob, size_t model_nbytes, const earl_mj_task* task, void** out);
int earl_mjs_destroy(void* h);
int earl_mjl_destroy(void* h);
int earl_mjs_obs_dim(const void* h);
int earl_mjl_obs_dim(const void* h);
int earl_mjs_action_dim(const void* h);
int earl_mjl_action_dim(const void* h);
int earl_mjs_nq(const void* h);
int earl_mjl_nq(const void* h);
int earl_mjs_nv(const void* h);
int earl_mjl_nv(const void* h);
int earl_mjs_set_goal_table(void* h, const double* rows_host, int32_t count);
int earl_mjl_set_goal_table(void* h, const double* rows_host, int32_t count);
int earl_mjs_build_reset_template(void* h, const double* hand_init_pos_host, const float* ctrl_host, int32_t steps);
int earl_mjl_build_reset_template(void* h, const double* hand_init_pos_host, const float* ctrl_host, int32_t steps);
int earl_mjs_set_reset_stream(void* h, const double* obj_qpos_host, const int32_t* goal_rows_host, int32_t rows, int32_t* goal_rows_dev);
int earl_mjl_set_reset_stream(void* h, const double* obj_qpos_host, const int32_t* goal_rows_host, int32_t rows, int32_t* goal_rows_dev);
int earl_mjs_reset(void* h, const uint8_t* mask_dev, const double* obj_qpos_dev, const int32_t* goal_idx_dev, float* obs_out_dev, void* stream);
int earl_mjl_reset(void* h, const uint8_t* mask_dev, const double* obj_qpos_dev, const int32_t* goal_idx_dev, float* obs_out_dev, void* stream);
int earl_mjs_step(void* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, void* stream);
int earl_mjl_step(void* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, void* stream);
int earl_mjs_step_host(void* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host, uint8_t* success_host);
int earl_mjl_step_host(void* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host, uint8_t* success_host);
int earl_mjs_get_obs(void* h, float* obs_dev, void* stream);
int earl_mjl_get_obs(void* h, float* obs_dev, void* stream);
int earl_mjs_get_state(void* h, double* qpos_host, double* qvel_host, double* warm_host, double* mocap_host);
int earl_mjl_get_state(void* h, double* qpos_host, double* qvel_host, double* warm_host, double* mocap_host);
int earl_mjs_set_state(void* h, const double* qpos_host, const double* qvel_host, const double* warm_host, const double* mocap_host);
int earl_mjl_set_state(void* h, const double* qpos_host, const double* qvel_host, const double* warm_host, const double* mocap_host);
int earl_mjs_counters(void* h, int64_t* total_steps_host, int64_t* num_interventions_dev, uint32_t* steps_since_reset_dev, double* lifelong_return_dev, void* stream);
int earl_mjl_counters(void* h, int64_t* total_steps_host, int64_t* num_interventions_dev, uint32_t* steps_since_reset_dev, double* lifelong_return_dev, void* stream);
int earl_mjs_eval_stats(void* h, double* out4_dev, void* stream);
int earl_mjl_eval_stats(void* h, double* out4_dev, void* stream);
int earl_mjs_work_counters(void* h, uint64_t* out7_host);
int earl_mjl_work_counters(void* h, uint64_t* out7_host);
int64_t earl_mjs_launch_count(const void* h);
int64_t earl_mjl_launch_count(const void* h);
int64_t earl_mjs_redo_count(void* h);
int64_t earl_mjl_redo_count(void* h);

int earl_mj_create(const earl_mj_config* cfg, const void* model_blob, size_t model_nbytes, const earl_mj_task* task,
                   earl_mj_handle** out) {
  if (!cfg || !out) return earl::set_error(EARL_ERR_INVALID, "null argument");
  *out = nullptr;
  // Both Sawyer tasks run on the SMALL set (16 envs in flight per SM): since the redo pass re-steps what overflows it
  // (peg: ~1 % of random-action env steps), the small set is the faster choice for the peg as well (65,536 envs, steady
  // window: 2.51e6 env-steps/s against 2.24e6 on the large set, overflow_states 0 either way).
  int set = 0;
  if (const char* e = getenv("EARL_MJ_CAPSET")) set = strcmp(e, "large") == 0 ? 1 : (strcmp(e, "small") == 0 ? 0 : set);
  void* impl = nullptr;
  const int rc = set ? earl_mjl_create(cfg, model_blob, model_nbytes, task, &impl) : earl_mjs_create(cfg, model_blob, model_nbytes, task, &impl);
  if (rc) return rc;
  earl_mj_handle* h = new (std::nothrow) earl_mj_handle{set, impl};
  if (!h) {
    if (set) earl_mjl_destroy(impl); else earl_mjs_destroy(impl);
    return earl::set_error(EARL_ERR_NOMEM, "out of host memory");
  }
  *out = h;
  return 0;
}

int earl_mj_destroy(earl_mj_handle* h) {
  if (!h) return 0;
  const int rc = h->set ? earl_mjl_destroy(h->impl) : earl_mjs_destroy(h->impl);
  delete h;
  return rc;
}

int earl_mj_obs_dim(const earl_mj_handle* h) {
  if (!h) return 0;
  return h->set ? earl_mjl_obs_dim(h->impl) : earl_mjs_obs_dim(h->impl);
}

int earl_mj_action_dim(const earl_mj_handle* h) {
  if (!h) return 0;
  return h->set ? earl_mjl_action_dim(h->impl) : earl_mjs_action_dim(h->impl);
}

int earl_mj_nq(const earl_mj_handle* h) {
  if (!h) return 0;
  return h->set ? earl_mjl_nq(h->impl) : earl_mjs_nq(h->impl);
}

int earl_mj_nv(const earl_mj_handle* h) {
  if (!h) return 0;
  return h->set ? earl_mjl_nv(h->impl) : earl_mjs_nv(h->impl);
}

int earl_mj_set_goal_table(earl_mj_handle* h, const double* rows_host, int32_t count) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_set_goal_table(h->impl, rows_host, count) : earl_mjs_set_goal_table(h->impl, rows_host, count);
}

int earl_mj_build_reset_template(earl_mj_handle* h, const double* hand_init_pos_host, const float* ctrl_host, int32_t steps) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_build_reset_template(h->impl, hand_init_pos_host, ctrl_host, steps) : earl_mjs_build_reset_template(h->impl, hand_init_pos_host, ctrl_host, steps);
}

int earl_mj_set_reset_stream(earl_mj_handle* h, const double* obj_qpos_host, const int32_t* goal_rows_host, int32_t rows, int32_t* goal_rows_dev) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_set_reset_stream(h->impl, obj_qpos_host, goal_rows_host, rows, goal_rows_dev) : earl_mjs_set_reset_stream(h->impl, obj_qpos_host, goal_rows_host, rows, goal_rows_dev);
}

int earl_mj_reset(earl_mj_handle* h, const uint8_t* mask_dev, const double* obj_qpos_dev, const int32_t* goal_idx_dev, float* obs_out_dev, void* stream) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_reset(h->impl, mask_dev, obj_qpos_dev, goal_idx_dev, obs_out_dev, stream) : earl_mjs_reset(h->impl, mask_dev, obj_qpos_dev, goal_idx_dev, obs_out_dev, stream);
}

int earl_mj_step(earl_mj_handle* h, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, void* stream) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_step(h->impl, actions_dev, obs_dev, reward_dev, done_dev, success_dev, stream) : earl_mjs_step(h->impl, actions_dev, obs_dev, reward_dev, done_dev, success_dev, stream);
}

int earl_mj_step_host(earl_mj_handle* h, const float* actions_host, float* obs_host, float* reward_host, uint8_t* done_host, uint8_t* success_host) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_step_host(h->impl, actions_host, obs_host, reward_host, done_host, success_host) : earl_mjs_step_host(h->impl, actions_host, obs_host, reward_host, done_host, success_host);
}

int earl_mj_get_obs(earl_mj_handle* h, float* obs_dev, void* stream) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_get_obs(h->impl, obs_dev, stream) : earl_mjs_get_obs(h->impl, obs_dev, stream);
}

int earl_mj_get_state(earl_mj_handle* h, double* qpos_host, double* qvel_host, double* warm_host, double* mocap_host) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_get_state(h->impl, qpos_host, qvel_host, warm_host, mocap_host) : earl_mjs_get_state(h->impl, qpos_host, qvel_host, warm_host, mocap_host);
}

int earl_mj_set_state(earl_mj_handle* h, const double* qpos_host, const double* qvel_host, const double* warm_host, const double* mocap_host) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_set_state(h->impl, qpos_host, qvel_host, warm_host, mocap_host) : earl_mjs_set_state(h->impl, qpos_host, qvel_host, warm_host, mocap_host);
}

int earl_mj_counters(earl_mj_handle* h, int64_t* total_steps_host, int64_t* num_interventions_dev, uint32_t* steps_since_reset_dev, double* lifelong_return_dev, void* stream) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_counters(h->impl, total_steps_host, num_interventions_dev, steps_since_reset_dev, lifelong_return_dev, stream) : earl_mjs_counters(h->impl, total_steps_host, num_interventions_dev, steps_since_reset_dev, lifelong_return_dev, stream);
}

int earl_mj_eval_stats(earl_mj_handle* h, double* out4_dev, void* stream) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_eval_stats(h->impl, out4_dev, stream) : earl_mjs_eval_stats(h->impl, out4_dev, stream);
}

int earl_mj_work_counters(earl_mj_handle* h, uint64_t* out7_host) {
  if (!h) return earl::set_error(EARL_ERR_INVALID, "null handle");
  return h->set ? earl_mjl_work_counters(h->impl, out7_host) : earl_mjs_work_counters(h->impl, out7_host);
}

int64_t earl_mj_launch_count(const earl_mj_handle* h) {
  if (!h) return 0;
  return h->set ? earl_mjl_launch_count(h->impl) : earl_mjs_launch_count(h->impl);
}

int64_t earl_mj_redo_count(earl_mj_handle* h) {
  if (!h) return -1;
  return h->set ? earl_mjl_redo_count(h->impl) : earl_mjs_redo_count(h->impl);
}

}  // extern "C"
