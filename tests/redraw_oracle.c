/*
 * redraw_oracle.c -- the CPU oracle's batched drivers with per-episode parameter redraws (mgym_set_param_redraw).
 * TEST INFRASTRUCTURE ONLY, built by tests/redraw_oracle.py.
 *
 * It includes tests/params_oracle.c (which includes the oracle), so the steps with per-env parameters, Philox, the
 * reset distributions and the f64 -> f32 uniform mapping are exactly theirs.  What is added is the redraw: the rows
 * are mutable, and every reset draws the env's parameters, parameter c = word c % 4 of the Philox block with
 * counter (g, k) and tag tag0 + c / 4, U[low[c], high[c]):
 *   auto-reset of step t ending an episode of `steps` steps   k = t + 1 - steps (its start), tag0 = 5
 *   explicit reset, reset call index r                          k = r, tag0 = 7
 * low == NULL (or high == NULL) means no redraw: the drivers are then oracle_vec_step_p / oracle_vec_rollout_p /
 * oracle_vec_reset.  Build with -ffp-contract=off, like the oracle.
 */
#include "params_oracle.c"

static void redraw_one(int kind, uint64_t seed, uint64_t g, uint64_t k, uint32_t tag0, const float *low,
                       const float *high, float *params, uint64_t ld, uint64_t i) {
  const int np = oracle_num_params(kind);
  for (int b = 0; b * 4 < np; ++b) {
    uint32_t w[4];
    philox_env(seed, g, k, tag0 + (uint32_t)b, w);
    for (int j = 0; j < 4 && 4 * b + j < np; ++j) {
      const int c = 4 * b + j;
      params[(uint64_t)c * ld + i] = uniform_f64_to_f32(w[j], (double)low[c], (double)high[c]);
    }
  }
}

/* one env of mgym_step with redraw: the step runs on the old row, a reset redraws it */
static inline uint32_t vec_step_one_r(int kind, const oracle_config *cfg, uint64_t i, uint64_t ld, uint64_t t,
                                      float *state, uint32_t *steps, uint32_t *sbt, float *ep_return, uint32_t au,
                                      float af, const float *reset_pool, uint64_t pool_len, float *obs_out,
                                      float *reward_out, uint8_t *flags_out, float *final_obs_out, oracle_stats *stats,
                                      float *params, const float *low, const float *high) {
  const uint32_t count = sat_inc(steps ? steps[i] : 0u); /* the episode length if this step ends it */
  const uint32_t flags = vec_step_one_p(kind, cfg, i, ld, t, state, steps, sbt, ep_return, au, af, reset_pool,
                                        pool_len, obs_out, reward_out, flags_out, final_obs_out, stats, params);
  if (params && low && high && cfg->auto_reset && flags)
    redraw_one(kind, cfg->seed, cfg->env_index_base + i, t + 1u - (uint64_t)count, 5u, low, high, params, ld, i);
  return flags;
}

/* oracle_vec_step_p with per-episode redraws into params [P][ld] (low / high: P values each, or NULL) */
ORACLE_HOT void oracle_vec_step_r(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t t,
                                  float *state, uint32_t *steps, uint32_t *sbt, float *ep_return, const void *actions,
                                  const float *reset_pool, uint64_t pool_len, float *obs_out, float *reward_out,
                                  uint8_t *flags_out, float *final_obs_out, oracle_stats *stats, float *params,
                                  const float *low, const float *high) {
  const int cont = oracle_action_is_continuous(kind);
  for (uint64_t i = 0; i < n; ++i) {
    uint32_t au = cont ? 0u : ((const uint8_t *)actions)[i];
    float af = cont ? ((const float *)actions)[i] : 0.0f;
    vec_step_one_r(kind, cfg, i, ld, t, state, steps, sbt, ep_return, au, af, reset_pool, pool_len, obs_out,
                   reward_out, flags_out, final_obs_out, stats, params, low, high);
  }
}

/* oracle_vec_rollout_p with per-episode redraws */
ORACLE_HOT void oracle_vec_rollout_r(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t t0,
                                     uint32_t K, float *state, uint32_t *steps, uint32_t *sbt, float *ep_return,
                                     const void *actions, const float *reset_pool, uint64_t pool_len, float *obs_traj,
                                     float *reward_traj, uint8_t *flags_traj, uint64_t *done_count,
                                     oracle_stats *stats, float *params, const float *low, const float *high) {
  const int cont = oracle_action_is_continuous(kind), od = oracle_obs_dim(kind);
  uint64_t dones = 0;
  for (uint32_t k = 0; k < K; ++k) {
    float *obs_k = obs_traj ? obs_traj + (uint64_t)k * od * ld : NULL;
    float *rew_k = reward_traj ? reward_traj + (uint64_t)k * ld : NULL;
    uint8_t *flg_k = flags_traj ? flags_traj + (uint64_t)k * ld : NULL;
    for (uint64_t i = 0; i < n; ++i) {
      uint8_t a8 = 0;
      float af = 0.0f;
      if (actions) {
        if (cont) af = ((const float *)actions)[(uint64_t)k * ld + i];
        else a8 = ((const uint8_t *)actions)[(uint64_t)k * ld + i];
      } else {
        oracle_sample_action(kind, cfg->seed, cfg->env_index_base + i, t0 + k, &a8, &af);
      }
      const uint32_t f = vec_step_one_r(kind, cfg, i, ld, t0 + k, state, steps, sbt, ep_return, a8, af, reset_pool,
                                        pool_len, obs_k, rew_k, flg_k, NULL, stats, params, low, high);
      dones += f ? 1 : 0;
    }
  }
  if (done_count) *done_count = dones;
}

/* oracle_vec_reset (reset call index r) with the reset envs' parameters redrawn from (g, r), tags 7 / 8 */
ORACLE_HOT void oracle_reset_r(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t r,
                               const uint8_t *mask, float *state, uint32_t *steps, uint32_t *sbt, float *ep_return,
                               const float *reset_pool, uint64_t pool_len, float *obs_out, float *params,
                               const float *low, const float *high) {
  oracle_vec_reset(kind, cfg, n, ld, r, mask, state, steps, sbt, ep_return, reset_pool, pool_len, obs_out);
  if (!params || !low || !high) return;
  for (uint64_t i = 0; i < n; ++i)
    if (!mask || mask[i]) redraw_one(kind, cfg->seed, cfg->env_index_base + i, r, 7u, low, high, params, ld, i);
}
