/*
 * episodes_oracle.c -- the CPU oracle's batched drivers with per-episode outputs (mgym_step_episodes,
 * mgym_rollout_episodes).  TEST INFRASTRUCTURE ONLY, built by tests/episodes_oracle.py.
 *
 * It includes tests/redraw_oracle.c (which includes tests/params_oracle.c and the oracle), so steps, resets, parameter
 * rows and redraws are exactly theirs.  What is added: where an env finishes, the episode's length and return are
 * stored at its flags index, before the reset clears them.  They are read from the oracle's own tally of that env
 * (its step counter after the finishing step and its f32 running return), i.e. the values its statistics add:
 *   ep_length  the step count the finishing step reached
 *   ep_return  CartPole the length (sutton_barto_reward: +1 if truncated, -1 if terminated), MountainCar-v0 -length,
 *              Acrobot (terminated ? 1 : 0) - length, MountainCarContinuous / Pendulum the running return
 * Entries of envs that did not finish are not written.  ep_return == NULL and ep_length == NULL give the bits of
 * oracle_vec_step_r / oracle_vec_rollout_r.  Build with -ffp-contract=off, like the oracle.
 */
#include "redraw_oracle.c"

static float episode_return(int kind, const oracle_config *cfg, uint32_t flags, uint32_t length, float ret) {
  const double term = (flags & ORACLE_FLAG_TERMINATED) ? 1.0 : 0.0, trunc = (flags & ORACLE_FLAG_TRUNCATED) ? 1.0 : 0.0;
  switch (kind) {
    case ORACLE_CARTPOLE_V1: return (float)(cfg->sutton_barto_reward ? trunc - term : (double)length);
    case ORACLE_MOUNTAIN_CAR_V0: return (float)(-(double)length);
    case ORACLE_ACROBOT_V1: return (float)(term - (double)length);
    default: return ret;
  }
}

/* one env of mgym_step_episodes: vec_step_one_r, tallied into a zeroed record of its own so that the finished
 * episode's length and return can be read back; that record is then added to `stats` as vec_step_one_r would have */
static inline uint32_t vec_step_one_e(int kind, const oracle_config *cfg, uint64_t i, uint64_t ld, uint64_t t,
                                      float *state, uint32_t *steps, uint32_t *sbt, float *ep_return, uint32_t au,
                                      float af, const float *reset_pool, uint64_t pool_len, float *obs_out,
                                      float *reward_out, uint8_t *flags_out, float *final_obs_out, oracle_stats *stats,
                                      float *params, const float *low, const float *high, float *ep_ret_out,
                                      uint32_t *ep_len_out, uint64_t out_i) {
  oracle_stats one = {0, 0, 0, 0, 0.0};
  const uint32_t flags = vec_step_one_r(kind, cfg, i, ld, t, state, steps, sbt, ep_return, au, af, reset_pool,
                                        pool_len, obs_out, reward_out, flags_out, final_obs_out, &one, params, low,
                                        high);
  if (cfg->auto_reset && flags) {
    const uint32_t length = (uint32_t)one.length_sum;
    if (ep_len_out) ep_len_out[out_i] = length;
    if (ep_ret_out) ep_ret_out[out_i] = episode_return(kind, cfg, flags, length, (float)one.return_sum);
    if (stats) {
      stats->episodes += one.episodes;
      stats->terminated += one.terminated;
      stats->truncated += one.truncated;
      stats->length_sum += one.length_sum;
      stats->return_sum += one.return_sum;
    }
  }
  return flags;
}

/* oracle_vec_step_r plus ep_return_out [n] / ep_length_out [n] (either may be NULL) */
ORACLE_HOT void oracle_vec_step_e(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t t,
                                  float *state, uint32_t *steps, uint32_t *sbt, float *ep_return, const void *actions,
                                  const float *reset_pool, uint64_t pool_len, float *obs_out, float *reward_out,
                                  uint8_t *flags_out, float *final_obs_out, oracle_stats *stats, float *params,
                                  const float *low, const float *high, float *ep_return_out, uint32_t *ep_length_out) {
  const int cont = oracle_action_is_continuous(kind);
  for (uint64_t i = 0; i < n; ++i) {
    uint32_t au = cont ? 0u : ((const uint8_t *)actions)[i];
    float af = cont ? ((const float *)actions)[i] : 0.0f;
    vec_step_one_e(kind, cfg, i, ld, t, state, steps, sbt, ep_return, au, af, reset_pool, pool_len, obs_out,
                   reward_out, flags_out, final_obs_out, stats, params, low, high, ep_return_out, ep_length_out, i);
  }
}

/* oracle_vec_rollout_r plus ep_return_traj [K][ld] and ep_length_traj [K][ld] (either may be NULL) */
ORACLE_HOT void oracle_vec_rollout_e(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t t0,
                                     uint32_t K, float *state, uint32_t *steps, uint32_t *sbt, float *ep_return,
                                     const void *actions, const float *reset_pool, uint64_t pool_len, float *obs_traj,
                                     float *reward_traj, uint8_t *flags_traj, uint64_t *done_count,
                                     oracle_stats *stats, float *params, const float *low, const float *high,
                                     float *ep_return_traj, uint32_t *ep_length_traj) {
  const int cont = oracle_action_is_continuous(kind), od = oracle_obs_dim(kind);
  uint64_t dones = 0;
  for (uint32_t k = 0; k < K; ++k) {
    float *obs_k = obs_traj ? obs_traj + (uint64_t)k * od * ld : NULL;
    float *rew_k = reward_traj ? reward_traj + (uint64_t)k * ld : NULL;
    uint8_t *flg_k = flags_traj ? flags_traj + (uint64_t)k * ld : NULL;
    float *ret_k = ep_return_traj ? ep_return_traj + (uint64_t)k * ld : NULL;
    uint32_t *len_k = ep_length_traj ? ep_length_traj + (uint64_t)k * ld : NULL;
    for (uint64_t i = 0; i < n; ++i) {
      uint8_t a8 = 0;
      float af = 0.0f;
      if (actions) {
        if (cont) af = ((const float *)actions)[(uint64_t)k * ld + i];
        else a8 = ((const uint8_t *)actions)[(uint64_t)k * ld + i];
      } else {
        oracle_sample_action(kind, cfg->seed, cfg->env_index_base + i, t0 + k, &a8, &af);
      }
      const uint32_t f = vec_step_one_e(kind, cfg, i, ld, t0 + k, state, steps, sbt, ep_return, a8, af, reset_pool,
                                        pool_len, obs_k, rew_k, flg_k, NULL, stats, params, low, high, ret_k, len_k, i);
      dones += f ? 1 : 0;
    }
  }
  if (done_count) *done_count = dones;
}
