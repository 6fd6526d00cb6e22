/*
 * params_oracle.c -- the CPU oracle's batched drivers with per-env physics parameters (mgym_set_params).
 * TEST INFRASTRUCTURE ONLY, built by tests/params_oracle.py.
 *
 * It includes oracle/mgym_oracle.c, so the restated glibc sinf/cosf, Philox, reset distributions, observations and
 * Acrobot are exactly the oracle's; what is restated here is each kind's step with its constants taken from a
 * parameter row (order and defaults of mgym_param_name / mgym_param_defaults), derived in f32 in the constructors'
 * operation order.  params == NULL means the constants, i.e. oracle_vec_step / oracle_vec_rollout.
 * Build with -ffp-contract=off, like the oracle.
 */
#include "../oracle/mgym_oracle.c"

int oracle_num_params(int kind) {
  static const int d[ORACLE_NUM_KINDS] = {6, 2, 2, 3, 0};
  return (kind >= 0 && kind < ORACLE_NUM_KINDS) ? d[kind] : -1;
}

/* prm: gravity, masscart, masspole, length, force_mag, tau (cartpole.rs:45-56 with these values) */
static inline uint32_t cartpole_step_p(const oracle_config *cfg, float *st, uint32_t *steps, uint32_t *sbt,
                                       uint32_t action, float *reward, const float *prm) {
  cartpole_params p = cartpole_new();
  if (prm) {
    p.gravity = prm[0];
    p.masspole = prm[2];
    p.total_mass = p.masspole + prm[1];
    p.length = prm[3];
    p.polemass_length = p.masspole * p.length;
    p.force_mag = prm[4];
    p.tau = prm[5];
  }
  float x = st[0], x_dot = st[1], theta = st[2], theta_dot = st[3];
  float force = (action == 0) ? -p.force_mag : p.force_mag;
  float costheta = ref_cosf(theta);
  float sintheta = ref_sinf(theta);
  float t0 = p.polemass_length * theta_dot;
  t0 = t0 * theta_dot;
  t0 = t0 * sintheta;
  float temp = (force + t0) / p.total_mass;
  float num = p.gravity * sintheta - costheta * temp;
  float d0 = p.masspole * costheta;
  d0 = d0 * costheta;
  d0 = d0 / p.total_mass;
  float four_thirds = 4.0f / 3.0f;
  float den = p.length * (four_thirds - d0);
  float thetaacc = num / den;
  float t1 = p.polemass_length * thetaacc;
  t1 = t1 * costheta;
  t1 = t1 / p.total_mass;
  float xacc = temp - t1;
  if (cfg->is_euler) {
    x = x + p.tau * x_dot;
    x_dot = x_dot + p.tau * xacc;
    theta = theta + p.tau * theta_dot;
    theta_dot = theta_dot + p.tau * thetaacc;
  } else {
    float half_tau = 0.5f * p.tau;
    x_dot = x_dot + half_tau * (xacc + temp);
    theta_dot = theta_dot + half_tau * (thetaacc + temp);
    theta = theta + (p.tau * theta_dot + (half_tau * p.tau) * thetaacc);
    theta_dot = theta_dot + half_tau * (thetaacc + temp);
  }
  st[0] = x;
  st[1] = x_dot;
  st[2] = theta;
  st[3] = theta_dot;
  int terminated = x < -p.x_threshold || x > p.x_threshold || theta < -p.theta_threshold ||
                   theta > p.theta_threshold;
  *steps = sat_inc(*steps);
  if (*steps >= 500) {
    *sbt = 1;
    *reward = 1.0f;
    return ORACLE_FLAG_TRUNCATED;
  }
  if (!terminated) {
    *reward = cfg->sutton_barto_reward ? 0.0f : 1.0f;
    return 0;
  } else if (*sbt == ORACLE_SBT_NONE) {
    *sbt = 1;
    *reward = cfg->sutton_barto_reward ? -1.0f : 1.0f;
    return ORACLE_FLAG_TERMINATED;
  } else {
    *reward = cfg->sutton_barto_reward ? -1.0f : 0.0f;
    *sbt = sat_inc(*sbt);
    return ORACLE_FLAG_TERMINATED;
  }
}

/* prm: force, gravity (mountain_car.rs:35-40); velocity += (a - 1) force + cos(3 p) (-gravity) */
static inline uint32_t mountain_car_step_p(const oracle_config *cfg, float *st, uint32_t *steps, uint32_t action,
                                           float *reward, const float *prm) {
  mountain_car_params p = mountain_car_new();
  if (prm) {
    p.force = prm[0];
    p.gravity = prm[1];
  }
  float position = st[0], velocity = st[1];
  float a = ((float)action - 1.0f) * p.force;
  float b = ref_cosf(3.0f * position) * (-p.gravity);
  velocity = velocity + (a + b);
  velocity = clampf(velocity, -p.max_speed, p.max_speed);
  position = position + velocity;
  position = clampf(position, p.min_position, p.max_position);
  if (position == p.min_position && velocity < 0.0f) velocity = 0.0f;
  st[0] = position;
  st[1] = velocity;
  int terminated = position >= p.goal_position && velocity >= cfg->goal_velocity;
  *reward = -1.0f;
  return (terminated ? ORACLE_FLAG_TERMINATED : 0u) | time_limit(cfg, steps);
}

/* prm: power, gravity; velocity += force power - gravity cos(3 p) */
static inline uint32_t mountain_car_continuous_step_p(const oracle_config *cfg, float *st, uint32_t *steps,
                                                      float action, float *reward, const float *prm) {
  const float min_position = -1.2f, max_position = 0.6f, max_speed = 0.07f, goal_position = 0.45f;
  const float power = prm ? prm[0] : 0.0015f, gravity = prm ? prm[1] : 0.0025f;
  float position = st[0], velocity = st[1];
  float force = action;
  if (force < -1.0f) force = -1.0f;
  if (force > 1.0f) force = 1.0f;
  velocity = velocity + (force * power - gravity * ref_cosf(3.0f * position));
  if (velocity > max_speed) velocity = max_speed;
  if (velocity < -max_speed) velocity = -max_speed;
  position = position + velocity;
  if (position > max_position) position = max_position;
  if (position < min_position) position = min_position;
  if (position == min_position && velocity < 0.0f) velocity = 0.0f;
  int terminated = position >= goal_position && velocity >= cfg->goal_velocity;
  float r = terminated ? 100.0f : 0.0f;
  r = r - (action * action) * 0.1f;
  st[0] = position;
  st[1] = velocity;
  *reward = r;
  return (terminated ? ORACLE_FLAG_TERMINATED : 0u) | time_limit(cfg, steps);
}

/* prm: g, m, l; the update uses 3g/(2l) (15 by default) and 3/(m l^2) (3 by default) */
static inline uint32_t pendulum_step_p(const oracle_config *cfg, float *st, uint32_t *steps, float action,
                                       float *reward, const float *prm) {
  const float dt = 0.05f, max_speed = 8.0f, max_torque = 2.0f;
  float c_sin = 15.0f, c_u = 3.0f;
  if (prm) {
    c_sin = (3.0f * prm[0]) / (2.0f * prm[2]);
    c_u = 3.0f / (prm[1] * (prm[2] * prm[2]));
  }
  float th = st[0], thdot = st[1];
  float u = clampf(action, -max_torque, max_torque);
  float an = angle_normalize(th);
  float costs = an * an + 0.1f * (thdot * thdot);
  costs = costs + 0.001f * (u * u);
  float acc = c_sin * ref_sinf(th) + c_u * u;
  float newthdot = thdot + acc * dt;
  newthdot = clampf(newthdot, -max_speed, max_speed);
  st[0] = th + newthdot * dt;
  st[1] = newthdot;
  *reward = -costs;
  return time_limit(cfg, steps);
}

static inline uint32_t env_step_p(int kind, const oracle_config *cfg, float *st, uint32_t *steps, uint32_t *sbt,
                                  uint32_t au, float af, float *reward, const float *prm) {
  switch (kind) {
    case ORACLE_CARTPOLE_V1: return cartpole_step_p(cfg, st, steps, sbt, au, reward, prm);
    case ORACLE_MOUNTAIN_CAR_V0: return mountain_car_step_p(cfg, st, steps, au, reward, prm);
    case ORACLE_MOUNTAIN_CAR_CONTINUOUS_V0: return mountain_car_continuous_step_p(cfg, st, steps, af, reward, prm);
    case ORACLE_PENDULUM_V1: return pendulum_step_p(cfg, st, steps, af, reward, prm);
    default: return acrobot_step(cfg, st, steps, au, reward); /* no parameters */
  }
}

/* one env of mgym_step (auto-reset or manual); returns the flags */
static inline uint32_t vec_step_one_p(int kind, const oracle_config *cfg, uint64_t i, uint64_t ld, uint64_t t,
                                      float *state, uint32_t *steps, uint32_t *sbt, float *ep_return, uint32_t au,
                                      float af, const float *reset_pool, uint64_t pool_len, float *obs_out,
                                      float *reward_out, uint8_t *flags_out, float *final_obs_out, oracle_stats *stats,
                                      const float *params) {
  const int sd = oracle_state_dim(kind), od = oracle_obs_dim(kind), np = oracle_num_params(kind);
  float st[4], obs[6], reward, prm[8];
  if (params)
    for (int c = 0; c < np; ++c) prm[c] = params[(uint64_t)c * ld + i];
  uint32_t my_steps = steps ? steps[i] : 0u;
  uint32_t my_sbt = sbt ? sbt[i] : ORACLE_SBT_NONE;
  for (int c = 0; c < sd; ++c) st[c] = state[(uint64_t)c * ld + i];
  if (cfg->auto_reset) my_sbt = ORACLE_SBT_NONE;
  uint32_t flags = env_step_p(kind, cfg, st, &my_steps, &my_sbt, au, af, &reward, params ? prm : NULL);
  float ret = 0.0f;
  if (ep_return) ret = ep_return[i] + reward;
  env_obs(kind, st, obs);
  if (final_obs_out)
    for (int c = 0; c < od; ++c) final_obs_out[(uint64_t)c * ld + i] = obs[c];
  if (cfg->auto_reset && flags) {
    if (stats) {
      stats->episodes += 1;
      stats->terminated += (flags & ORACLE_FLAG_TERMINATED) ? 1 : 0;
      stats->truncated += (flags & ORACLE_FLAG_TRUNCATED) ? 1 : 0;
      stats->length_sum += my_steps;
      stats->return_sum += (double)ret;
    }
    uint64_t g = cfg->env_index_base + i;
    if (reset_pool && pool_len) {
      uint64_t j = (g + t) % pool_len;
      for (int c = 0; c < sd; ++c) st[c] = reset_pool[(uint64_t)c * pool_len + j];
    } else {
      oracle_reset_state(kind, cfg->seed, g, t + 1u - (uint64_t)my_steps, 0u, st);
    }
    my_steps = 0;
    my_sbt = ORACLE_SBT_NONE;
    ret = 0.0f;
    env_obs(kind, st, obs);
  }
  for (int c = 0; c < sd; ++c) state[(uint64_t)c * ld + i] = st[c];
  if (steps) steps[i] = my_steps;
  if (sbt) sbt[i] = my_sbt;
  if (ep_return) ep_return[i] = ret;
  if (obs_out)
    for (int c = 0; c < od; ++c) obs_out[(uint64_t)c * ld + i] = obs[c];
  if (reward_out) reward_out[i] = reward;
  if (flags_out) flags_out[i] = (uint8_t)flags;
  return flags;
}

/* oracle_vec_step with params [oracle_num_params(kind)][ld] (NULL = the constants) */
ORACLE_HOT void oracle_vec_step_p(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t t,
                                  float *state, uint32_t *steps, uint32_t *sbt, float *ep_return, const void *actions,
                                  const float *reset_pool, uint64_t pool_len, float *obs_out, float *reward_out,
                                  uint8_t *flags_out, float *final_obs_out, oracle_stats *stats, const float *params) {
  const int cont = oracle_action_is_continuous(kind);
  for (uint64_t i = 0; i < n; ++i) {
    uint32_t au = cont ? 0u : ((const uint8_t *)actions)[i];
    float af = cont ? ((const float *)actions)[i] : 0.0f;
    vec_step_one_p(kind, cfg, i, ld, t, state, steps, sbt, ep_return, au, af, reset_pool, pool_len, obs_out,
                   reward_out, flags_out, final_obs_out, stats, params);
  }
}

/* oracle_vec_rollout with params (NULL = the constants) */
ORACLE_HOT void oracle_vec_rollout_p(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, uint64_t t0,
                                     uint32_t K, float *state, uint32_t *steps, uint32_t *sbt, float *ep_return,
                                     const void *actions, const float *reset_pool, uint64_t pool_len, float *obs_traj,
                                     float *reward_traj, uint8_t *flags_traj, uint64_t *done_count,
                                     oracle_stats *stats, const float *params) {
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
      const uint32_t f = vec_step_one_p(kind, cfg, i, ld, t0 + k, state, steps, sbt, ep_return, a8, af, reset_pool,
                                        pool_len, obs_k, rew_k, flg_k, NULL, stats, params);
      dones += f ? 1 : 0;
    }
  }
  if (done_count) *done_count = dones;
}

/* mgym_sample_params: parameter c of env i (g = env_index_base + i) is word c % 4 of the Philox block with counter
 * (g, key) and tag 3 + c / 4, U[low[c], high[c]) in f64 cast to f32; envs with mask[i] == 0 are untouched */
void oracle_sample_params(int kind, const oracle_config *cfg, uint64_t n, uint64_t ld, const float *low,
                          const float *high, const uint8_t *mask, uint64_t key, float *params) {
  const int np = oracle_num_params(kind);
  for (uint64_t i = 0; i < n; ++i) {
    if (mask && !mask[i]) continue;
    const uint64_t g = cfg->env_index_base + i;
    for (int b = 0; b * 4 < np; ++b) {
      uint32_t w[4];
      philox_env(cfg->seed, g, key, 3u + (uint32_t)b, w);
      for (int j = 0; j < 4 && 4 * b + j < np; ++j) {
        const int c = 4 * b + j;
        params[(uint64_t)c * ld + i] = uniform_f64_to_f32(w[j], (double)low[c], (double)high[c]);
      }
    }
  }
}
