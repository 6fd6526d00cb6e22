/*
 * mgym.h -- C ABI of the B200-native batched classic-control simulator.
 *
 * This is the drop-in boundary for the hot path of ModuRL/ModuRL_Gym: the
 * `Gym::reset` / `Gym::step` dynamics of src/classic_control/{cartpole,
 * mountain_car}.rs, batched over N independent envs that live in HBM.
 * Citations below are relative to /root/reference.
 *
 * Reference interface each entry point replaces
 * ---------------------------------------------
 *   mgym_create      CartPoleV1::builder().build()      cartpole.rs:34-96
 *                    MountainCarV0::builder().build()   mountain_car.rs:25-69
 *   mgym_reset       <T as Gym>::reset                  cartpole.rs:238-249, mountain_car.rs:279-291
 *   mgym_step        <T as Gym>::step -> StepInfo       cartpole.rs:251-348, mountain_car.rs:293-330
 *   mgym_rollout     the caller's step loop             cartpole.rs:460-471, mountain_car.rs:425-439
 *   mgym_set_state   Testable::set_state / reset_deterministic   cartpole.rs:436-447, mountain_car.rs:402-413
 *   mgym_space_*     Gym::observation_space/action_space          cartpole.rs:58-69,:350-356; mountain_car.rs:42-48,:332-338
 *   mgym_sample_actions   Space::sample(device)         cartpole.rs:461, mountain_car.rs:427
 *
 * Layout (all buffers are DEVICE memory owned by the caller unless named *_host)
 * -----------------------------------------------------------------------------
 *   state / obs   structure of arrays, component-major: obs[c * N + i], f32
 *   actions       discrete kinds: uint8_t[N];  continuous kinds: float[N]
 *   reward        float[N]
 *   flags         uint8_t[N]; bit0 = StepInfo.done (terminated), bit1 = StepInfo.truncated
 *   trajectories  time-major: obs[k][c][N], reward[k][N], flags[k][N], actions[k][N]
 * Fastest path (TMA-staged step kernel): auto_reset, N % 1024 == 0, 16-byte aligned pointers.
 * N % 4 == 0 with aligned pointers takes the 128-bit vector kernel, anything else the
 * scalar-lane instantiation of the same kernel: same results bit for bit, lower throughput.
 *
 * Semantics
 * ---------
 *   auto_reset = 0  reference-faithful: the handle keeps `steps_since_reset` and
 *                   `steps_beyond_terminated` per env exactly like cartpole.rs:24-28 and
 *                   the caller resets (mgym_reset / mgym_reset_masked) as in cartpole.rs:468-470.
 *   auto_reset = 1  the caller loop `if done { env.reset() }` is folded into the step:
 *                   an env whose step returns terminated or truncated is reset in the
 *                   same call; obs_out holds the post-reset observation, reward/flags the
 *                   finishing step's values, final_obs_out (optional) the pre-reset obs.
 *                   mgym_rollout_final keeps the same pre-reset obs for a fused rollout, stored only
 *                   where an env finished.
 *   Reset states come from a counter-based Philox4x32-10 stream keyed by the seed; the counter is
 *   (global env index, reset call index) for mgym_reset and (global env index, step index at which
 *   the episode that just finished BEGAN) for a same-step auto-reset, so results do not depend on
 *   launch geometry, on the mix of mgym_step / mgym_rollout calls or on how envs are sharded over
 *   GPUs -- and the state an env will restart from is known as soon as its episode starts, which
 *   lets the rollout kernel draw it ahead of time.  Or they come from an injected pool
 *   (mgym_set_reset_pool) for parity runs.
 *
 * Errors: every function returns 0 on success or a negative mgym_status; the message is
 * kept per thread (mgym_last_error).  Nothing aborts or throws across this boundary.  The
 * reference panics on an invalid action (assert!, cartpole.rs:252, mountain_car.rs:294);
 * here validate_actions=1 (a debug mode: one small pre-pass launch and a stream synchronisation per call)
 * makes the offending mgym_step / mgym_rollout / mgym_step_host call itself return MGYM_ERR_INVALID_ACTION
 * BEFORE anything is stepped: state, counters, statistics and step index are untouched, so the caller can
 * correct the batch and retry, exactly as the reference asserts before any mutation.  Without it CartPole
 * treats 0 as left and anything else as right (cartpole.rs:258-262) and MountainCar computes
 * (a as f32) - 1.0 (mountain_car.rs:302).
 *
 * Threading: one handle = one GPU; calls on a handle must be serialised by the caller
 * (the reference's `&mut self`).  Different handles are independent.
 *
 * There is no CPU fallback: without a CUDA device mgym_create fails with MGYM_ERR_CUDA.
 */
#ifndef MGYM_H
#define MGYM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGYM_ABI_VERSION 1

typedef struct mgym_env mgym_env; /* opaque handle */

typedef enum mgym_kind {
  MGYM_CARTPOLE_V1 = 0,                /* cartpole.rs */
  MGYM_MOUNTAIN_CAR_V0 = 1,            /* mountain_car.rs */
  MGYM_MOUNTAIN_CAR_CONTINUOUS_V0 = 2, /* not in the reference; Gymnasium semantics */
  MGYM_PENDULUM_V1 = 3,                /* not in the reference; Gymnasium semantics */
  MGYM_ACROBOT_V1 = 4,                 /* not in the reference; Gymnasium semantics */
  MGYM_NUM_KINDS = 5
} mgym_kind;

typedef enum mgym_status {
  MGYM_OK = 0,
  MGYM_ERR_BAD_ARGUMENT = -1,
  MGYM_ERR_CUDA = -2,
  MGYM_ERR_NCCL = -3,
  MGYM_ERR_INVALID_ACTION = -4, /* the reference's assert!(action_space.contains(&action)) */
  MGYM_ERR_OUT_OF_MEMORY = -5
} mgym_status;

#define MGYM_FLAG_TERMINATED 1u /* StepInfo.done */
#define MGYM_FLAG_TRUNCATED 2u  /* StepInfo.truncated */

/* Builder parameters (cartpole.rs:36-44, mountain_car.rs:27-34) plus batching options. */
typedef struct mgym_config {
  uint32_t struct_size;        /* sizeof(mgym_config), for ABI growth */
  int32_t auto_reset;          /* default 1 */
  int32_t max_episode_steps;   /* 0 = none.  CartPole ignores it: 500 is hard-coded (cartpole.rs:297).
                                  Defaults: MountainCar 0 (reference never truncates, mountain_car.rs:328),
                                  MountainCarContinuous 999, Pendulum 200, Acrobot 500 (Gymnasium) */
  int32_t sutton_barto_reward; /* cartpole.rs:39, default 0 */
  int32_t is_euler;            /* cartpole.rs:40, default 1 */
  float goal_velocity;         /* mountain_car.rs:33, default 0.0 */
  int32_t track_stats;         /* default 1: episode count, terminated / truncated counts and length sum
                                  (auto_reset only), and the return sum for the kinds whose return follows from
                                  those (CartPole, MountainCar, Acrobot: constant rewards).  Costs no per-step
                                  traffic: the episode length comes from a per-env START STAMP that a step only
                                  reads (2 bytes, kinds with a time limit) or does not touch at all (no limit). */
  int32_t validate_actions;    /* default 0: debug mode, see Errors above */
  uint64_t env_index_base;     /* global index of this handle's env 0 (multi-GPU slices) */
  int32_t device_clock;        /* default 0.  1 = keep the step index and the tile-ticket base in device memory,
                                  advanced on the device by the last CTA of each launch (mgym_step_host's chunked
                                  launches enqueue a one-thread kernel instead): mgym_step, mgym_rollout and
                                  mgym_sample_actions then carry no per-call launch parameter and may be captured
                                  into a CUDA graph and replayed (same results as the eager calls).
                                  mgym_step_index then synchronises the device. */
  int32_t track_returns;       /* default 0.  1 = also accumulate the return sum of the kinds whose rewards are not
                                  constants (MountainCarContinuous, Pendulum): a per-env running return, i.e. 4 bytes
                                  read and 4 written per env-step in the per-call step kernel (free in mgym_rollout,
                                  which keeps it in registers).  Needs track_stats.  Without it those kinds report
                                  return_sum = 0. */
} mgym_config;

/* Episode statistics accumulated on the device since creation / mgym_stats_reset. */
typedef struct mgym_stats {
  uint64_t episodes;   /* finished episodes */
  uint64_t terminated; /* of which ended with bit0 */
  uint64_t truncated;  /* of which ended with bit1 */
  uint64_t length_sum; /* sum of episode lengths */
  double return_sum;   /* sum of episode returns */
} mgym_stats_t;

/* ---- metadata -------------------------------------------------------------------- */
int mgym_abi_version(void);
const char *mgym_last_error(void);
const char *mgym_kind_name(int kind);
int mgym_state_dim(int kind);
int mgym_obs_dim(int kind);
int mgym_action_is_continuous(int kind); /* 0: Discrete(n), uint8 actions; 1: Box, float actions */
int mgym_num_actions(int kind);          /* Discrete(n): n; continuous: 0 */
/* observation_space / action_space bounds (BoxSpace low/high; +-inf where unbounded). */
int mgym_space_observation(int kind, float *low, float *high);
int mgym_space_action(int kind, float *low, float *high);

/* ---- lifecycle -------------------------------------------------------------------- */
int mgym_config_default(int kind, mgym_config *cfg);
int mgym_create(int kind, uint64_t num_envs, int device_ordinal, uint64_t seed, const mgym_config *cfg,
                mgym_env **out);
int mgym_destroy(mgym_env *env);
uint64_t mgym_num_envs(const mgym_env *env);
int mgym_kind_of(const mgym_env *env);
uint64_t mgym_step_index(const mgym_env *env); /* steps executed since creation (Philox counter) */

/* ---- reset ------------------------------------------------------------------------ */
/* Gym::reset for every env (mask == NULL) or for envs with mask[i] != 0.  obs_out optional. */
int mgym_reset(mgym_env *env, float *obs_out, void *stream);
int mgym_reset_masked(mgym_env *env, const uint8_t *mask, float *obs_out, void *stream);
/* Injected reset states, SoA [state_dim][pool_len] (copied).  Entry (global_env + step_index) % pool_len
 * replaces the Philox draw.  pool_len = 0 restores Philox. */
int mgym_set_reset_pool(mgym_env *env, const float *pool, uint64_t pool_len, void *stream);

/* ---- state injection / checkpoint (Testable::set_state) --------------------------- */
/* state: SoA [state_dim][N]; steps, sbt: uint32[N] or NULL (-> 0 / None); device or host pointers.
 * sbt encodes steps_beyond_terminated: 0 = None, k+1 = Some(k).  steps = episode step counts
 * (cartpole.rs:24 steps_since_reset); an auto-reset handle of a kind with a time limit <= 65535 keeps them in 16
 * bits, so injected counts above 65535 are stored as 65535 (either way "past the limit": the next step truncates). */
int mgym_set_state(mgym_env *env, const float *state, const uint32_t *steps, const uint32_t *sbt, void *stream);
int mgym_get_state(mgym_env *env, float *state, uint32_t *steps, uint32_t *sbt, void *stream);
int mgym_get_obs(mgym_env *env, float *obs_out, void *stream); /* current observation, [obs_dim][N]; device or host */
/* Zero-copy view of the resident state rows ([state_dim][N]); for kinds whose observation is the
 * state (CartPole, MountainCar, MountainCarContinuous) this IS the observation buffer. */
float *mgym_state_ptr(mgym_env *env);

/* Checkpoint / resume: the whole handle (state rows, counters, running returns, statistics, step and reset
 * indices, per-env parameters and redraw ranges if set) as one opaque HOST blob.  mgym_checkpoint_size gives the byte
 * count; a handle created with the same kind, num_envs and config continues bit-identically after
 * mgym_checkpoint_load, which restores exactly the parameters and ranges the blob carries (a blob without them clears
 * the handle's). */
size_t mgym_checkpoint_size(const mgym_env *env);
int mgym_checkpoint_save(mgym_env *env, void *host_blob, size_t blob_bytes, void *stream);
int mgym_checkpoint_load(mgym_env *env, const void *host_blob, size_t blob_bytes, void *stream);

/* ---- the hot path ------------------------------------------------------------------ */
/* One Gym::step for all N envs.  obs_out, reward_out, flags_out, final_obs_out may be NULL.
 * final_obs_out is DENSE: every env's entry is written (the pre-reset observation where the env finished, the
 * observation itself elsewhere).  mgym_rollout_final's final_obs_traj is SPARSE: only finished envs are written.
 * CUDA graphs: by default the step index that keys the Philox resets and the tile tickets are per-call launch
 * parameters, so on a capturing stream mgym_step / mgym_rollout / mgym_sample_actions return
 * MGYM_ERR_BAD_ARGUMENT instead of recording a launch whose replay would be wrong.  A handle created with
 * cfg.device_clock = 1 keeps both on the device and IS capturable (launch-bound small batches: capture
 * [policy, mgym_step] once, replay it per step).  mgym_reset, mgym_step_host and the state accessors are never
 * capturable. */
int mgym_step(mgym_env *env, const void *actions, float *obs_out, float *reward_out, uint8_t *flags_out,
              float *final_obs_out, void *stream);
/* K fused steps with state held in registers; only the trajectory is written.
 * actions == NULL: uniform random policy sampled on the device (Space::sample).
 * done_count_out (device uint64, optional) receives the number of finished env-steps. */
int mgym_rollout(mgym_env *env, uint32_t K, const void *actions, float *obs_traj, float *reward_traj,
                 uint8_t *flags_traj, unsigned long long *done_count_out, void *stream);
/* mgym_rollout plus the observation every finished episode ended on.
 * final_obs_traj: device float[K][obs_dim][N], time-major like obs_traj.  Where flags_traj[k][i] != 0 (env i
 * finished at step k), final_obs_traj[k][c][i] = the observation step k produced BEFORE the auto-reset: the value
 * mgym_step's final_obs_out would hold for that env at that step.  Every other entry is NOT written: it keeps what
 * the caller put there (unlike mgym_step's dense final_obs_out: a dense copy would write every observation twice,
 * sparse stores cost only where an env finished).  next_obs of transition k is therefore
 * flags[k] ? final_obs_traj[k] : obs_traj[k].
 * final_obs_traj == NULL: exactly mgym_rollout.  Everything else (obs_traj, reward_traj, flags_traj, done_count,
 * state, counters, running returns, statistics, parameter rows and redraws, step index) is bit-identical to
 * mgym_rollout with the same arguments.  The finishing step runs on the env's old parameters, so with redraw ranges
 * the final observation is the one those produced; a reset pool changes reset states only.  Needs 4-byte alignment
 * only.  auto_reset = 0 handles: MGYM_ERR_BAD_ARGUMENT (nothing resets inside the rollout; obs_traj already holds the
 * final observations).  final_obs_traj == obs_traj: MGYM_ERR_BAD_ARGUMENT.  validate_actions = 1 rejects a bad batch
 * before anything, final_obs_traj included, is written.  Capturable under the same rules as mgym_rollout
 * (device_clock handles). */
int mgym_rollout_final(mgym_env *env, uint32_t K, const void *actions, float *obs_traj, float *reward_traj,
                       uint8_t *flags_traj, float *final_obs_traj, unsigned long long *done_count_out, void *stream);
/* Space::sample for all envs at the current step index (same stream mgym_rollout uses). */
int mgym_sample_actions(mgym_env *env, void *actions_out, void *stream);

/* Host-buffer convenience used for end-to-end timing: pinned or pageable host pointers;
 * H2D actions, step, D2H results, synchronises the stream.  Any output may be NULL. */
int mgym_step_host(mgym_env *env, const void *actions_host, float *obs_host, float *reward_host,
                   uint8_t *flags_host, void *stream);

/* ---- per-env physics parameters (domain randomisation, system identification) ------------
 * A handle may carry one row per parameter, SoA float[P][N] (P = mgym_num_params), owned by the handle and
 * allocated on first use.  Without them every env runs the kind's constants (the defaults below) on the same
 * kernels as before, bit for bit; with them step, rollout and step_host read each env's own constants.
 * Derived constants are computed per env in f32 in the host's operation order, so defaults set explicitly give
 * the same bits as no parameters.  Termination thresholds, spaces, time limits and reset distributions do not
 * depend on parameters.
 *   CartPole-v1               gravity 9.8, masscart 1.0, masspole 0.1, length 0.5 (half-pole), force_mag 10.0,
 *                             tau 0.02 (masses, length and tau > 0)
 *   MountainCar-v0            force 0.001, gravity 0.0025
 *   MountainCarContinuous-v0  power 0.0015, gravity 0.0025
 *   Pendulum-v1               g 10.0, m 1.0, l 1.0 (m, l > 0)
 *   Acrobot-v1                none (P = 0; mgym_set_params / mgym_sample_params return MGYM_ERR_BAD_ARGUMENT)
 * Every parameter must be finite. */
int mgym_num_params(int kind);                      /* P, or a negative status for an unknown kind */
const char *mgym_param_name(int kind, int i);       /* NULL outside [0, P) */
int mgym_param_defaults(int kind, float *out);      /* P floats */
/* params: [P][N], host or device; NULL = back to the constants.  Checked before anything is copied: a rejected
 * set returns MGYM_ERR_BAD_ARGUMENT and leaves the handle untouched.  Synchronises; not capturable. */
int mgym_set_params(mgym_env *env, const float *params, void *stream);
/* out: [P][N], host or device; the defaults when no parameters are set. */
int mgym_get_params(mgym_env *env, float *out, void *stream);
/* Draws parameter c of env i uniformly from [low[c], high[c]) (host arrays of P; f64 draw cast to f32, like the
 * reset states): word c % 4 of the Philox block with counter (global env index, key mod 2^56) and tag 3 + c / 4,
 * so the draws do not depend on sharding or launch geometry.  mask (device uint8[N] or NULL) limits the draw to
 * envs with mask[i] != 0 (e.g. `mask = flags != 0` after a step; mgym_set_param_redraw does per-episode draws
 * on the device instead).  Rows not set before start from the defaults.  Capturable into a CUDA graph once the rows
 * exist (the key is the caller's). */
int mgym_sample_params(mgym_env *env, const float *low, const float *high, const uint8_t *mask, uint64_t key,
                       void *stream);
/* Per-episode redraw (domain randomisation per episode): with ranges set, EVERY reset of an env also draws its
 * parameters, parameter c uniformly from [low[c], high[c]) with the mapping of mgym_sample_params, from the Philox
 * block with the counter of the new episode's reset state:
 *   auto-reset in mgym_step / mgym_step_host / mgym_rollout   (global env index, step at which the finished episode
 *                                                              began), tags 5 (parameters 0-3) and 6 (4-7)
 *   mgym_reset / mgym_reset_masked, reset call index r        (global env index, r), tags 7 and 8
 * so the draws do not depend on launch geometry, sharding or the mix of step and rollout calls.  The finishing step
 * runs on the old parameters.  Nothing else redraws: not mgym_set_state, not a manual-mode (auto_reset = 0) step, and
 * a reset pool (mgym_set_reset_pool) replaces only the reset STATES.  low[c] == high[c] draws exactly low[c].
 * low, high: host arrays of P (finite, low <= high, low > 0 for masses, lengths and tau), or both NULL = off.
 * Checked before anything changes: a rejected call leaves the handle untouched.  Setting ranges allocates the rows
 * with the defaults if none are set and leaves the current episodes alone; `mgym_set_param_redraw(lo, hi);
 * mgym_reset()` starts every env on drawn parameters.  mgym_set_params(NULL) clears the ranges with the rows,
 * mgym_set_params(rows) keeps them; checkpoints carry them.  Acrobot: MGYM_ERR_BAD_ARGUMENT.  Not capturable.
 * CUDA graphs: the ranges are launch parameters of the captured step / rollout, so a graph replays the ranges it was
 * captured with -- recapture after changing them. */
int mgym_set_param_redraw(mgym_env *env, const float *low, const float *high, void *stream);
/* *enabled = 0 / 1; low, high (P floats each, may be NULL) receive the ranges when enabled. */
int mgym_get_param_redraw(const mgym_env *env, int *enabled, float *low, float *high);

/* ---- statistics --------------------------------------------------------------------- */
int mgym_stats_get(mgym_env *env, mgym_stats_t *out, void *stream); /* synchronises */
int mgym_stats_reset(mgym_env *env, void *stream);
/* Writes {episodes, terminated, truncated, length_sum, return_sum} as 5 doubles into a caller-owned
 * DEVICE buffer: this is the vector a host layer all-reduces (sum) across GPUs. */
int mgym_stats_export(mgym_env *env, double *device_vec5_out, void *stream);
/* mgym_stats_export followed by ncclAllReduce(sum) in place on `comm` (an ncclComm_t).  NCCL is
 * resolved at run time from the process (dlsym), so the library carries no NCCL link dependency.  A single
 * thread that drives several GPUs brackets the calls with ncclGroupStart/ncclGroupEnd as usual. */
int mgym_stats_allreduce(mgym_env *env, void *nccl_comm, double *device_vec5_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MGYM_H */
