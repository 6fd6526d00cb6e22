//! Raw declarations of include/mgym.h (what `bindgen` would emit).  NOT COMPILED in the build image.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct mgym_env {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct mgym_config {
    pub struct_size: u32,
    pub auto_reset: i32,
    pub max_episode_steps: i32,
    pub sutton_barto_reward: i32, // cartpole.rs:39
    pub is_euler: i32,            // cartpole.rs:40
    pub goal_velocity: f32,       // mountain_car.rs:33
    pub track_stats: i32,
    pub validate_actions: i32,
    pub env_index_base: u64,
    pub device_clock: i32, // 1 = CUDA-graph-capturable handle (step index + tile tickets on the device)
    pub track_returns: i32, // 1 = per-env running return for MountainCarContinuous / Pendulum statistics
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct mgym_stats {
    pub episodes: u64,
    pub terminated: u64,
    pub truncated: u64,
    pub length_sum: u64,
    pub return_sum: f64,
}

pub const MGYM_CARTPOLE_V1: c_int = 0;
pub const MGYM_MOUNTAIN_CAR_V0: c_int = 1;
pub const MGYM_MOUNTAIN_CAR_CONTINUOUS_V0: c_int = 2;
pub const MGYM_PENDULUM_V1: c_int = 3;
pub const MGYM_ACROBOT_V1: c_int = 4;
pub const MGYM_OK: c_int = 0;
pub const MGYM_ERR_INVALID_ACTION: c_int = -4;
pub const MGYM_FLAG_TERMINATED: u8 = 1;
pub const MGYM_FLAG_TRUNCATED: u8 = 2;

extern "C" {
    pub fn mgym_abi_version() -> c_int;
    pub fn mgym_last_error() -> *const c_char;
    pub fn mgym_kind_name(kind: c_int) -> *const c_char;
    pub fn mgym_state_dim(kind: c_int) -> c_int;
    pub fn mgym_obs_dim(kind: c_int) -> c_int;
    pub fn mgym_action_is_continuous(kind: c_int) -> c_int;
    pub fn mgym_num_actions(kind: c_int) -> c_int;
    pub fn mgym_space_observation(kind: c_int, low: *mut f32, high: *mut f32) -> c_int;
    pub fn mgym_space_action(kind: c_int, low: *mut f32, high: *mut f32) -> c_int;
    pub fn mgym_config_default(kind: c_int, cfg: *mut mgym_config) -> c_int;
    pub fn mgym_create(kind: c_int, num_envs: u64, device: c_int, seed: u64, cfg: *const mgym_config,
                       out: *mut *mut mgym_env) -> c_int;
    pub fn mgym_destroy(env: *mut mgym_env) -> c_int;
    pub fn mgym_num_envs(env: *const mgym_env) -> u64;
    pub fn mgym_kind_of(env: *const mgym_env) -> c_int;
    pub fn mgym_step_index(env: *const mgym_env) -> u64;
    pub fn mgym_reset(env: *mut mgym_env, obs_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn mgym_reset_masked(env: *mut mgym_env, mask: *const u8, obs_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn mgym_set_reset_pool(env: *mut mgym_env, pool: *const f32, pool_len: u64, stream: *mut c_void) -> c_int;
    pub fn mgym_set_state(env: *mut mgym_env, state: *const f32, steps: *const u32, sbt: *const u32,
                          stream: *mut c_void) -> c_int;
    pub fn mgym_get_state(env: *mut mgym_env, state: *mut f32, steps: *mut u32, sbt: *mut u32,
                          stream: *mut c_void) -> c_int;
    pub fn mgym_get_obs(env: *mut mgym_env, obs_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn mgym_state_ptr(env: *mut mgym_env) -> *mut f32;
    pub fn mgym_reward_ptr(env: *mut mgym_env) -> *mut f32;
    pub fn mgym_reward_constant(env: *mut mgym_env, value: *mut f32) -> c_int;
    pub fn mgym_checkpoint_size(env: *const mgym_env) -> usize;
    pub fn mgym_checkpoint_save(env: *mut mgym_env, blob: *mut c_void, bytes: usize, stream: *mut c_void) -> c_int;
    pub fn mgym_checkpoint_load(env: *mut mgym_env, blob: *const c_void, bytes: usize, stream: *mut c_void) -> c_int;
    pub fn mgym_step(env: *mut mgym_env, actions: *const c_void, obs_out: *mut f32, reward_out: *mut f32,
                     flags_out: *mut u8, final_obs_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn mgym_rollout(env: *mut mgym_env, k: u32, actions: *const c_void, obs_traj: *mut f32,
                        reward_traj: *mut f32, flags_traj: *mut u8, done_count_out: *mut u64,
                        stream: *mut c_void) -> c_int;
    pub fn mgym_rollout_final(env: *mut mgym_env, k: u32, actions: *const c_void, obs_traj: *mut f32,
                              reward_traj: *mut f32, flags_traj: *mut u8, final_obs_traj: *mut f32,
                              done_count_out: *mut u64, stream: *mut c_void) -> c_int;
    pub fn mgym_step_episodes(env: *mut mgym_env, actions: *const c_void, obs_out: *mut f32, reward_out: *mut f32,
                              flags_out: *mut u8, final_obs_out: *mut f32, ep_return_out: *mut f32,
                              ep_length_out: *mut u32, stream: *mut c_void) -> c_int;
    pub fn mgym_rollout_episodes(env: *mut mgym_env, k: u32, actions: *const c_void, obs_traj: *mut f32,
                                 reward_traj: *mut f32, flags_traj: *mut u8, final_obs_traj: *mut f32,
                                 ep_return_traj: *mut f32, ep_length_traj: *mut u32, done_count_out: *mut u64,
                                 stream: *mut c_void) -> c_int;
    pub fn mgym_sample_actions(env: *mut mgym_env, actions_out: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn mgym_step_host(env: *mut mgym_env, actions_host: *const c_void, obs_host: *mut f32,
                          reward_host: *mut f32, flags_host: *mut u8, stream: *mut c_void) -> c_int;
    pub fn mgym_num_params(kind: c_int) -> c_int;
    pub fn mgym_param_name(kind: c_int, i: c_int) -> *const c_char;
    pub fn mgym_param_defaults(kind: c_int, out: *mut f32) -> c_int;
    pub fn mgym_set_params(env: *mut mgym_env, params: *const f32, stream: *mut c_void) -> c_int;
    pub fn mgym_get_params(env: *mut mgym_env, out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn mgym_sample_params(env: *mut mgym_env, low: *const f32, high: *const f32, mask: *const u8, key: u64,
                              stream: *mut c_void) -> c_int;
    pub fn mgym_set_param_redraw(env: *mut mgym_env, low: *const f32, high: *const f32, stream: *mut c_void) -> c_int;
    pub fn mgym_get_param_redraw(env: *const mgym_env, enabled: *mut c_int, low: *mut f32, high: *mut f32) -> c_int;
    pub fn mgym_stats_get(env: *mut mgym_env, out: *mut mgym_stats, stream: *mut c_void) -> c_int;
    pub fn mgym_stats_reset(env: *mut mgym_env, stream: *mut c_void) -> c_int;
    pub fn mgym_stats_export(env: *mut mgym_env, device_vec5_out: *mut f64, stream: *mut c_void) -> c_int;
    pub fn mgym_stats_allreduce(env: *mut mgym_env, nccl_comm: *mut c_void, device_vec5_out: *mut f64,
                                stream: *mut c_void) -> c_int;
}
