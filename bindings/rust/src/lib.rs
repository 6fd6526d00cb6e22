//! `GpuVecEnv`: the batched counterpart of `impl Gym for CartPoleV1` (src/classic_control/cartpole.rs:234-357
//! of ModuRL_Gym) over the C ABI of libmgym.so.  NOT COMPILED in the build image (no cargo/rustc).
//!
//! The scalar trait is `fn reset(&mut self) -> Result<Tensor>` / `fn step(&mut self, action: Tensor) ->
//! Result<StepInfo>`; here the tensors gain an env axis and are raw device pointers the embedding crate owns
//! (candle's CUDA storage exposes them), so this crate has no tensor-library dependency.
pub mod scalar;
pub mod sys;

use std::ffi::CStr;
use std::os::raw::c_void;
use std::ptr;

#[derive(Debug)]
pub struct MgymError {
    pub code: i32,
    pub message: String,
}
impl std::fmt::Display for MgymError {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "mgym error {}: {}", self.code, self.message)
    }
}
impl std::error::Error for MgymError {}

fn check(rc: i32) -> Result<(), MgymError> {
    if rc == sys::MGYM_OK {
        return Ok(());
    }
    let message = unsafe { CStr::from_ptr(sys::mgym_last_error()) }.to_string_lossy().into_owned();
    Err(MgymError { code: rc, message })
}

#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum Kind {
    CartPoleV1 = 0,
    MountainCarV0 = 1,
    MountainCarContinuousV0 = 2,
    PendulumV1 = 3,
    AcrobotV1 = 4,
}

/// Builder options keep the reference's names (cartpole.rs:36-44, mountain_car.rs:27-34).
pub struct Builder {
    kind: Kind,
    num_envs: u64,
    device: i32,
    seed: u64,
    cfg: sys::mgym_config,
}
impl Builder {
    pub fn device(mut self, ordinal: i32) -> Self { self.device = ordinal; self }
    pub fn seed(mut self, seed: u64) -> Self { self.seed = seed; self }
    pub fn sutton_barto_reward(mut self, v: bool) -> Self { self.cfg.sutton_barto_reward = v as i32; self }
    pub fn is_euler(mut self, v: bool) -> Self { self.cfg.is_euler = v as i32; self }
    pub fn goal_velocity(mut self, v: f32) -> Self { self.cfg.goal_velocity = v; self }
    pub fn auto_reset(mut self, v: bool) -> Self { self.cfg.auto_reset = v as i32; self }
    pub fn validate_actions(mut self, v: bool) -> Self { self.cfg.validate_actions = v as i32; self }
    pub fn track_stats(mut self, v: bool) -> Self { self.cfg.track_stats = v as i32; self }
    pub fn track_returns(mut self, v: bool) -> Self { self.cfg.track_returns = v as i32; self }
    pub fn env_index_base(mut self, v: u64) -> Self { self.cfg.env_index_base = v; self }
    pub fn graph_capturable(mut self, v: bool) -> Self { self.cfg.device_clock = v as i32; self }
    pub fn build(self) -> Result<GpuVecEnv, MgymError> {
        let mut h = ptr::null_mut();
        check(unsafe { sys::mgym_create(self.kind as i32, self.num_envs, self.device, self.seed, &self.cfg, &mut h) })?;
        Ok(GpuVecEnv { h, kind: self.kind, num_envs: self.num_envs, stream: ptr::null_mut() })
    }
}

/// StepInfo { state, reward, done, truncated } (cartpole.rs:300-305), batched: device pointers to
/// `[obs_dim][N]` f32, `[N]` f32 and `[N]` u8 flags (bit0 = done, bit1 = truncated).
pub struct VecStepInfo {
    pub state: *const f32,
    pub reward: *const f32,
    pub flags: *const u8,
}

/// Host-side actions of one step: Discrete kinds take bytes, Box kinds (MountainCarContinuous, Pendulum) floats.
pub enum HostActions<'a> {
    Discrete(&'a [u8]),
    Box(&'a [f32]),
}

pub struct GpuVecEnv {
    h: *mut sys::mgym_env,
    kind: Kind,
    num_envs: u64,
    stream: *mut c_void,
}
// One handle = one GPU; calls are serialised by `&mut self`, as with the reference's envs.
unsafe impl Send for GpuVecEnv {}

impl GpuVecEnv {
    pub fn builder(kind: Kind, num_envs: u64) -> Result<Builder, MgymError> {
        let mut cfg = unsafe { std::mem::zeroed::<sys::mgym_config>() };
        check(unsafe { sys::mgym_config_default(kind as i32, &mut cfg) })?;
        Ok(Builder { kind, num_envs, device: 0, seed: 0, cfg })
    }
    pub fn num_envs(&self) -> u64 { self.num_envs }
    pub fn obs_dim(&self) -> usize { unsafe { sys::mgym_obs_dim(self.kind as i32) as usize } }
    pub fn is_continuous(&self) -> bool { unsafe { sys::mgym_action_is_continuous(self.kind as i32) == 1 } }
    /// Discrete(n): n; Box action spaces: 0.
    pub fn num_actions(&self) -> i32 { unsafe { sys::mgym_num_actions(self.kind as i32) } }
    /// observation_space() bounds (cartpole.rs:58-64, mountain_car.rs:42-43): (low, high), obs_dim values each.
    pub fn observation_bounds(&self) -> (Vec<f32>, Vec<f32>) {
        let (mut low, mut high) = (vec![0f32; self.obs_dim()], vec![0f32; self.obs_dim()]);
        unsafe { sys::mgym_space_observation(self.kind as i32, low.as_mut_ptr(), high.as_mut_ptr()) };
        (low, high)
    }
    /// action_space() bounds: Box kinds (low, high); Discrete(n) kinds (0, n - 1).
    pub fn action_bounds(&self) -> (f32, f32) {
        let (mut low, mut high) = (0f32, 0f32);
        unsafe { sys::mgym_space_action(self.kind as i32, &mut low, &mut high) };
        (low, high)
    }
    /// The current observation of every env as a host vector, component-major [obs_dim][N] (mgym_get_obs accepts
    /// host pointers).
    pub fn get_obs_host(&mut self) -> Result<Vec<f32>, MgymError> {
        let mut obs = vec![0f32; self.obs_dim() * self.num_envs as usize];
        check(unsafe { sys::mgym_get_obs(self.h, obs.as_mut_ptr(), self.stream) })?;
        Ok(obs)
    }
    pub fn set_stream(&mut self, stream: *mut c_void) { self.stream = stream; }

    /// Gym::reset for every env; `obs_out` is a device buffer of obs_dim * N floats.
    pub fn reset(&mut self, obs_out: *mut f32) -> Result<(), MgymError> {
        check(unsafe { sys::mgym_reset(self.h, obs_out, self.stream) })
    }
    /// Gym::step for every env.  `actions`: device u8[N] (Discrete) or f32[N] (Box).
    pub fn step(&mut self, actions: *const c_void, obs_out: *mut f32, reward_out: *mut f32,
                flags_out: *mut u8) -> Result<VecStepInfo, MgymError> {
        check(unsafe { sys::mgym_step(self.h, actions, obs_out, reward_out, flags_out, ptr::null_mut(), self.stream) })?;
        Ok(VecStepInfo { state: obs_out, reward: reward_out, flags: flags_out })
    }
    /// K fused steps (the caller's loop of cartpole.rs:460-471); `actions` null = device-side random policy.
    pub fn rollout(&mut self, k: u32, actions: *const c_void, obs_traj: *mut f32, reward_traj: *mut f32,
                   flags_traj: *mut u8, done_count: *mut u64) -> Result<(), MgymError> {
        check(unsafe { sys::mgym_rollout(self.h, k, actions, obs_traj, reward_traj, flags_traj, done_count, self.stream) })
    }
    /// `rollout` plus the observation every finished episode ended on (auto-reset handles): where flags_traj[k][i]
    /// != 0, final_obs_traj[k][c][i] is env i's observation before its reset at step k; other entries are not
    /// written.  `final_obs_len` is the length in floats of the device buffer `final_obs_traj`, checked against the
    /// k * obs_dim * N the kernel may write.
    pub fn rollout_final(&mut self, k: u32, actions: *const c_void, obs_traj: *mut f32, reward_traj: *mut f32,
                         flags_traj: *mut u8, final_obs_traj: *mut f32, final_obs_len: usize, done_count: *mut u64)
                         -> Result<(), MgymError> {
        assert!(!final_obs_traj.is_null(), "final_obs_traj: a device buffer (use rollout without one)");
        assert!(final_obs_len >= k as usize * self.obs_dim() * self.num_envs as usize,
                "final_obs_traj: K * obs_dim * N floats, time-major");
        check(unsafe {
            sys::mgym_rollout_final(self.h, k, actions, obs_traj, reward_traj, flags_traj, final_obs_traj, done_count,
                                    self.stream)
        })
    }
    /// `step` plus the return and length of every episode that ended in it (auto-reset handles): where
    /// flags_out[i] != 0, ep_return[i] / ep_length[i] are env i's finished episode; other entries are not written.
    /// Either buffer may be null; `ep_return_len` / `ep_length_len` are the lengths in elements of the device buffers,
    /// checked against the N the kernel may write.
    pub fn step_episodes(&mut self, actions: *const c_void, obs_out: *mut f32, reward_out: *mut f32,
                         flags_out: *mut u8, ep_return: *mut f32, ep_return_len: usize, ep_length: *mut u32,
                         ep_length_len: usize) -> Result<VecStepInfo, MgymError> {
        let n = self.num_envs as usize;
        assert!(ep_return.is_null() || ep_return_len >= n, "ep_return: N floats");
        assert!(ep_length.is_null() || ep_length_len >= n, "ep_length: N u32");
        check(unsafe {
            sys::mgym_step_episodes(self.h, actions, obs_out, reward_out, flags_out, ptr::null_mut(), ep_return,
                                    ep_length, self.stream)
        })?;
        Ok(VecStepInfo { state: obs_out, reward: reward_out, flags: flags_out })
    }
    /// `rollout` plus the return and length of every episode that ended in it (auto-reset handles): where
    /// flags_traj[k][i] != 0, ep_return_traj[k][i] / ep_length_traj[k][i] are the episode env i finished at step k;
    /// other entries are not written.  Either buffer may be null; their lengths in elements are checked against the
    /// K * N the kernel may write.
    pub fn rollout_episodes(&mut self, k: u32, actions: *const c_void, obs_traj: *mut f32, reward_traj: *mut f32,
                            flags_traj: *mut u8, ep_return_traj: *mut f32, ep_return_len: usize,
                            ep_length_traj: *mut u32, ep_length_len: usize, done_count: *mut u64)
                            -> Result<(), MgymError> {
        let kn = k as usize * self.num_envs as usize;
        assert!(ep_return_traj.is_null() || ep_return_len >= kn, "ep_return_traj: K * N floats, time-major");
        assert!(ep_length_traj.is_null() || ep_length_len >= kn, "ep_length_traj: K * N u32, time-major");
        check(unsafe {
            sys::mgym_rollout_episodes(self.h, k, actions, obs_traj, reward_traj, flags_traj, ptr::null_mut(),
                                       ep_return_traj, ep_length_traj, done_count, self.stream)
        })
    }
    /// Host-buffer step for scalar adapters and tests: H2D actions, step, D2H results, synchronises.
    /// Every slice length is checked against what the C side reads or writes (N actions of the kind's own type,
    /// obs_dim * N observations, N rewards, N flags), so this safe function cannot reach out of bounds.
    pub fn step_host(&mut self, actions: HostActions<'_>, obs: &mut [f32], reward: &mut [f32], flags: &mut [u8])
                     -> Result<(), MgymError> {
        let n = self.num_envs as usize;
        let continuous = unsafe { sys::mgym_action_is_continuous(self.kind as i32) } == 1;
        let act_ptr = match actions {
            HostActions::Discrete(a) => {
                assert!(!continuous, "this kind takes Box (f32) actions");
                assert_eq!(a.len(), n, "actions: one u8 per env");
                a.as_ptr() as *const c_void
            }
            HostActions::Box(a) => {
                assert!(continuous, "this kind takes Discrete (u8) actions");
                assert_eq!(a.len(), n, "actions: one f32 per env");
                a.as_ptr() as *const c_void
            }
        };
        assert_eq!(obs.len(), self.obs_dim() * n, "obs: obs_dim * N floats, component-major");
        assert_eq!(reward.len(), n, "reward: N floats");
        assert_eq!(flags.len(), n, "flags: N bytes");
        check(unsafe { sys::mgym_step_host(self.h, act_ptr, obs.as_mut_ptr(), reward.as_mut_ptr(), flags.as_mut_ptr(),
                                           self.stream) })
    }
    /// Testable::set_state (cartpole.rs:444-446) from a HOST array of state_dim * N floats, component-major.
    pub fn set_state(&mut self, state_soa: &[f32]) -> Result<(), MgymError> {
        let sd = unsafe { sys::mgym_state_dim(self.kind as i32) } as usize;
        assert_eq!(state_soa.len(), sd * self.num_envs as usize, "state: state_dim * N floats");
        check(unsafe { sys::mgym_set_state(self.h, state_soa.as_ptr(), ptr::null(), ptr::null(), self.stream) })
    }
    /// Number of per-env physics parameters of this kind (0 for Acrobot).
    pub fn num_params(&self) -> usize { unsafe { sys::mgym_num_params(self.kind as i32).max(0) as usize } }
    /// Per-env physics parameters from a HOST array of num_params * N floats, parameter-major; `None` returns to
    /// the kind's constants.  Rejected values leave the handle untouched.
    pub fn set_params(&mut self, params_soa: Option<&[f32]>) -> Result<(), MgymError> {
        let p = match params_soa {
            Some(p) => {
                assert_eq!(p.len(), self.num_params() * self.num_envs as usize, "params: num_params * N floats");
                p.as_ptr()
            }
            None => ptr::null(),
        };
        check(unsafe { sys::mgym_set_params(self.h, p, self.stream) })
    }
    pub fn get_params(&mut self) -> Result<Vec<f32>, MgymError> {
        let mut v = vec![0f32; self.num_params() * self.num_envs as usize];
        check(unsafe { sys::mgym_get_params(self.h, v.as_mut_ptr(), self.stream) })?;
        Ok(v)
    }
    /// Draws each env's parameters (those with mask[i] != 0; `mask` a device u8[N] or null) from [low, high).
    pub fn sample_params(&mut self, low: &[f32], high: &[f32], mask: *const u8, key: u64) -> Result<(), MgymError> {
        assert!(low.len() == self.num_params() && high.len() == self.num_params(), "low, high: num_params each");
        check(unsafe { sys::mgym_sample_params(self.h, low.as_ptr(), high.as_ptr(), mask, key, self.stream) })
    }
    /// Per-episode redraw: every reset of an env draws its parameters from [low, high) (num_params values each);
    /// `None` stops redrawing.  Rejected ranges leave the handle untouched.
    pub fn set_param_redraw(&mut self, ranges: Option<(&[f32], &[f32])>) -> Result<(), MgymError> {
        let (lo, hi) = match ranges {
            Some((low, high)) => {
                assert!(low.len() == self.num_params() && high.len() == self.num_params(), "low, high: num_params each");
                (low.as_ptr(), high.as_ptr())
            }
            None => (ptr::null(), ptr::null()),
        };
        check(unsafe { sys::mgym_set_param_redraw(self.h, lo, hi, self.stream) })
    }
    /// The redraw ranges (low, high), or `None` when the handle does not redraw.
    pub fn param_redraw(&self) -> Result<Option<(Vec<f32>, Vec<f32>)>, MgymError> {
        let (mut lo, mut hi) = (vec![0f32; self.num_params()], vec![0f32; self.num_params()]);
        let mut on: std::os::raw::c_int = 0;
        check(unsafe { sys::mgym_get_param_redraw(self.h, &mut on, lo.as_mut_ptr(), hi.as_mut_ptr()) })?;
        Ok(if on != 0 { Some((lo, hi)) } else { None })
    }
    pub fn stats(&mut self) -> Result<sys::mgym_stats, MgymError> {
        let mut s = sys::mgym_stats::default();
        check(unsafe { sys::mgym_stats_get(self.h, &mut s, self.stream) })?;
        Ok(s)
    }
    pub fn checkpoint(&mut self) -> Result<Vec<u8>, MgymError> {
        let n = unsafe { sys::mgym_checkpoint_size(self.h) };
        let mut blob = vec![0u8; n];
        check(unsafe { sys::mgym_checkpoint_save(self.h, blob.as_mut_ptr() as *mut c_void, n, self.stream) })?;
        Ok(blob)
    }
    pub fn restore(&mut self, blob: &[u8]) -> Result<(), MgymError> {
        check(unsafe { sys::mgym_checkpoint_load(self.h, blob.as_ptr() as *const c_void, blob.len(), self.stream) })
    }
}

impl Drop for GpuVecEnv {
    fn drop(&mut self) {
        unsafe { sys::mgym_destroy(self.h) };
    }
}
