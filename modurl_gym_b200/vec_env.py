"""GpuVecEnv: host-side mirror of the reference's `Gym` trait for N batched envs on one B200.

The reference exposes, per scalar env (cartpole.rs:234-357, mountain_car.rs:275-339):
    reset() -> Tensor            step(action: Tensor) -> StepInfo{state, reward, done, truncated}
    observation_space()          action_space()
GpuVecEnv keeps those names and meanings, batched: tensors gain a trailing env axis
(observations are component-major [obs_dim, N]) and live in device memory.  All arithmetic
happens in the CUDA library behind the C ABI of include/mgym.h; PyTorch is used only to
own device buffers and streams.  There is no CPU or PyTorch fallback.
"""
import ctypes as C
from collections import namedtuple

import torch

from . import _lib, spaces

CARTPOLE, MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS, PENDULUM, ACROBOT = range(5)
KINDS = {
    "CartPole-v1": CARTPOLE,
    "MountainCar-v0": MOUNTAIN_CAR,
    "MountainCarContinuous-v0": MOUNTAIN_CAR_CONTINUOUS,
    "Pendulum-v1": PENDULUM,
    "Acrobot-v1": ACROBOT,
}
FLAG_TERMINATED, FLAG_TRUNCATED = 1, 2

class StepInfo:
    """StepInfo { state, reward, done, truncated } (cartpole.rs:300-305), batched.

    state [obs_dim, N] f32, reward [N] f32, flags [N] u8 (bit0 = done, bit1 = truncated) are views of buffers the
    next step overwrites; `done` / `truncated` are boolean tensors derived from `flags` on first use."""

    __slots__ = ("state", "reward", "flags", "_done", "_truncated")

    def __init__(self, state, reward, flags):
        self.state, self.reward, self.flags = state, reward, flags
        self._done = self._truncated = None

    @property
    def done(self):
        if self._done is None:
            self._done = (self.flags & FLAG_TERMINATED) != 0
        return self._done

    @property
    def truncated(self):
        if self._truncated is None:
            self._truncated = (self.flags & FLAG_TRUNCATED) != 0
        return self._truncated

    def __iter__(self):  # state, reward, done, truncated = env.step(a)
        return iter((self.state, self.reward, self.done, self.truncated))


class _DeviceArray:
    """Zero-copy torch view of memory the C library owns (CUDA array interface)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False),
                                         "version": 3, "strides": None}

Rollout = namedtuple("Rollout", ["obs", "reward", "flags", "done_count"])
EpisodeStats = namedtuple("EpisodeStats", ["episodes", "terminated", "truncated", "length_sum", "return_sum"])
# Return (float32) and length (int32 view of the library's uint32) of every episode that ended, aligned with the
# flags of the same call: valid only where flags != 0, e.g. `ep.ret[flags != 0]`
Episodes = namedtuple("Episodes", ["ret", "length"])


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class GpuVecEnv:
    """N independent classic-control envs stepped by hand-written sm_100a kernels.

    kind: one of KINDS (name or index).  Builder parameters keep the reference's names:
    sutton_barto_reward, is_euler (cartpole.rs:39-40), goal_velocity (mountain_car.rs:33).
    """

    def __init__(self, kind, num_envs, device=0, seed=0, auto_reset=True, max_episode_steps=None,
                 sutton_barto_reward=False, is_euler=True, goal_velocity=0.0, track_stats=True,
                 validate_actions=False, env_index_base=0, graph_capturable=False, track_returns=False):
        self._lib = _lib.load()
        self.kind = KINDS[kind] if isinstance(kind, str) else int(kind)
        if isinstance(device, torch.device):
            device = device.index or 0
        self.device = torch.device("cuda", int(device))
        self.num_envs = int(num_envs)
        cfg = _lib.Config()
        _lib.check(self._lib.mgym_config_default(self.kind, C.byref(cfg)))
        cfg.auto_reset = int(bool(auto_reset))
        if max_episode_steps is not None:
            cfg.max_episode_steps = int(max_episode_steps)
        cfg.sutton_barto_reward = int(bool(sutton_barto_reward))
        cfg.is_euler = int(bool(is_euler))
        cfg.goal_velocity = float(goal_velocity)
        cfg.track_stats = int(bool(track_stats))
        cfg.validate_actions = int(bool(validate_actions))
        # per-env running return: gives MountainCarContinuous / Pendulum statistics a return sum (8 more bytes per
        # env-step in the per-call step kernel; free in rollouts)
        cfg.track_returns = int(bool(track_returns))
        cfg.env_index_base = int(env_index_base)
        # device_clock: step index and tile tickets live on the device, so step / rollout / sample_actions can be
        # captured into a CUDA graph (torch.cuda.graph) and replayed; one extra one-thread launch per call
        cfg.device_clock = int(bool(graph_capturable))
        self.config = cfg
        self.auto_reset = bool(auto_reset)
        self._h = C.c_void_p()
        _lib.check(self._lib.mgym_create(self.kind, self.num_envs, self.device.index, int(seed), C.byref(cfg),
                                         C.byref(self._h)))
        self.state_dim = self._lib.mgym_state_dim(self.kind)
        self.obs_dim = self._lib.mgym_obs_dim(self.kind)
        self.continuous = bool(self._lib.mgym_action_is_continuous(self.kind))
        self.action_dtype = torch.float32 if self.continuous else torch.uint8
        self._obs_space = spaces.observation_space(self.kind)
        self._act_space = spaces.action_space(self.kind)
        n = self.num_envs
        with torch.cuda.device(self.device):
            # the handle's own reward row [N].  Where every reward is one value (CartPole-v1 with auto-reset and the
            # default rewards, MountainCar-v0) the library filled it at creation and a step given it stores nothing
            # (36 instead of 40 bytes per CartPole env-step); reward_constant is that value, else None
            self._reward = torch.as_tensor(_DeviceArray(self._lib.mgym_reward_ptr(self._h), (n,)), device=self.device)
            value = C.c_float()
            rc = self._lib.mgym_reward_constant(self._h, C.byref(value))
            if rc < 0:
                _lib.check(rc)
            self.reward_constant = value.value if rc == 1 else None
            self._flags = torch.empty(n, dtype=torch.uint8, device=self.device)
            # the resident state rows [state_dim, N] as a tensor (valid while this env is open)
            self.state_view = torch.as_tensor(_DeviceArray(self._lib.mgym_state_ptr(self._h), (self.state_dim, n)),
                                              device=self.device)
            # kinds whose observation IS the state (CartPole, MountainCar, MountainCarContinuous) return that view:
            # no separate observation buffer is written (42 instead of 58 bytes per CartPole env-step)
            self.obs_is_state = self.kind in (CARTPOLE, MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS)
            self._obs = self.state_view if self.obs_is_state else torch.empty((self.obs_dim, n), dtype=torch.float32,
                                                                              device=self.device)
            # device pointers of the handle's own output buffers, marshalled once (a step is launch-bound for
            # small batches: every microsecond of argument marshalling shows)
            self._p_obs = None if self.obs_is_state else _ptr(self._obs)
            self._p_reward, self._p_flags = _ptr(self._reward), _ptr(self._flags)

    # -- lifecycle ---------------------------------------------------------------------------
    def close(self):
        """Frees the handle; `state_view`, observations returned for obs_is_state kinds and rewards returned by step
        dangle afterwards."""
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.mgym_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # -- Gym trait -----------------------------------------------------------------------------
    def observation_space(self):
        return self._obs_space

    def action_space(self):
        return self._act_space

    def reset(self, mask=None, out=None):
        """Gym::reset for all envs (or those with mask != 0).  Returns obs [obs_dim, N]."""
        obs = self._obs if out is None else out
        dst = None if (self.obs_is_state and out is None) else _ptr(obs)
        if mask is None:
            _lib.check(self._lib.mgym_reset(self._h, dst, self._stream()))
        else:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            _lib.check(self._lib.mgym_reset_masked(self._h, _ptr(mask), dst, self._stream()))
        return obs

    def _check_actions(self, actions, lead=()):
        if not isinstance(actions, torch.Tensor):
            raise TypeError("actions must be a torch.Tensor on the env's device")
        if actions.dtype != self.action_dtype or actions.device != self.device:
            raise TypeError(f"actions must be {self.action_dtype} on {self.device}, got {actions.dtype} on "
                            f"{actions.device}")
        if tuple(actions.shape) != tuple(lead) + (self.num_envs,) or not actions.is_contiguous():
            raise ValueError(f"actions must be contiguous with shape {tuple(lead) + (self.num_envs,)}")

    def _check_buffer(self, t, name, dtype, shape):
        if t.dtype != dtype or t.device != self.device or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
            raise ValueError(f"{name} must be contiguous {str(dtype).replace('torch.', '')} on {self.device} with "
                             f"shape {tuple(shape)}")

    def step(self, actions, want_final_obs=False, want_episodes=False):
        """Gym::step for all envs.  actions: uint8[N] (Discrete) or float32[N] (Box).

        Returns StepInfo(state=[obs_dim, N] f32, reward=[N] f32, done=[N] bool, truncated=[N] bool).
        The tensors are views of buffers reused by the next call.  For obs_is_state kinds `state` is `state_view`, the
        resident state rows.  `reward` is a view of the handle's reward row; on a handle whose rewards are all one
        value (reward_constant is not None) that row is filled once at creation and no step stores into it, so it is
        live: writing into it changes what later steps return.

        want_final_obs=True also returns final [obs_dim, N], the observation before the auto-reset (dense).
        want_episodes=True (auto-reset handles) also returns Episodes(ret [N] f32, length [N] i32): the return and
        length of the episode each env finished in this step (RecordEpisodeStatistics' info["episode"]), the values
        the statistics add.  Valid only where info.flags != 0, e.g. `ep.ret[info.flags != 0]`; the other entries keep
        what an earlier step left (the buffers are reused by the next call).  MountainCarContinuous and Pendulum need
        track_returns=True for ret.  Returns info, (info, final), (info, episodes) or (info, final, episodes)."""
        self._check_actions(actions)
        final = None
        if want_final_obs:
            final = torch.empty_like(self._obs)
        if not want_episodes:
            _lib.check(self._lib.mgym_step(self._h, _ptr(actions), self._p_obs, self._p_reward, self._p_flags,
                                           _ptr(final), self._stream()))
            info = StepInfo(self._obs, self._reward, self._flags)
            return (info, final) if want_final_obs else info
        if getattr(self, "_episodes", None) is None:
            n = self.num_envs
            self._episodes = Episodes(torch.zeros(n, dtype=torch.float32, device=self.device),
                                      torch.zeros(n, dtype=torch.int32, device=self.device))
        ep = self._episodes
        _lib.check(self._lib.mgym_step_episodes(self._h, _ptr(actions), self._p_obs, self._p_reward, self._p_flags,
                                                _ptr(final), _ptr(ep.ret), _ptr(ep.length), self._stream()))
        info = StepInfo(self._obs, self._reward, self._flags)
        return (info, final, ep) if want_final_obs else (info, ep)

    def step_raw(self, actions, obs_out=None, reward_out=None, flags_out=None, final_obs_out=None):
        """mgym_step with caller-owned (possibly absent) outputs; returns nothing."""
        _lib.check(self._lib.mgym_step(self._h, _ptr(actions), _ptr(obs_out), _ptr(reward_out), _ptr(flags_out),
                                       _ptr(final_obs_out), self._stream()))

    def rollout(self, K, actions=None, obs=None, reward=None, flags=None, want_obs=True, count_done=True,
                final_obs=None, want_final_obs=False, ep_return=None, ep_length=None, want_episodes=False):
        """K fused steps (the caller's step loop, cartpole.rs:460-471).  actions: [K, N] or None for the
        device-side uniform random policy.  Returns time-major trajectories.

        want_final_obs=True (auto-reset handles): returns (Rollout, final_obs), where final_obs [K, obs_dim, N]
        (`final_obs`, or a new buffer) holds the observation each episode ended on, before its auto-reset.  Only the
        entries of envs that finished at that step (flags != 0) are written; the others keep what the buffer held.
        The next observation of every transition is then
            next_obs = torch.where((out.flags != 0).unsqueeze(1), final_obs, out.obs)

        want_episodes=True (auto-reset handles): also returns Episodes(ret [K, N] f32, length [K, N] i32)
        (`ep_return` / `ep_length`, or new buffers): the return and length of the episode env i finished at step k,
        the values the statistics add.  Valid only where out.flags != 0, e.g. `ep.ret[out.flags != 0]`; the other
        entries keep what the buffers held.  MountainCarContinuous and Pendulum need track_returns=True.  Returns
        (Rollout, episodes), or (Rollout, final_obs, episodes) with want_final_obs."""
        K = int(K)
        n = self.num_envs
        if final_obs is not None and not want_final_obs:
            raise ValueError("final_obs is the buffer of want_final_obs=True")
        if (ep_return is not None or ep_length is not None) and not want_episodes:
            raise ValueError("ep_return / ep_length are the buffers of want_episodes=True")
        if actions is not None:
            self._check_actions(actions, (K,))
        if obs is None and want_obs:
            obs = torch.empty((K, self.obs_dim, n), dtype=torch.float32, device=self.device)
        if reward is None:
            reward = torch.empty((K, n), dtype=torch.float32, device=self.device)
        if flags is None:
            flags = torch.empty((K, n), dtype=torch.uint8, device=self.device)
        dc = torch.zeros(1, dtype=torch.int64, device=self.device) if count_done else None
        if want_final_obs:
            if final_obs is None:
                final_obs = torch.empty((K, self.obs_dim, n), dtype=torch.float32, device=self.device)
            else:
                self._check_buffer(final_obs, "final_obs", torch.float32, (K, self.obs_dim, n))
        if want_episodes:
            if ep_return is None:
                ep_return = torch.empty((K, n), dtype=torch.float32, device=self.device)
            else:
                self._check_buffer(ep_return, "ep_return", torch.float32, (K, n))
            if ep_length is None:
                ep_length = torch.empty((K, n), dtype=torch.int32, device=self.device)
            else:
                self._check_buffer(ep_length, "ep_length", torch.int32, (K, n))
            _lib.check(self._lib.mgym_rollout_episodes(self._h, K, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(flags),
                                                       _ptr(final_obs), _ptr(ep_return), _ptr(ep_length), _ptr(dc),
                                                       self._stream()))
            out, ep = Rollout(obs, reward, flags, dc), Episodes(ep_return, ep_length)
            return (out, final_obs, ep) if want_final_obs else (out, ep)
        if want_final_obs:
            _lib.check(self._lib.mgym_rollout_final(self._h, K, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(flags),
                                                    _ptr(final_obs), _ptr(dc), self._stream()))
            return Rollout(obs, reward, flags, dc), final_obs
        _lib.check(self._lib.mgym_rollout(self._h, K, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(flags), _ptr(dc),
                                          self._stream()))
        return Rollout(obs, reward, flags, dc)

    def iter_rollout(self, total_steps, chunk=32, actions=None, want_obs=True, want_final_obs=False,
                     want_episodes=False):
        """A long rollout (e.g. MountainCar's 1000 steps, BASELINE configs[2]) as fused launches of `chunk` steps
        over ONE reused trajectory ring: the full trajectory of 2^24 envs x 1000 steps would be 218 GB.
        Yields (first_step, Rollout) per launch; the Rollout tensors are overwritten by the next launch.
        actions: None (device policy) or a callable first_step, n_steps -> [n_steps, N] tensor.
        want_final_obs=True yields (first_step, (Rollout, final_obs)) with one reused [chunk, obs_dim, N] final buffer
        (see rollout: only entries with flags != 0 are valid).  want_episodes=True appends Episodes to that tuple,
        over one reused [chunk, N] pair (valid only where flags != 0: `ep.ret[out.flags != 0]`)."""
        n, K = self.num_envs, int(chunk)
        obs = torch.empty((K, self.obs_dim, n), dtype=torch.float32, device=self.device) if want_obs else None
        reward = torch.empty((K, n), dtype=torch.float32, device=self.device)
        flags = torch.empty((K, n), dtype=torch.uint8, device=self.device)
        final = torch.empty((K, self.obs_dim, n), dtype=torch.float32, device=self.device) if want_final_obs else None
        ep_ret = torch.empty((K, n), dtype=torch.float32, device=self.device) if want_episodes else None
        ep_len = torch.empty((K, n), dtype=torch.int32, device=self.device) if want_episodes else None
        done = 0
        while done < total_steps:
            k = min(K, total_steps - done)
            a = None if actions is None else actions(done, k)
            out = self.rollout(k, a, obs=None if obs is None else obs[:k], reward=reward[:k], flags=flags[:k],
                               want_obs=want_obs, final_obs=None if final is None else final[:k],
                               want_final_obs=want_final_obs, ep_return=None if ep_ret is None else ep_ret[:k],
                               ep_length=None if ep_len is None else ep_len[:k], want_episodes=want_episodes)
            yield done, out
            done += k

    def sample_actions(self, out=None):
        """action_space().sample(device) for every env (cartpole.rs:461)."""
        if out is None:
            out = torch.empty(self.num_envs, dtype=self.action_dtype, device=self.device)
        _lib.check(self._lib.mgym_sample_actions(self._h, _ptr(out), self._stream()))
        return out

    def step_host(self, actions_host, obs_host=None, reward_host=None, flags_host=None):
        """End-to-end step with HOST buffers (numpy arrays or pinned CPU tensors): H2D, step, D2H, sync."""
        _lib.check(self._lib.mgym_step_host(self._h, _hptr(actions_host), _hptr(obs_host), _hptr(reward_host),
                                            _hptr(flags_host), self._stream()))

    # -- Testable hooks (cartpole.rs:436-447) and checkpointing ---------------------------------
    def set_state(self, state, steps=None, sbt=None):
        state = state.to(device=self.device, dtype=torch.float32).contiguous()
        assert tuple(state.shape) == (self.state_dim, self.num_envs)
        steps = None if steps is None else steps.to(device=self.device, dtype=torch.int32).contiguous()
        sbt = None if sbt is None else sbt.to(device=self.device, dtype=torch.int32).contiguous()
        _lib.check(self._lib.mgym_set_state(self._h, _ptr(state), _ptr(steps), _ptr(sbt), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()  # inputs may be temporaries

    def get_state(self):
        n = self.num_envs
        state = torch.empty((self.state_dim, n), dtype=torch.float32, device=self.device)
        steps = torch.empty(n, dtype=torch.int32, device=self.device)
        sbt = torch.empty(n, dtype=torch.int32, device=self.device)
        _lib.check(self._lib.mgym_get_state(self._h, _ptr(state), _ptr(steps), _ptr(sbt), self._stream()))
        return state, steps, sbt

    def get_obs(self, out=None):
        obs = torch.empty((self.obs_dim, self.num_envs), dtype=torch.float32, device=self.device) if out is None else out
        _lib.check(self._lib.mgym_get_obs(self._h, _ptr(obs), self._stream()))
        return obs

    def get_obs_host(self):
        """The current observation as a host array [obs_dim, N] (mgym_get_obs also takes host pointers)."""
        import numpy as np

        out = np.empty((self.obs_dim, self.num_envs), dtype=np.float32)
        _lib.check(self._lib.mgym_get_obs(self._h, _hptr(out), self._stream()))
        return out

    def checkpoint(self):
        """The whole handle (state, counters, running returns, statistics, step/reset indices) as bytes."""
        size = self._lib.mgym_checkpoint_size(self._h)
        buf = (C.c_uint8 * size)()
        _lib.check(self._lib.mgym_checkpoint_save(self._h, buf, size, self._stream()))
        return bytes(buf)

    def restore(self, blob):
        """Resume from `checkpoint()` of a handle with the same kind, size and config: continues bit-identically."""
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        _lib.check(self._lib.mgym_checkpoint_load(self._h, buf, len(blob), self._stream()))

    def set_reset_pool(self, pool):
        """Injected reset states [state_dim, P] (parity runs); None restores Philox."""
        if pool is None:
            _lib.check(self._lib.mgym_set_reset_pool(self._h, None, 0, self._stream()))
            return
        pool = pool.to(device=self.device, dtype=torch.float32).contiguous()
        assert pool.shape[0] == self.state_dim
        _lib.check(self._lib.mgym_set_reset_pool(self._h, _ptr(pool), pool.shape[1], self._stream()))

    # -- per-env physics parameters (domain randomisation) ---------------------------------------
    @staticmethod
    def param_names(kind):
        """Names of the per-env parameters of `kind` (name or index), in row order; () for Acrobot."""
        lib = _lib.load()
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        n = lib.mgym_num_params(k)
        if n < 0:
            raise ValueError(f"unknown kind {kind!r}")
        return tuple(lib.mgym_param_name(k, i).decode() for i in range(n))

    @staticmethod
    def param_defaults(kind):
        """The kind's constants, in the order of param_names(kind)."""
        lib = _lib.load()
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        names = GpuVecEnv.param_names(k)
        out = (C.c_float * max(1, len(names)))()
        _lib.check(lib.mgym_param_defaults(k, out))
        return tuple(float(out[i]) for i in range(len(names)))

    def set_params(self, params):
        """Per-env physics parameters.  params: a [P, N] tensor (rows in param_names order), a dict name -> scalar or
        [N] tensor (unnamed parameters keep their current values), or None to return to the kind's constants.
        Rejected values (not finite, or a non-positive mass / length / time step) raise and change nothing."""
        if params is None:
            _lib.check(self._lib.mgym_set_params(self._h, None, self._stream()))
            return
        names = self.param_names(self.kind)
        if isinstance(params, dict):
            unknown = set(params) - set(names)
            if unknown:
                raise KeyError(f"{sorted(unknown)} are not parameters of {self.kind}: {names}")
            rows = self.get_params()
            for c, name in enumerate(names):
                if name in params:
                    rows[c] = torch.as_tensor(params[name], dtype=torch.float32, device=self.device)
            params = rows
        params = torch.as_tensor(params, dtype=torch.float32).to(self.device).contiguous()
        if tuple(params.shape) != (len(names), self.num_envs):
            raise ValueError(f"params must have shape {(len(names), self.num_envs)}")
        _lib.check(self._lib.mgym_set_params(self._h, _ptr(params), self._stream()))

    def get_params(self, out=None):
        """The per-env parameters as [P, N] (the defaults while none are set)."""
        if out is None:
            out = torch.empty((len(self.param_names(self.kind)), self.num_envs), dtype=torch.float32,
                              device=self.device)
        _lib.check(self._lib.mgym_get_params(self._h, _ptr(out), self._stream()))
        return out

    def sample_params(self, low, high, mask=None, key=0):
        """Draw every env's parameters (or those with mask != 0) uniformly from [low, high) (P values each):
        Philox-keyed by (global env index, key), so independent of sharding.  Capturable into a CUDA graph once
        parameters exist.  For new parameters at every new episode use set_param_redraw instead: it draws them on
        the device inside the resets of step, rollout and reset, keyed by the episode rather than by the caller."""
        np_ = len(self.param_names(self.kind))
        if len(low) != np_ or len(high) != np_:
            raise ValueError(f"low and high need {np_} values each")
        lo = (C.c_float * max(1, np_))(*[float(x) for x in low])
        hi = (C.c_float * max(1, np_))(*[float(x) for x in high])
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self._lib.mgym_sample_params(self._h, lo, hi, _ptr(mask), int(key), self._stream()))

    def set_param_redraw(self, low, high=None):
        """Per-episode domain randomisation: every reset of an env (auto-reset in step / rollout / step_host, and
        reset()) also draws its parameters uniformly from [low, high), on the device, keyed by the episode (DESIGN.md
        section 11).  low, high: P values each; or one dict name -> (low, high), where missing names keep their
        default value ([default, default]); or None to stop redrawing (the rows stay).  Current episodes keep their
        parameters: set_param_redraw(lo, hi); reset() starts every env on drawn ones.  Bad ranges raise and change
        nothing.  A captured CUDA graph replays the ranges it was captured with."""
        if low is None:
            _lib.check(self._lib.mgym_set_param_redraw(self._h, None, None, self._stream()))
            return
        names = self.param_names(self.kind)
        if isinstance(low, dict):
            unknown = set(low) - set(names)
            if unknown:
                raise KeyError(f"{sorted(unknown)} are not parameters of {self.kind}: {names}")
            d = self.param_defaults(self.kind)
            pairs = [low.get(name, (d[c], d[c])) for c, name in enumerate(names)]
            low, high = [p[0] for p in pairs], [p[1] for p in pairs]
        if high is None or len(low) != len(names) or len(high) != len(names):
            raise ValueError(f"low and high need {len(names)} values each")
        lo = (C.c_float * max(1, len(names)))(*[float(x) for x in low])
        hi = (C.c_float * max(1, len(names)))(*[float(x) for x in high])
        _lib.check(self._lib.mgym_set_param_redraw(self._h, lo, hi, self._stream()))

    def param_redraw(self):
        """The redraw ranges as (low, high) tuples of P floats, or None when the handle does not redraw."""
        np_ = max(1, len(self.param_names(self.kind)))
        on, lo, hi = C.c_int(0), (C.c_float * np_)(), (C.c_float * np_)()
        _lib.check(self._lib.mgym_get_param_redraw(self._h, C.byref(on), lo, hi))
        if not on.value:
            return None
        p = len(self.param_names(self.kind))
        return tuple(lo[:p]), tuple(hi[:p])

    @property
    def step_index(self):
        return int(self._lib.mgym_step_index(self._h))

    # -- statistics ------------------------------------------------------------------------------
    def stats(self):
        s = _lib.Stats()
        _lib.check(self._lib.mgym_stats_get(self._h, C.byref(s), self._stream()))
        return EpisodeStats(s.episodes, s.terminated, s.truncated, s.length_sum, s.return_sum)

    def reset_stats(self):
        _lib.check(self._lib.mgym_stats_reset(self._h, self._stream()))

    def stats_tensor(self):
        """The 5-double device vector {episodes, terminated, truncated, length_sum, return_sum}."""
        out = torch.empty(5, dtype=torch.float64, device=self.device)
        _lib.check(self._lib.mgym_stats_export(self._h, _ptr(out), self._stream()))
        return out

    def all_reduce_stats(self, group=None):
        """Sum the episode statistics over all ranks (NCCL all-reduce of 5 doubles)."""
        from .distributed import all_reduce_stats_vector

        return EpisodeStats(*all_reduce_stats_vector(self.stats_tensor(), group))

    def all_reduce_stats_native(self, comm):
        """The same sum through the C ABI's own collective: mgym_stats_allreduce on a raw ncclComm_t
        (`comm`: distributed.NativeNcclComm).  Returns the reduced 5-double device vector."""
        out = torch.empty(5, dtype=torch.float64, device=self.device)
        _lib.check(self._lib.mgym_stats_allreduce(self._h, comm.handle, _ptr(out), self._stream()))
        return out


def _hptr(a):
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        assert a.device.type == "cpu" and a.is_contiguous()
        return C.c_void_p(a.data_ptr())
    return a.ctypes.data_as(C.c_void_p)  # numpy
