"""ctypes binding of the C ABI declared in include/mgym.h.

This is the same set of entry points a Rust `extern "C"` block would bind (INTEGRATION.md).
There is no fallback: if libmgym.so is missing the import fails loudly."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# MGYM_LIB selects an alternative build of the same library (tuning experiments only)
LIB_PATH = os.environ.get("MGYM_LIB") or os.path.join(HERE, "libmgym.so")

OK = 0
ERR_BAD_ARGUMENT, ERR_CUDA, ERR_NCCL, ERR_INVALID_ACTION, ERR_OUT_OF_MEMORY = -1, -2, -3, -4, -5


class MgymError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"mgym error {code}: {message}")
        self.code = code


class InvalidActionError(MgymError):
    """The reference panics here: assert!(self.action_space.contains(&action)) (cartpole.rs:252)."""


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("auto_reset", C.c_int32),
        ("max_episode_steps", C.c_int32),
        ("sutton_barto_reward", C.c_int32),
        ("is_euler", C.c_int32),
        ("goal_velocity", C.c_float),
        ("track_stats", C.c_int32),
        ("validate_actions", C.c_int32),
        ("env_index_base", C.c_uint64),
        ("device_clock", C.c_int32),
        ("track_returns", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("episodes", C.c_uint64),
        ("terminated", C.c_uint64),
        ("truncated", C.c_uint64),
        ("length_sum", C.c_uint64),
        ("return_sum", C.c_double),
    ]


# every symbol include/mgym.h declares: name -> (restype, argtypes)
_vp, _u64, _i = C.c_void_p, C.c_uint64, C.c_int
SYMBOLS = {
    "mgym_abi_version": (_i, []),
    "mgym_last_error": (C.c_char_p, []),
    "mgym_kind_name": (C.c_char_p, [_i]),
    "mgym_state_dim": (_i, [_i]),
    "mgym_obs_dim": (_i, [_i]),
    "mgym_action_is_continuous": (_i, [_i]),
    "mgym_num_actions": (_i, [_i]),
    "mgym_space_observation": (_i, [_i, _vp, _vp]),
    "mgym_space_action": (_i, [_i, _vp, _vp]),
    "mgym_config_default": (_i, [_i, C.POINTER(Config)]),
    "mgym_create": (_i, [_i, _u64, _i, _u64, C.POINTER(Config), C.POINTER(_vp)]),
    "mgym_destroy": (_i, [_vp]),
    "mgym_num_envs": (_u64, [_vp]),
    "mgym_kind_of": (_i, [_vp]),
    "mgym_step_index": (_u64, [_vp]),
    "mgym_reset": (_i, [_vp, _vp, _vp]),
    "mgym_reset_masked": (_i, [_vp, _vp, _vp, _vp]),
    "mgym_set_reset_pool": (_i, [_vp, _vp, _u64, _vp]),
    "mgym_set_state": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "mgym_get_state": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "mgym_get_obs": (_i, [_vp, _vp, _vp]),
    "mgym_state_ptr": (_vp, [_vp]),
    "mgym_checkpoint_size": (C.c_size_t, [_vp]),
    "mgym_checkpoint_save": (_i, [_vp, _vp, C.c_size_t, _vp]),
    "mgym_checkpoint_load": (_i, [_vp, _vp, C.c_size_t, _vp]),
    "mgym_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mgym_rollout": (_i, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mgym_rollout_final": (_i, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mgym_sample_actions": (_i, [_vp, _vp, _vp]),
    "mgym_step_host": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "mgym_num_params": (_i, [_i]),
    "mgym_param_name": (C.c_char_p, [_i, _i]),
    "mgym_param_defaults": (_i, [_i, _vp]),
    "mgym_set_params": (_i, [_vp, _vp, _vp]),
    "mgym_get_params": (_i, [_vp, _vp, _vp]),
    "mgym_sample_params": (_i, [_vp, _vp, _vp, _vp, _u64, _vp]),
    "mgym_set_param_redraw": (_i, [_vp, _vp, _vp, _vp]),
    "mgym_get_param_redraw": (_i, [_vp, C.POINTER(_i), _vp, _vp]),
    "mgym_stats_get": (_i, [_vp, C.POINTER(Stats), _vp]),
    "mgym_stats_reset": (_i, [_vp, _vp]),
    "mgym_stats_export": (_i, [_vp, _vp, _vp]),
    "mgym_stats_allreduce": (_i, [_vp, _vp, _vp, _vp]),
}
# test probes, not part of the public header
PROBES = {
    "mgym_probe_trig": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _vp]),
    "mgym_probe_philox": (_i, [_vp, _vp, _u64, _vp]),
    "mgym_probe_trig_checksum": (_i, [C.c_uint32, _u64, C.c_uint32, _vp]),
    "mgym_probe_fast_exhaustive": (_i, [_i, _u64, _u64, _vp]),
    "mgym_probe_fast_div_random": (_i, [_u64, _u64, _vp]),
    "mgym_probe_cartpole_fast": (_i, [_u64, _u64, _vp]),
}

_lib = None


def load():
    """Load libmgym.so.  Raises if the CUDA extension has not been built: no fallback exists."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  modurl_gym_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in {**SYMBOLS, **PROBES}.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != OK:
        msg = load().mgym_last_error().decode("utf-8", "replace")
        raise (InvalidActionError if rc == ERR_INVALID_ACTION else MgymError)(rc, msg)
    return rc
