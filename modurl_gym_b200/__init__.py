"""modurl_gym_b200 -- B200-native batched classic-control simulator (drop-in for the
reset/step hot path of ModuRL/ModuRL_Gym).  See DESIGN.md and include/mgym.h."""
from ._lib import InvalidActionError, MgymError, load as load_library  # noqa: F401
from .spaces import BoxSpace, Discrete  # noqa: F401


def __getattr__(name):
    # GpuVecEnv needs torch; keep `import modurl_gym_b200` light for symbol/ABI checks.
    if name in ("GpuVecEnv", "StepInfo", "Rollout", "EpisodeStats", "Episodes", "KINDS", "CARTPOLE", "MOUNTAIN_CAR",
                "MOUNTAIN_CAR_CONTINUOUS", "PENDULUM", "ACROBOT", "FLAG_TERMINATED", "FLAG_TRUNCATED"):
        from . import vec_env

        return getattr(vec_env, name)
    raise AttributeError(name)
