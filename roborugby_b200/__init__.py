"""roborugby_b200 — B200-native batched simulator for the RoboRugby gym environments.

Only the step()/reset() hot path of harman097/RoboRugby is implemented (SURVEY.md §8), as
hand-written sm_100a CUDA kernels behind the C ABI in include/rr_b200.h.  There is no CPU
fallback: importing this package works anywhere, constructing an env needs a CUDA device and the
built librr_b200.so.
"""
from .constants import ENV_IDS, GAME, PRESETS, TEAM_GRUMPY, TEAM_HAPPY, TRAIN, get_preset  # noqa: F401
from .stats import allreduce_stats, shard_envs, summarize  # noqa: F401


def __getattr__(name):  # torch-dependent modules are imported lazily
    if name in ("RoboRugbyVecEnv", "ResetPool"):
        from . import vec_env
        return getattr(vec_env, name)
    if name in ("og_twitchy_actions",):
        from .players import og_twitchy_actions
        return og_twitchy_actions
    if name in ("make", "spec", "RoboRugbyEnv", "DebugInfo"):
        from . import gym_env
        return getattr(gym_env, name)
    raise AttributeError(name)
