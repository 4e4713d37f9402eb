"""ctypes loader for librr_b200.so (C ABI declared in include/rr_b200.h).

The library is CUDA-only; there is no CPU fallback.  Loading fails loudly if the shared object
has not been built (run `python -c "import __graft_entry__ as g; g.build()"`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RR_B200_LIB", os.path.join(_HERE, "librr_b200.so"))

ABI_VERSION = 2
PRESET_GAME, PRESET_TRAIN = 0, 1
REW_CHASE, REW_PUSHPOS, REW_NAUGHTY = 1, 2, 4
OBS_NONE, OBS_BASIC_LIDAR, OBS_LIDAR6_V2, OBS_ALLCOORDS, OBS_ALLCOORDS_PRIOR, OBS_LIDAR6_V1 = 0, 1, 2, 3, 4, 5
NUM_STATS = 8
STAT_NAMES = ("episodes", "return_happy", "return_grumpy", "length", "naughty", "errors", "steps", "squeeze_replays")
FLAG_NO_SQUEEZE_MEMO = 1

ERR_BITS = {
    1: "Game is over. Go home.",                                   # RR_EnvBase.py:262
    2: "more commands than robot engines",                        # :271 / :622
    4: "UNABLE TO RESOLVE BOT/BOT COLLISIONS",                    # :313
    8: "UNABLE TO UNDO MOVE FOR ROBOT",                           # :325
    16: "ROBOTS STUCK FROM PRIOR FRAME.",                         # :328
    32: "UNABLE TO RESOLVE ALL COLLISIONS FOR FRAME",             # :421
    64: "Really tho?? The balls are in the EXACT same spot????",  # RR_TrashyPhysics.py:250
    128: "Numerator AND Denominator are both 0.",                 # MyUtils.py:25
    256: "reset placement loop exceeded its bound",
    512: "invalid action: a discrete id outside 0..7 (KeyError), or a thrust whose int(round(x)) is NaN, infinite or "
         "outside [-8, 7]",                                         # RR_EnvBase.py:593-606, RR_Robot.py:100-102
}


class Config(C.Structure):
    """struct rr_config (include/rr_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("preset", C.c_int32), ("reward_mask", C.c_uint32),
        ("observer", C.c_int32), ("discrete", C.c_int32), ("time_limit", C.c_int32),
        ("auto_reset", C.c_int32), ("out_f64", C.c_int32), ("strict_reset", C.c_int32),
        ("reward_order", C.c_uint32), ("seed", C.c_uint64), ("env_offset", C.c_int64),
        ("flags", C.c_uint32), ("goal_scoring", C.c_int32),
    ]


# name -> (restype, argtypes); kept in one table so tests can check it against the header
_vp, _i32, _i64 = C.c_void_p, C.c_int32, C.c_int64
SIGNATURES = {
    "rr_default_config": (C.c_int, [C.POINTER(Config), C.c_int, C.c_char_p]),
    "rr_check_config": (C.c_int, [C.POINTER(Config)]),
    "rr_create": (C.c_int, [C.POINTER(Config), _i64, C.c_int, C.POINTER(_vp)]),
    "rr_destroy": (C.c_int, [_vp]),
    "rr_last_error": (C.c_char_p, []),
    "rr_num_envs": (C.c_int, [_vp, C.POINTER(_i64)]),
    "rr_num_robots": (C.c_int, [_vp]),
    "rr_num_balls": (C.c_int, [_vp]),
    "rr_obs_dim": (C.c_int, [_vp]),
    "rr_max_steps": (C.c_int, [_vp]),
    "rr_reset": (C.c_int, [_vp, _vp, _vp]),
    "rr_reset_fixed": (C.c_int, [_vp, _vp, _i32, _vp]),
    "rr_set_starting_positions": (C.c_int, [_vp, _vp, _vp]),
    "rr_get_starting_positions": (C.c_int, [_vp, _vp, _vp]),
    "rr_observe": (C.c_int, [_vp, _vp, _vp, _vp]),
    "rr_observe_entity": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "rr_assign_balls": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "rr_step": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "rr_step_host": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "rr_set_pipeline": (C.c_int, [_vp, _i32]),
    "rr_join": (C.c_int, [_vp, _vp]),
    "rr_set_flush_buffer": (C.c_int, [_vp, _vp, _i64]),
    "rr_step_host_begin": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, C.POINTER(_i32)]),
    "rr_step_host_end": (C.c_int, [_vp, _i32]),
    "rr_set_state": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "rr_get_state": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "rr_goal_state": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "rr_error_mask": (C.c_int, [_vp, _vp, _i32]),
    "rr_last_naughty": (C.c_int, [_vp, _vp]),
    "rr_get_stats": (C.c_int, [_vp, _vp]),
    "rr_stats_device_ptr": (C.c_int, [_vp, C.POINTER(_vp)]),
    "rr_clear_stats": (C.c_int, [_vp, _vp]),
    "rr_set_stats_buffer": (C.c_int, [_vp, _vp]),
    "rr_launch_count": (_i64, [_vp]),
    "rr_state_bytes_per_env": (_i64, [_vp]),
    "rr_selftest": (C.c_int, [_i32, _i32, _i64, C.c_uint64, _vp]),
}

_lib = None


class RRError(Exception):
    """Raised for any non-zero status of the C ABI (message = rr_last_error())."""


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built. roborugby_b200 has no CPU "
                "fallback; build it with `python -c 'import __graft_entry__ as g; g.build()'`.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here == header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise RRError(load().rr_last_error().decode() or f"rr error {rc}")


def check_config(cfg):
    """rr_check_config: ValueError naming the field if rr_create would refuse cfg."""
    if load().rr_check_config(C.byref(cfg)) != 0:
        raise ValueError(load().rr_last_error().decode())


def default_config(preset, env_id):
    cfg = Config()
    check(load().rr_default_config(C.byref(cfg), int(preset), env_id.encode()))
    return cfg
