"""ctypes binding of the CPU oracle (oracle/rr_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the cpu_baseline /
--impl reference legs of bench.py.  Nothing under roborugby_b200/ may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "librr_oracle.so")

REW_CHASE, REW_PUSHPOS, REW_NAUGHTY = 1, 2, 4
OBS_NONE, OBS_BASIC_LIDAR, OBS_LIDAR6_V2, OBS_ALLCOORDS, OBS_ALLCOORDS_PRIOR, OBS_LIDAR6_V1 = 0, 1, 2, 3, 4, 5

ERR_BITS = {
    1: "STEP_AFTER_DONE", 2: "TOO_MANY_COMMANDS", 4: "BOT_COLLISIONS", 8: "UNDO_FAILED",
    16: "ROBOTS_STUCK", 32: "UNRESOLVED_FRAME", 64: "COINCIDENT_BALLS", 128: "DIV0", 512: "BAD_ACTION",
}


class Config(C.Structure):
    _fields_ = [
        ("arena_w", C.c_int), ("arena_h", C.c_int),
        ("n_happy", C.c_int), ("n_grumpy", C.c_int),
        ("n_pos", C.c_int), ("n_neg", C.c_int),
        ("game_length_steps", C.c_int), ("game_mode", C.c_int),
        ("reward_mask", C.c_uint32), ("observer", C.c_int),
        ("discrete", C.c_int), ("time_limit", C.c_int), ("reward_order", C.c_uint32),
        ("goal_scoring", C.c_int),
    ]


def build(force=False):
    """Compile the oracle in place (gcc + make only)."""
    src = os.path.join(_HERE, "rr_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < max(
            os.path.getmtime(src), os.path.getmtime(os.path.join(_HERE, "rr_oracle.h"))):
        subprocess.check_call(["make", "-s", "-C", _HERE, "librr_oracle.so"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        L.rro_default_config.argtypes = [C.POINTER(Config), C.c_int, C.c_char_p]
        L.rro_create.argtypes = [C.POINTER(Config)]
        L.rro_create.restype = C.c_void_p
        L.rro_destroy.argtypes = [C.c_void_p]
        for f in (L.rro_obs_dim, L.rro_num_robots, L.rro_num_balls):
            f.argtypes = [C.c_void_p]
            f.restype = C.c_int
        L.rro_set_state.argtypes = [C.c_void_p, dp, dp, ip, dp, C.c_int32]
        L.rro_get_state.argtypes = [C.c_void_p, dp, dp, ip, dp, ip]
        L.rro_step.argtypes = [C.c_void_p, dp, C.c_int, dp, dp, dp, ip, ip]
        L.rro_step.restype = C.c_uint32
        L.rro_observe.argtypes = [C.c_void_p, C.c_int, dp]
        L.rro_observe.restype = C.c_uint32
        L.rro_observe_entity.argtypes = [C.c_void_p, C.c_int, C.c_int, dp]
        L.rro_observe_entity.restype = C.c_uint32
        L.rro_assign_balls.argtypes = [C.c_void_p, ip, C.c_int, ip]
        L.rro_reset_draws.argtypes = [C.c_void_p, C.c_int, ip, C.c_int]
        L.rro_reset_draws.restype = C.c_int
        L.rro_reset_philox.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32]
        L.rro_reset_philox_mode.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int]
        L.rro_set_starting_positions.argtypes = [C.c_void_p, dp, dp]
        L.rro_rollout.argtypes = [C.c_void_p, C.c_long, C.c_uint64]
        L.rro_rollout.restype = C.c_long
        L.rro_goal_state.argtypes = [C.c_void_p, ip, ip, ip, ip, ip]
        L.rro_debug_failed_frames.argtypes = [C.c_int]
        L.rro_debug_failed_frames.restype = C.c_long
        L.rro_scratch_mode.argtypes = [C.c_int]
        L.rro_scratch_reset.argtypes = []
        L.rro_philox4x32.argtypes = [C.POINTER(C.c_uint32)] * 3
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def default_config(preset, env_id, time_limit=False):
    cfg = Config()
    lib().rro_default_config(C.byref(cfg), 1 if preset == "GAME" else 0, env_id.encode())
    cfg.time_limit = int(time_limit)
    return cfg


class OracleEnv:
    """One reference-equivalent env on the CPU."""

    def __init__(self, preset="GAME", env_id="RoboRugbySimpleDuel-v2", cfg=None, time_limit=False):
        self.cfg = cfg if cfg is not None else default_config(preset, env_id, time_limit)
        self._h = lib().rro_create(C.byref(self.cfg))
        if not self._h:
            raise RuntimeError("rro_create failed")
        self.R = lib().rro_num_robots(self._h)
        self.B = lib().rro_num_balls(self._h)
        self.obs_dim = lib().rro_obs_dim(self._h)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().rro_destroy(self._h)
            self._h = None

    def set_state(self, st):
        rob = np.ascontiguousarray(st["rob"], np.float64)
        rhist = np.ascontiguousarray(st["rhist"], np.float64)
        rflag = np.ascontiguousarray(st["rflag"], np.int32)
        ball = np.ascontiguousarray(st["ball"], np.float64)
        assert rob.shape == (self.R, 7) and ball.shape == (self.B, 8), (rob.shape, ball.shape)
        lib().rro_set_state(self._h, _dp(rob), _dp(rhist), _ip(rflag), _dp(ball), int(st["step"]))

    def get_state(self):
        rob = np.zeros((self.R, 7)); rhist = np.zeros((self.R, 3)); rflag = np.zeros((self.R, 3), np.int32)
        ball = np.zeros((self.B, 8)); step = np.zeros(1, np.int32)
        lib().rro_get_state(self._h, _dp(rob), _dp(rhist), _ip(rflag), _dp(ball), _ip(step))
        return dict(rob=rob, rhist=rhist, rflag=rflag, ball=ball, step=np.int32(step[0]))

    def step(self, actions):
        a = np.ascontiguousarray(np.asarray(actions, np.float64).reshape(-1))
        oh = np.full(max(self.obs_dim, 1), np.nan); og = np.full(max(self.obs_dim, 1), np.nan)
        rew = np.zeros(2); done = np.zeros(1, np.int32); nc = np.zeros(1, np.int32)
        err = lib().rro_step(self._h, _dp(a), a.size, _dp(oh), _dp(og), _dp(rew), _ip(done), _ip(nc))
        return dict(obs_h=oh[:self.obs_dim], obs_g=og[:self.obs_dim], rew=rew, done=int(done[0]),
                    naughty=int(nc[0]), err=int(err))

    def observe(self, team):
        o = np.full(max(self.obs_dim, 1), np.nan)
        lib().rro_observe(self._h, int(team), _dp(o))
        return o[:self.obs_dim]

    def goal_state(self):
        """alive[B], score[2] (happy goal, grumpy goal), destroyed[2], dwell[2, B], delta of the last step."""
        alive = np.zeros(self.B, np.int32); score = np.zeros(2, np.int32); destroyed = np.zeros(2, np.int32)
        dwell = np.zeros((2, self.B), np.int32); delta = np.zeros(1, np.int32)
        lib().rro_goal_state(self._h, _ip(alive), _ip(score), _ip(destroyed), _ip(dwell), _ip(delta))
        return dict(alive=alive, score=score, destroyed=destroyed, dwell=dwell, delta=int(delta[0]))

    def observe_entity(self, robot, ball=-1):
        """get_game_state(obj_robot=lstRobots[robot], obj_ball=lstBalls[ball]); ball=-1 is the default ball."""
        o = np.full(max(self.obs_dim, 1), np.nan)
        err = lib().rro_observe_entity(self._h, int(robot), int(ball), _dp(o))
        if err == 0xffffffff:
            raise NotImplementedError("Robot-specific state output not supported.")
        return o[:self.obs_dim]

    def assign_balls(self, robots):
        """Stephen.__ponder: greedy nearest-ball assignment for the players driving `robots`; -1 = no ball."""
        r = np.ascontiguousarray(robots, np.int32)
        out = np.zeros(len(r), np.int32)
        lib().rro_assign_balls(self._h, _ip(r), len(r), _ip(out))
        return out

    def reset_draws(self, draws, randomize=True):
        d = np.ascontiguousarray(draws, np.int32)
        return lib().rro_reset_draws(self._h, int(randomize), _ip(d), d.size)

    def reset_philox(self, seed, env_index, episode, relaxed=False):
        """Placement from the product's counter-based stream; relaxed=True adds the strict_reset=0 rejection rules."""
        lib().rro_reset_philox_mode(self._h, int(seed), int(env_index), int(episode), int(bool(relaxed)))

    def rollout(self, n_steps, seed):
        """n_steps random-action env-steps entirely in C (timing leg of bench.py)."""
        return int(lib().rro_rollout(self._h, int(n_steps), int(seed)))

    def set_starting_positions(self, rob3, ball2):
        r = np.ascontiguousarray(rob3, np.float64); b = np.ascontiguousarray(ball2, np.float64)
        lib().rro_set_starting_positions(self._h, _dp(r), _dp(b))


def scratch_mode(fresh):
    lib().rro_scratch_mode(int(fresh))


def failed_frames(clear=False):
    """Pinned-ball frames (ten failed resolve passes + undo) executed since the last clear."""
    return int(lib().rro_debug_failed_frames(int(clear)))


def scratch_reset():
    lib().rro_scratch_reset()


def philox4x32(ctr, key):
    c = (C.c_uint32 * 4)(*ctr); k = (C.c_uint32 * 2)(*key); o = (C.c_uint32 * 4)()
    lib().rro_philox4x32(c, k, o)
    return list(o)


def _rollout_worker(args):
    import time
    preset, env_id, n_steps, seed = args
    env = OracleEnv(preset, env_id, time_limit=True)
    env.rollout(min(200, n_steps), seed)  # warm-up
    t0 = time.perf_counter()
    env.rollout(n_steps, seed + 1)
    return n_steps, time.perf_counter() - t0


def timed_rollout(preset, env_id, n_steps_per_core, cores):
    """Random-action rollouts of the C oracle on `cores` processes; returns (env_steps/s aggregate, seconds).

    Runs oracle/time_oracle.py in a child interpreter so that the caller's CUDA context (bench.py)
    is never forked."""
    import json
    import sys
    build()
    out = subprocess.run([sys.executable, os.path.join(_HERE, "time_oracle.py"), preset, env_id,
                          str(int(n_steps_per_core)), str(int(cores))], check=True, capture_output=True, text=True,
                         timeout=900)
    d = json.loads(out.stdout.strip().splitlines()[-1])
    return d["steps_per_s"], d["wall_s"]
