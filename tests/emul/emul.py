"""ctypes binding of tests/emul/librr_emul.so: the device simulator source compiled for the HOST.

TEST INFRASTRUCTURE ONLY (CPU-side verification of the kernel logic); see rr_emul.cu.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from roborugby_b200._lib import Config, ABI_VERSION

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = os.path.join(_HERE, "librr_emul.so")
_SRCS = [os.path.join(_HERE, "rr_emul.cu"), os.path.join(_ROOT, "include", "rr_b200.h")] + [
    os.path.join(_ROOT, "roborugby_b200", "csrc", f) for f in ("rr_sim.cuh", "rr_sincos.cuh", "rr_sincos_grid.inc")]


def build(force=False):
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(p) for p in _SRCS):
        tmp = f"{_LIB}.{os.getpid()}.tmp"   # (pytest-xdist workers may all find the library stale at once)
        subprocess.check_call([
            "nvcc", "-O2", "-std=c++17", "--fmad=false", "-Wno-deprecated-gpu-targets",
            "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-builtin", "-shared", "-o", tmp, _SRCS[0]])
        os.replace(tmp, _LIB)
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        vp = C.c_void_p
        L.emul_step.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, vp, C.c_int, vp, vp, vp, vp, vp]
        L.emul_step.restype = C.c_uint
        L.emul_reset.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, C.c_uint64, C.c_uint32, C.c_int]
        L.emul_reset.restype = C.c_uint
        L.emul_observe.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, C.c_int, vp]
        L.emul_observe.restype = C.c_uint
        L.emul_reset_fixed.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, vp, C.c_int]
        L.emul_reset_fixed.restype = None
        L.emul_use_libm_sincos.argtypes = [C.c_int]
        L.emul_use_libm_sincos.restype = None
        L.emul_sincos.argtypes = [vp, C.c_int, vp, vp]
        L.emul_sincos.restype = None
        L.emul_sincos2.argtypes = [vp, C.c_int, vp, vp, C.c_int]
        L.emul_sincos2.restype = None
        L.emul_predicates.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, vp, vp]
        L.emul_predicates.restype = None
        L.emul_observe_entity.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, C.c_int, C.c_int, vp]
        L.emul_observe_entity.restype = C.c_uint
        L.emul_assign_balls.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, vp, C.c_int, vp]
        L.emul_assign_balls.restype = None
        L.emul_goal_rollout.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, vp, vp, vp, vp]
        L.emul_goal_rollout.restype = C.c_uint
        L.emul_step_k.argtypes = [C.POINTER(Config), vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, vp, vp]
        L.emul_step_k.restype = C.c_uint
        i64 = C.c_int64
        L.emul_cols_dims.argtypes = [C.POINTER(Config), vp]
        L.emul_cols_dims.restype = None
        L.emul_cols_set_state.argtypes = [C.POINTER(Config), vp, vp, i64, i64, vp, vp, vp, vp, C.c_int32]
        L.emul_cols_set_state.restype = None
        L.emul_cols_get_state.argtypes = [C.POINTER(Config), vp, vp, i64, i64, vp, vp, vp, vp, vp]
        L.emul_cols_get_state.restype = None
        L.emul_cols_reset.argtypes = [C.POINTER(Config), vp, vp, i64, vp, C.c_int]
        L.emul_cols_reset.restype = None
        L.emul_launch.argtypes = [C.POINTER(Config), vp, vp, i64, vp, C.c_int, C.c_int] + [vp] * 7
        L.emul_launch.restype = None
        L.emul_reward_config_valid.argtypes = [vp, vp, i64, vp]
        L.emul_reward_config_valid.restype = None
        L.emul_last_replays.argtypes = []
        L.emul_last_replays.restype = C.c_double
        L.emul_last_whole_frames.argtypes = []
        L.emul_last_whole_frames.restype = C.c_double
        L.emul_last_stuck_replays.argtypes = []
        L.emul_last_stuck_replays.restype = C.c_double
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class EmulEnv:
    """One env advanced by the host build of the CUDA simulator source."""

    def __init__(self, cfg, R, B, obs_dim):
        self.cfg, self.R, self.B, self.obs_dim = cfg, R, B, obs_dim
        self.rob = np.zeros((R, 7)); self.rhist = np.zeros((R, 3)); self.rflag = np.zeros((R, 3), np.int32)
        self.ball = np.zeros((B, 8)); self.stepc = np.zeros(1, np.int32)

    def set_state(self, st):
        self.rob[...] = st["rob"]; self.rhist[...] = st["rhist"]; self.rflag[...] = st["rflag"]
        self.ball[...] = st["ball"]; self.stepc[0] = st["step"]

    def get_state(self):
        return dict(rob=self.rob.copy(), rhist=self.rhist.copy(), rflag=self.rflag.copy(), ball=self.ball.copy(),
                    step=np.int32(self.stepc[0]))

    def step(self, actions):
        a = np.ascontiguousarray(np.asarray(actions, np.float64).reshape(-1))
        d = max(self.obs_dim, 1)
        oh = np.full(d, np.nan); og = np.full(d, np.nan); rew = np.zeros(2)
        done = np.zeros(1, np.int32); ng = np.zeros(1, np.int32)
        err = lib().emul_step(C.byref(self.cfg), _p(self.rob), _p(self.rhist), _p(self.rflag), _p(self.ball),
                              _p(self.stepc), _p(a), a.size, _p(oh), _p(og), _p(rew), _p(done), _p(ng))
        return dict(obs_h=oh[:self.obs_dim], obs_g=og[:self.obs_dim], rew=rew, done=int(done[0]), naughty=int(ng[0]),
                    err=int(err))

    def step_k(self, actions):
        """K discrete steps on one Env object (memo state persists across the steps, as in a fused GPU launch).
        actions [K, A]; returns (error bits, rewards [K, 2], (replays, whole-frame replays, stuck-pair replays))."""
        a = np.ascontiguousarray(np.asarray(actions, np.float64))
        K, A = a.shape
        rew = np.zeros((K, 2)); cnt = np.zeros(3)
        err = lib().emul_step_k(C.byref(self.cfg), _p(self.rob), _p(self.rhist), _p(self.rflag), _p(self.ball),
                                _p(self.stepc), _p(a), A, K, _p(rew), _p(cnt))
        return int(err), rew, cnt

    def goal_rollout(self, actions):
        """K steps on one Env object with the goal bookkeeping recorded after every step.  actions [K, A] with NaN for
        absent commands.  Returns dict(err, steps (completed), rew [K, 2], alive [K] (mask), scored [K] (masks), done [K],
        dwell [2, B] (final))."""
        a = np.ascontiguousarray(np.asarray(actions, np.float64))
        K, A = a.shape
        n_act = np.ascontiguousarray((~np.isnan(a)).sum(1).astype(np.int32))
        a = np.nan_to_num(a, nan=0.0)
        rew = np.zeros((K, 2)); goal = np.zeros((K, 3), np.int32); dwell = np.zeros((2, self.B), np.int32)
        done_steps = np.zeros(1, np.int32)
        err = lib().emul_goal_rollout(C.byref(self.cfg), _p(self.rob), _p(self.rhist), _p(self.rflag), _p(self.ball),
                                      _p(self.stepc), _p(a), _p(n_act), A, K, _p(rew), _p(goal), _p(dwell), _p(done_steps))
        return dict(err=int(err), steps=int(done_steps[0]), rew=rew, alive=goal[:, 0], scored=goal[:, 1], done=goal[:, 2],
                    dwell=dwell)

    def reset(self, env_index, episode, construct=False):
        return lib().emul_reset(C.byref(self.cfg), _p(self.rob), _p(self.rhist), _p(self.rflag), _p(self.ball),
                                _p(self.stepc), int(env_index), int(episode), int(construct))

    def reset_fixed(self, start, as_constructed=False):
        st = np.ascontiguousarray(start, np.float64)
        lib().emul_reset_fixed(C.byref(self.cfg), _p(self.rob), _p(self.rhist), _p(self.rflag), _p(self.ball),
                               _p(self.stepc), _p(st), int(as_constructed))

    def observe(self, team):
        o = np.full(max(self.obs_dim, 1), np.nan)
        lib().emul_observe(C.byref(self.cfg), _p(self.rob), _p(self.rhist), _p(self.rflag), _p(self.ball),
                           _p(self.stepc), int(team), _p(o))
        return o[:self.obs_dim]


class EmulBatch:
    """M envs whose complete state persists between calls in the kernels' HBM layout (rr::Columns in rr_sim.cuh):
    launch() does what one k_step launch does, with the bookkeeping and auto-reset of the kernel source."""

    def __init__(self, cfg, M, R, B, obs_dim):
        self.cfg, self.M, self.R, self.B, self.obs_dim = cfg, M, R, B, obs_dim
        dims = np.zeros(5, np.int32)
        lib().emul_cols_dims(C.byref(cfg), _p(dims))
        nf, ni, self._episode_row, self._err_row, self._naughty_row = (int(d) for d in dims)
        self.sf = np.zeros((nf, M)); self.si = np.zeros((ni, M), np.int32)
        self.reset(create=True)

    def reset(self, mask=None, create=False):
        """rr_create (create=True) or rr_reset of the envs whose mask entry is true (None: all)."""
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        lib().emul_cols_reset(C.byref(self.cfg), _p(self.sf), _p(self.si), self.M, None if m is None else _p(m),
                              int(create))

    def set_state(self, i, st):
        """rr_set_state for env i."""
        rob = np.ascontiguousarray(st["rob"], np.float64); rhist = np.ascontiguousarray(st["rhist"], np.float64)
        rflag = np.ascontiguousarray(st["rflag"], np.int32); ball = np.ascontiguousarray(st["ball"], np.float64)
        lib().emul_cols_set_state(C.byref(self.cfg), _p(self.sf), _p(self.si), self.M, int(i), _p(rob), _p(rhist),
                                  _p(rflag), _p(ball), int(st["step"]))

    def get_state(self, i):
        """rr_get_state of env i."""
        rob = np.zeros((self.R, 7)); rhist = np.zeros((self.R, 3)); rflag = np.zeros((self.R, 3), np.int32)
        ball = np.zeros((self.B, 8)); step = np.zeros(1, np.int32)
        lib().emul_cols_get_state(C.byref(self.cfg), _p(self.sf), _p(self.si), self.M, int(i), _p(rob), _p(rhist),
                                  _p(rflag), _p(ball), _p(step))
        return dict(rob=rob, rhist=rhist, rflag=rflag, ball=ball, step=np.int32(step[0]))

    @property
    def episode(self):
        return self.si[self._episode_row].copy()

    def error_mask(self, clear=False):
        """rr_error_mask."""
        m = self.si[self._err_row].astype(np.uint32)
        if clear:
            self.si[self._err_row] = 0
        return m

    def last_naughty(self):
        return self.si[self._naughty_row].copy()

    def launch(self, actions, observe=False):
        """One launch of K steps; actions [K, M, A].  Returns dict(rew [K, M, 2], done, err (the row's error bits),
        naughty [K, M], obs_h / obs_g [K, M, D] (observe=True), stats [M, RR_NUM_STATS]: each env's contribution)."""
        a = np.ascontiguousarray(actions, np.float64)
        K, M, A = a.shape
        assert M == self.M
        rew = np.zeros((K, M, 2)); done = np.zeros((K, M), np.int32); err = np.zeros((K, M), np.int32)
        ng = np.zeros((K, M), np.int32); stats = np.zeros((M, 8))
        oh = og = None
        if observe and self.obs_dim:
            oh = np.full((K, M, self.obs_dim), np.nan); og = np.full((K, M, self.obs_dim), np.nan)
        lib().emul_launch(C.byref(self.cfg), _p(self.sf), _p(self.si), M, _p(a), A, K, _p(rew), _p(done), _p(err),
                          _p(ng), None if oh is None else _p(oh), None if og is None else _p(og), _p(stats))
        return dict(rew=rew, done=done, err=err, naughty=ng, obs_h=oh, obs_g=og, stats=stats)


def observe_entity(cfg, st, robot, ball, obs_dim):
    rob = np.ascontiguousarray(st["rob"], np.float64); rhist = np.ascontiguousarray(st["rhist"], np.float64)
    rflag = np.ascontiguousarray(st["rflag"], np.int32); bl = np.ascontiguousarray(st["ball"], np.float64)
    step = np.zeros(1, np.int32)
    o = np.full(max(obs_dim, 1), np.nan)
    lib().emul_observe_entity(C.byref(cfg), _p(rob), _p(rhist), _p(rflag), _p(bl), _p(step), int(robot), int(ball), _p(o))
    return o[:obs_dim]


def assign_balls(cfg, st, robots):
    rob = np.ascontiguousarray(st["rob"], np.float64); rhist = np.ascontiguousarray(st["rhist"], np.float64)
    rflag = np.ascontiguousarray(st["rflag"], np.int32); bl = np.ascontiguousarray(st["ball"], np.float64)
    step = np.zeros(1, np.int32)
    r = np.ascontiguousarray(robots, np.int32); out = np.zeros(len(r), np.int32)
    lib().emul_assign_balls(C.byref(cfg), _p(rob), _p(rhist), _p(rflag), _p(bl), _p(step), _p(r), len(r), _p(out))
    return out


def predicates(cfg, st):
    """(rr[6], br[32]) int arrays: bit0 = cheap rejection fired, bit1 = reference predicate True."""
    rob = np.ascontiguousarray(st["rob"], np.float64); rhist = np.ascontiguousarray(st["rhist"], np.float64)
    rflag = np.ascontiguousarray(st["rflag"], np.int32); ball = np.ascontiguousarray(st["ball"], np.float64)
    step = np.zeros(1, np.int32)
    rr = np.zeros(6, np.int32); br = np.zeros(32, np.int32)
    lib().emul_predicates(C.byref(cfg), _p(rob), _p(rhist), _p(rflag), _p(ball), _p(step), _p(rr), _p(br))
    return rr, br


def reward_config_valid(mask, order):
    """rr_reward_config_valid (rr_sim.cuh) element-wise over two integer arrays -> bool array."""
    m = np.ascontiguousarray(mask, np.uint32).reshape(-1); o = np.ascontiguousarray(order, np.uint32).reshape(-1)
    assert m.shape == o.shape
    ok = np.zeros(m.size, np.uint8)
    lib().emul_reward_config_valid(_p(m), _p(o), m.size, _p(ok))
    return ok.astype(bool)


def sincos(x, dd_only=False):
    """The simulator's sin/cos on the host: rr_sincos_grid (grid fast path + rr_sincos_dd), or rr_sincos_dd alone."""
    x = np.ascontiguousarray(x, np.float64)
    s = np.empty_like(x); c = np.empty_like(x)
    lib().emul_sincos2(_p(x), x.size, _p(s), _p(c), int(bool(dd_only)))
    return s, c


def use_libm_sincos(on):
    """True: the host build calls glibc sin/cos (bit-identical trig to the oracle, isolates the kernel
    LOGIC); False (default): rr_sincos_dd, the routine the GPU executes."""
    lib().emul_use_libm_sincos(int(bool(on)))
