"""ctypes binding of tests/emul/librr_emul_pool.so: rr_step_pool's launch (auto-reset from a reset pool) and its draw in the
host build of the device simulator source.

TEST INFRASTRUCTURE ONLY; see rr_emul_pool.cu.  The library is rr_emul.cu plus emul_launch_pool and emul_pool_draw, so
it carries its own copy of the sin/cos switch: use_libm_sincos here sets it in this library and the others.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from roborugby_b200._lib import Config

from . import emul, emul_info

_LIB = os.path.join(emul._HERE, "librr_emul_pool.so")
_SRCS = [os.path.join(emul._HERE, "rr_emul_pool.cu")] + emul._SRCS


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
        vp, i64 = C.c_void_p, C.c_int64
        L.emul_launch_pool.argtypes = [C.POINTER(Config), vp, vp, vp, i64, vp, C.c_int, C.c_int] + [vp] * 11 + [
            i64, vp, C.c_double, vp]
        L.emul_launch_pool.restype = None
        L.emul_pool_draw.argtypes = [C.c_uint64, vp, vp, i64, i64, vp, C.c_double, vp]
        L.emul_pool_draw.restype = None
        L.emul_use_libm_sincos.argtypes = [C.c_int]
        L.emul_use_libm_sincos.restype = None
        _lib = L
    return _lib


def use_libm_sincos(on):
    """emul.use_libm_sincos for every test library."""
    emul_info.use_libm_sincos(on)
    lib().emul_use_libm_sincos(int(bool(on)))


def _opt(x):
    return None if x is None else emul._p(x)


def draw(seed, env, episode, m, cdf=None, p=1.0):
    """rr_sim.cuh pool_draw for arrays of global env indices and (incremented) episode counters -> int64 slots (-1:
    random reset)."""
    env = np.ascontiguousarray(env, np.uint64)
    episode = np.ascontiguousarray(np.broadcast_to(episode, env.shape), np.uint32)
    cdf = None if cdf is None else np.ascontiguousarray(cdf, np.float64)
    out = np.empty(env.size, np.int64)
    lib().emul_pool_draw(int(seed), emul._p(env), emul._p(episode), env.size, int(m), _opt(cdf), float(p), emul._p(out))
    return out.reshape(env.shape)


def launch(batch, start, actions, rows, cdf=None, p=1.0):
    """emul_info.launch through rr_step_pool's launch on an EmulBatch and its start columns [3R + 2B, M] (updated by
    pool resets): the same dict plus slot [K, M] (int32)."""
    a = np.ascontiguousarray(actions, np.float64)
    K, M, A = a.shape
    assert M == batch.M and start.flags.c_contiguous and start.shape[1] == M
    rows = np.ascontiguousarray(rows, np.uint8)
    cdf = None if cdf is None else np.ascontiguousarray(cdf, np.float64)
    D = batch.obs_dim
    rew = np.zeros((K, M, 2)); done = np.zeros((K, M), np.int32); err = np.zeros((K, M), np.int32)
    ng = np.zeros((K, M), np.int32); stats = np.zeros((M, 8)); slot = np.full((K, M), -7, np.int32)
    oh = og = fh = fg = None
    if D:
        oh = np.full((K, M, D), np.nan); og = np.full((K, M, D), np.nan)
        fh = np.full((K, M, D), emul_info.FINAL_CANARY); fg = np.full((K, M, D), emul_info.FINAL_CANARY)
    fl = np.full((K, M), emul_info.FLAGS_CANARY, np.int32)
    p_ = emul._p
    lib().emul_launch_pool(C.byref(batch.cfg), p_(batch.sf), p_(batch.si), p_(start), M, p_(a), A, K, p_(rew), p_(done),
                           p_(err), p_(ng), _opt(oh), _opt(og), p_(stats), _opt(fh), _opt(fg), p_(fl), p_(rows),
                           rows.shape[0], _opt(cdf), float(p), p_(slot))
    return dict(rew=rew, done=done, err=err, naughty=ng, obs_h=oh, obs_g=og, stats=stats, final_h=fh, final_g=fg,
                flags=fl, slot=slot)
