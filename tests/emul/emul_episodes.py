"""ctypes binding of tests/emul/librr_emul_episodes.so: rr_step_episodes' launch (each row's episode return, length and goal
words, with or without a reset pool) in the host build of the device simulator source.

TEST INFRASTRUCTURE ONLY; see rr_emul_episodes.cu.  The library is rr_emul.cu plus emul_launch_episodes, so it carries
its own copy of the sin/cos switch: use_libm_sincos here sets it in this library and the others.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from roborugby_b200._lib import Config

from . import emul, emul_info, emul_pool

_LIB = os.path.join(emul._HERE, "librr_emul_episodes.so")
_SRCS = [os.path.join(emul._HERE, "rr_emul_episodes.cu")] + emul._SRCS

# what launch() puts in the episode rows before the launch, so that a row the launch does not write shows
EP_CANARY = -3333.5


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
        L.emul_launch_episodes.argtypes = [C.POINTER(Config), vp, vp, vp, i64, vp, C.c_int, C.c_int] + [vp] * 11 + [
            i64, vp, C.c_double, vp, vp, vp, vp]
        L.emul_launch_episodes.restype = None
        L.emul_use_libm_sincos.argtypes = [C.c_int]
        L.emul_use_libm_sincos.restype = None
        _lib = L
    return _lib


def use_libm_sincos(on):
    """emul.use_libm_sincos for every test library."""
    emul_pool.use_libm_sincos(on)
    lib().emul_use_libm_sincos(int(bool(on)))


def launch(batch, actions, start=None, rows=None, cdf=None, p=1.0):
    """emul_pool.launch without a pool (rows None: rr_step_info's reset; start may then be None) or with one, plus
    ep_return [K, M, 2] (float64), ep_length [K, M] (int32) and, with goal scoring, ep_goals [K, M, 4] (int32; None
    otherwise)."""
    a = np.ascontiguousarray(actions, np.float64)
    K, M, A = a.shape
    assert M == batch.M
    if start is None:
        assert rows is None
        start = np.zeros((3 * batch.R + 2 * batch.B, M))
    assert start.flags.c_contiguous and start.shape[1] == M
    if rows is not None:
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
    er = np.full((K, M, 2), EP_CANARY); el = np.full((K, M), -7, np.int32)
    eg = np.full((K, M, 4), -7, np.int32) if batch.cfg.goal_scoring else None
    p_ = emul._p
    opt = lambda x: None if x is None else p_(x)
    lib().emul_launch_episodes(C.byref(batch.cfg), p_(batch.sf), p_(batch.si), p_(start), M, p_(a), A, K, p_(rew),
                               p_(done), p_(err), p_(ng), opt(oh), opt(og), p_(stats), opt(fh), opt(fg), p_(fl), opt(rows),
                               0 if rows is None else rows.shape[0], opt(cdf), float(p), p_(slot), p_(er), p_(el), opt(eg))
    return dict(rew=rew, done=done, err=err, naughty=ng, obs_h=oh, obs_g=og, stats=stats, final_h=fh, final_g=fg,
                flags=fl, slot=slot, ep_return=er, ep_length=el, ep_goals=eg)
