"""ctypes binding of tests/emul/librr_emul_info.so: rr_step_info's launch (terminal observations, RR_ROW_* flags) in the
host build of the device simulator source.

TEST INFRASTRUCTURE ONLY; see rr_emul_info.cu.  The library is rr_emul.cu plus emul_launch_info, so it carries its own
copy of the sin/cos switch: use_libm_sincos here sets it in both test libraries.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from roborugby_b200._lib import Config

from . import emul

_LIB = os.path.join(emul._HERE, "librr_emul_info.so")
_SRCS = [os.path.join(emul._HERE, "rr_emul_info.cu")] + emul._SRCS

# what launch() puts in the rows the launch does not write
FINAL_CANARY = -7777.25
FLAGS_CANARY = 0x55


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
        L.emul_launch_info.argtypes = [C.POINTER(Config), vp, vp, C.c_int64, vp, C.c_int, C.c_int] + [vp] * 10
        L.emul_launch_info.restype = None
        L.emul_use_libm_sincos.argtypes = [C.c_int]
        L.emul_use_libm_sincos.restype = None
        _lib = L
    return _lib


def use_libm_sincos(on):
    """emul.use_libm_sincos for both test libraries."""
    emul.use_libm_sincos(on)
    lib().emul_use_libm_sincos(int(bool(on)))


def launch(batch, actions, observe=False):
    """EmulBatch.launch through rr_step_info's launch: the same dict, plus final_h / final_g [K, M, D] (done rows
    written, the others keep FINAL_CANARY; None without an observer) and flags [K, M] (RR_ROW_*)."""
    p = emul._p
    a = np.ascontiguousarray(actions, np.float64)
    K, M, A = a.shape
    assert M == batch.M
    D = batch.obs_dim
    rew = np.zeros((K, M, 2)); done = np.zeros((K, M), np.int32); err = np.zeros((K, M), np.int32)
    ng = np.zeros((K, M), np.int32); stats = np.zeros((M, 8))
    oh = og = fh = fg = None
    if observe and D:
        oh = np.full((K, M, D), np.nan); og = np.full((K, M, D), np.nan)
    if D:
        fh = np.full((K, M, D), FINAL_CANARY); fg = np.full((K, M, D), FINAL_CANARY)
    fl = np.full((K, M), FLAGS_CANARY, np.int32)
    opt = lambda x: None if x is None else p(x)
    lib().emul_launch_info(C.byref(batch.cfg), p(batch.sf), p(batch.si), M, p(a), A, K, p(rew), p(done), p(err), p(ng),
                           opt(oh), opt(og), p(stats), opt(fh), opt(fg), p(fl))
    return dict(rew=rew, done=done, err=err, naughty=ng, obs_h=oh, obs_g=og, stats=stats, final_h=fh, final_g=fg, flags=fl)
