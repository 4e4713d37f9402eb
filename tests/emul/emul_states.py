"""ctypes binding of tests/emul/librr_emul_states.so: rr_save_states / rr_load_states in the host build of the device
simulator source.

TEST INFRASTRUCTURE ONLY; see rr_emul_states.cu.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from roborugby_b200._lib import Config

from . import emul

_LIB = os.path.join(emul._HERE, "librr_emul_states.so")
_SRCS = [os.path.join(emul._HERE, "rr_emul_states.cu")] + emul._SRCS


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
        L.emul_row_bytes.argtypes = [C.POINTER(Config)]
        L.emul_row_bytes.restype = i64
        L.emul_save_rows.argtypes = [C.POINTER(Config), vp, vp, vp, i64, vp, i64, vp]
        L.emul_save_rows.restype = None
        L.emul_load_rows.argtypes = [C.POINTER(Config), vp, i64, vp, i64, vp, vp, vp]
        L.emul_load_rows.restype = None
        _lib = L
    return _lib


def row_bytes(cfg):
    return int(lib().emul_row_bytes(C.byref(cfg)))


def _idx(a):
    return None if a is None else emul._p(np.ascontiguousarray(a, np.int64))


def save(batch, start, envs=None, rows=None):
    """rr_save_states on an EmulBatch and its start columns [3R + 2B, M]: rows uint8 [m, S] (m = len(envs), or M).
    `rows` (written in place) keeps whatever the skip rule leaves unwritten."""
    envs = None if envs is None else np.ascontiguousarray(envs, np.int64)
    m = batch.M if envs is None else len(envs)
    if rows is None:
        rows = np.zeros((m, row_bytes(batch.cfg)), np.uint8)
    assert rows.shape == (m, row_bytes(batch.cfg)) and rows.flags.c_contiguous
    p = emul._p
    lib().emul_save_rows(C.byref(batch.cfg), p(batch.sf), p(start), p(batch.si), batch.M, _idx(envs), m, p(rows))
    return rows


def load(batch, start, rows, slots=None):
    """rr_load_states into an EmulBatch and its start columns."""
    slots = None if slots is None else np.ascontiguousarray(slots, np.int64)
    assert rows.dtype == np.uint8 and rows.flags.c_contiguous and rows.shape[1] == row_bytes(batch.cfg)
    p = emul._p
    lib().emul_load_rows(C.byref(batch.cfg), p(rows), rows.shape[0], _idx(slots), batch.M, p(batch.sf), p(start),
                         p(batch.si))
