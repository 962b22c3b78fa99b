"""ctypes wrapper of the plain-C restatement of closed-array scans (oracle/cport/qd_cport_closed.c).  TEST INFRASTRUCTURE
(oracle/__init__.py): used by tests/ to cross-check the CUDA closed path and by tools/closed_bench.py as its CPU baseline."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import time

import numpy as np

from . import ALG

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "qd_cport_closed.c")
_DEPS = (_SRC, os.path.join(_HERE, "qd_cport.c"))          # it includes the open restatement
_LIB = os.path.join(_HERE, "libqd_cport_closed.so")
_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(_LIB) < os.path.getmtime(s) for s in _DEPS):
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-shared", "-o", _LIB, _SRC, "-lm"])
    return _LIB


def _load():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        vp = C.c_void_p
        lib.qd_cport_scans_closed.argtypes = [C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, C.c_uint, vp, vp, vp, vp, vp,
                                              vp, vp, C.c_int]
        lib.qd_cport_scans_closed.restype = C.c_int
        _lib = lib
    return _lib


def run_scans_closed(mb, scans, n_charge, flags: int, threads: int = 0, want_n: bool = True, want_margin: bool = False):
    """``oracle.cport.run_scans`` for closed arrays: scan i with total charge ``n_charge[i]`` (broadcast from a scalar) on
    the dots.  Returns (z float32 [pixels], n float64 [pixels, N] or None, seconds[, margin float64 [pixels]])."""
    lib = _load()
    scans = np.ascontiguousarray(scans)
    q = np.ascontiguousarray(np.broadcast_to(np.asarray(n_charge, dtype=np.int32), (len(scans),)))
    pixels = int((scans["pix_offset"] + scans["nx"].astype(np.int64) * scans["ny"]).max())
    n_dot = mb.cdd_inv_gs.shape[-1]
    z = np.empty(pixels, dtype=np.float32)
    n = np.empty((pixels, n_dot), dtype=np.float64) if want_n else None
    margin = np.full(pixels, np.inf) if want_margin else None
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (mb.cdd_inv_gs, mb.cdd_inv_full, mb.cgd_full)]
    params = np.ascontiguousarray(mb.params)
    t0 = time.perf_counter()
    rc = lib.qd_cport_scans_closed(len(scans), scans.ctypes.data, q.ctypes.data, n_dot, mb.cgd_full.shape[-1],
                                   ALG[mb.algorithm], flags, *[a.ctypes.data for a in arrs], params.ctypes.data,
                                   z.ctypes.data, None if n is None else n.ctypes.data,
                                   None if margin is None else margin.ctypes.data, threads)
    dt = time.perf_counter() - t0
    if rc != 0:
        raise ValueError(f"qd_cport_scans_closed failed: {rc} (algorithm {mb.algorithm}, n_charge {sorted(set(q.tolist()))})")
    if want_margin:
        return z, n, dt, margin
    return z, n, dt
