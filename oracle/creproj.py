"""TEST INFRASTRUCTURE ONLY — ctypes loader for oracle/reproj_exact.c (the PnP reprojection-error checker)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "reproj_exact.c")
_SO = os.path.join(_HERE, "_build", "liboracle_reproj.so")
# the flags of oracle/Makefile: -ffp-contract=off keeps every product and sum a separate IEEE operation
_CFLAGS = ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-Wall"]
_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        tmp = _SO + ".tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), *_CFLAGS, "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, _SO)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_SO)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _cols(X, x):
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    return [np.ascontiguousarray(c) for c in (X[:, 0], X[:, 1], X[:, 2], x[:, 0], x[:, 1])]


def projection(K, Rt):
    """P = K [R | t] in the pinned order of the device (pnp_projection)."""
    K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    Rt = np.ascontiguousarray(Rt, dtype=np.float64).reshape(12)
    P = np.empty(12, dtype=np.float64)
    lib().oracle_pnp_projection(_p(K), _p(Rt), _p(P))
    return P.reshape(3, 4)


def reproj_exact_many(Rt, K, X, x, thr):
    """(mask, value) of every record under one [R | t] (3x4), in the device's pinned evaluation order."""
    Rt = np.ascontiguousarray(Rt, dtype=np.float64).reshape(12)
    K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    cols = _cols(X, x)
    n = len(cols[0])
    mask = np.empty(n, dtype=np.uint8)
    val = np.empty(n, dtype=np.float64)
    lib().oracle_reproj_exact_many(_p(Rt), _p(K), *(_p(c) for c in cols), ctypes.c_int64(n), ctypes.c_double(thr),
                                   _p(mask), _p(val))
    return mask.astype(bool), val


def reproj_score_batch(Rt, K, X, x, thr, table=None, valid=None, nthreads=1):
    """(count_extra, S1, S2) per pose [h,3,4]: the 4 samples (table columns 0-3) are never counted and always summed."""
    Rt = np.ascontiguousarray(Rt, dtype=np.float64).reshape(-1, 12)
    K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    h = Rt.shape[0]
    cols = _cols(X, x)
    cnt = np.empty(h, dtype=np.int32)
    s1 = np.empty(h, dtype=np.float64)
    s2 = np.empty(h, dtype=np.float64)
    if table is not None:
        table = np.ascontiguousarray(table, dtype=np.int32).reshape(h, 8)
    if valid is not None:
        valid = np.ascontiguousarray(valid, dtype=np.uint8)
    lib().oracle_reproj_score_batch(
        _p(Rt), _p(valid) if valid is not None else None, _p(K), *(_p(c) for c in cols), ctypes.c_int64(len(cols[0])),
        ctypes.c_int64(h), _p(table) if table is not None else None, ctypes.c_double(thr), _p(cnt), _p(s1), _p(s2),
        ctypes.c_int(nthreads))
    return cnt, s1, s2
