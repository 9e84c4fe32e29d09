"""TEST INFRASTRUCTURE ONLY — ctypes loader for oracle/transfer_exact.c (the homography transfer-error checker)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "transfer_exact.c")
_SO = os.path.join(_HERE, "_build", "liboracle_transfer.so")
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


def transfer_exact_many(H, xa, ya, xb, yb, thr):
    """(mask, value) of the homography transfer error for one H over arrays of pixel coordinates, in the pinned
    evaluation order of the device kernels (see oracle_transfer_exact in sed_exact.c)."""
    H = np.ascontiguousarray(H, dtype=np.float64).reshape(9)
    xa, ya, xb, yb = (np.ascontiguousarray(v, dtype=np.float64) for v in (xa, ya, xb, yb))
    mask = np.empty(len(xa), dtype=np.uint8)
    val = np.empty(len(xa), dtype=np.float64)
    lib().oracle_transfer_exact_many(_p(H), _p(xa), _p(ya), _p(xb), _p(yb), ctypes.c_int64(len(xa)),
                                     ctypes.c_double(thr), _p(mask), _p(val))
    return mask.astype(bool), val


def transfer_score_batch(H, xa, ya, xb, yb, thr, table=None, valid=None, nthreads=1):
    """(count_extra, S1, S2) per homography: the 4 samples (table columns 0-3) are never counted and always summed."""
    H = np.ascontiguousarray(H, dtype=np.float64).reshape(-1, 9)
    h = H.shape[0]
    xa, ya, xb, yb = (np.ascontiguousarray(v, dtype=np.float64) for v in (xa, ya, xb, yb))
    cnt = np.empty(h, dtype=np.int32)
    s1 = np.empty(h, dtype=np.float64)
    s2 = np.empty(h, dtype=np.float64)
    if table is not None:
        table = np.ascontiguousarray(table, dtype=np.int32).reshape(h, 8)
    if valid is not None:
        valid = np.ascontiguousarray(valid, dtype=np.uint8)
    lib().oracle_transfer_score_batch(
        _p(H), _p(valid) if valid is not None else None, _p(xa), _p(ya), _p(xb), _p(yb),
        ctypes.c_int64(len(xa)), ctypes.c_int64(h), _p(table) if table is not None else None,
        ctypes.c_double(thr), _p(cnt), _p(s1), _p(s2), ctypes.c_int(nthreads))
    return cnt, s1, s2
