"""TEST INFRASTRUCTURE ONLY — ctypes loader for oracle/select_exact.c (the essential-matrix / homography model scores)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "select_exact.c")
_SO = os.path.join(_HERE, "_build", "liboracle_select.so")
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
        _lib.oracle_score_models.restype = ctypes.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def fundamental(E, K):
    """F = K^-T E K^-1 in the kernel's order."""
    E, K = (np.ascontiguousarray(m, dtype=np.float64).reshape(9) for m in (E, K))
    F = np.empty(9, dtype=np.float64)
    lib().oracle_fundamental(_p(E), _p(K), _p(F))
    return F.reshape(3, 3)


def score_models(K, pts_a, pts_b, E=None, H=None, sigma=1.0, ratio=0.45):
    """dict(per_point [n,4], fixed_e, fixed_h, count_e, count_h, score_e, score_h, ratio_h, model) in the pinned
    evaluation order of k_score_models (see select_exact.c)."""
    pa = np.asarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pb = np.asarray(pts_b, dtype=np.float64).reshape(-1, 2)
    xa, ya, xb, yb = (np.ascontiguousarray(v) for v in (pa[:, 0], pa[:, 1], pb[:, 0], pb[:, 1]))
    n = xa.shape[0]
    Ea = None if E is None else np.ascontiguousarray(E, dtype=np.float64).reshape(9)
    Ha = None if H is None else np.ascontiguousarray(H, dtype=np.float64).reshape(9)
    Ka = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    pp = np.empty((n, 4), dtype=np.float64)
    fixed = np.zeros(2, dtype=np.uint64)
    count = np.zeros(2, dtype=np.int64)
    scores = np.zeros(3, dtype=np.float64)
    model = lib().oracle_score_models(_p(Ea), _p(Ha), _p(Ka), _p(xa), _p(ya), _p(xb), _p(yb), ctypes.c_int64(n),
                                      ctypes.c_double(sigma), ctypes.c_double(ratio), _p(pp), _p(fixed), _p(count),
                                      _p(scores))
    return dict(per_point=pp, fixed_e=int(fixed[0]), fixed_h=int(fixed[1]), count_e=int(count[0]),
                count_h=int(count[1]), score_e=float(scores[0]), score_h=float(scores[1]), ratio_h=float(scores[2]),
                model=int(model))
