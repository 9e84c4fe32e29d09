"""ctypes binding of include/sfm_b200.h and the per-process engine.

There is NO CPU fallback: if the shared library is missing or no sm_100 device is visible
the calls raise ``NativeUnavailableError``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SFM_B200_LIB") or os.path.join(_HERE, "libsfm_b200.so")  # override: A/B experiments only

AGG = {"sum": 0, "square": 1, "mean": 2, "rms": 3}
SELECT = {"min_error": 0, "max_inliers": 1, "msac": 2}
VARIANT = {"screen": 0, "full": 1, "screen32": 2, "auto": 3}


class NativeUnavailableError(RuntimeError):
    """libsfm_b200.so is missing / not loadable, or there is no B200 to run it on."""


class NativeError(RuntimeError):
    """A C-ABI call returned a non-zero status."""


class Best(C.Structure):
    _fields_ = [("err", C.c_double), ("index", C.c_int64), ("count_extra", C.c_int32),
                ("reserved", C.c_int32), ("num_invalid", C.c_int64), ("first_invalid", C.c_int64),
                ("E", C.c_double * 9), ("sample", C.c_int32 * 8)]


class Poses(C.Structure):
    _fields_ = [("R", (C.c_double * 9) * 4), ("t", (C.c_double * 3) * 4), ("sv", C.c_double * 3),
                ("counts", C.c_int64 * 4), ("best", C.c_int32), ("reserved", C.c_int32)]


class HPoses(C.Structure):
    _fields_ = [("R", (C.c_double * 9) * 4), ("t", (C.c_double * 3) * 4), ("n", (C.c_double * 3) * 4),
                ("d", C.c_double * 4), ("sv", C.c_double * 3), ("counts", C.c_int64 * 4), ("best", C.c_int32),
                ("rotation_only", C.c_int32)]


class ModelScores(C.Structure):
    _fields_ = [("score_e", C.c_double), ("score_h", C.c_double), ("ratio_h", C.c_double), ("fixed_e", C.c_uint64),
                ("fixed_h", C.c_uint64), ("count_e", C.c_int64), ("count_h", C.c_int64), ("model", C.c_int32),
                ("reserved", C.c_int32)]


class Refinement(C.Structure):
    _fields_ = [("model", C.c_double * 9), ("cost_ransac", C.c_double), ("cost_start", C.c_double),
                ("cost_final", C.c_double), ("num", C.c_int64), ("iterations", C.c_int32), ("status", C.c_int32),
                ("rejected", C.c_int32), ("reserved", C.c_int32)]


REFINE_STATUS = {0: "converged", 1: "max_iterations", 2: "stalled", 3: "no_model", 4: "nonfinite"}

_P = C.c_void_p
_SIGNATURES = {
    "sfm_version": (C.c_int, []),
    "sfm_last_error": (C.c_char_p, []),
    "sfm_device_count": (C.c_int, []),
    "sfm_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "sfm_destroy": (C.c_int, [_P]),
    "sfm_set_stream": (C.c_int, [_P, _P]),
    "sfm_use_default_stream": (C.c_int, [_P]),
    "sfm_synchronize": (C.c_int, [_P]),
    "sfm_set_score_variant": (C.c_int, [_P, C.c_int, C.c_int, C.c_int]),
    "sfm_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(_P)]),
    "sfm_host_free": (C.c_int, [_P]),
    "sfm_mt_shuffle_table": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int64, _P]),
    "sfm_mt_shuffle_resume": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P]),
    "sfm_mt_shuffle_snapshots": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int64, _P, _P]),
    "sfm_set_table": (C.c_int, [_P, _P, C.c_int64]),
    "sfm_sample_device": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_int64, C.c_int64]),
    "sfm_get_table": (C.c_int, [_P, _P, C.c_int64, C.c_int64]),
    "sfm_upload_pairs": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int64, _P]),
    "sfm_upload_pairs_async": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int64, _P]),
    "sfm_upload_pairs_d": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int64, _P]),
    "sfm_get_normalised": (C.c_int, [_P, _P, C.c_int64]),
    "sfm_fit": (C.c_int, [_P, _P, _P, _P]),
    "sfm_set_models": (C.c_int, [_P, _P, _P, C.c_int64]),
    "sfm_get_models": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P]),
    "sfm_score": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P]),
    "sfm_get_best": (C.c_int, [_P, C.POINTER(Best)]),
    "sfm_set_winner": (C.c_int, [_P, C.c_int64, _P]),
    "sfm_near_ties": (C.c_int, [_P, C.c_double, C.c_int64, _P, C.POINTER(C.c_int64)]),
    "sfm_get_rescored": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "sfm_inlier_mask": (C.c_int, [_P, C.c_double, _P, _P]),
    "sfm_ransac_essential": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.POINTER(Best), _P, _P]),
    "sfm_fit_homography": (C.c_int, [_P, _P, _P]),
    "sfm_ransac_homography": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.POINTER(Best), _P, _P, _P, _P]),
    "sfm_homography_mask": (C.c_int, [_P, _P, C.c_double, _P, _P]),
    "sfm_decompose_essential": (C.c_int, [_P, _P, C.POINTER(Poses)]),
    "sfm_recover_pose": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_double, C.POINTER(Poses), _P]),
    "sfm_recover_pose_pixels": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_double,
                                          C.POINTER(Poses), _P]),
    "sfm_triangulate": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, _P]),
    "sfm_pose_and_triangulate": (C.c_int, [_P, C.c_double, C.c_double, C.POINTER(Poses), C.c_int64,
                                           C.POINTER(C.c_int64), _P, _P, _P]),
    "sfm_two_view": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, C.POINTER(Best), C.POINTER(Poses),
                               C.c_int64, C.POINTER(C.c_int64), _P, _P, _P, _P, _P]),
    "sfm_two_view_async": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, _P, _P]),
    "sfm_two_view_fetch": (C.c_int, [_P, C.POINTER(Best), C.POINTER(Poses), C.c_int64, C.POINTER(C.c_int64), _P, _P, _P]),
    "sfm_decompose_homography": (C.c_int, [_P, _P, _P, C.c_double, C.POINTER(HPoses)]),
    "sfm_homography_pose_and_triangulate": (C.c_int, [_P, _P, C.c_double, C.c_double, C.c_double, C.POINTER(HPoses),
                                                      C.c_int64, C.POINTER(C.c_int64), _P, _P, _P]),
    "sfm_two_view_homography": (C.c_int, [_P, _P, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double,
                                          C.POINTER(Best), C.POINTER(HPoses), C.c_int64, C.POINTER(C.c_int64), _P, _P,
                                          _P, _P, _P]),
    "sfm_score_models": (C.c_int, [_P, _P, _P, _P, C.c_double, C.c_double, C.POINTER(ModelScores), _P]),
    "sfm_set_refinement": (C.c_int, [_P, C.c_int]),
    "sfm_get_refinement": (C.c_int, [_P, C.POINTER(Refinement), C.c_int64]),
    "sfm_score_async": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_int, C.POINTER(_P)]),
    "sfm_sharded_tail": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_double, C.c_double]),
    "sfm_sharded_fetch": (C.c_int, [_P, C.POINTER(Best), C.POINTER(C.c_int32), C.POINTER(Poses), C.c_int64,
                                    C.POINTER(C.c_int64), _P, _P, _P]),
    "sfm_nccl_unique_id": (C.c_int, [_P]),
    "sfm_nccl_init": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "sfm_nccl_destroy": (C.c_int, [_P]),
    "sfm_two_view_sharded": (C.c_int, [_P, C.c_uint64, C.c_int64, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double]),
    "sfm_batch_ransac": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, _P, C.c_int64, _P, C.c_int64, C.c_uint64,
                                   C.c_uint64, C.c_double, C.c_double, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "sfm_batch_two_view": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, _P, C.c_int64, _P, C.c_int64, C.c_uint64,
                                     C.c_uint64, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, _P, _P, _P, _P, _P,
                                     _P, _P, C.c_int64, _P, _P, _P]),
    "sfm_batch_two_view_homography": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, _P, C.c_int64, _P, C.c_int64, C.c_uint64,
                                                C.c_uint64, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double,
                                                C.c_double, _P, _P, _P, _P, _P, _P, _P, C.c_int64, _P, _P, _P]),
    "sfm_batch_score_models": (C.c_int, [_P, _P, _P, _P, _P, C.c_double, C.c_double, _P, _P]),
    "sfm_match_brute_force": (C.c_int, [_P, _P, _P, C.c_int, C.c_int64, C.c_int64, _P, C.c_int64, _P, C.c_int64, C.c_int,
                                        C.c_int, C.c_int, C.c_double, _P, _P, _P, _P]),
    "sfm_match_from_scores": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int, C.c_double, _P, _P, _P]),
    "sfm_cross_correlate": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int64, _P, C.c_int, _P]),
    "sfm_harris_output_shape": (C.c_int, [C.c_int64, C.c_int64, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "sfm_harris_corners": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_double, _P, _P,
                                     C.POINTER(C.c_int64), _P, C.POINTER(C.c_int32)]),
    "sfm_enable_timing": (C.c_int, [_P, C.c_int]),
    "sfm_get_timing": (C.c_int, [_P, _P, C.POINTER(C.c_int64)]),
    "sfm_measure_fp64_peak": (C.c_int, [_P, C.POINTER(C.c_double)]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lib_lock = threading.Lock()


def load_library():
    """Load libsfm_b200.so and declare every prototype of include/sfm_b200.h."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeUnavailableError(
                f"{LIB_PATH} is missing — build it with `python -m structure_from_motion_b200.build` "
                "(or __graft_entry__.build()); there is no CPU fallback.")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as exc:  # pragma: no cover
            raise NativeUnavailableError(f"cannot load {LIB_PATH}: {exc}") from exc
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def _ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(_P)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _split_xy(pa):
    """Accept [n,2] arrays (interleaved, stride 2) and return (x_ptr_array, y_view, stride)."""
    pa = _f64(pa)
    if pa.ndim != 2 or pa.shape[1] != 2:
        raise ValueError(f"expected an [n,2] coordinate array, got shape {pa.shape}")
    return pa


class Engine:
    """One context (one GPU, one stream).  Thin, stateful mirror of the C ABI."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = _P()
        rc = self.lib.sfm_create(int(device), C.byref(h))
        if rc != 0:
            msg = self.lib.sfm_last_error().decode()
            if rc == -4:
                raise NativeUnavailableError(f"sfm_create(device={device}): {msg}; there is no CPU fallback.")
            raise NativeError(f"sfm_create(device={device}) -> {rc}: {msg}")
        self.h = h
        self.device = int(device)
        self._keep = None  # host arrays an un-synchronised upload still reads from
        self._out_ptr, self._out_cap, self._out = None, 0, None  # pinned landing buffers of the async path
        self.n = 0
        self.batch_pairs = 0  # pairs of the current batched upload (0: none)

    # -- helpers -------------------------------------------------------------------------
    def _ck(self, rc, what):
        if rc != 0:
            raise NativeError(f"{what} -> {rc}: {self.lib.sfm_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.sfm_destroy(self.h)
            self.h = None
        if getattr(self, "_out_ptr", None):
            self.lib.sfm_host_free(self._out_ptr)
            self._out_ptr, self._out_cap, self._out = None, 0, None

    def pinned_out(self, n: int):
        """(uint8[n], float64[n]) views of engine-owned pinned memory for the results of two_view_async: allocated
        once, grown geometrically, freed with the engine.  Valid until the next call that lands results in them."""
        n = int(n)
        if n > self._out_cap:
            if self._out_ptr:
                self.synchronize()
                self.lib.sfm_host_free(self._out_ptr)
            cap = max(n, self._out_cap + self._out_cap // 2, 1024)
            p = _P()
            self._ck(self.lib.sfm_host_alloc(9 * cap + 64, C.byref(p)), "sfm_host_alloc")
            self._out_ptr, self._out_cap = p, cap
            sed = np.frombuffer((C.c_char * (8 * cap)).from_address(p.value), dtype=np.float64, count=cap)
            mask = np.frombuffer((C.c_char * cap).from_address(p.value + 8 * cap), dtype=np.uint8, count=cap)
            self._out = (mask, sed)
        return self._out[0][:n], self._out[1][:n]

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        """Run on an external stream: a cudaStream_t handle, 0 = the legacy default stream (what
        ``torch.cuda.default_stream().cuda_stream`` is), None = back to the engine's own non-blocking stream.  The
        engine must share a stream with whatever it has to be ordered with (NCCL collectives, timing events)."""
        if cuda_stream_ptr is None:
            self._ck(self.lib.sfm_set_stream(self.h, None), "sfm_set_stream")
        elif int(cuda_stream_ptr) == 0:
            self._ck(self.lib.sfm_use_default_stream(self.h), "sfm_use_default_stream")
        else:
            self._ck(self.lib.sfm_set_stream(self.h, _P(int(cuda_stream_ptr))), "sfm_set_stream")

    def synchronize(self):
        self._ck(self.lib.sfm_synchronize(self.h), "sfm_synchronize")

    def set_score_variant(self, variant="auto", hyps_per_thread=0, group=0):
        self._ck(self.lib.sfm_set_score_variant(self.h, VARIANT[variant], int(hyps_per_thread), int(group)),
                 "sfm_set_score_variant")

    def set_refinement(self, max_iterations=0):
        """Refine the winner over its inliers before the pose in every later tail call (0 = off).  The calls below
        take ``refine_iterations`` and set this for themselves, because engines are shared."""
        n = int(max_iterations)
        if n < 0:
            raise ValueError(f"refine_iterations must be >= 0, got {n}")
        self._ck(self.lib.sfm_set_refinement(self.h, n), "sfm_set_refinement")

    def get_refinement(self, pairs=1):
        """The refinement reports of the last tail call (a ctypes array of ``pairs`` Refinement)."""
        out = (Refinement * max(int(pairs), 1))()
        self._ck(self.lib.sfm_get_refinement(self.h, C.cast(out, C.POINTER(Refinement)), int(pairs)), "sfm_get_refinement")
        return out

    # -- correspondences ------------------------------------------------------------------
    def upload_pairs(self, pts_a, pts_b, K, sync=True):
        """pts_a, pts_b: [n,2] pixel coordinates; K: 3x3.  sync=False only enqueues the copies: the arrays (kept
        referenced by the engine) must not change until the next synchronising call."""
        pa, pb = _split_xy(pts_a), _split_xy(pts_b)
        if pa.shape != pb.shape:
            raise ValueError("pts_a and pts_b must have the same shape")
        K = _f64(K).reshape(3, 3)
        n = pa.shape[0]
        base_a, base_b = pa.ctypes.data, pb.ctypes.data
        fn = self.lib.sfm_upload_pairs if sync else self.lib.sfm_upload_pairs_async
        self._ck(fn(self.h, _P(base_a), _P(base_a + 8), _P(base_b), _P(base_b + 8), 2, n, _ptr(K)), "sfm_upload_pairs")
        self._keep = None if sync else (pa, pb)
        self.n, self.batch_pairs = n, 0

    def upload_pairs_soa(self, xa, ya, xb, yb, K):
        xa, ya, xb, yb = (_f64(v).reshape(-1) for v in (xa, ya, xb, yb))
        K = _f64(K).reshape(3, 3)
        n = xa.shape[0]
        self._ck(self.lib.sfm_upload_pairs(self.h, _ptr(xa), _ptr(ya), _ptr(xb), _ptr(yb), 1, n, _ptr(K)),
                 "sfm_upload_pairs")
        self.n, self.batch_pairs = n, 0

    def upload_pairs_device(self, xa_ptr, ya_ptr, xb_ptr, yb_ptr, stride, n, K):
        K = _f64(K).reshape(3, 3)
        self._ck(self.lib.sfm_upload_pairs_d(self.h, _P(xa_ptr), _P(ya_ptr), _P(xb_ptr), _P(yb_ptr), int(stride),
                                             int(n), _ptr(K)), "sfm_upload_pairs_d")
        self.n, self.batch_pairs = int(n), 0

    def get_normalised(self):
        out = np.empty((self.n, 4), dtype=np.float64)
        self._ck(self.lib.sfm_get_normalised(self.h, _ptr(out), self.n), "sfm_get_normalised")
        return out

    # -- sampling -------------------------------------------------------------------------
    def set_table(self, table):
        table = np.ascontiguousarray(table, dtype=np.int32).reshape(-1, 8)
        self._ck(self.lib.sfm_set_table(self.h, _ptr(table), table.shape[0]), "sfm_set_table")
        self.h_count = table.shape[0]

    def sample_device(self, seed, h, stream=0, hyp_offset=0):
        self._ck(self.lib.sfm_sample_device(self.h, int(seed), int(stream), int(hyp_offset), int(h)),
                 "sfm_sample_device")
        self.h_count = int(h)

    def get_table(self, h=None, first=0):
        h = self.h_count - first if h is None else h
        out = np.empty((h, 8), dtype=np.int32)
        self._ck(self.lib.sfm_get_table(self.h, _ptr(out), int(first), int(h)), "sfm_get_table")
        return out

    # -- fit / score ----------------------------------------------------------------------
    def fit(self, want_E=True, want_eig=False):
        h = self.h_count
        E = np.empty((h, 3, 3), dtype=np.float64) if want_E else None
        valid = np.empty(h, dtype=np.uint8)
        eig = np.empty((h, 9), dtype=np.float64) if want_eig else None
        self._ck(self.lib.sfm_fit(self.h, _ptr(E), _ptr(valid), _ptr(eig)), "sfm_fit")
        return E, valid.astype(bool), eig

    def get_models(self, first=0, count=None):
        count = self.h_count - first if count is None else int(count)
        E = np.empty((count, 3, 3), dtype=np.float64)
        valid = np.empty(count, dtype=np.uint8)
        self._ck(self.lib.sfm_get_models(self.h, int(first), count, _ptr(E), _ptr(valid)), "sfm_get_models")
        return E, valid.astype(bool)

    def set_models(self, E, valid=None):
        E = _f64(E).reshape(-1, 9)
        v = None if valid is None else np.ascontiguousarray(valid, dtype=np.uint8)
        self._ck(self.lib.sfm_set_models(self.h, _ptr(E), _ptr(v), E.shape[0]), "sfm_set_models")
        self.h_count = E.shape[0]

    def score(self, threshold, min_extra=0.0, aggregation="rms", selection="min_error", use_table=True,
              idx_offset=0, want_arrays=True):
        h = self.h_count
        if want_arrays:
            cnt = np.empty(h, dtype=np.int32)
            s1 = np.empty(h, dtype=np.float64)
            s2 = np.empty(h, dtype=np.float64)
            err = np.empty(h, dtype=np.float64)
        else:
            cnt = s1 = s2 = err = None
        self._ck(self.lib.sfm_score(self.h, float(threshold), float(min_extra), AGG[aggregation], SELECT[selection],
                                    1 if use_table else 0, int(idx_offset), _ptr(cnt), _ptr(s1), _ptr(s2), _ptr(err)),
                 "sfm_score")
        return cnt, s1, s2, err

    def get_best(self):
        b = Best()
        self._ck(self.lib.sfm_get_best(self.h, C.byref(b)), "sfm_get_best")
        return b

    def set_winner(self, local_index, E=None):
        Ea = None if E is None else _f64(E).reshape(9)
        self._ck(self.lib.sfm_set_winner(self.h, int(local_index), _ptr(Ea)), "sfm_set_winner")

    def near_ties(self, rel_tol=1e-12, cap=64):
        """Local indices (ascending) of the hypotheses whose error is within rel_tol of the winner's, and their
        total number (which may exceed ``cap``)."""
        idx = np.empty(cap, dtype=np.int64)
        n = C.c_int64(0)
        self._ck(self.lib.sfm_near_ties(self.h, float(rel_tol), int(cap), _ptr(idx), C.byref(n)), "sfm_near_ties")
        return np.sort(idx[:min(int(n.value), cap)]), int(n.value)

    def rescored(self) -> int:
        n = C.c_int64(0)
        self._ck(self.lib.sfm_get_rescored(self.h, C.byref(n)), "sfm_get_rescored")
        return int(n.value)

    def inlier_mask(self, threshold, want_sed=True):
        mask = np.empty(self.n, dtype=np.uint8)
        sed = np.empty(self.n, dtype=np.float64) if want_sed else None
        self._ck(self.lib.sfm_inlier_mask(self.h, float(threshold), _ptr(mask), _ptr(sed)), "sfm_inlier_mask")
        return mask.astype(bool), sed

    def ransac_essential(self, threshold, min_extra=0.0, aggregation="rms", selection="min_error",
                         want_mask=True, want_sed=True, mask_out=None, sed_out=None):
        b = Best()
        mask = mask_out if mask_out is not None else (np.empty(self.n, dtype=np.uint8) if want_mask else None)
        sed = sed_out if sed_out is not None else (np.empty(self.n, dtype=np.float64) if want_sed else None)
        self._ck(self.lib.sfm_ransac_essential(self.h, float(threshold), float(min_extra), AGG[aggregation],
                                               SELECT[selection], C.byref(b), _ptr(mask), _ptr(sed)),
                 "sfm_ransac_essential")
        return b, mask, sed

    # -- homography --------------------------------------------------------------------------
    def fit_homography(self):
        """The 4-point solve for every row of the current table / device draw -> (H [h,3,3], valid bool[h])."""
        h = self.h_count
        H = np.empty((h, 3, 3), dtype=np.float64)
        valid = np.empty(h, dtype=np.uint8)
        self._ck(self.lib.sfm_fit_homography(self.h, _ptr(H), _ptr(valid)), "sfm_fit_homography")
        return H, valid.astype(bool)

    def ransac_homography(self, threshold, min_extra=0.0, aggregation="rms", selection="min_error",
                          want_mask=True, want_arrays=False):
        """fit -> score -> select -> mask in one call.  Returns (best, mask uint8[n], err[n], count_extra[h], err[h]);
        the per-hypothesis arrays are None unless want_arrays."""
        b = Best()
        mask = np.empty(self.n, dtype=np.uint8) if want_mask else None
        err = np.empty(self.n, dtype=np.float64) if want_mask else None
        cnt = np.empty(self.h_count, dtype=np.int32) if want_arrays else None
        err_h = np.empty(self.h_count, dtype=np.float64) if want_arrays else None
        self._ck(self.lib.sfm_ransac_homography(self.h, float(threshold), float(min_extra), AGG[aggregation],
                                                SELECT[selection], C.byref(b), _ptr(mask), _ptr(err), _ptr(cnt),
                                                _ptr(err_h)), "sfm_ransac_homography")
        return b, mask, err, cnt, err_h

    def homography_mask(self, H, threshold):
        """(decision bool[n], transfer error [n]) under H (3x3), or under the last estimate's winner when H is None."""
        Ha = None if H is None else _f64(H).reshape(9)
        mask = np.empty(self.n, dtype=np.uint8)
        err = np.empty(self.n, dtype=np.float64)
        self._ck(self.lib.sfm_homography_mask(self.h, _ptr(Ha), float(threshold), _ptr(mask), _ptr(err)),
                 "sfm_homography_mask")
        return mask.astype(bool), err

    def decompose_homography(self, H, K, rotation_tolerance=1e-2):
        """The four (R, t, n, d) candidates of H (3x3, pixels) with K -> HPoses (sfm_hposes)."""
        Ha, Ka = _f64(H).reshape(9), _f64(K).reshape(9)
        p = HPoses()
        self._ck(self.lib.sfm_decompose_homography(self.h, _ptr(Ha), _ptr(Ka), float(rotation_tolerance), C.byref(p)),
                 "sfm_decompose_homography")
        return p

    def homography_pose_and_triangulate(self, K, threshold, distance_threshold=50.0, rotation_tolerance=1e-2, cap=None,
                                        refine_iterations=0):
        """Tail of the current homography winner -> (HPoses, num_inliers, inlier_idx, pass_bits, X).  With
        refine_iterations > 0 the winner is refined first and the tail describes the refined H (get_refinement())."""
        self.set_refinement(refine_iterations)
        cap = self.n if cap is None else int(cap)
        Ka = _f64(K).reshape(9)
        p = HPoses()
        num = C.c_int64(0)
        idx = np.empty(cap, dtype=np.int64)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        self._ck(self.lib.sfm_homography_pose_and_triangulate(self.h, _ptr(Ka), float(threshold), float(distance_threshold),
                                                              float(rotation_tolerance), C.byref(p), cap, C.byref(num),
                                                              _ptr(idx), _ptr(ok), _ptr(X)),
                 "sfm_homography_pose_and_triangulate")
        m = min(int(num.value), cap)
        return p, int(num.value), idx[:m], ok[:m], X[:m]

    def two_view_homography(self, K, threshold, min_extra=0.0, aggregation="rms", selection="min_error",
                            distance_threshold=50.0, rotation_tolerance=1e-2, cap=None, refine_iterations=0):
        """ransac_homography + homography_pose_and_triangulate in one C call (one synchronisation for the fixed-size
        results).  Returns (best, mask, err, HPoses, num_inliers, inlier_idx, pass_bits, X)."""
        self.set_refinement(refine_iterations)
        cap = self.n if cap is None else int(cap)
        Ka = _f64(K).reshape(9)
        b, p = Best(), HPoses()
        num = C.c_int64(0)
        idx = np.empty(cap, dtype=np.int64)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        mask = np.empty(self.n, dtype=np.uint8)
        err = np.empty(self.n, dtype=np.float64)
        self._ck(self.lib.sfm_two_view_homography(self.h, _ptr(Ka), float(threshold), float(min_extra), AGG[aggregation],
                                                  SELECT[selection], float(distance_threshold), float(rotation_tolerance),
                                                  C.byref(b), C.byref(p), cap, C.byref(num), _ptr(idx), _ptr(ok), _ptr(X),
                                                  _ptr(mask), _ptr(err)), "sfm_two_view_homography")
        m = min(int(num.value), cap)
        return b, mask, err, p, int(num.value), idx[:m], ok[:m], X[:m]

    # -- essential matrix or homography -------------------------------------------------------
    def model_scores(self, E, H, K, sigma=1.0, homography_ratio=0.45, per_point=False):
        """Scores of E and / or H (3x3 or None) on the current single-pair upload -> (ModelScores, per-point
        [n,4] errors (d2_A,E, d2_B,E, d2_A,H, d2_B,H) in px^2 or None)."""
        Ea = None if E is None else _f64(E).reshape(9)
        Ha = None if H is None else _f64(H).reshape(9)
        Ka = _f64(K).reshape(9)
        s = ModelScores()
        pp = np.empty((self.n, 4), dtype=np.float64) if per_point else None
        self._ck(self.lib.sfm_score_models(self.h, _ptr(Ea), _ptr(Ha), _ptr(Ka), float(sigma), float(homography_ratio),
                                           C.byref(s), _ptr(pp)), "sfm_score_models")
        return s, pp

    # -- pose / triangulation ---------------------------------------------------------------
    def decompose_essential(self, E):
        E = _f64(E).reshape(9)
        p = Poses()
        self._ck(self.lib.sfm_decompose_essential(self.h, _ptr(E), C.byref(p)), "sfm_decompose_essential")
        return p

    def recover_pose(self, E, norm_a, norm_b, distance_threshold=50.0, camera_matrix=None):
        """norm_a, norm_b: [m,2] K-normalised coordinates — or pixel coordinates when ``camera_matrix`` is given
        (they are then normalised on the device)."""
        E = _f64(E).reshape(9)
        na, nb = _split_xy(norm_a), _split_xy(norm_b)
        m = na.shape[0]
        p = Poses()
        pass4 = np.zeros(m, dtype=np.uint8)
        a, b = na.ctypes.data, nb.ctypes.data
        if camera_matrix is None:
            self._ck(self.lib.sfm_recover_pose(self.h, _ptr(E), _P(a), _P(a + 8), _P(b), _P(b + 8), 2, m,
                                               float(distance_threshold), C.byref(p), _ptr(pass4)), "sfm_recover_pose")
        else:
            K = _f64(camera_matrix).reshape(9)
            self._ck(self.lib.sfm_recover_pose_pixels(self.h, _ptr(E), _ptr(K), _P(a), _P(a + 8), _P(b), _P(b + 8), 2, m,
                                                      float(distance_threshold), C.byref(p), _ptr(pass4)),
                     "sfm_recover_pose_pixels")
        return p, pass4

    def triangulate(self, P1, P2, pts_a, pts_b):
        P1 = _f64(np.asarray(P1)[:3, :]).reshape(12)
        P2 = _f64(np.asarray(P2)[:3, :]).reshape(12)
        pa, pb = _split_xy(pts_a), _split_xy(pts_b)
        m = pa.shape[0]
        X = np.empty((m, 3), dtype=np.float64)
        a, b = pa.ctypes.data, pb.ctypes.data
        self._ck(self.lib.sfm_triangulate(self.h, _ptr(P1), _ptr(P2), _P(a), _P(a + 8), _P(b), _P(b + 8), 2, m,
                                          _ptr(X)), "sfm_triangulate")
        return X

    def pose_and_triangulate(self, threshold, distance_threshold=50.0, cap=None, refine_iterations=0):
        self.set_refinement(refine_iterations)
        cap = self.n if cap is None else int(cap)
        p = Poses()
        num = C.c_int64(0)
        idx = np.empty(cap, dtype=np.int64)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        self._ck(self.lib.sfm_pose_and_triangulate(self.h, float(threshold), float(distance_threshold), C.byref(p),
                                                   cap, C.byref(num), _ptr(idx), _ptr(ok), _ptr(X)),
                 "sfm_pose_and_triangulate")
        m = min(int(num.value), cap)
        return p, int(num.value), idx[:m], ok[:m], X[:m]

    def two_view(self, threshold, min_extra=0.0, aggregation="rms", selection="min_error", distance_threshold=50.0,
                 cap=None, want_mask=True, want_sed=True, refine_iterations=0):
        """ransac_essential + pose_and_triangulate in one C call (one synchronisation for the fixed-size results).
        Returns (best, mask, sed, poses, num_inliers, inlier_idx, pass_bits, X)."""
        self.set_refinement(refine_iterations)
        cap = self.n if cap is None else int(cap)
        b, p = Best(), Poses()
        num = C.c_int64(0)
        idx = np.empty(cap, dtype=np.int64)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        mask = np.empty(self.n, dtype=np.uint8) if want_mask else None
        sed = np.empty(self.n, dtype=np.float64) if want_sed else None
        self._ck(self.lib.sfm_two_view(self.h, float(threshold), float(min_extra), AGG[aggregation], SELECT[selection],
                                       float(distance_threshold), C.byref(b), C.byref(p), cap, C.byref(num), _ptr(idx),
                                       _ptr(ok), _ptr(X), _ptr(mask), _ptr(sed)), "sfm_two_view")
        m = min(int(num.value), cap)
        return b, mask, sed, p, int(num.value), idx[:m], ok[:m], X[:m]

    def two_view_async(self, threshold, min_extra=0.0, aggregation="rms", selection="min_error", distance_threshold=50.0,
                       want_mask=True, want_sed=True, out=None, refine_iterations=0):
        """Enqueue fit -> score -> select -> tail; nothing synchronises.  Returns the (mask, sed) arrays that the
        enqueued copies will fill - valid after two_view_fetch().  ``out``: (uint8[n], float64[n]) to fill, ideally
        pinned and reused (page-locking fresh memory per call costs more than the estimate's transfers)."""
        self.set_refinement(refine_iterations)
        mask, sed = out if out is not None else self.pinned_out(self.n)
        if not want_mask:
            mask = None
        if not want_sed:
            sed = None
        self._ck(self.lib.sfm_two_view_async(self.h, float(threshold), float(min_extra), AGG[aggregation],
                                             SELECT[selection], float(distance_threshold), _ptr(mask), _ptr(sed)),
                 "sfm_two_view_async")
        return mask, sed

    def two_view_fetch(self, cap=None):
        cap = self.n if cap is None else int(cap)
        b, p = Best(), Poses()
        num = C.c_int64(0)
        idx = np.empty(cap, dtype=np.int64)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        self._ck(self.lib.sfm_two_view_fetch(self.h, C.byref(b), C.byref(p), cap, C.byref(num), _ptr(idx), _ptr(ok),
                                             _ptr(X)), "sfm_two_view_fetch")
        self._keep = None
        m = min(int(num.value), cap)
        return b, p, int(num.value), idx[:m], ok[:m], X[:m]

    # -- hypothesis-sharded runs: nothing synchronises between scoring and the final fetch ----
    RECORD_BYTES = 144  # include/sfm_b200.h SFM_RECORD_BYTES

    def score_async(self, threshold, min_extra=0.0, aggregation="rms", selection="min_error") -> int:
        """fit + score + select, enqueued only.  Returns the DEVICE address of this rank's selection record."""
        ptr = _P()
        self._ck(self.lib.sfm_score_async(self.h, float(threshold), float(min_extra), AGG[aggregation], SELECT[selection],
                                          C.byref(ptr)), "sfm_score_async")
        return int(ptr.value)

    def sharded_tail(self, gathered_dev_ptr: int, world: int, rank: int, hyps_per_rank: int, threshold,
                     distance_threshold=50.0, selection="min_error"):
        self._ck(self.lib.sfm_sharded_tail(self.h, _P(gathered_dev_ptr), int(world), int(rank), int(hyps_per_rank),
                                           SELECT[selection], float(threshold), float(distance_threshold)),
                 "sfm_sharded_tail")

    def sharded_fetch(self, cap=None):
        cap = self.n if cap is None else int(cap)
        b, p = Best(), Poses()
        owner, num = C.c_int32(-1), C.c_int64(0)
        idx = np.empty(cap, dtype=np.int64)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        self._ck(self.lib.sfm_sharded_fetch(self.h, C.byref(b), C.byref(owner), C.byref(p), cap, C.byref(num), _ptr(idx),
                                            _ptr(ok), _ptr(X)), "sfm_sharded_fetch")
        m = min(int(num.value), cap)
        return b, int(owner.value), p, int(num.value), idx[:m], ok[:m], X[:m]

    # -- the collective behind the C ABI (no torch needed on the data path) --------------------------
    def nccl_init(self, rank: int, world: int, unique_id: bytes):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._ck(self.lib.sfm_nccl_init(self.h, int(rank), int(world), C.cast(buf, _P)), "sfm_nccl_init")
        self.nccl_world = int(world)

    def nccl_destroy(self):
        self._ck(self.lib.sfm_nccl_destroy(self.h), "sfm_nccl_destroy")

    def two_view_sharded(self, seed, hyps_per_rank, threshold, min_extra=0.0, aggregation="rms", selection="min_error",
                         distance_threshold=50.0):
        """Enqueue one hypothesis-sharded estimate on the communicator of nccl_init; results via sharded_fetch()."""
        self._ck(self.lib.sfm_two_view_sharded(self.h, int(seed), int(hyps_per_rank), float(threshold), float(min_extra),
                                               AGG[aggregation], SELECT[selection], float(distance_threshold)),
                 "sfm_two_view_sharded")

    # -- batches ----------------------------------------------------------------------------
    def batch_ransac(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra=0.0, aggregation="rms",
                     selection="min_error", pair_id0=0):
        pa, pb = _split_xy(pts_a), _split_xy(pts_b)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        P = offsets.shape[0] - 1
        Ks = _f64(Ks).reshape(P, 9)
        E = np.empty((P, 3, 3), dtype=np.float64)
        bi = np.empty(P, dtype=np.int64)
        be = np.empty(P, dtype=np.float64)
        ce = np.empty(P, dtype=np.int32)
        ni = np.empty(P, dtype=np.int64)
        a, b = pa.ctypes.data, pb.ctypes.data
        self._ck(self.lib.sfm_batch_ransac(self.h, _P(a), _P(a + 8), _P(b), _P(b + 8), 2, _ptr(offsets), P, _ptr(Ks),
                                           int(h), int(seed), int(pair_id0), float(threshold), float(min_extra),
                                           AGG[aggregation], SELECT[selection], _ptr(E), _ptr(bi), _ptr(be), _ptr(ce),
                                           _ptr(ni)), "sfm_batch_ransac")
        self.n, self.batch_pairs = int(offsets[-1]), P
        return dict(E=E, best_index=bi, best_err=be, count_extra=ce, num_invalid=ni)

    def batch_two_view(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra=0.0, aggregation="rms",
                       selection="min_error", distance_threshold=50.0, pair_id0=0, refine_iterations=0):
        """batch_ransac + per pair: inlier list, pose vote, triangulation.  Returns the batch_ransac dict plus
        R [P,3,3], t [P,3] (NaN without a model), counts [P,4], pose_index [P], inlier_offsets [P+1], inlier_idx
        (pair-relative), pass_bits, points [total,3].  With refine_iterations > 0 the pose and everything after it
        describe the refined E, and the dict gains refined_E and the refine_* reports (_refine_keys)."""
        return self._batch_two_view(pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra, aggregation, selection,
                                    distance_threshold, pair_id0, refine_iterations)[0]

    def _refine_keys(self, out, P, model_key):
        """The per-pair refinement reports of the last batch tail as dict entries."""
        rep = self.get_refinement(P)
        raw = np.frombuffer(rep, dtype=np.uint8).reshape(P, C.sizeof(Refinement))
        dbl = raw[:, :12 * 8].copy().view(np.float64)
        out[model_key] = dbl[:, :9].reshape(P, 3, 3).copy()
        out["refine_cost_ransac"], out["refine_cost_start"], out["refine_cost_final"] = (dbl[:, 9].copy(), dbl[:, 10].copy(),
                                                                                        dbl[:, 11].copy())
        out["refine_num"] = raw[:, 96:104].copy().view(np.int64).reshape(P)
        ints = raw[:, 104:116].copy().view(np.int32).reshape(P, 3)
        out["refine_iterations"], out["refine_status"], out["refine_rejected"] = (ints[:, 0].copy(), ints[:, 1].copy(),
                                                                                  ints[:, 2].copy())
        return out

    def _batch_two_view(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra, aggregation, selection,
                        distance_threshold, pair_id0, refine_iterations=0):
        """batch_two_view's dict and the smallest singular value of every pair's winning E ([P], NaN without one)."""
        self.set_refinement(refine_iterations)
        pa, pb = _split_xy(pts_a), _split_xy(pts_b)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        P = offsets.shape[0] - 1
        Ks = _f64(Ks).reshape(P, 9)
        E = np.empty((P, 3, 3), dtype=np.float64)
        bi = np.empty(P, dtype=np.int64)
        be = np.empty(P, dtype=np.float64)
        ce = np.empty(P, dtype=np.int32)
        ni = np.empty(P, dtype=np.int64)
        poses = (Poses * P)()
        ioff = np.empty(P + 1, dtype=np.int64)
        cap = int(offsets[-1])
        idx = np.empty(cap, dtype=np.int32)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        a, b = pa.ctypes.data, pb.ctypes.data
        self._ck(self.lib.sfm_batch_two_view(self.h, _P(a), _P(a + 8), _P(b), _P(b + 8), 2, _ptr(offsets), P, _ptr(Ks),
                                             int(h), int(seed), int(pair_id0), float(threshold), float(min_extra),
                                             AGG[aggregation], SELECT[selection], float(distance_threshold), _ptr(E),
                                             _ptr(bi), _ptr(be), _ptr(ce), _ptr(ni), C.cast(poses, _P), _ptr(ioff), cap,
                                             _ptr(idx), _ptr(ok), _ptr(X)), "sfm_batch_two_view")
        self.n, self.batch_pairs = cap, P
        raw = np.frombuffer(poses, dtype=np.uint8).reshape(P, C.sizeof(Poses))
        dbl = raw[:, :(36 + 12 + 3) * 8].copy().view(np.float64)
        R4, t4 = dbl[:, :36].reshape(P, 4, 3, 3), dbl[:, 36:48].reshape(P, 4, 3)
        counts = raw[:, 51 * 8:55 * 8].copy().view(np.int64).reshape(P, 4)
        pose_index = raw[:, 55 * 8:55 * 8 + 4].copy().view(np.int32).reshape(P)
        sel = np.clip(pose_index, 0, 3)
        R = R4[np.arange(P), sel].copy()
        t = t4[np.arange(P), sel].copy()
        R[pose_index < 0] = np.nan
        t[pose_index < 0] = np.nan
        sv = dbl[:, 48:51].copy()
        total = int(ioff[-1])
        out = dict(E=E, best_index=bi, best_err=be, count_extra=ce, num_invalid=ni, R=R, t=t, counts=counts,
                   pose_index=pose_index, inlier_offsets=ioff, inlier_idx=idx[:total], pass_bits=ok[:total],
                   points=X[:total])
        if int(refine_iterations) > 0:
            self._refine_keys(out, P, "refined_E")
        return out, np.where(pose_index[:, None] == -2, np.nan, sv)[:, 2]

    def batch_two_view_homography(self, pts_a, pts_b, offsets, Ks, h, seed, threshold, min_extra=0.0,
                                  aggregation="rms", selection="min_error", distance_threshold=50.0,
                                  rotation_tolerance=1e-2, pair_id0=0, refine_iterations=0):
        """batch_two_view for homographies (threshold: symmetric transfer error in px^2; Ks: each upper triangular with
        K[2,2] = 1).  The keys of batch_two_view with H [P,3,3] in place of E, plus n [P,3], d [P] and
        rotation_only bool[P] of the voted candidate.  R, t, n, d are NaN without a model; on a rotation-only pair R is
        the nearest rotation, t = 0, n NaN, d inf, pose_index -1 and no inlier passes.  refine_iterations > 0: as in
        batch_two_view, with refined_H."""
        self.set_refinement(refine_iterations)
        pa, pb = _split_xy(pts_a), _split_xy(pts_b)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        P = offsets.shape[0] - 1
        Ks = _f64(Ks).reshape(P, 9)
        H = np.empty((P, 3, 3), dtype=np.float64)
        bi = np.empty(P, dtype=np.int64)
        be = np.empty(P, dtype=np.float64)
        ce = np.empty(P, dtype=np.int32)
        ni = np.empty(P, dtype=np.int64)
        poses = (HPoses * P)()
        ioff = np.empty(P + 1, dtype=np.int64)
        cap = int(offsets[-1])
        idx = np.empty(cap, dtype=np.int32)
        ok = np.empty(cap, dtype=np.uint8)
        X = np.empty((cap, 3), dtype=np.float64)
        a, b = pa.ctypes.data, pb.ctypes.data
        self._ck(self.lib.sfm_batch_two_view_homography(
            self.h, _P(a), _P(a + 8), _P(b), _P(b + 8), 2, _ptr(offsets), P, _ptr(Ks), int(h), int(seed), int(pair_id0),
            float(threshold), float(min_extra), AGG[aggregation], SELECT[selection], float(distance_threshold),
            float(rotation_tolerance), _ptr(H), _ptr(bi), _ptr(be), _ptr(ce), _ptr(ni), C.cast(poses, _P), _ptr(ioff), cap,
            _ptr(idx), _ptr(ok), _ptr(X)), "sfm_batch_two_view_homography")
        self.n, self.batch_pairs = cap, P
        raw = np.frombuffer(poses, dtype=np.uint8).reshape(P, C.sizeof(HPoses))
        dbl = raw[:, :67 * 8].copy().view(np.float64)  # R 36, t 12, n 12, d 4, sv 3
        R4, t4 = dbl[:, :36].reshape(P, 4, 3, 3), dbl[:, 36:48].reshape(P, 4, 3)
        n4, d4 = dbl[:, 48:60].reshape(P, 4, 3), dbl[:, 60:64]
        counts = raw[:, 67 * 8:71 * 8].copy().view(np.int64).reshape(P, 4)
        ints = raw[:, 71 * 8:72 * 8].copy().view(np.int32).reshape(P, 2)
        pose_index, rot = ints[:, 0].copy(), ints[:, 1] != 0
        sel = np.clip(pose_index, 0, 3)  # a rotation-only pair's one candidate is candidate 0
        rows = np.arange(P)
        R, t, n, d = R4[rows, sel].copy(), t4[rows, sel].copy(), n4[rows, sel].copy(), d4[rows, sel].copy()
        none = pose_index == -2
        R[none], t[none], n[none], d[none] = np.nan, np.nan, np.nan, np.nan
        total = int(ioff[-1])
        out = dict(H=H, best_index=bi, best_err=be, count_extra=ce, num_invalid=ni, R=R, t=t, counts=counts,
                   pose_index=pose_index, inlier_offsets=ioff, inlier_idx=idx[:total], pass_bits=ok[:total],
                   points=X[:total], n=n, d=d, rotation_only=rot)
        if int(refine_iterations) > 0:
            self._refine_keys(out, P, "refined_H")
        return out

    def batch_score_models(self, E, H, have_e=None, have_h=None, sigma=1.0, homography_ratio=0.45, per_point=False):
        """model_scores for every pair of the current batched upload: E / H [P,3,3] or None, given for pair p where
        have_e[p] / have_h[p] (None = all), each pair scored with its own K of the upload.  Returns (ModelScores array
        [P], per-point [n_total,4] errors or None); a pair with neither model has model -1."""
        P = self.batch_pairs
        Ea = None if E is None else _f64(E).reshape(P, 9)
        Ha = None if H is None else _f64(H).reshape(P, 9)
        fe = None if have_e is None else np.ascontiguousarray(have_e, dtype=np.uint8).reshape(P)
        fh = None if have_h is None else np.ascontiguousarray(have_h, dtype=np.uint8).reshape(P)
        out = (ModelScores * max(P, 1))()
        pp = np.empty((self.n, 4), dtype=np.float64) if per_point else None
        self._ck(self.lib.sfm_batch_score_models(self.h, _ptr(Ea), _ptr(fe), _ptr(Ha), _ptr(fh), float(sigma),
                                                 float(homography_ratio), C.cast(out, _P), _ptr(pp)),
                 "sfm_batch_score_models")
        return out, pp

    # -- front end: brute-force matcher (N1) ---------------------------------------------------
    def match_brute_force(self, image_a, image_b, feats_a, feats_b, kind="ncc", window=None, ratio_test=False,
                          crosscheck=False, ratio_threshold=0.5, want_scores=False):
        """feats_*: [n,2] (x, y).  Returns (best_b int32[na], best_score[na], keep bool[na], scores|None)."""
        image_a, image_b = np.asarray(image_a), np.asarray(image_b)
        if image_a.shape != image_b.shape:
            raise ValueError("the images must have the same shape")  # ncc.py:22-23
        if image_a.ndim != 2:
            raise ValueError("grayscale (2-D) images expected")
        if image_a.dtype == np.uint8 and image_b.dtype == np.uint8:
            dt, ia, ib = 0, np.ascontiguousarray(image_a), np.ascontiguousarray(image_b)
        else:
            dt, ia, ib = 1, _f64(image_a), _f64(image_b)
        fa = _f64(np.asarray(feats_a, dtype=np.float64).reshape(-1, 2))
        fb = _f64(np.asarray(feats_b, dtype=np.float64).reshape(-1, 2))
        na, nb = fa.shape[0], fb.shape[0]
        if window is None:
            window = 3 if kind == "ncc" else 5
        best_b = np.full(na, -1, dtype=np.int32)
        best_s = np.full(na, np.inf, dtype=np.float64)
        keep = np.zeros(na, dtype=np.uint8)
        S = np.empty((na, nb), dtype=np.float64) if want_scores else None
        self._ck(self.lib.sfm_match_brute_force(self.h, _ptr(ia), _ptr(ib), dt, ia.shape[0], ia.shape[1], _ptr(fa), na,
                                                _ptr(fb), nb, {"ncc": 0, "ssd": 1}[kind], int(window),
                                                (1 if ratio_test else 0) | (2 if crosscheck else 0),
                                                float(ratio_threshold), _ptr(best_b), _ptr(best_s), _ptr(keep),
                                                _ptr(S)), "sfm_match_brute_force")
        return best_b, best_s, keep.astype(bool), S

    def match_from_scores(self, scores, ratio_test=False, crosscheck=False, ratio_threshold=0.5):
        """The selection + validations of match_brute_force on a caller-supplied score matrix [na, nb]."""
        S = _f64(scores)
        if S.ndim != 2:
            raise ValueError("a [na, nb] score matrix is expected")
        na, nb = S.shape
        best_b = np.full(na, -1, dtype=np.int32)
        best_s = np.full(na, np.inf, dtype=np.float64)
        keep = np.zeros(na, dtype=np.uint8)
        self._ck(self.lib.sfm_match_from_scores(self.h, _ptr(S), na, nb, (1 if ratio_test else 0) | (2 if crosscheck else 0),
                                                float(ratio_threshold), _ptr(best_b), _ptr(best_s), _ptr(keep)),
                 "sfm_match_from_scores")
        return best_b, best_s, keep.astype(bool)

    # -- front end: Harris corners (N2) ---------------------------------------------------------
    @staticmethod
    def _image(image):
        image = np.asarray(image)
        if image.ndim != 2:
            raise ValueError("Only 2D single channel images are supported")
        if image.dtype == np.uint8:
            return 0, np.ascontiguousarray(image)
        return 1, _f64(image)

    def cross_correlate(self, image, kernel):
        dt, img = self._image(image)
        kernel = _f64(kernel)
        out = np.empty(img.shape, dtype=np.float64)
        self._ck(self.lib.sfm_cross_correlate(self.h, _ptr(img), dt, img.shape[0], img.shape[1], _ptr(kernel),
                                              kernel.shape[0], _ptr(out)), "sfm_cross_correlate")
        return out

    def harris_corners(self, image, num_corners=50, block_size=2, k=0.04, want_cornerness=False):
        """Returns (xy [m,2] = (x, y), cornerness score [m], dict(cornerness=..., nms_sweeps=...))."""
        dt, img = self._image(image)
        orows, ocols = C.c_int64(0), C.c_int64(0)
        self._ck(self.lib.sfm_harris_output_shape(img.shape[0], img.shape[1], int(block_size), C.byref(orows),
                                                  C.byref(ocols)), "sfm_harris_output_shape")
        if orows.value <= 0 or ocols.value <= 0:
            raise ValueError("negative dimensions are not allowed")  # np.zeros at harris_detector.py:66-72
        cap = max(1, min(int(num_corners), orows.value * ocols.value))
        xy = np.empty((cap, 2), dtype=np.float64)
        score = np.empty(cap, dtype=np.float64)
        found, sweeps = C.c_int64(0), C.c_int32(0)
        cim = np.empty((orows.value, ocols.value), dtype=np.float64) if want_cornerness else None
        self._ck(self.lib.sfm_harris_corners(self.h, _ptr(img), dt, img.shape[0], img.shape[1], int(num_corners),
                                             int(block_size), float(k), _ptr(xy), _ptr(score), C.byref(found), _ptr(cim),
                                             C.byref(sweeps)), "sfm_harris_corners")
        m = int(found.value)
        return xy[:m], score[:m], dict(cornerness=cim, nms_sweeps=int(sweeps.value))

    # -- measurement ------------------------------------------------------------------------
    def enable_timing(self, on=True):
        self._ck(self.lib.sfm_enable_timing(self.h, 1 if on else 0), "sfm_enable_timing")

    def get_timing(self):
        ms = (C.c_float * 8)()
        n = C.c_int64(0)
        self._ck(self.lib.sfm_get_timing(self.h, C.cast(ms, _P), C.byref(n)), "sfm_get_timing")
        names = ["upload", "sample", "fit", "score", "select", "mask", "pose", "triangulate"]
        return {k: float(v) for k, v in zip(names, ms)}, int(n.value)

    def measure_fp64_peak(self):
        v = C.c_double(0)
        self._ck(self.lib.sfm_measure_fp64_peak(self.h, C.byref(v)), "sfm_measure_fp64_peak")
        return float(v.value)


def mt_shuffle_table(state625: np.ndarray, n: int, h: int, perm_at: int = -1):
    """CPython-exact sampler (host).  state625 is updated in place.  Returns (table, perm|None)."""
    lib = load_library()
    st = np.ascontiguousarray(state625, dtype=np.uint32)
    assert st.shape == (625,)
    table = np.empty((h, 8), dtype=np.int32)
    perm = np.empty(n, dtype=np.int32) if perm_at >= 0 else None
    rc = lib.sfm_mt_shuffle_table(_ptr(st), int(n), int(h), _ptr(table), int(perm_at), _ptr(perm))
    if rc != 0:
        raise NativeError(f"sfm_mt_shuffle_table -> {rc}: {lib.sfm_last_error().decode()}")
    if st is not state625:
        state625[...] = st
    return table, perm


class ReferenceSampler:
    """The reference's sampling (cumulative ``random.shuffle`` + first 8, lib/ransac/ransac.py:62-63) for H iterations
    over n items, with (state, permutation) snapshots every ``stride`` iterations so that the permutation — or the RNG
    state — after any given iteration is recovered by replaying at most ``stride`` iterations instead of the whole run."""

    SNAPSHOT_BYTES = 64 << 20
    MAX_SNAPSHOTS = 64

    def __init__(self, state625: np.ndarray, n: int, h: int):
        lib = load_library()
        self.n, self.h = int(n), int(h)
        # at most MAX_SNAPSHOTS snapshots (each costs a call and two copies) and at most SNAPSHOT_BYTES of them
        self.stride = max(1, -(-self.h // self.MAX_SNAPSHOTS), -(-(self.h * self.n * 4) // self.SNAPSHOT_BYTES))
        self.table = np.empty((self.h, 8), dtype=np.int32)
        st = np.ascontiguousarray(state625, dtype=np.uint32).copy()
        assert st.shape == (625,)
        ns = -(-self.h // self.stride)
        self._states = np.empty((ns, 625), dtype=np.uint32)
        self._perms = np.empty((ns, self.n), dtype=np.int32)
        rc = lib.sfm_mt_shuffle_snapshots(_ptr(st), self.n, self.h, _ptr(self.table), self.stride, _ptr(self._states),
                                          _ptr(self._perms))  # one C call: table + snapshots
        if rc != 0:
            raise NativeError(f"sfm_mt_shuffle_snapshots -> {rc}: {lib.sfm_last_error().decode()}")
        self.final_state = st

    def after(self, iteration: int):
        """(state625, permutation) right after 0-based ``iteration``."""
        lib = load_library()
        k = int(iteration) // self.stride
        st, perm = self._states[k].copy(), self._perms[k].copy()
        count = int(iteration) - k * self.stride + 1
        rc = lib.sfm_mt_shuffle_resume(_ptr(st), self.n, count, None, _ptr(perm))
        if rc != 0:
            raise NativeError(f"sfm_mt_shuffle_resume -> {rc}: {lib.sfm_last_error().decode()}")
        return st, perm


def nccl_unique_id() -> bytes:
    """ncclGetUniqueId through the C ABI: 128 bytes that rank 0 hands to its peers (any transport)."""
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.sfm_nccl_unique_id(C.cast(buf, _P))
    if rc != 0:
        raise NativeError(f"sfm_nccl_unique_id -> {rc}: {lib.sfm_last_error().decode()}")
    return buf.raw


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by pinned (page-locked) host memory from sfm_host_alloc.  The memory lives until
    ``pinned_free(array)`` (or the end of the process): meant for long-lived staging buffers, not per-call use."""
    lib = load_library()
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = _P()
    rc = lib.sfm_host_alloc(max(nbytes, 1), C.byref(p))
    if rc != 0:
        raise NativeError(f"sfm_host_alloc -> {rc}: {lib.sfm_last_error().decode()}")
    buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


def pinned_free(arr) -> None:
    """Release an array obtained from pinned_empty (the array must not be used afterwards)."""
    p = _PINNED.pop(arr.ctypes.data, None)
    if p is not None:
        load_library().sfm_host_free(p)


_PINNED: dict = {}
_engines: dict = {}
_engine_lock = threading.Lock()


def default_device() -> int:
    return int(os.environ.get("SFM_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def get_engine(device: int | None = None) -> Engine:
    """The calling THREAD's engine for a device (created on first use).  An Engine is a stateful context (upload ->
    table -> estimate -> fetch on one stream with shared buffers) and is not thread-safe, so every thread that goes
    through the module-level API gets its own; pass ``engine=`` explicitly to share one under your own lock."""
    dev = default_device() if device is None else int(device)
    key = (dev, threading.get_ident())
    with _engine_lock:
        eng = _engines.get(key)
        if eng is None:
            eng = Engine(dev)
            _engines[key] = eng
        return eng
