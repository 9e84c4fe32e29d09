"""Time the bundle adjustment (sfm_bundle_adjust) on the GPU.

Workloads (make_multi_view_scene, track lengths 2-8, 0.5 px noise, 10 % outlier observations; the start is the truth
with every pose but view 0 rotated by about 0.05 degrees and moved by 0.2 % of |t|, every point by 0.2 % of its depth;
threshold 16 px^2; view 0 fixed, view 1 anchored):
  A   16 views x 10^5 points;
  B   64 views x 10^6 points (about 5 * 10^6 observations);
  C   256 views x 2 * 10^5 points (the largest reduced camera system, 1530 x 1530).
Per workload: the device time of each kernel (CUPTI activity records through torch.profiler, in a run of its own).
The kernels are chained (programmatic dependent launch): a kernel's blocks are resident and waiting while its
predecessor runs, so its recorded duration includes that wait.  Each kernel is charged its exclusive time, from the
later of its start and the end of everything before it to its end; these add up to the device span of the call.  Per
round: summed over the call and divided by the LM rounds that did work (the evaluated proposals; launches after the
problem finished exit at once and are counted with them); the call time (median of a host clock around the call, profiler off;
it includes the host's structure pass and the copies); the FP64 rate of k_ba_schur (108 FMA per observation pair of
the list) and of k_ba_chol (n^3 / 6 useful FMA) against the 18.38e12 DFMA/s of DESIGN.md section 7f; the bytes of
k_ba_eval against 7.7 TB/s.  --scipy times scipy least_squares(method="trf", jac_sparsity=...) on workload A for
the same number of iterations on the host CPU (no GPU needed; the CPU model is recorded).

    python tools/time_ba.py [--iters 10] [--steps 3] [--out profiles/bundle_time_b200.json]
    python tools/time_ba.py --scipy [--iters 10] [--out ...]
"""
from __future__ import annotations

import argparse
import json
import os
import platform
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

THR = 16.0
DFMA_PEAK = 18.38e12
HBM = 7.7e12
WORKLOADS = {"A": (16, 100_000), "B": (64, 1_000_000), "C": (256, 200_000)}
KERNELS = ["k_ba_init", "k_ba_list", "k_ba_eval", "k_ba_views", "k_ba_views_sum", "k_ba_schur_pts", "k_ba_schur_obs",
           "k_ba_schur", "k_ba_schur_sum", "k_ba_chol", "k_ba_backsolve", "k_ba_points", "k_ba_finish", "k_ba_mask"]
ONCE = ("k_ba_init", "k_ba_list", "k_ba_finish", "k_ba_mask")


def scene(V, N, seed=0):
    import numpy as np

    from oracle.refine import rodrigues
    from structure_from_motion_b200.scenes import make_multi_view_scene

    K, R, t, X, off, view, x, _ = make_multi_view_scene(N, V, seed, noise_px=0.5, outlier_frac=0.1)
    rng = np.random.default_rng(seed + 1)
    R0, t0 = R.copy(), t.copy()
    for c in range(1, V):
        w = rng.normal(size=3)
        R0[c] = R[c] @ rodrigues(w / np.linalg.norm(w) * np.radians(0.05))
        t0[c] = t[c] + rng.normal(size=3) * 0.002 * np.linalg.norm(t[c]) / np.sqrt(3)
    k = int(np.argmax(np.abs(t[1])))
    t0[1, k] = t[1, k]
    X0 = X + rng.normal(size=X.shape) * 0.002 * X[:, 2:] / np.sqrt(3)
    return K, R0, t0, X0, off, view, x


def _kernel(name):
    for k in KERNELS:
        if k + "(" in name or name.endswith(k):
            return k
    return None


def gpu_main(args):
    import numpy as np
    import torch

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.multiview import bundle_adjust_arrays
    from tools.time_homography import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("time_ba.py needs a CUDA device")
    eng = _native.get_engine(0)
    out = {"gpu": gpu_info(0), "threshold_px2": THR, "max_iterations": args.iters, "steps": args.steps}
    for name in args.workloads:
        V, N = WORKLOADS[name]
        K, R0, t0, X0, off, view, x = scene(V, N)
        res = {}

        def call():
            res["r"] = bundle_adjust_arrays(K, R0, t0, X0, off, view, x, THR, fixed=(0,), scale_view=1,
                                            max_iterations=args.iters, engine=eng)

        call()  # warm-up
        host = []
        for _ in range(args.steps):
            torch.cuda.synchronize()
            t_0 = time.perf_counter()
            call()
            host.append(time.perf_counter() - t_0)
        rep = res["r"].report
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        tot = {k: 0.0 for k in KERNELS}
        cnt = {k: 0 for k in KERNELS}
        evs = []
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                k = _kernel(ev.name)
                if k:
                    evs.append((ev.time_range.start, ev.time_range.end, k))
        evs.sort()
        done_to = evs[0][0] if evs else 0.0
        for s0, e0, k in evs:
            tot[k] += max(0.0, e0 - max(s0, done_to))
            done_to = max(done_to, e0)
            cnt[k] += 1
        span = evs[-1][1] - evs[0][0] if evs else 0.0
        rounds = rep.iterations + 1
        per_round = {k: tot[k] / rounds for k in KERNELS if k not in ONCE}
        # operation and byte counts of the list actually solved (its decisions are the start's)
        from oracle import bundle as oba
        inlist, param = oba.start_list(K, np.concatenate([R0, t0[:, :, None]], axis=2), X0, off, view, x, THR)
        pt = np.repeat(np.arange(len(off) - 1), np.diff(off))
        nf = np.bincount(pt[inlist & (view != 0)], minlength=len(off) - 1).astype(np.int64)
        pairs = int((nf * (nf + 1) // 2).sum())  # one observation per view in these scenes
        n = 6 * (V - 1)
        schur_fma = 108 * pairs
        chol_fma = n ** 3 / 6
        L, T, M = int(inlist.sum()), len(off) - 1, len(view)
        eval_bytes = L * (160 + 16 + 4) + M * 1 + T * (24 + 8 + 1 + 80)
        us = lambda k: per_round[k] * 1e-6  # noqa: E731
        w = {"views": V, "points": N, "observations": M, "list": L, "parameter_points": rep.num_points,
             "iterations": rep.iterations, "status": _native.REFINE_STATUS[rep.status] if isinstance(rep.status, int)
             else rep.status, "cost_start": rep.cost_start, "cost_final": rep.cost_final,
             "call_ms_median": 1e3 * float(np.median(host)),
             "call_ms_spread": [1e3 * float(np.min(host)), 1e3 * float(np.max(host))],
             "kernel_us_per_round": per_round, "kernel_launches": cnt,
             "kernel_us_once": {k: tot[k] for k in ONCE}, "device_span_us": span,
             "device_us_per_round": float(sum(per_round.values())),
             "schur_pairs": pairs, "schur_fma": schur_fma, "reduced_system_n": n, "chol_fma_useful": chol_fma,
             "schur_dfma_rate": schur_fma / us("k_ba_schur") if per_round["k_ba_schur"] else None,
             "chol_dfma_rate": chol_fma / us("k_ba_chol") if per_round["k_ba_chol"] else None,
             "eval_bytes": eval_bytes, "eval_bytes_per_s": eval_bytes / us("k_ba_eval") if per_round["k_ba_eval"] else None}
        w["schur_share_of_dfma_peak"] = w["schur_dfma_rate"] / DFMA_PEAK if w["schur_dfma_rate"] else None
        w["chol_share_of_dfma_peak"] = w["chol_dfma_rate"] / DFMA_PEAK if w["chol_dfma_rate"] else None
        w["eval_share_of_hbm"] = w["eval_bytes_per_s"] / HBM if w["eval_bytes_per_s"] else None
        out[name] = w
        print(name, json.dumps(w), flush=True)
    return out


def scipy_main(args):
    """scipy trf with a sparsity pattern (finite-difference Jacobian by column groups) on workload A, on the host."""
    import numpy as np
    import scipy.sparse as sp
    from scipy.optimize import least_squares

    from oracle import bundle as oba
    from oracle.refine import rodrigues

    V, N = WORKLOADS["A"]
    K, R0, t0, X0, off, view, x = scene(V, N)
    Rt0 = np.concatenate([R0, t0[:, :, None]], axis=2)
    fixed = np.arange(V) == 0
    prob = oba.problem(K, Rt0, X0, off, view, x, THR, fixed, 1)
    cols = oba._cam_columns(prob)
    L = len(prob.obs_track)
    pidx = np.full(len(off) - 1, -1)
    pidx[prob.points] = np.arange(len(prob.points))
    rows, cidx = [], []
    for c, col in cols.items():
        m = np.flatnonzero(prob.obs_view == c)
        for q in col:
            if q >= 0:
                for k in range(2):
                    rows.append(2 * m + k)
                    cidx.append(np.full(len(m), q))
    for j in range(3):
        for k in range(2):
            rows.append(2 * np.arange(L) + k)
            cidx.append(prob.n_cam + 3 * pidx[prob.obs_track] + j)
    rows, cidx = np.concatenate(rows), np.concatenate(cidx)
    S = sp.csr_matrix((np.ones(len(rows)), (rows, cidx)), shape=(2 * L, prob.n))
    Kv = prob.K[prob.obs_view]

    def fun(z):
        R, tt = prob.R.copy(), prob.t.copy()
        for c, col in cols.items():
            v = np.array([z[q] if q >= 0 else 0.0 for q in col])
            R[c] = prob.R[c] @ rodrigues(v[:3])
            tt[c] = prob.t[c] + v[3:]
        Xp = prob.X[prob.obs_track] + z[prob.n_cam:].reshape(-1, 3)[pidx[prob.obs_track]]
        p = np.einsum("mij,mj->mi", Kv, np.einsum("mij,mj->mi", R[prob.obs_view], Xp) + tt[prob.obs_view])
        return (p[:, :2] / p[:, 2:] - prob.obs_x).ravel()

    t_0 = time.perf_counter()
    res = least_squares(fun, np.zeros(prob.n), jac_sparsity=S, method="trf", tr_solver="lsmr", x_scale="jac",
                        max_nfev=args.iters + 1, xtol=1e-15, ftol=1e-15, gtol=1e-15)
    dt = time.perf_counter() - t_0
    cpu = platform.processor() or platform.machine()
    try:
        with open("/proc/cpuinfo") as f:
            cpu = next(l.split(":", 1)[1].strip() for l in f if l.startswith("model name"))
    except (OSError, StopIteration):
        pass
    return {"scipy_trf_A": {"cpu": cpu, "cpus": os.cpu_count(), "parameters": prob.n, "residuals": 2 * L,
                            "max_nfev": args.iters + 1, "nfev": int(res.nfev), "seconds": dt,
                            "cost_start": float(np.sum(fun(np.zeros(prob.n)) ** 2)), "cost_final": 2 * float(res.cost)}}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--workloads", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--scipy", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    out = scipy_main(args) if args.scipy else gpu_main(args)
    line = json.dumps(out)
    print(line)
    if args.out:
        prev = {}
        if os.path.exists(args.out):
            with open(args.out) as f:
                prev = json.loads(f.read() or "{}")
        prev.update(out)
        with open(args.out, "w") as f:
            f.write(json.dumps(prev) + "\n")


if __name__ == "__main__":
    main()
