"""Time the essential-matrix / homography choice on one GPU.

1. k_score_models alone at N = 100 000 (E and H, pixel coordinates of make_scene): kernel time from torch.profiler
   (CUDA activities, in a run of its own) and the whole sfm_score_models call (staging copy, kernel, result copy,
   synchronisation) from CUDA events, averaged over many calls.
2. two_view_select_arrays end to end on the homography timing scene (make_planar_scene, N = 100 000, H = 65 536 from
   the device sampler, 40 % outliers, 4 px^2 on the transfer error, 1e-5 on the SED, minimum 30 000 extra inliers,
   RMS) against the two calls it makes, two_view_arrays and two_view_homography_arrays, timed alone.  Host clock
   around each call (every call ends in a synchronisation), the three alternated step by step.

Prints one JSON line with the card's name, power limit and maximum SM clock read in the same run.

    python tools/time_model_select.py [--steps 10] [--calls 200] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.time_homography import gpu_info  # noqa: E402

N, H, OUTLIERS, H_THR, E_THR, MIN_EXTRA = 100_000, 65_536, 0.4, 4.0, 1e-5, 30_000


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200 import homography as hg
    from structure_from_motion_b200 import two_view
    from structure_from_motion_b200.errors import EightPointCalculationError
    from structure_from_motion_b200.model_selection import two_view_select_arrays
    from structure_from_motion_b200.scenes import make_planar_scene, make_scene

    if not torch.cuda.is_available():
        raise SystemExit("time_model_select.py needs a CUDA device")
    torch.cuda.set_device(0)
    eng = _native.get_engine(0)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)

    # 1. the kernel
    K, x1, x2, R, t, _ = make_scene(N, 0.3, seed=0)
    tx = np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]])
    E = tx @ R
    Hm = K @ (R + np.outer(t, [0.0, 0.0, 1.0]) / 6.0) @ np.linalg.inv(K)
    eng.upload_pairs(x1, x2, K)
    for _ in range(20):
        eng.model_scores(E, Hm, K)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(args.calls):
        s, _ = eng.model_scores(E, Hm, K)
    b.record(stream)
    torch.cuda.synchronize()
    call_ms = a.elapsed_time(b) / args.calls
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.calls):
            eng.model_scores(E, Hm, K)
        torch.cuda.synchronize()
    kern = [e for e in prof.events() if e.name.startswith("_ZN3sfm14k_score_models") or "k_score_models" in e.name]
    kernel_ms = sum(getattr(e, "device_time", 0.0) for e in kern) / max(len(kern), 1) / 1e3 if kern else None

    # 2. end to end
    K, x1, x2, _, _ = make_planar_scene(N, OUTLIERS, seed=0)
    common = dict(sampler="device", engine=eng)

    def run_e(seed):
        return two_view.two_view_arrays(K, x1, x2, E_THR, MIN_EXTRA, "rms", H, seed=seed, on_degenerate="skip", **common)

    def run_h(seed):
        return hg.two_view_homography_arrays(K, x1, x2, H_THR, MIN_EXTRA, "rms", H, seed=seed, **common)

    def run_sel(seed):
        return two_view_select_arrays(K, x1, x2, E_THR, H_THR, MIN_EXTRA, "rms", H, seed=seed, **common)

    arms = {"essential": run_e, "homography": run_h, "select": run_sel}
    for f in arms.values():
        try:
            f(1000)
        except (ValueError, EightPointCalculationError):
            pass
    times = {k: [] for k in arms}
    last = None
    for step in range(args.steps):
        for k, f in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            try:
                r = f(step)
            except (ValueError, EightPointCalculationError) as exc:  # still a timed call: it ran to the end
                r = exc
            times[k].append((time.perf_counter() - t0) * 1e3)
            if k == "select":
                last = r
    rec = {
        "what": "essential matrix or homography: k_score_models and two_view_select_arrays",
        "k_score_models": {"n": N, "calls": args.calls, "kernel_ms": kernel_ms, "profiled_launches": len(kern),
                           "sfm_score_models_call_ms": round(call_ms, 5), "bytes_read": N * 32,
                           "model": int(s.model), "ratio_h": s.ratio_h},
        "end_to_end": {"scene": "make_planar_scene", "n": N, "h": H, "outlier_frac": OUTLIERS, "threshold_px2": H_THR,
                       "sed_threshold": E_THR, "min_extra": MIN_EXTRA, "sampler": "device", "steps": args.steps,
                       "ms": {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}
                              for k, v in times.items()},
                       "select_minus_both_ms": float(np.median(times["select"]) - np.median(times["essential"])
                                                     - np.median(times["homography"])),
                       "model": getattr(last, "model", repr(last)), "ratio_h": getattr(getattr(last, "scores", None), "ratio_h", None)},
        "gpu": gpu_info(torch.cuda.current_device()),
    }
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
