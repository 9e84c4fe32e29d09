"""Time the multi-view triangulation of tracks (sfm_triangulate_tracks) on the GPU.

Workloads (make_multi_view_scene, threshold 4 px^2):
  tracks      10^6 tracks over 16 views, lengths uniform in 2-8, 10 % outlier observations, refinement off;
  refined     the same with refine_iterations = 10;
  two_obs     10^6 two-observation tracks over 2 views, next to k_triangulate (sfm_triangulate, Engine.triangulate) on the
              same 10^6 correspondences with P = K [R | t] of the same two views.
Kernel times: the device duration of each kernel (CUPTI activity records through torch.profiler, in a run of their own),
with the 126 MB L2 overwritten by a 512 MB device fill between passes; the median over the passes.  Call times: the
median of a host clock around each call (the call synchronises; it includes the copies in and out), profiler off.
The bar: the two-observation tracks' kernels (k_track_views + k_track_pairs + k_track_solve) take at most twice
k_triangulate's time.  Writes one JSON object with the GPU's name, power limit and maximum SM clock read in the same run.

    python tools/time_tracks.py [--steps 10] [--warmup 2] [--out profiles/tracks_time_b200.json]
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

THR = 4.0
N = 1_000_000


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.multiview import triangulate_tracks_arrays
    from structure_from_motion_b200.scenes import make_multi_view_scene

    if not torch.cuda.is_available():
        raise SystemExit("time_tracks.py needs a CUDA device")
    eng = _native.get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    out = {"gpu": gpu_info(0), "threshold_px2": THR, "tracks": N, "steps": args.steps}

    def measure(call, names):
        for _ in range(args.warmup):
            call()
        host = []
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call()
            host.append(time.perf_counter() - t0)
        per = {k: [] for k in names}
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                flush.fill_(1)
                torch.cuda.synchronize()
                call()
            torch.cuda.synchronize()
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                for k in names:
                    if k in ev.name:
                        per[k].append(ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total)
        kern = {k: float(np.median(v)) if v else None for k, v in per.items()}
        return {"call_ms_median": 1e3 * float(np.median(host)),
                "call_ms_spread": [1e3 * float(np.min(host)), 1e3 * float(np.max(host))],
                "kernel_us_median": kern, "kernel_samples": {k: len(v) for k, v in per.items()}}

    track_kernels = ["k_track_views", "k_track_pairs", "k_track_solve"]
    K, R, t, X, off, view, x, _ = make_multi_view_scene(N, 16, 0, noise_px=0.5, outlier_frac=0.1)
    pairs = int((np.diff(off) * (np.diff(off) - 1) // 2).sum())
    for name, it in (("tracks", 0), ("refined", 10)):
        res = {}

        def call():
            res["r"] = triangulate_tracks_arrays(K, R, t, off, view, x, THR, refine_iterations=it, engine=eng)

        out[name] = measure(call, track_kernels)
        out[name].update({"views": 16, "observations": int(off[-1]), "pairs": pairs, "refine_iterations": it,
                          "ok_share": float((res["r"].status == "ok").mean())})
        print(name, json.dumps(out[name]), flush=True)

    K2, R2, t2, X2, off2, view2, x2, _ = make_multi_view_scene(N, 2, 1, noise_px=0.5, min_len=2, max_len=2)
    xa, xb = np.ascontiguousarray(x2[0::2]), np.ascontiguousarray(x2[1::2])
    P = [K2 @ np.column_stack([R2[c], t2[c]]) for c in range(2)]

    def call_tracks():
        triangulate_tracks_arrays(K2, R2, t2, off2, view2, x2, THR, engine=eng)

    def call_tri():
        eng.triangulate(P[0], P[1], xa, xb)

    a = measure(call_tracks, track_kernels)
    b = measure(call_tri, ["k_triangulate"])
    tracks_us = sum(v for v in a["kernel_us_median"].values() if v)
    tri_us = b["kernel_us_median"]["k_triangulate"]
    out["two_obs"] = {"tracks": a, "k_triangulate": b, "tracks_kernels_us": tracks_us, "k_triangulate_us": tri_us,
                      "ratio": tracks_us / tri_us if tri_us else None}
    print("two_obs", json.dumps(out["two_obs"]), flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
