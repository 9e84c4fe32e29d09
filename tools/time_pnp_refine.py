"""Time the PnP pose refinement (sfm_refine_pnp): what refine_iterations=20 adds to ransac_pnp_arrays(sampler="device").

Large shape (the tools/time_pnp.py scene): make_pnp_scene, N = 100 000 records, H = 65 536 device-sampled hypotheses,
40 % outliers, threshold 4 px^2, minimum 30 000 extra inliers, RMS.  Small shape: 1 000 records, 500 hypotheses, 40 %
outliers, minimum 300 extra inliers.  Each shape alternates calls with the refinement off and on (same seed) and takes
the median of a host clock around each call (the call synchronises; it includes the upload).  The refinement's device
time is the summed duration of its kernels (k_refine_*, and the k_pnp_mask under the refined pose) in a separate
torch.profiler run.  Writes one JSON object with the GPU's name, power limit and maximum SM clock read in the same run.

    python tools/time_pnp_refine.py [--steps 20] [--warmup 3] [--out profiles/pnp_refine_time_b200.json]
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

SHAPES = {"large": (100_000, 65_536, 30_000), "small": (1_000, 500, 300)}
OUTLIERS, THR, ITERS = 0.4, 4.0, 20


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.pnp import ransac_pnp_arrays
    from structure_from_motion_b200.scenes import make_pnp_scene

    if not torch.cuda.is_available():
        raise SystemExit("time_pnp_refine.py needs a CUDA device")
    eng = _native.get_engine(0)
    out = {"gpu": gpu_info(0), "refine_iterations": ITERS, "threshold_px2": THR, "outliers": OUTLIERS}
    for name, (n, h, extra) in SHAPES.items():
        K, X, x, R, t, _ = make_pnp_scene(n, OUTLIERS, seed=0)

        def call(it, seed):
            t0 = time.perf_counter()
            res = ransac_pnp_arrays(K, X, x, THR, extra, "rms", h, sampler="device", seed=seed, engine=eng,
                                    refine_iterations=it)
            return time.perf_counter() - t0, res

        for w in range(args.warmup):
            call(0, w)
            call(ITERS, w)
        off, on, statuses = [], [], []
        for s in range(args.steps):
            a, _ = call(0, 100 + s)
            b, res = call(ITERS, 100 + s)
            off.append(a)
            on.append(b)
            statuses.append((res.refinement.status, res.refinement.iterations, res.refinement.num))
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for s in range(5):
                call(ITERS, 100 + s)
            torch.cuda.synchronize()
        dev = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                dev.setdefault(ev.name, []).append(ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total)
        refine_us = sum(sum(v) for k, v in dev.items() if "k_refine_" in k) / 5
        mask_us = sum(sum(v) for k, v in dev.items() if "k_pnp_mask" in k) / 5 / 2  # one of the two masks per call
        step_us = [np.mean(v) for k, v in dev.items() if "k_refine_step" in k]
        off_ms, on_ms = 1e3 * float(np.median(off)), 1e3 * float(np.median(on))
        out[name] = {
            "records": n, "hypotheses": h, "min_extra": extra,
            "call_ms_off_median": off_ms, "call_ms_on_median": on_ms,
            "call_ms_off_spread": [1e3 * float(np.min(off)), 1e3 * float(np.max(off))],
            "call_ms_on_spread": [1e3 * float(np.min(on)), 1e3 * float(np.max(on))],
            "added_share": (on_ms - off_ms) / off_ms,
            "refine_kernels_us_per_call": refine_us, "refined_mask_us_per_call": mask_us,
            "step_us_each": float(step_us[0]) if step_us else None,
            "statuses": sorted(set(map(str, statuses)))[:8],
        }
        print(name, json.dumps(out[name]), flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
