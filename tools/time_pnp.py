"""Time the absolute-pose (PnP) path on one GPU: k_score_pnp alone, the whole estimate, and the whole
ransac_pnp_arrays(sampler="device") call.

Scene: make_pnp_scene, N = 100 000 records, H = 65 536 hypotheses from the device sampler, 40 % outliers, threshold
4 px^2 on the squared reprojection error, minimum 30 000 extra inliers, RMS.  Every timed step starts from a flushed L2 (a 256 MB buffer is zeroed
first).  Times come from CUDA events: torch events around the whole estimate (sample -> fit -> score -> select -> mask
-> copies to the host), the library's stage events (sfm_get_timing) for the scorer and the other stages, and a host
clock around ransac_pnp_arrays (which synchronises; it includes the upload of the records).

Prints one JSON line: evaluations/s of the scorer against the pipe floor implied by the 16 counted FP64 slots per
evaluation (sfm_measure_fp64_peak), the stage times, and the GPU's name, power limit and maximum SM clock read in the
same run.

    python tools/time_pnp.py [--steps 20] [--warmup 3] [--out FILE]
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

N, H, OUTLIERS, THR, MIN_EXTRA = 100_000, 65_536, 0.4, 4.0, 30_000
SLOTS = 16  # FP64 issue slots per evaluation (csrc/sfm_pnp.cuh)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.pnp import ransac_pnp_arrays
    from structure_from_motion_b200.scenes import make_pnp_scene

    if not torch.cuda.is_available():
        raise SystemExit("time_pnp.py needs a CUDA device")
    torch.cuda.set_device(0)
    eng = _native.get_engine(0)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    K, X, x, R, t, _ = make_pnp_scene(N, OUTLIERS, seed=0)
    eng.upload_pnp(X, x, K)
    peak_dfma = eng.measure_fp64_peak()

    def step(seed):
        eng.sample_device(seed, H)
        best, Rt, *_ = eng.ransac_pnp(THR, MIN_EXTRA, "rms", "min_error")
        if best.index < 0:
            raise RuntimeError("no model found")
        return best, Rt

    for w in range(max(args.warmup, 1)):
        step(1000 + w)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for s in range(args.steps):
        flush_buf.zero_()
        ev[s][0].record(stream)
        best, Rt = step(s)
        ev[s][1].record(stream)
    torch.cuda.synchronize()
    whole_ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps

    eng.enable_timing(True)
    stage = {}
    for s in range(args.steps):
        flush_buf.zero_()
        step(s)
        tm, _ = eng.get_timing()
        for k, v in tm.items():
            stage[k] = stage.get(k, 0.0) + v / args.steps
    eng.enable_timing(False)
    torch.cuda.synchronize()

    api_ms = []
    for s in range(args.steps):
        flush_buf.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = ransac_pnp_arrays(K, X, x, THR, MIN_EXTRA, "rms", H, sampler="device", seed=s, engine=eng)
        api_ms.append((time.perf_counter() - t0) * 1e3)

    evals = float(N) * H
    score_rate = evals / (stage["score"] * 1e-3)
    floor_rate = peak_dfma / SLOTS
    rec = {
        "what": "PnP RANSAC (P3P, reprojection error), make_pnp_scene",
        "n": N, "h": H, "outlier_frac": OUTLIERS, "threshold_px2": THR, "min_extra": MIN_EXTRA, "sampler": "device",
        "steps": args.steps, "l2": "flushed before every step",
        "k_score_pnp_ms": round(stage["score"], 4),
        "k_score_pnp_evals_per_s": score_rate,
        "whole_estimate_ms": round(whole_ms, 4),
        "ransac_pnp_arrays_ms_median": round(float(np.median(api_ms)), 4),
        "fp64_peak_dfma_per_s": peak_dfma,
        "fp64_slots_per_eval": SLOTS,
        "pipe_floor_evals_per_s": floor_rate,
        "share_of_pipe_floor": score_rate / floor_rate,
        "stage_ms": {k: round(v, 4) for k, v in stage.items()},
        "winner": {"index": int(best.index), "count_extra": int(best.count_extra), "error": float(best.err),
                   "max_abs_dev_R": float(np.abs(Rt[:, :3] - R).max()), "max_abs_dev_t": float(np.abs(Rt[:, 3] - t).max()),
                   "api_count_extra": int(res.count_extra)},
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
