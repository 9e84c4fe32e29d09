"""Time the homography path on one GPU: k_score_homography alone and the whole estimate.

Scene: planar (make_planar_scene), N = 100 000 correspondences, H = 65 536 hypotheses from the device sampler,
40 % outliers, threshold 4 px^2 on the symmetric transfer error, minimum 30 000 extra inliers, RMS.  Every timed step
starts from a flushed L2 (a 256 MB buffer is zeroed first, as bench.py does).  Times come from CUDA events: torch
events around the whole estimate (sample -> fit -> score -> select -> mask -> one D2H of the record), the library's
stage events (sfm_get_timing) for the scorer and the other stages.

Prints one JSON line: evaluations/s of the scorer and of the whole estimate, the share of the FP64 pipe floor
implied by the 27 counted FP64 slots per evaluation (against sfm_measure_fp64_peak), the stage times, and the GPU's
name, power limit and maximum SM clock read in the same run.

--tail times the fused call sfm_two_view_homography instead: the same estimate followed by the pose tail (T1 inlier
mask + compaction + decomposition of K^-1 H K, T2 cheirality vote, T3 triangulation) and the copies of the mask, the
errors and the per-inlier results to the host.  The stage times "mask", "pose" and "triangulate" are T1, T2 and T3.

    python tools/time_homography.py [--steps 20] [--warmup 3] [--tail] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N, H, OUTLIERS, THR, MIN_EXTRA = 100_000, 65_536, 0.4, 4.0, 30_000
SLOTS = 27  # FP64 issue slots per evaluation of the division-free decision (csrc/sfm_homography.cuh)


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [v.strip() for v in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--tail", action="store_true", help="time estimate + pose tail (sfm_two_view_homography)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.scenes import make_planar_scene

    if not torch.cuda.is_available():
        raise SystemExit("time_homography.py needs a CUDA device")
    torch.cuda.set_device(0)
    eng = _native.get_engine(0)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)  # the flush, the events and the engine in one stream order
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB of L2

    K, x1, x2, H_true, _ = make_planar_scene(N, OUTLIERS, seed=0)
    eng.upload_pairs(x1, x2, np.eye(3))
    peak_dfma = eng.measure_fp64_peak()

    tail = {}

    def step(seed):
        eng.sample_device(seed, H)
        if args.tail:
            best, _, _, p, num, *_ = eng.two_view_homography(K, THR, MIN_EXTRA, "rms", "min_error")
            tail.update(num_inliers=num, counts=list(p.counts), best=int(p.best), rotation_only=int(p.rotation_only))
        else:
            best, *_ = eng.ransac_homography(THR, MIN_EXTRA, "rms", "min_error", want_mask=True)
        if best.index < 0:
            raise RuntimeError("no model found")
        return best

    for w in range(max(args.warmup, 1)):
        step(1000 + w)
    torch.cuda.synchronize()

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for s in range(args.steps):
        flush_buf.zero_()
        ev[s][0].record(stream)
        best = step(s)
        ev[s][1].record(stream)
    torch.cuda.synchronize()
    whole_ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps

    eng.enable_timing(True)
    stage = {}
    for s in range(args.steps):
        flush_buf.zero_()
        step(s)
        t, _ = eng.get_timing()
        for k, v in t.items():
            stage[k] = stage.get(k, 0.0) + v / args.steps
    eng.enable_timing(False)
    torch.cuda.synchronize()

    H_est = np.array(best.E).reshape(3, 3)
    evals = float(N) * H
    score_rate = evals / (stage["score"] * 1e-3)
    floor_rate = peak_dfma / SLOTS
    rec = {
        "what": "homography RANSAC + pose tail, planar scene" if args.tail else "homography RANSAC, planar scene",
        "n": N, "h": H, "outlier_frac": OUTLIERS, "threshold_px2": THR, "min_extra": MIN_EXTRA, "sampler": "device",
        "steps": args.steps, "l2": "flushed before every step",
        "k_score_homography_ms": round(stage["score"], 4),
        "k_score_homography_evals_per_s": score_rate,
        "whole_estimate_ms": round(whole_ms, 4),
        "whole_estimate_evals_per_s": evals / (whole_ms * 1e-3),
        "fp64_peak_dfma_per_s": peak_dfma,
        "fp64_slots_per_eval": SLOTS,
        "pipe_floor_evals_per_s": floor_rate,
        "share_of_pipe_floor": score_rate / floor_rate,
        "stage_ms": {k: round(v, 4) for k, v in stage.items()},
        **({"tail_ms": round(stage["mask"] + stage["pose"] + stage["triangulate"], 4), "tail": tail} if args.tail else {}),
        "winner": {"index": int(best.index), "count_extra": int(best.count_extra), "error": float(best.err),
                   "rel_dev_from_true_H": float(np.max(np.abs(H_est - H_true)) / np.max(np.abs(H_true)))},
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
