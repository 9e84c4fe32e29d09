"""Time the least-squares refinement (sfm_set_refinement) against the same calls with refinement off, on one GPU.

Workloads (each timed with refinement off and on, alternated step by step, host clock around calls that end in a
synchronisation; medians):
  config3      make_scene(100 000, 40 % outliers) x 65 536 device-sampler hypotheses through
               two_view.two_view_arrays(sampler="device"), SED threshold 1.5e-6, RMS, min_extra 10 (bench.py's config 3)
  homography   the planar timing scene of DESIGN.md section 7a (make_planar_scene(100 000, 40 %), 65 536 hypotheses,
               4 px^2, min_extra 30 000) through homography.two_view_homography_arrays(sampler="device")
  config4_e    512 pairs x 2 000 correspondences x 2 000 hypotheses (tools/time_batch_select.py's pairs) through
               Engine.batch_two_view
  config4_sel  the same through model_selection.batch_two_view_select_arrays
Per workload:
  host      the median call time off and on, and the time of the report fetch (sfm_get_refinement: one synchronisation
            and a D2H copy, which only the "on" call makes); ms_refinement = on - off - fetch, and its share of the call
  device    from a separate run under torch.profiler (CUDA activities, every kernel of the process): the summed device
            time of the refinement's kernels (k_refine_init, the k_refine_step launches, k_refine_finish) and of the
            extra T1 pass (k_tail_mask on minus off) in one "on" call, and that stage time as a share of the host "on" call
  the kernels launched per call off and on, the list sizes (refine_num), and the iterations and rejected proposals of
  the refined pairs (median / max) with their statuses.

Prints one JSON line with the card's name, power limit and maximum SM clock read in the same run.

    python tools/time_refine.py [--steps 7] [--warmup 2] [--iterations 20] [--out FILE]
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

from tools.time_batch_select import E_THR as B_E_THR, H_THR as B_H_THR, H as B_H, MIN_EXTRA as B_MIN_EXTRA  # noqa: E402
from tools.time_batch_select import scenes as batch_scenes  # noqa: E402
from tools.time_homography import gpu_info  # noqa: E402


def main() -> None:
    import numpy as np

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.homography import two_view_homography_arrays
    from structure_from_motion_b200.model_selection import batch_two_view_select_arrays
    from structure_from_motion_b200.scenes import make_planar_scene, make_scene
    from structure_from_motion_b200.two_view import two_view_arrays

    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iterations", type=int, default=20, help="refine_iterations of the timed calls")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    eng = _native.Engine(0)
    eng.enable_timing(False)
    it = args.iterations

    K3, a3, b3, *_ = make_scene(100_000, 0.4, seed=0)
    Kh, ah, bh, *_ = make_planar_scene(100_000, 0.4, seed=0)
    xa, xb, offsets, Ks = batch_scenes()

    fetch = {}

    def timed_fetch(name, pairs):
        t0 = time.perf_counter()
        eng.get_refinement(pairs)
        fetch.setdefault(name, []).append(time.perf_counter() - t0)

    def config3(r):
        res = two_view_arrays(K3, a3, b3, 1.5e-6, 10, "rms", 65_536, sampler="device", seed=1, on_degenerate="skip",
                              engine=eng, refine_iterations=r)
        if r:
            timed_fetch("config3", 1)
        return [res.refinement] if res.refinement else []

    def homography(r):
        res = two_view_homography_arrays(Kh, ah, bh, 4.0, 30_000, "rms", 65_536, sampler="device", seed=1, engine=eng,
                                         refine_iterations=r)
        if r:
            timed_fetch("homography", 1)
        return [res.refinement] if res.refinement else []

    def config4_e(r):
        out = eng.batch_two_view(xa, xb, offsets, Ks, B_H, 1, B_E_THR, B_MIN_EXTRA, refine_iterations=r)
        if r:
            timed_fetch("config4_e", len(offsets) - 1)
        return _batch_reports(out) if r else []

    def config4_sel(r):
        out = batch_two_view_select_arrays(xa, xb, offsets, Ks, B_E_THR, B_H_THR, B_H, 1, min_extra=B_MIN_EXTRA,
                                           engine=eng, refine_iterations=r)
        if r:  # the selection fetches two reports (E batch and H batch)
            timed_fetch("config4_sel", len(offsets) - 1)
            fetch["config4_sel"][-1] *= 2
        return _batch_reports(out["essential"]) + _batch_reports(out["homography"]) if r else []

    def _batch_reports(d):
        return [dict(iterations=int(i), rejected=int(j), num=int(n), status=_native.REFINE_STATUS[int(s)])
                for i, j, n, s in zip(d["refine_iterations"], d["refine_rejected"], d["refine_num"], d["refine_status"])]

    def device_times(fn, r):
        """Device time of the refinement's kernels and of the extra T1 pass in one call (torch.profiler)."""
        try:
            import torch
            from torch.profiler import ProfilerActivity, profile

            torch.cuda.init()

            def kernels(rr):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    fn(rr)
                    torch.cuda.synchronize()
                out = {}
                for ev in prof.events():
                    us = getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0)
                    out.setdefault(ev.name, []).append(float(us))
                return out

            on_k, off_k = kernels(r), kernels(0)
            refine = sum(sum(v) for k, v in on_k.items() if "k_refine_" in k) / 1e3
            mask = lambda d: sum(sum(v) for k, v in d.items() if "k_tail_mask" in k) / 1e3
            steps = sum(len(v) for k, v in on_k.items() if "k_refine_step" in k)
            return {"refine_kernels_ms": refine, "extra_tail_mask_ms": mask(on_k) - mask(off_k), "step_launches": steps,
                    "step_ms_each": (sum(sum(v) for k, v in on_k.items() if "k_refine_step" in k) / 1e3 / steps
                                     if steps else None)}
        except Exception as exc:  # the host figures stand on their own
            return {"error": repr(exc)[:200], "refine_kernels_ms": 0.0, "extra_tail_mask_ms": 0.0}

    record = {"tool": "tools/time_refine.py", "gpu": gpu_info(0), "refine_iterations": it, "steps": args.steps,
              "warmup": args.warmup, "workloads": {}}
    for name, fn in (("config3", config3), ("homography", homography), ("config4_e", config4_e),
                     ("config4_sel", config4_sel)):
        for _ in range(args.warmup):
            fn(0), fn(it)
        t = {0: [], it: []}
        launches = {}
        reports = []
        for _ in range(args.steps):
            for r in (0, it):  # alternated
                l0 = eng.get_timing()[1]
                t0 = time.perf_counter()
                rep = fn(r)
                t[r].append(time.perf_counter() - t0)
                launches[r] = eng.get_timing()[1] - l0
                if r:
                    reports = rep
        off, on = float(np.median(t[0])) * 1e3, float(np.median(t[it])) * 1e3
        fetch_ms = float(np.median(fetch[name])) * 1e3
        reps = [x if isinstance(x, dict) else dict(iterations=x.iterations, rejected=x.rejected, num=x.num,
                                                   status=x.status) for x in reports]
        refined = [x for x in reps if x["status"] not in ("no_model", "nonfinite")]
        iters = [x["iterations"] for x in refined]
        rej = [x["rejected"] for x in refined]
        nums = [x["num"] for x in refined]
        status = [x["status"] for x in reps]
        dev = device_times(fn, it)
        dev_stage = dev["refine_kernels_ms"] + dev["extra_tail_mask_ms"] if "error" not in dev else None
        record["workloads"][name] = {
            "ms_off": off, "ms_on": on, "ms_fetch": fetch_ms, "ms_refinement": on - off - fetch_ms,
            "share_of_call": (on - off - fetch_ms) / on,
            "device_ms_stage": dev_stage, "device_share_of_call": dev_stage / on if dev_stage is not None else None, "device": dev,
            "spread_off_ms": [float(np.min(t[0])) * 1e3, float(np.max(t[0])) * 1e3],
            "spread_on_ms": [float(np.min(t[it])) * 1e3, float(np.max(t[it])) * 1e3],
            "launches_off": int(launches[0]), "launches_on": int(launches[it]),
            "iterations_median": float(np.median(iters)) if iters else None,
            "iterations_max": int(max(iters)) if iters else None,
            "rejected_median": float(np.median(rej)) if rej else None, "rejected_max": int(max(rej)) if rej else None,
            "num_median": float(np.median(nums)) if nums else None, "num_min": int(min(nums)) if nums else None,
            "num_max": int(max(nums)) if nums else None,
            "status": {s: status.count(s) for s in sorted(set(status))},
        }
        print(name, json.dumps(record["workloads"][name]), flush=True)
    eng.close()
    line = json.dumps(record)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
