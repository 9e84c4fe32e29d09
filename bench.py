#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: fp64 hypothesis x correspondence
evaluations per second of RANSAC essential-matrix estimation (+ cheirality vote and
triangulation of the inliers), BASELINE.json configs[2]: 100k correspondences x 64k hypotheses.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload ...] [--dump-outputs DIR]

One "step" = one complete estimate on a synthetic two-view scene (40 % outliers): device
sampler -> eight-point fit of every hypothesis -> scoring -> selection -> inlier mask of the
winner -> decomposition + cheirality vote -> triangulation of the passing inliers.

* ``value``     whole-step throughput, correspondences already resident in HBM.
* ``e2e``       the same estimate through the public Python API (two_view.two_view_arrays) from
                pinned HOST arrays: H2D of the correspondences and D2H of every result are inside
                the timed region.
* ``roofline``  the scoring kernel (k_score) against the FP64 pipe: algorithmic work
                (SURVEY.md §8(d): 35 flop per evaluation) / its CUDA-event duration, against an FP64
                FMA peak measured on this GPU in this run (MEASURED_PEAKS.json has no fp64 entry).
* ``cpu_baseline`` the oracle port (numpy eight-point + threaded C scorer) on the host cores, on a
                bounded sample of the same workload.
N > 1 (torchrun): hypotheses are sharded — every rank scores its own 64k hypotheses of the same
pair (weak scaling); the 144-byte selection records are all-gathered device-to-device by NCCL (the one collective),
merged by a kernel, and the tail runs behind it without a host round trip.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "hyp x point evals/sec (fp64)"
UNIT = "evals/s"
THR, MIN_EXTRA, AGG = 1.5e-6, 10, "rms"  # apps/config/config.yaml:6-9, apps/sfm.py:116
FLOP_PER_EVAL = 35.0                      # SURVEY.md §8(d): 14 DFMA + 7 DMUL/DADD
BYTES_PER_CORR = 32.0

WORKLOADS = {
    # name: (correspondences, hypotheses per GPU, outlier fraction)
    "config2": (10_000, 16_384, 0.4),
    "config3": (100_000, 65_536, 0.4),
    "config5": (1_048_576, 1_048_576, 0.4),  # hypotheses are split over the ranks (strong scaling)
}


_REAL_STDOUT = None


def quiet_stdout():
    """Everything libraries print to stdout during the run (NCCL's version banner, for one) goes to stderr; the
    one JSON line is written to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="config3", choices=list(WORKLOADS) + ["config1", "config4", "frontend"])
    ap.add_argument("--variant", default=os.environ.get("SFM_SCORE_VARIANT", "auto"), choices=["auto", "screen", "full", "screen32"])
    ap.add_argument("--hpt", type=int, default=int(os.environ.get("SFM_SCORE_HPT", "2")))
    ap.add_argument("--group", type=int, default=int(os.environ.get("SFM_SCORE_GROUP", "16")))
    ap.add_argument("--pairs", type=int, default=512, help="config4: image pairs per GPU per step")
    ap.add_argument("--cpu-sample-hyps", type=int, default=0, help="reference arm: hypotheses per step (0 = auto)")
    ap.add_argument("--cpu-step-seconds", type=float, default=2.0, help="reference arm: target seconds per step")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=12.0, help="native arm: cpu_baseline sample length")
    ap.add_argument("--true-reference-seconds", type=float, default=10.0,
                    help="CPU legs: budget for timing the unmodified reference on one core")
    ap.add_argument("--no-true-reference", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the sub-records (config3_strong, config5_strong, config4_pairs, parity_multi)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fp32-variant", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="config4: one context instead of the two-context pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="native arm: write the results of the last timed step as DIR/<name>.npy (float64; rank 0's on "
                         "several GPUs); the inputs depend only on the arguments, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the native arm")
    return args


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(directory, arrays):
    """Save each array as directory/<name>.npy in float64 (integers up to 2^53 stay exact).  Every value must be
    finite: placeholders such as the NaN of an untriangulated point are left out by the caller, not written."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes + 128 for a in arrays.values())  # + the .npy header
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
    bad = [k for k, a in arrays.items() if not np.isfinite(a).all()]
    if bad:
        raise SystemExit(f"--dump-outputs: non-finite values in {bad}")
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def two_view_outputs(res):
    """One estimate's results, from Engine.two_view's tuple (one GPU) or two_view_sharded's dict (several GPUs): the
    winner, the four poses of its decomposition with their cheirality votes, the inlier list, the cheirality pass bits
    of every inlier (bit b: passes pose b) and the points triangulated for the inliers that pass the voted pose (the
    library returns NaN rows for the others)."""
    if isinstance(res, tuple):
        best, _, _, poses, num, idx, ok, X = res
        res = dict(err=best.err, index=best.index, count=best.count_extra, E=best.E, num_invalid=best.num_invalid,
                   poses=poses, num_inliers=num, inlier_idx=idx, pass_bits=ok, points=X)
    p = res["poses"]
    ok = res["pass_bits"]
    passing = ((ok >> p.best) & 1).astype(bool) if p.best >= 0 else np.zeros(len(ok), dtype=bool)
    return {"E": np.reshape(res["E"], (3, 3)), "best_err": res["err"], "best_index": res["index"],
            "count_extra": res["count"], "num_invalid": res["num_invalid"], "num_inliers": res["num_inliers"],
            "pose_R": np.reshape(p.R, (4, 3, 3)), "pose_t": np.reshape(p.t, (4, 3)), "pose_sv": p.sv,
            "pose_counts": p.counts, "pose_best": p.best, "inlier_idx": res["inlier_idx"], "pass_bits": res["pass_bits"],
            "points": res["points"][passing]}


# ----------------------------------------------------------------------------------------------
# clocks (nvidia-smi sampled DURING the timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 20 ms from before the warm-up; only samples whose timestamp falls
    inside [mark_begin, mark_end] (the timed region) are reported."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.path = tempfile.mktemp(prefix="sfm_clocks_", suffix=".csv")
        self.proc = None
        self.index = index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime

        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "power_w_max": None}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), float(f[3]),
                                 [nm for nm, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        inside = [r for r in rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or 1e30)]
        window = "timed region"
        if not inside:  # timestamps unusable (time zone / clock skew): fall back to every sample of the run
            inside, window = rows, "whole run"
        if inside:
            out.update(sm_mhz=statistics.median(r[1] for r in inside), sm_max_mhz=max(r[2] for r in inside),
                       power_w_max=max(r[3] for r in inside), reasons=sorted({x for r in inside for x in r[4]}),
                       samples=len(inside), window=window)
        return out


# ----------------------------------------------------------------------------------------------
# CPU legs (oracle port; the only places bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------
_CPU_CTX = {}


def _cpu_worker_init(K, x1, x2):
    from oracle import csed
    from oracle import restatement as o

    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    _CPU_CTX.update(nxa=nxa, nya=nya, nxb=nxb, nyb=nyb, ca=np.stack([nxa, nya], 1), cb=np.stack([nxb, nyb], 1))
    csed.lib()


def _cpu_worker(job):
    """One shard of hypotheses on one host core: numpy eight-point fit per hypothesis
    (oracle/restatement.py: np.linalg.eig 9x9 + svd 3x3, as the reference) + exact C scorer
    (oracle/sed_exact.c) over all correspondences + the candidate/error rule."""
    from oracle import csed
    from oracle import restatement as o

    seed, hyps = job
    c = _CPU_CTX
    n = len(c["nxa"])
    rng = np.random.default_rng(seed)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(hyps)]).astype(np.int32)
    E = np.zeros((hyps, 9))
    valid = np.ones(hyps, dtype=np.uint8)
    for i in range(hyps):
        try:
            E[i] = o.eight_point(c["ca"][table[i]], c["cb"][table[i]]).reshape(9)
        except o.OracleEightPointError:
            valid[i] = 0
    cnt, s1, s2 = csed.score_batch(E, c["nxa"], c["nya"], c["nxb"], c["nyb"], THR, table=table, valid=valid, nthreads=1)
    err = np.where((cnt >= MIN_EXTRA) & (valid > 0), np.sqrt(s2 / (8 + cnt)), np.inf)
    j = int(np.argmin(err))
    return float(err[j]), j


class CpuPort:
    """The oracle port, hypothesis-sharded over all host cores (one process per core; the path has
    no exchange step other than picking the minimum-error winner)."""

    def __init__(self, K, x1, x2, procs: int):
        import multiprocessing as mp

        self.n = x1.shape[0]
        self.procs = procs
        self.pool = mp.get_context("fork").Pool(procs, initializer=_cpu_worker_init, initargs=(K, x1, x2))

    def rate(self, hyps: int, seed: int):
        per = max(1, hyps // self.procs)
        jobs = [(seed * 100003 + p, per) for p in range(self.procs)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, jobs)
        min(res)
        dt = time.perf_counter() - t0
        return per * self.procs, dt

    def close(self):
        self.pool.close()
        self.pool.join()


def time_true_reference(K, x1, x2, budget_s: float):
    """The UNMODIFIED reference (baseline/_ref or /root/reference, through oracle/reference_shims.py) on ONE core:
    estimate_essential_mat_with_ransac (lib/epipolar/epipolar_ransac.py:45-70) as is - list-of-Feature inputs, its own
    random.shuffle per iteration - on ALL correspondences of the workload for a bounded number of iterations, reported
    as hypothesis x correspondence evaluations per second (linear in H, so this is the rate of the full run)."""
    import random

    from oracle import reference_shims

    if not reference_shims.reference_available():
        return None
    ref = reference_shims.load()
    F, M = ref.feature.Feature, ref.matching.Match
    n = x1.shape[0]
    fa = [F(x=float(p[0]), y=float(p[1])) for p in x1]
    fb = [F(x=float(p[0]), y=float(p[1])) for p in x2]
    ms = [M(a_index=i, b_index=i) for i in range(n)]

    def run(iters):
        random.seed(5)
        t0 = time.perf_counter()
        try:
            ref.epipolar_ransac.estimate_essential_mat_with_ransac(
                K, fa, fb, ms, THR, min_num_extra_inliers=MIN_EXTRA,
                error_aggregation_method=ref.ransac.ErrorAggregationMethod.RMS, max_iterations=iters)
        except ValueError:
            pass  # "No model could be found" after so few iterations: the work was done all the same
        return time.perf_counter() - t0

    t1 = run(1)
    iters = int(max(2, min(32, budget_s / max(t1, 1e-3))))
    dt = run(iters)
    return {"value": iters * float(n - 8) / dt, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"the unmodified reference ({os.path.relpath(reference_shims.REFERENCE_ROOT, ROOT)}), "
                      f"{iters} iterations x all {n} correspondences incl. its shuffle, {dt:.1f} s; the full run is "
                      "this rate extrapolated linearly in the iteration count"}


def run_reference_arm(args):
    """--impl reference: the CPU implementation of the path on the host cores.  The reference is
    pure Python (2.5e4 evals/s on one core, SURVEY.md §6), has nothing to compile into oracle/_ref,
    and cannot travel to the GPU box; the arm times the oracle port (numpy eight-point fit + exact C
    scorer, one process per host core), which is ~4 orders of magnitude faster than the reference
    itself — a generous CPU baseline.  Each step = a bounded sample of the workload's hypotheses
    against ALL its correspondences."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from structure_from_motion_b200.scenes import make_scene

    wl = args.workload if args.workload in WORKLOADS else "config3"
    n, h, frac = WORKLOADS[wl]
    procs = os.cpu_count() or 1
    K, x1, x2, *_ = make_scene(n, frac, seed=0)
    port = CpuPort(K, x1, x2, procs)
    # size a step to ~args.cpu_step_seconds from a short calibration run (also the warm-up)
    hyps0 = 16 * procs
    done, dt = port.rate(hyps0, seed=999)
    for w in range(max(0, args.warmup - 1)):
        done, dt = port.rate(hyps0, seed=1000 + w)
    sample_h = args.cpu_sample_hyps or int(done / dt * args.cpu_step_seconds)
    sample_h = max(procs, min(sample_h, h))
    secs, evals = 0.0, 0.0
    for s in range(args.steps):
        done, dt = port.rate(sample_h, seed=s)
        secs += dt
        evals += float(done) * n
    port.close()
    value = evals / secs
    sample_h = done
    true_ref = None if args.no_true_reference else time_true_reference(K, x1, x2, args.true_reference_seconds)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{wl}: {n} correspondences x {h} hypotheses, 40% outliers, thr 1.5e-6, RMS, "
                               f"min_extra 10 (each step a sample of {sample_h} hypotheses x all correspondences)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port",
                         "sample": f"{sample_h} of {h} hypotheses x {n} correspondences per step, "
                                   f"{args.steps} steps, {secs:.1f} s"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if true_ref is not None:
        line["cpu_baseline"]["reference"] = true_ref
    else:
        line["cpu_baseline"]["reference"] = {"unavailable": "no baseline/_ref and no /root/reference on this box"}
    emit(line)
    return line


def cpu_baseline_subprocess(args, workload):
    """cpu_baseline leg of the native arm: the reference arm in a fresh process (no CUDA context to
    fork), one step of ~args.cpu_baseline_seconds."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--steps", "1",
           "--warmup", "1", "--cpu-step-seconds", str(args.cpu_baseline_seconds),
           "--true-reference-seconds", str(args.true_reference_seconds)]
    if args.no_true_reference:
        cmd.append("--no-true-reference")
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    for ln in reversed(out.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    raise RuntimeError("cpu baseline failed: " + out.stderr[-2000:])



# ----------------------------------------------------------------------------------------------
# sub-records of the default line: the north_star's other multi-GPU configurations + multi-rank parity
# ----------------------------------------------------------------------------------------------
def _timed(torch, dist, world, stream, barrier, flush_l2, steps, fn):
    """steps timed calls of fn(step) bracketed by barrier + synchronize, L2 flushed between steps; ms total, max over ranks."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    for s in range(steps):
        flush_l2()
        stream.synchronize()
        ev[s][0].record(stream)
        fn(s)
        ev[s][1].record(stream)
    barrier()
    ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.cpu()[0])


def run_extras(args, eng, world, rank, barrier, flush_l2, torch, dist, per_gpu_rate):
    """config3_strong (65 536 hypotheses split over the ranks), config5_strong (1M x 1M split over the ranks),
    config4_pairs (4 096 pairs split over the ranks, host buffers, pose + triangulation per pair) and parity_multi
    (the merged multi-rank result against a single-rank evaluation of the union of the hypotheses, untimed).
    ``per_gpu_rate`` = evaluations/s of ONE GPU on config 3 measured in this run (the denominator of `efficiency`)."""
    from structure_from_motion_b200 import _native, distributed
    from structure_from_motion_b200.scenes import make_scene

    out = {}
    stream = torch.cuda.current_stream()

    def sharded_step(h_rank, seed):
        if world == 1:
            eng.sample_device(seed, h_rank)
            best, *_rest = eng.two_view(THR, MIN_EXTRA, AGG, "min_error", 50.0, want_mask=False, want_sed=False)
            return int(best.index)
        r = distributed.two_view_sharded(THR, MIN_EXTRA, AGG, h_rank, seed, engine=eng, rank=rank, world=world, native=True)
        return int(r["index"])

    # ---- parity_multi: every rank must return the single-GPU answer for the union of the hypotheses ----
    if world > 1:
        ok = 1
        K, x1, x2, *_ = make_scene(100_000, 0.4, seed=0)
        eng.upload_pairs(x1, x2, K)
        hs = 4096
        for seed in (11, 12, 13):
            r = distributed.two_view_sharded(THR, MIN_EXTRA, AGG, hs, seed, engine=eng, rank=rank, world=world, native=True)
            eng.sample_device(seed, hs * world)  # the union on this one GPU (the sampler is keyed by the global index)
            best, _, _, poses, num, idx, okb, X = eng.two_view(THR, MIN_EXTRA, AGG, "min_error", 50.0, want_mask=False,
                                                                want_sed=False)
            same = (r["index"] == best.index and r["err"] == best.err and r["count"] == best.count_extra
                    and np.array_equal(r["E"].reshape(9), np.array(best.E)) and r["num_inliers"] == num
                    and np.array_equal(r["inlier_idx"], idx) and np.array_equal(r["pass_bits"], okb)
                    and np.array_equal(r["points"], X, equal_nan=True) and int(r["poses"].best) == int(poses.best)
                    and list(r["poses"].counts) == list(poses.counts))
            ok &= int(bool(same))
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out["parity_multi"] = bool(int(flag.cpu()[0]))
        out["parity_multi_note"] = (f"3 estimates, {hs} hypotheses per rank x {world} ranks over NCCL: (index, error, count, E, "
                                    "inlier list, cheirality bits, vote, triangulated points) bit-identical on EVERY rank "
                                    "to one GPU evaluating the union")

    # ---- latency of the small configurations (one GPU): config 2 resident, config 1 through the reference signature ----
    if world == 1:
        n2, h2, frac2 = WORKLOADS["config2"]
        K, x1, x2, *_ = make_scene(n2, frac2, seed=0)
        eng.upload_pairs(x1, x2, K)
        for w in range(3):
            sharded_step(h2, 800 + w)
        steps = 20
        ms = _timed(torch, dist, world, stream, barrier, flush_l2, steps, lambda s: sharded_step(h2, s))
        out["config2_latency"] = {"workload": f"{n2} correspondences x {h2} hypotheses + tail, resident, device sampler",
                                  "ms_per_estimate": ms / steps, "value": float(n2) * h2 * steps / (ms * 1e-3), "unit": UNIT,
                                  "steps": steps}
        import random

        from lib.common.feature import Feature
        from lib.epipolar.epipolar_ransac import estimate_essential_mat_with_ransac
        from lib.feature_matching.matching import Match
        from lib.ransac.ransac import ErrorAggregationMethod

        n1, h1 = 500, 1000
        K, x1, x2, *_ = make_scene(n1, 0.3, seed=0)
        fa = [Feature(x=float(p[0]), y=float(p[1])) for p in x1]
        fb = [Feature(x=float(p[0]), y=float(p[1])) for p in x2]
        mt = [Match(a_index=i, b_index=i) for i in range(n1)]

        def list_step():
            random.seed(5)
            return estimate_essential_mat_with_ransac(K, fa, fb, mt, THR, min_num_extra_inliers=MIN_EXTRA,
                                                      error_aggregation_method=ErrorAggregationMethod.RMS, max_iterations=h1)

        for w in range(3):
            e, pairs = list_step()
        t0 = time.perf_counter()
        steps = 20
        for s in range(steps):
            e, pairs = list_step()
        dt = (time.perf_counter() - t0) * 1e3 / steps
        golden = json.load(open(os.path.join(ROOT, "tests", "golden", "config1_known_answer.json")))
        coords = {(f.x, f.y): i for i, f in enumerate(fa)}
        out["config1_list_api"] = {
            "workload": f"BASELINE configs[0]: {n1} correspondences x {h1} iterations through estimate_essential_mat_with_ransac("
                        "list[Feature], list[Match]) with the CPython-exact sampler; host wall clock incl. marshalling",
            "ms_per_estimate": dt, "value": float(n1 - 8) * h1 / (dt * 1e-3), "unit": UNIT, "steps": steps,
            "parity_golden": bool(np.allclose(e, np.array(golden["E"]), rtol=1e-6, atol=1e-9)
                                  and [coords[(p[0].x, p[0].y)] for p in pairs] == golden["inlier_indices"]),
            "golden": "tests/golden/config1_known_answer.json (the unmodified reference: iteration 87, 23 inliers, same order)"}

    # ---- config3_strong: BASELINE configs[2] with its 65 536 hypotheses split over the ranks ----
    n, h, frac = WORKLOADS["config3"]
    K, x1, x2, *_ = make_scene(n, frac, seed=0)
    eng.upload_pairs(x1, x2, K)
    h_rank = h // world
    for w in range(3):
        sharded_step(h_rank, 500 + w)
    steps = max(5, min(args.steps, 20))
    ms = _timed(torch, dist, world, stream, barrier, flush_l2, steps, lambda s: sharded_step(h_rank, s))
    rate = float(n) * h_rank * world * steps / (ms * 1e-3)
    out["config3_strong"] = {"workload": f"{n} correspondences x {h} hypotheses split over {world} GPU(s) ({h_rank} each) + tail",
                             "ms_per_estimate": ms / steps, "value": rate, "unit": UNIT, "steps": steps, "scaling": "strong",
                             "efficiency_vs_one_gpu": rate / (world * per_gpu_rate)}

    # ---- config5_strong: 1M correspondences x 1M hypotheses split over the ranks ----
    n, h, frac = WORKLOADS["config5"]
    K, x1, x2, *_ = make_scene(n, frac, seed=0)
    eng.upload_pairs(x1, x2, K)
    h_rank = h // world
    sharded_step(h_rank, 600)
    steps = 2
    ms = _timed(torch, dist, world, stream, barrier, flush_l2, steps, lambda s: sharded_step(h_rank, s))
    rate = float(n) * h_rank * world * steps / (ms * 1e-3)
    out["config5_strong"] = {"workload": f"{n} correspondences x {h} hypotheses split over {world} GPU(s) ({h_rank} each) + tail",
                             "ms_per_estimate": ms / steps, "value": rate, "unit": UNIT, "steps": steps, "scaling": "strong",
                             "efficiency_vs_one_gpu": rate / (world * per_gpu_rate)}

    # ---- config4_pairs: 4 096 image pairs x 2 000 matches x 2 000 hypotheses, pair-sharded, host buffers ----
    P_total, n, h = 4096, 2000, 2000
    P = P_total // world
    base = make_scene(n, 0.4, seed=0)
    rng = np.random.default_rng(rank)
    pa = _native.pinned_empty((P * n, 2))
    pb = _native.pinned_empty((P * n, 2))
    for p in range(P):  # cheap per-pair variation of one scene (generation is not what is measured)
        perm = rng.permutation(n)
        pa[p * n:(p + 1) * n] = base[1][perm]
        pb[p * n:(p + 1) * n] = base[2][perm]
    offsets = np.arange(P + 1, dtype=np.int64) * n
    Ks = np.stack([base[0]] * P)
    # four to eight contexts, chunks of up to 512 pairs: H2D of one chunk, kernels of another and D2H of a third overlap
    # (profiles/r2_pair_pipeline_depth.txt: 4 096 pairs 0.634e12 with 4 contexts, 0.663e12 with 8 - one per chunk;
    #  0.56e12 with two contexts and 256-pair chunks)
    depth = int(min(8, max(4, P // 512)))
    chunk = int(min(512, max(128, P // depth)))
    pipe = distributed.PairPipeline(depth=depth)
    try:
        def pstep(seed):
            return pipe.batch_two_view(pa, pb, offsets, Ks, h, seed, THR, MIN_EXTRA, AGG, pair_id0=rank * P, chunk_pairs=chunk)

        for w in range(2):
            res = pstep(700 + w)
        steps = 5
        ms = _timed(torch, dist, world, stream, barrier, flush_l2, steps, pstep)
    finally:
        pipe.close()
    rate = float(P) * n * h * world * steps / (ms * 1e-3)
    out["config4_pairs"] = {"workload": f"{P_total} image pairs x {n} correspondences x {h} hypotheses, pair-sharded over {world} "
                                        f"GPU(s) ({P} each), HOST buffers (H2D inside the timed region), per pair: E, inlier "
                                        f"mask, 4-pose cheirality vote, triangulated inliers back on the host; {depth} contexts x "
                                        f"{chunk}-pair chunks",
                            "ms_per_step": ms / steps, "value": rate, "unit": UNIT, "steps": steps, "scaling": "strong",
                            "models_found": int((res["best_index"] >= 0).sum()), "pairs_per_s": P * world * steps / (ms * 1e-3),
                            "efficiency_vs_one_gpu_config3": rate / (world * per_gpu_rate)}
    return out


# ----------------------------------------------------------------------------------------------
# native arm
# ----------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    quiet_stdout()
    import torch
    import torch.distributed as dist

    from structure_from_motion_b200 import _native, distributed, two_view
    from structure_from_motion_b200.scenes import make_scene

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the native arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = _native.get_engine(local_rank)
    eng.set_score_variant(args.variant, args.hpt, args.group)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)  # torch's default stream: the flush, the timing events and the engine in one order
    if world > 1:
        # the data-path collective (one all-gather of the selection records) runs on the library's OWN communicator,
        # behind the C ABI; torch.distributed only does the plumbing here (rendezvous, barriers, max over ranks)
        uid = [_native.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.nccl_init(rank, world, uid[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def flush_l2():
        flush_buf.zero_()

    if args.workload == "config4":
        return bench_pairs(args, eng, world, rank, barrier, flush_l2, torch, dist)
    if args.workload == "frontend":
        return bench_frontend(args, eng, world, rank, barrier, flush_l2, torch, dist)
    if args.workload == "config1":
        return bench_config1(args, eng, world, rank, barrier, flush_l2, torch, dist)

    n, h_cfg, frac = WORKLOADS[args.workload]
    strong = args.workload == "config5"
    h_rank = h_cfg // world if strong else h_cfg
    K, x1, x2, *_ = make_scene(n, frac, seed=0)
    # pinned host copies for the e2e leg
    pa = _native.pinned_empty((n, 2))
    pb = _native.pinned_empty((n, 2))
    pa[...] = x1
    pb[...] = x2

    eng.upload_pairs(pa, pb, K)  # resident correspondences for the `value` leg
    fp64_peak_dfma = eng.measure_fp64_peak()

    def step_resident(seed):
        if world == 1:  # one GPU: no merge step, so selection -> mask -> pose vote -> triangulation is one C call
            eng.sample_device(seed, h_rank)
            res = eng.two_view(THR, MIN_EXTRA, AGG, "min_error", 50.0, want_mask=False, want_sed=False)
            best, num = res[0], res[4]
            if best.index < 0:
                raise RuntimeError("no model found")
            return {"index": int(best.index)}, num, res
        # several GPUs: records all-gathered device-to-device (the one collective), merged by a kernel, tail enqueued
        # behind it - the host synchronises once per estimate
        r = distributed.two_view_sharded(THR, MIN_EXTRA, AGG, h_rank, seed, engine=eng, rank=rank, world=world, native=True)
        if r["owner"] < 0:
            raise RuntimeError("no model found")
        return r, r["num_inliers"], r

    def step_e2e(seed):
        if world == 1:
            res = two_view.two_view_arrays(K, pa, pb, THR, MIN_EXTRA, AGG, h_rank, sampler="device", seed=seed,
                                           on_degenerate="skip", engine=eng)
            return res.points.shape[0]
        eng.upload_pairs(pa, pb, K)  # every rank uploads the (replicated) correspondences from its host buffers
        r = distributed.two_view_sharded(THR, MIN_EXTRA, AGG, h_rank, seed, engine=eng, rank=rank, world=world, native=True)
        mask, sed = eng.inlier_mask(THR)
        return r["num_inliers"]

    # ---- warm-up -------------------------------------------------------------------------------
    clocks = ClockSampler(local_rank)
    clocks.start()
    for w in range(max(args.warmup, 3)):
        step_resident(1000 + w)
    barrier()

    # ---- timed: resident ---------------------------------------------------------------------
    # the library's per-stage event timers are instrumentation (16 extra event records per step): OFF while `value` is
    # measured, ON in a second pass of the same steps that yields the stage breakdown and the k_score launch duration
    _, launches0 = eng.get_timing()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    num_inl = 0
    barrier()
    clocks.mark_begin()
    for s in range(args.steps):
        flush_l2()
        ev[s][0].record(stream)
        _, num_inl, last = step_resident(s)
        ev[s][1].record(stream)
    barrier()
    clocks.mark_end()
    clk = clocks.stop()
    _, launches1 = eng.get_timing()
    ms_total = sum(a.elapsed_time(b) for a, b in ev)
    eng.enable_timing(True)
    stage_ms = {}
    for s in range(args.steps):
        flush_l2()
        step_resident(s)
        t, _ = eng.get_timing()
        for k, v in t.items():
            stage_ms[k] = stage_ms.get(k, 0.0) + v
    barrier()
    eng.enable_timing(False)

    # ---- timed: end to end through the public API (host buffers) ---------------------------------
    e2e_ms = None
    if not args.no_e2e:
        for w in range(2):
            step_e2e(2000 + w)
        barrier()
        ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for s in range(args.steps):
            flush_l2()
            ev2[s][0].record(stream)
            m = step_e2e(s)
            ev2[s][1].record(stream)
        barrier()
        e2e_ms = sum(a.elapsed_time(b) for a, b in ev2)

    # ---- the same through the streaming API: two contexts, the transfers of estimate s+1 behind the kernels of s ----
    e2e_stream_ms = None
    if not args.no_e2e and world == 1:
        ts = two_view.TwoViewStream(depth=2, device=local_rank)
        ts.set_score_variant(args.variant, args.hpt, args.group)
        try:
            def submit(seed):
                return ts.submit(K, pa, pb, THR, MIN_EXTRA, AGG, h_rank, 50.0, seed=seed)

            for w in range(2):
                ts.result(submit(4000 + w))
            barrier()
            t0 = time.perf_counter()
            flush_l2()
            stream.synchronize()
            prev = submit(0)
            for s in range(1, args.steps):
                cur = submit(s)
                rs = ts.result(prev)
                prev = cur
            rs = ts.result(prev)
            torch.cuda.synchronize()
            e2e_stream_ms = (time.perf_counter() - t0) * 1e3
            stream_ok = bool(rs.points.shape[0] == rs.inlier_indices.shape[0] > 0)
        finally:
            ts.close()

    # ---- reported separately: the fp32 pre-filter variant (bit-identical results, see sfm_score.cuh) ---
    f32 = None
    if not args.no_fp32_variant:
        eng.set_score_variant("screen32")
        try:
            for w in range(3):
                step_resident(3000 + w)
            barrier()
            eng.enable_timing(True)
            ev3 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            sc = 0.0
            for s in range(args.steps):
                flush_l2()
                ev3[s][0].record(stream)
                r32, _, _ = step_resident(s)
                ev3[s][1].record(stream)
                t, _ = eng.get_timing()
                sc += t.get("score", 0.0)
            barrier()
            eng.enable_timing(False)
            f32 = (sum(a.elapsed_time(b) for a, b in ev3), sc, r32["index"])
        finally:
            eng.set_score_variant(args.variant, args.hpt, args.group)

    # ---- max over ranks ----------------------------------------------------------------------------
    vals = torch.tensor([ms_total, e2e_ms if e2e_ms is not None else 0.0, stage_ms.get("score", 0.0),
                         f32[0] if f32 else 0.0, f32[1] if f32 else 0.0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms_total, e2e_max, score_ms, f32_ms, f32_score_ms = (float(v) for v in vals.cpu())

    extras = {}
    if args.workload == "config3" and not args.no_extras:
        # one GPU's config-3 rate in this run: every rank did the full config 3 in the (weak) headline leg
        extras = run_extras(args, eng, world, rank, barrier, flush_l2, torch, dist,
                            float(n) * h_rank * args.steps / (ms_total * 1e-3))

    if rank == 0:
        evals_per_step = float(n) * h_rank * world
        value = evals_per_step * args.steps / (ms_total * 1e-3)
        score_ms_per_launch = score_ms / args.steps
        kern_evals = float(n) * h_rank / (score_ms_per_launch * 1e-3)
        fp64_peak_tflops = 2.0 * fp64_peak_dfma / 1e12
        achieved_tflops = kern_evals * FLOP_PER_EVAL / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "k_score_dram_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get(args.workload)
            except Exception:
                traffic = None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        algo_bytes = BYTES_PER_CORR * n * ((h_rank + 32 * args.hpt - 1) // (32 * args.hpt)) + 72.0 * h_rank  # one pass per hypothesis group
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": f"{args.workload}: {n} correspondences x {h_rank} hypotheses per GPU "
                            f"({h_rank * world} total), 40% outliers, thr 1.5e-6, RMS, min_extra 10, + cheirality "
                            f"vote + triangulation of the {num_inl} inliers",
                "sampler": "device (Philox)", "score_variant": args.variant + (" (device pilot: survivor rate 1.6 % -> 11-slot one-sided screen)" if args.variant == "auto" else ""), "hyps_per_thread": args.hpt, "group": args.group,
                "l2": "flushed (256 MiB memset) between timed steps",
                "parallelism": f"hypothesis-sharded x{world}, one 144 B/rank ncclAllGather issued by the library (C ABI) + merge kernel" if world > 1 else "single GPU",
            },
            "ms_per_estimate": ms_total / args.steps,
            "stage_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
            "kernel_evals_per_s": kern_evals,
            "roofline": {
                "bound": "fp64", "kernel": "k_score", "achieved": achieved_tflops, "peak": fp64_peak_tflops,
                "unit": "TFLOP/s", "frac": achieved_tflops / fp64_peak_tflops if fp64_peak_tflops else None,
                "traffic": traffic,
                "peak_source": "DFMA microbenchmark in this run (sfm_measure_fp64_peak); MEASURED_PEAKS.json has no fp64 entry",
                "algorithmic_flop_per_eval": FLOP_PER_EVAL,
                "executed_fp64_slots_per_eval": 21.0 if args.variant == "full" else 11.0,
                "fp64_pipe_busy_frac_est": kern_evals * (21.0 if args.variant == "full" else 11.0) / fp64_peak_dfma,
                "l2_to_smem_stream_gbs": algo_bytes / (score_ms_per_launch * 1e-3) / 1e9,
                "l2_to_smem_note": "32 B per correspondence per hypothesis-group pass, served by L2 (the working set is L2-resident); NOT HBM traffic",
                "dram_gbs": (traffic / (score_ms_per_launch * 1e-3) / 1e9) if traffic else None,
                "dram_note": "traffic = dram__bytes_read+write per k_score launch from the committed ncu --set full capture (profiles/k_score_dram_traffic.json), divided by this run's launch duration",
                "hbm_peak_gbs": peaks.get("hbm_gbs"),
            },
            "clocks": clk,
            "gpu_launches": launches1 - launches0,
        }
        if f32:
            line["fp32_prefilter"] = {
                "value": evals_per_step * args.steps / (f32_ms * 1e-3), "unit": UNIT, "ms_per_step": f32_ms / args.steps,
                "kernel_evals_per_s": float(n) * h_rank / (f32_score_ms / args.steps * 1e-3),
                "note": "score_variant screen32: the 11-slot screen in fp32 as a pre-filter (guard band 1.0316 thr + kappa32), "
                        "every survivor decided and summed by the exact fp64 scorer - results bit-identical to the fp64 "
                        "variants (tests/test_gpu_configs.py); NOT the headline value"}
        if e2e_ms is not None:
            d2h = 8 + 72 + 48 + n * 1 + n * 8 + num_inl * (8 + 1 + 24) + 392
            line["e2e"] = {"value": evals_per_step * args.steps / (e2e_max * 1e-3), "unit": UNIT,
                           "ms_per_step": e2e_max / args.steps,
                           "h2d_bytes_per_step": int(n * 32 + 72), "d2h_bytes_per_step": int(d2h),
                           "api": "two_view.two_view_arrays: one blocking call per estimate (upload, estimate, results back)"}
            if e2e_stream_ms is not None:
                line["e2e_stream"] = {"value": evals_per_step * args.steps / (e2e_stream_ms * 1e-3), "unit": UNIT,
                                      "ms_per_step": e2e_stream_ms / args.steps, "h2d_bytes_per_step": int(n * 32 + 72),
                                      "d2h_bytes_per_step": int(d2h), "timing": "host wall clock over all steps",
                                      "api": "two_view.TwoViewStream: back-to-back estimates from host buffers on two contexts - "
                                             "the H2D of estimate s+1 and the unpacking of s-1 overlap the kernels of s; every "
                                             "step's H2D and D2H are inside the timed region", "ok": stream_ok}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_subprocess(args, args.workload)
        line.update(extras)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, two_view_outputs(last))
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def bench_pairs(args, eng, world, rank, barrier, flush_l2, torch, dist):
    """config4: a batch of independent image pairs, sharded by pair, no communication."""
    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.scenes import make_scene

    P, n, h = args.pairs, 2000, 2000
    xs1, xs2, Ks = [], [], []
    base = make_scene(n, 0.4, seed=0)
    rng = np.random.default_rng(rank)
    for p in range(P):  # cheap per-pair variation of one scene (generation is not what is measured)
        perm = rng.permutation(n)
        xs1.append(base[1][perm])
        xs2.append(base[2][perm])
        Ks.append(base[0])
    pa = _native.pinned_empty((P * n, 2))
    pb = _native.pinned_empty((P * n, 2))
    pa[...] = np.concatenate(xs1)
    pb[...] = np.concatenate(xs2)
    offsets = np.arange(P + 1, dtype=np.int64) * n
    Ks = np.stack(Ks)
    stream = torch.cuda.current_stream()

    from structure_from_motion_b200.distributed import PairPipeline

    pipe = None if args.no_pipeline else PairPipeline(depth=2)

    def step(seed):
        if pipe is not None:  # H2D of one chunk of pairs overlaps the kernels of another (two contexts, two streams)
            return pipe.batch_ransac(pa, pb, offsets, Ks, h, seed, THR, MIN_EXTRA, AGG, pair_id0=rank * P)
        return eng.batch_ransac(pa, pb, offsets, Ks, h, seed, THR, MIN_EXTRA, AGG, pair_id0=rank * P)

    clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    clocks.start()
    for w in range(max(args.warmup, 3)):
        step(100 + w)
    barrier()
    if pipe is None:
        eng.enable_timing(True)
    count_launches = (lambda: pipe.launches()) if pipe is not None else (lambda: eng.get_timing()[1])
    l0 = count_launches()
    clocks.mark_begin()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stage = {}
    for s in range(args.steps):
        flush_l2()
        if pipe is not None:
            stream.synchronize()  # the pipeline's own streams do not wait for the flush on torch's stream
        ev[s][0].record(stream)
        out = step(s)             # returns when every result is back on the host
        ev[s][1].record(stream)
        if pipe is None:
            t, _ = eng.get_timing()
            for k, v in t.items():
                stage[k] = stage.get(k, 0.0) + v
    barrier()
    clocks.mark_end()
    clk = clocks.stop()
    l1 = count_launches()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    vals = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms = float(vals.cpu()[0])
    if rank == 0:
        evals = float(P) * n * h * world * args.steps
        found = int((out["best_index"] >= 0).sum())
        line = {
            "metric": METRIC, "value": evals / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"config4: {P} image pairs per GPU x {n} correspondences x {h} hypotheses, "
                                   f"pair-sharded, host buffers (H2D inside the timed region), models found {found}/{P}",
                       "pipeline": "one context" if pipe is None else "2 contexts x 4 chunks of pairs: H2D of a chunk overlaps the kernels of another",
                       "l2": "flushed between timed steps", "parallelism": f"pair-sharded x{world}, no collective"},
            "stage_ms_per_step": {k: v / args.steps for k, v in stage.items()},
            "clocks": clk,
            "gpu_launches": l1 - l0,
        }
        if args.dump_outputs:
            found = out["best_index"] >= 0  # a pair without a model has no E and an infinite error (best_index -1)
            dump_outputs(args.dump_outputs, dict(out, E=out["E"][found], best_err=out["best_err"][found]))
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def bench_config1(args, eng, world, rank, barrier, flush_l2, torch, dist):
    """--workload config1 (BASELINE.json configs[0], the reference's own CPU-runnable case): 500 correspondences, 30 %
    outliers, 1000 iterations through the REFERENCE SIGNATURE — lists of Feature / Match objects in, (E, list of
    inlier pairs) out, the CPython-exact sampler on the global ``random`` state.  Everything (marshalling, sampler, H2D,
    kernels, D2H, rebuilding the inlier list) is inside the timed region.  Ranks run independent replicas."""
    import random

    from lib.common.feature import Feature
    from lib.epipolar.epipolar_ransac import estimate_essential_mat_with_ransac
    from lib.feature_matching.matching import Match
    from lib.ransac.ransac import ErrorAggregationMethod
    from structure_from_motion_b200.scenes import make_scene

    n, h = 500, 1000
    K, x1, x2, *_ = make_scene(n, 0.3, seed=0)
    fa = [Feature(x=float(p[0]), y=float(p[1])) for p in x1]
    fb = [Feature(x=float(p[0]), y=float(p[1])) for p in x2]
    ms = [Match(a_index=i, b_index=i) for i in range(n)]

    def step():
        random.seed(5)
        return estimate_essential_mat_with_ransac(K, fa, fb, ms, THR, min_num_extra_inliers=MIN_EXTRA,
                                                  error_aggregation_method=ErrorAggregationMethod.RMS, max_iterations=h)

    clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    clocks.start()
    for _ in range(max(args.warmup, 3)):
        e, pairs = step()
    barrier()
    _, l0 = eng.get_timing()
    clocks.mark_begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush_l2()
        e, pairs = step()
    barrier()
    ms_total = (time.perf_counter() - t0) * 1e3
    clocks.mark_end()
    clk = clocks.stop()
    _, l1 = eng.get_timing()
    vals = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms_total = float(vals.cpu()[0])
    if rank == 0:
        evals = float(n - 8) * h * world * args.steps
        golden = json.load(open(os.path.join(ROOT, "tests", "golden", "config1_known_answer.json")))
        line = {
            "metric": METRIC, "value": evals / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"config1: {n} correspondences x {h} iterations, 30% outliers, thr 1.5e-6, RMS, min_extra 10, "
                                   "through estimate_essential_mat_with_ransac(list[Feature], list[Match]) with the CPython-exact "
                                   "sampler; wall clock incl. marshalling (this workload is host-bound: ~5e5 evaluations)",
                       "l2": "flushed between timed steps", "parallelism": f"{world} independent replicas"},
            "clocks": clk, "gpu_launches": l1 - l0,
            "parity": {"inliers": len(pairs), "E_matches_reference_1e-6": bool(np.allclose(e, np.array(golden["E"]), rtol=1e-6, atol=1e-9)),
                       "golden": "tests/golden/config1_known_answer.json (unmodified reference: iteration 87, 23 inliers)"},
        }
        line["e2e"] = {"value": line["value"], "unit": UNIT, "ms_per_step": line["ms_per_step"],
                       "h2d_bytes_per_step": n * 32 + h * 32 + 72, "d2h_bytes_per_step": n * 9 + 136}
        tp = os.path.join(ROOT, "profiles", "r1_true_reference_config1.json")
        if os.path.exists(tp):
            t = json.load(open(tp))
            line["cpu_baseline"] = {"value": t["evals_per_s"], "unit": UNIT, "cores": 1, "kind": "reference",
                                    "sample": f"the UNMODIFIED reference on this exact workload: {t['seconds']:.1f} s per estimate, "
                                              "recorded in the build container by tools/time_true_reference.py (the reference "
                                              "cannot travel to the GPU box)"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"E": e, "inlier_pairs": np.reshape([[a.x, a.y, b.x, b.y] for a, b in pairs], (-1, 4))})
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def bench_frontend(args, eng, world, rank, barrier, flush_l2, torch, dist):
    """--workload frontend (SURVEY.md §8(f) N1+N2, not the headline): the stages in front of the hot path at the
    sizes of apps/config/config.yaml — Harris corners (600 per image, 640x480) on both images + brute-force 9x9 NCC
    matching with ratio test and cross-check.  Host images in, host results out (the only API these stages have);
    image pairs are independent, so ranks simply process their own pairs."""
    from structure_from_motion_b200.scenes import make_image_pair

    img1, img2, *_ = make_image_pair(rank)
    stream = torch.cuda.current_stream()

    def step():
        c1, s1, _ = eng.harris_corners(img1, 600, 2, 0.04)
        c2, s2, _ = eng.harris_corners(img2, 600, 2, 0.04)
        bb, bs, keep, _ = eng.match_brute_force(img1, img2, c1, c2, kind="ncc", window=9, ratio_test=True, crosscheck=True,
                                                ratio_threshold=0.7)
        return c1, s1, c2, s2, bb, bs, keep

    clocks = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    clocks.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    _, l0 = eng.get_timing()
    clocks.mark_begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = 0.0
    for _ in range(args.steps):
        flush_l2()
        ev0.record(stream)
        c1, s1, c2, s2, bb, bs, keep = step()
        ev1.record(stream)
        ev1.synchronize()
        ms += ev0.elapsed_time(ev1)
    barrier()
    clocks.mark_end()
    clk = clocks.stop()
    _, l1 = eng.get_timing()
    vals = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    ms = float(vals.cpu()[0])
    if rank == 0:
        line = {
            "metric": "front-end image pairs/sec (2 x Harris 640x480 -> 600 corners, 600x600 9x9 NCC match)",
            "value": world * args.steps / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "frontend: rendered 640x480 uint8 image pair, 600 Harris corners per image, "
                                   f"9x9 NCC, ratio 0.7 + cross-check ({int(keep.sum())} matches kept), host buffers",
                       "l2": "flushed between timed steps", "parallelism": f"pair-sharded x{world}, no collective"},
            "clocks": clk, "gpu_launches": l1 - l0,
            "e2e": {"value": world * args.steps / (ms * 1e-3), "unit": "pairs/s",
                    "h2d_bytes_per_step": int(4 * img1.size + 2 * 16 * 600), "d2h_bytes_per_step": int(2 * 600 * 24 + 600 * 13)},
        }
        if not args.no_cpu_baseline:
            from oracle import front_end as fe

            t0 = time.perf_counter()
            o1, _, _, _ = fe.harris_corners_vectorised(img1, 600)
            o2, _, _, _ = fe.harris_corners_vectorised(img2, 600)
            t_h = time.perf_counter() - t0
            rows = 24  # a bounded sample of the 600 rows of the score matrix (Python loop, as the reference)
            t0 = time.perf_counter()
            fe.score_matrix(img1, img2, o1[:rows], o2, "ncc", 9)
            t_m = (time.perf_counter() - t0) * len(o1) / rows
            line["cpu_baseline"] = {"value": 1.0 / (t_h + t_m), "unit": "pairs/s", "cores": 1, "kind": "port",
                                    "sample": f"vectorised-numpy Harris on both images ({t_h:.2f} s) + {rows} of {len(o1)} rows "
                                              f"of the per-pair NCC loop, extrapolated ({t_m:.1f} s)"}
            line["parity"] = bool(np.array_equal(o1, c1) and np.array_equal(o2, c2))
        if args.dump_outputs:
            kept = np.flatnonzero(keep)  # (a, b, score) of every kept match, as the matcher's list of Match
            dump_outputs(args.dump_outputs, {"corners_a": c1, "corner_scores_a": s1, "corners_b": c2, "corner_scores_b": s2,
                                             "matches": np.stack([kept, bb[kept], bs[kept]], 1)})
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
