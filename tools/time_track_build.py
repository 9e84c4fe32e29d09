"""Time the track building from pairwise matches (sfm_build_tracks) on the GPU.

Workloads:
  W       make_match_graph(10^6 points, 64 views, span 3, 2 % wrong matches, 25 % distractors): about 6.6 M features
          and 10^7 matches over 189 pairs; next to it sfm_triangulate_tracks on W's ok tracks (threshold 4 px^2,
          refinement off), the bar being build device time <= 25 % of the triangulation's kernel time.
  chain   10^6 features alternating between two views, joined into one chain by 10^6 - 1 matches in random order (one
          conflicting track: the longest finds the union-find can meet).
Kernel times: the device duration of every kernel of the call (CUPTI activity records through torch.profiler, in a run
of their own), summed per call and per kernel name (mean over the steps: the radix sort launches its one-sweep kernel
once per 8-bit digit), with the 126 MB L2 overwritten by a 512 MB device fill between calls.  Call times: the median of
a host clock around each synchronising call (host validation and the copies included), profiler off.  Compulsory bytes:
the matches read once (8 B each) and the outputs written once (offsets 8 B and status 4 B per track, view and feature
4 B per observation, track 4 B per feature), over the build's device time, against 7.7 TB/s.  The host's
scipy.sparse.csgraph.connected_components on the same edges is timed for the record.  Writes one JSON object with the
GPU's name, power limit and maximum SM clock read in the same run.

    python tools/time_track_build.py [--steps 10] [--warmup 2] [--out profiles/track_build_time_b200.json]
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

HBM = 7.7e12
BUILD = ("k_tb_", "DeviceRadixSort", "DeviceScan")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import scipy.sparse as sp
    import torch
    from scipy.sparse.csgraph import connected_components

    from oracle import track_build as otb
    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.multiview import build_tracks_arrays, triangulate_tracks_arrays
    from structure_from_motion_b200.scenes import make_match_graph

    if not torch.cuda.is_available():
        raise SystemExit("time_track_build.py needs a CUDA device")
    eng = _native.get_engine(0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    out = {"gpu": gpu_info(0), "steps": args.steps, "hbm_bytes_per_s": HBM}

    def measure(call, keys):
        for _ in range(args.warmup):
            call()
        host = []
        for _ in range(args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call()
            host.append(time.perf_counter() - t0)
        per = {}
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                flush.fill_(1)
                torch.cuda.synchronize()
                call()
            torch.cuda.synchronize()
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and any(k in ev.name for k in keys):
                name = next(k for k in ("k_tb_init", "k_tb_hook", "k_tb_compress", "k_tb_flag", "k_tb_select",
                                        "k_tb_heads", "k_tb_obs", "k_tb_status", "k_track_views", "k_track_pairs",
                                        "k_track_solve", "DeviceRadixSort", "DeviceScan") if k in ev.name)
                t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                per[name] = per.get(name, 0.0) + t
        kern = {k: v / args.steps for k, v in sorted(per.items())}
        return {"call_ms_median": 1e3 * float(np.median(host)),
                "call_ms_spread": [1e3 * float(np.min(host)), 1e3 * float(np.max(host))],
                "kernel_us_mean_per_call": kern, "device_us_per_call": float(sum(kern.values()))}

    def arrays(features, pairs, matches):
        fo = np.zeros(len(features) + 1, dtype=np.int64)
        np.cumsum([len(f) for f in features], out=fo[1:])
        mo = np.zeros(len(matches) + 1, dtype=np.int64)
        np.cumsum([len(m) for m in matches], out=mo[1:])
        return fo, np.asarray(pairs, dtype=np.int32), mo, np.concatenate(matches).astype(np.int32)

    def workload(name, fo, pv, mo, m):
        res = {}

        def call():
            res["r"] = eng.build_tracks(fo, pv, mo, m)

        r = measure(call, BUILD)
        offsets, status, view, feature, track = res["r"]
        ref = otb.build_tracks(fo, pv, mo, m)
        same = all(np.array_equal(a, ref[k]) for a, k in zip(res["r"], ("offsets", "status", "view", "feature", "track")))
        N, E, T, M = int(fo[-1]), int(mo[-1]), len(offsets) - 1, len(view)
        nbytes = 8 * E + 12 * T + 8 + 8 * M + 4 * N
        e = otb.global_edges(fo, pv, mo, m)
        g = sp.coo_matrix((np.ones(E, dtype=np.int8), (e[:, 0], e[:, 1])), shape=(N, N)).tocsr()
        t0 = time.perf_counter()
        connected_components(g, directed=False)
        scipy_ms = 1e3 * (time.perf_counter() - t0)
        r.update({"features": N, "matches": E, "pairs": len(pv), "tracks": T, "observations": M,
                  "status_counts": {s: int((status == k).sum()) for k, s in _native.BUILT_TRACK_STATUS.items()},
                  "equal_to_oracle": bool(same), "compulsory_bytes": nbytes,
                  "compulsory_bytes_per_s": nbytes / (r["device_us_per_call"] * 1e-6),
                  "share_of_hbm": nbytes / (r["device_us_per_call"] * 1e-6) / HBM,
                  "scipy_connected_components_ms_on_csr": scipy_ms})
        print(name, json.dumps(r), flush=True)
        return r

    t0 = time.perf_counter()
    gw = make_match_graph(1_000_000, 64, 0, span=3, wrong_frac=0.02, distractor_frac=0.25)
    out["W_generation_s"] = time.perf_counter() - t0
    fo, pv, mo, m = arrays(gw.features, gw.pairs, gw.matches)
    out["W"] = workload("W", fo, pv, mo, m)
    ok = build_tracks_arrays(gw.features, gw.pairs, gw.matches, engine=eng).ok()

    def call_tri():
        triangulate_tracks_arrays(gw.K, gw.R, gw.t, ok.offsets, ok.view, ok.x, 4.0, engine=eng)

    tri = measure(call_tri, ("k_track_",))
    tri.update({"tracks": len(ok.offsets) - 1, "observations": len(ok.view)})
    out["W_triangulate_ok_tracks"] = tri
    print("W_triangulate", json.dumps(tri), flush=True)
    out["bar"] = {"build_device_us": out["W"]["device_us_per_call"], "triangulate_kernels_us": tri["device_us_per_call"],
                  "ratio": out["W"]["device_us_per_call"] / tri["device_us_per_call"], "limit": 0.25}

    n = 1_000_000
    rng = np.random.default_rng(1)
    k = np.arange(n - 1)
    # feature k of the chain is local k // 2 of view k % 2; pair (0, 1) holds every edge
    i = np.where(k % 2 == 0, k // 2, (k + 1) // 2)
    j = np.where(k % 2 == 0, k // 2, (k - 1) // 2)
    chain = np.column_stack([i, j])[rng.permutation(n - 1)]
    fo = np.array([0, (n + 1) // 2, n], dtype=np.int64)
    out["chain"] = workload("chain", fo, np.array([[0, 1]], dtype=np.int32), np.array([0, n - 1], dtype=np.int64),
                            chain.astype(np.int32))
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
