"""Dump every output of the homography path on a seeded planar scene, and compare two such dumps bit for bit.

--dump DIR runs ransac_homography_arrays and two_view_homography_arrays with the reference, table and device samplers
on make_planar_scene(N, 0.4, seed=0) at the size of tools/time_homography.py (N = 100 000, H = 65 536, threshold
4 px^2, 30 000 extra inliers, RMS) and saves each field as DIR/<sampler>_<call>_<field>.npy.  The global random state
after each call is saved too: the reference sampler must advance it exactly as the reference does.  The table sampler
gets the device sampler's rows, first four columns only (the [H,4] form).

--compare A B checks that two directories hold the same .npy files with the same dtype, shape and bytes (NaN payloads
and signed zeros included); bench.py --dump-outputs directories compare the same way.  Exit status 1 on any difference.

    python tools/homography_outputs.py --dump DIR [--n N] [--h H]
    python tools/homography_outputs.py --compare A B
"""
from __future__ import annotations

import argparse
import dataclasses
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

THR, MIN_EXTRA = 4.0, 30_000


def _fields(prefix, obj, out):
    for f in dataclasses.fields(obj):
        v = getattr(obj, f.name)
        if dataclasses.is_dataclass(v):
            _fields(f"{prefix}_{f.name}", v, out)
        elif f.name == "candidates":
            for i, cand in enumerate(v):
                for j, a in enumerate(cand):
                    out[f"{prefix}_cand{i}_{j}"] = np.asarray(a)
        else:
            out[f"{prefix}_{f.name}"] = np.asarray(v)


def dump(directory, n, h):
    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.homography import ransac_homography_arrays, two_view_homography_arrays
    from structure_from_motion_b200.scenes import make_planar_scene

    K, x1, x2, _, _ = make_planar_scene(n, 0.4, seed=0)
    eng = _native.get_engine()
    eng.upload_pairs(x1, x2, np.eye(3))
    eng.sample_device(7, h)
    table = eng.get_table()[:, :4].copy()
    out = {}
    for sampler in ("reference", "table", "device"):
        kw = dict(sampler=sampler, seed=3, engine=eng, table=table if sampler == "table" else None)
        random.seed(11)
        res = ransac_homography_arrays(x1, x2, THR, MIN_EXTRA, "rms", h, **kw)
        _fields(f"{sampler}_ransac", res, out)
        out[f"{sampler}_ransac_random_state"] = np.array(random.getstate()[1], dtype=np.uint64)
        random.seed(11)
        tv = two_view_homography_arrays(K, x1, x2, THR, MIN_EXTRA, "rms", h, **kw)
        _fields(f"{sampler}_two_view", tv, out)
        out[f"{sampler}_two_view_random_state"] = np.array(random.getstate()[1], dtype=np.uint64)
    os.makedirs(directory, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(directory, k + ".npy"), a)
    print(f"{len(out)} arrays written to {directory}")


def compare(a, b) -> bool:
    names = sorted(set(os.listdir(a)) | set(os.listdir(b)))
    bad = []
    for name in names:
        pa, pb = os.path.join(a, name), os.path.join(b, name)
        if not (os.path.exists(pa) and os.path.exists(pb)):
            bad.append(f"{name}: missing on one side")
            continue
        x, y = np.load(pa), np.load(pb)
        if x.dtype != y.dtype or x.shape != y.shape or x.tobytes() != y.tobytes():
            bad.append(f"{name}: differs ({x.dtype}{x.shape} vs {y.dtype}{y.shape})")
    print(f"{a} vs {b}: {len(names)} arrays, {len(names) - len(bad)} bit-identical")
    for line in bad:
        print("  " + line)
    return not bad


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump", metavar="DIR")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--h", type=int, default=65_536)
    args = ap.parse_args()
    if args.dump:
        dump(args.dump, args.n, args.h)
    if args.compare and not compare(*args.compare):
        sys.exit(1)


if __name__ == "__main__":
    main()
