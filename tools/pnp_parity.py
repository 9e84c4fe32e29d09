"""Compare the PnP path of two builds of libsfm_b200.so bit for bit.

    SFM_B200_LIB=/path/to/other/libsfm_b200.so python tools/pnp_parity.py dump A.npz
    python tools/pnp_parity.py dump B.npz
    python tools/pnp_parity.py compare A.npz B.npz

``dump`` runs, on cuda:0, two make_pnp_scene estimates (2 049 records x 4 096 and 100 000 x 8 192 device-sampled
hypotheses, 40 % outliers, 1 px noise, threshold 4 px^2) under three aggregation / selection pairs, and fits 600
random samples of make_pnp_samples (1 px noise) one at a time.  It saves every pose, validity flag, count, mask,
per-record error and aggregated error.  ``compare`` prints how many of the saved arrays differ in any bit and which.
"""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def dump(path: str) -> None:
    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.scenes import make_pnp_samples, make_pnp_scene

    eng = _native.Engine(0)
    out = {}
    for seed, n, h in ((1, 2049, 4096), (2, 100_000, 8192)):
        K, X, x, R, t, _ = make_pnp_scene(n, 0.4, seed=seed, noise_px=1.0)
        eng.upload_pnp(X, x, K)
        eng.sample_device(seed, h)
        for j, (agg, sel) in enumerate((("rms", "min_error"), ("sum", "msac"), ("mean", "max_inliers"))):
            best, Rt_w, mask, err, cnt, err_h = eng.ransac_pnp(4.0, 0.0, agg, sel, want_arrays=True)
            models, valid = eng.get_pnp_models()
            for k, v in dict(best=np.int64(best.index), Rt=Rt_w, mask=mask, err=err, cnt=cnt, err_h=err_h,
                             models=models, valid=valid).items():
                out[f"scene{seed}_{agg}_{sel}_{k}"] = np.asarray(v)
    one = np.array([[0, 1, 2, 3, 0, 1, 2, 3]], dtype=np.int32)
    for i, (K, Xs, xs, R, t) in enumerate(make_pnp_samples(600, seed=5, noise_px=1.0)):
        eng.upload_pnp(Xs, xs, K)
        eng.set_table(one)
        Rt, v = eng.fit_pnp()
        out[f"sample{i}_Rt"], out[f"sample{i}_valid"] = Rt, v
    np.savez(path, **out)


def compare(a_path: str, b_path: str) -> int:
    a, b = np.load(a_path), np.load(b_path)
    keys = sorted(set(a.files) | set(b.files))
    diff = [k for k in keys if k not in a.files or k not in b.files or a[k].tobytes() != b[k].tobytes()]
    print(f"arrays: {len(keys)}  differing in any bit: {len(diff)}", *diff[:50])
    return 1 if diff else 0


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "dump":
        dump(sys.argv[2])
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        raise SystemExit(__doc__)
