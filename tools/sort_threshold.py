"""One upload plus one estimate (device sampler, fit, K2, K3, tail) of a single pair, against the pair size: the cost
the upload-time sort of K2's copy adds (kK2SortMin in csrc/sfm_ransac.cu) against what the 9-slot screen saves.  Run it in
two trees and compare; prints the median wall time of 20 calls per (N, H) after 3 warm-up calls."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_scene  # noqa: E402

eng = _native.get_engine(0)
print("N        H        ms (upload + estimate, median of 20)")
for n in (32_768, 65_536, 131_072):
    K, x1, x2, *_ = make_scene(n, 0.4, seed=0)
    pa, pb = _native.pinned_empty((n, 2)), _native.pinned_empty((n, 2))
    pa[...] = x1
    pb[...] = x2
    for h in (16_384, 65_536):
        ts = []
        for s in range(23):
            t0 = time.perf_counter()
            eng.upload_pairs(pa, pb, K)
            eng.sample_device(s, h)
            res = eng.two_view(1.5e-6, 10, "rms", "min_error", 50.0, want_mask=False, want_sed=False)
            ts.append(time.perf_counter() - t0)
        print(f"{n:<8d} {h:<8d} {np.median(ts[3:]) * 1e3:.4f}")
