"""Small end-to-end case for compute-sanitizer: upload -> device sampler -> fit -> score (every variant)
-> select -> mask -> pose vote -> triangulation, plus a ragged batch.  usage: compute-sanitizer --tool memcheck python tools/sanitize_case.py"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from structure_from_motion_b200 import _native, two_view  # noqa: E402
from structure_from_motion_b200.scenes import make_scene  # noqa: E402

K, x1, x2, *_ = make_scene(3003, 0.4, seed=0)
eng = _native.get_engine(0)
for variant, hpt, g, thr in (("screen", 2, 16, 1.5e-6), ("screen32", 4, 8, 1.5e-6), ("full", 2, 16, 1.5e-6), ("auto", 2, 16, 1.5e-6),
                            ("full", 2, 16, 1e-3), ("auto", 2, 16, 0.5), ("screen", 2, 16, 1e-3)):
    eng.set_score_variant(variant, hpt, g)
    res = two_view.two_view_arrays(K, x1, x2, thr, 10, "rms", 1000, sampler="device", seed=1, on_degenerate="skip",
                                   engine=eng)
    print(variant, hpt, thr, res.ransac.best_index, len(res.inlier_indices), int(res.passing.sum()))
eng.set_score_variant("auto", 2, 16)
sizes = [700, 5, 0, 333, 64]
scenes = [make_scene(max(s, 8), 0.4, seed=10 + p) for p, s in enumerate(sizes)]
xa = np.concatenate([sc[1][:s] for sc, s in zip(scenes, sizes)])
xb = np.concatenate([sc[2][:s] for sc, s in zip(scenes, sizes)])
off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
out = eng.batch_ransac(xa, xb, off, np.stack([K] * len(sizes)), 300, 3, 1.5e-6, 10, "rms")
print("batch", out["best_index"].tolist())
