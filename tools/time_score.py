"""Time the scoring kernel alone (CUDA events inside the library) for a threshold / variant sweep.
usage: python tools/time_score.py [config3] ; prints ms per launch"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_scene  # noqa: E402

n, h = {"config2": (10_000, 16_384), "config3": (100_000, 65_536)}[sys.argv[1] if len(sys.argv) > 1 else "config3"]
K, x1, x2, *_ = make_scene(n, 0.4, seed=0)
eng = _native.get_engine(0)
eng.upload_pairs(x1, x2, K)
eng.sample_device(0, h)
eng.fit(want_E=False)
eng.enable_timing(True)
cfgs = [("screen32", 4, 8), ("screen32", 2, 16), ("screen", 2, 16), ("full", 2, 16), ("auto", 2, 16)]
if len(sys.argv) > 2:
    cfgs = [tuple([sys.argv[2], int(sys.argv[3]), int(sys.argv[4])])]
for thr in (1.5e-6, 1.5e-8, 1e-30):
    for v, hpt, g in cfgs:
        eng.set_score_variant(v, hpt, g)
        ts = []
        for r in range(4):
            eng.score(thr, 10, "rms", want_arrays=False)
            t, _ = eng.get_timing()
            ts.append(t["score"])
        print(f"thr {thr:8.1e} {v:12s} hpt {hpt} G {g}: score {min(ts[1:]):7.3f} ms  -> {n * h / min(ts[1:]) * 1e3:.3e} evals/s")
