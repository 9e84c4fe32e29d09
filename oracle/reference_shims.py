"""TEST INFRASTRUCTURE ONLY — load the UNMODIFIED reference behind import shims.

The reference (Bazs/structure_from_motion) is pure Python.  It lives at ``/root/reference`` in the
build container; ``baseline/install_reference.py`` pip-installs it, unmodified, into the git-ignored
``baseline/_ref/`` so that a copy travels to the GPU box.  This loader is used (a) by
``tests/golden/make_golden.py`` to generate the committed golden vectors, which pin
``oracle/restatement.py`` and ``oracle/front_end.py`` against the real thing, and (b) by
``bench.py``'s CPU legs, which time the reference itself beside the GPU.

Four shims are needed because of dependency drift (SURVEY.md §8(c)); none of them
touches hot-path arithmetic:

* ``transforms3d.affines.compose``  — not installed; only call site is
  lib/transforms/transforms.py:30 with unit zooms.
* ``np.Infinity``                   — removed in numpy 2 (lib/feature_matching/matching.py:20).
* ``matplotlib`` / ``tkinter``      — only needed by the reference's *tests*.

The reference modules are imported under a private package name (``_sfm_reference``)
so that they never collide with this repository's own drop-in ``lib`` package.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))
_PKG = "_sfm_reference"


def _find_root() -> str:
    """SFM_REFERENCE_ROOT, else baseline/_ref (the pip-staged copy that travels to the GPU box, see
    baseline/install_reference.py), else /root/reference (build container)."""
    cands = [os.environ.get("SFM_REFERENCE_ROOT"), os.path.join(os.path.dirname(_HERE), "baseline", "_ref"),
             "/root/reference"]
    for c in cands:
        if c and os.path.isfile(os.path.join(c, "lib", "ransac", "ransac.py")):
            return c
    return "/root/reference"


REFERENCE_ROOT = _find_root()


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "lib", "ransac", "ransac.py"))


def _install_shims() -> None:
    import numpy as np

    if not hasattr(np, "Infinity"):
        np.Infinity = np.inf  # matching.py:20
    if "transforms3d" not in sys.modules:
        t3d = types.ModuleType("transforms3d")
        aff = types.ModuleType("transforms3d.affines")

        def compose(T, R, Z, S=None):  # transforms.py:30 — Z is always ones(3)
            A = np.eye(4)
            A[:3, :3] = np.asarray(R) @ np.diag(np.asarray(Z, dtype=float))
            A[:3, 3] = np.asarray(T)
            return A

        aff.compose = compose
        t3d.affines = aff
        sys.modules["transforms3d"] = t3d
        sys.modules["transforms3d.affines"] = aff


def load():
    """Return a namespace with the reference's hot-path modules.

    Attributes: ransac, epipolar_ransac, eight_point, sed, triangulation, feature,
    matching, transforms.
    """
    if not reference_available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    _install_shims()
    if _PKG + ".loaded" in sys.modules:
        return sys.modules[_PKG + ".loaded"]

    # Temporarily make `lib` resolve to the reference tree, import, then restore.
    saved = {k: v for k, v in sys.modules.items() if k == "lib" or k.startswith("lib.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        mods = {}
        for short, name in [
            ("feature", "lib.common.feature"),
            ("matching", "lib.feature_matching.matching"),
            ("transforms", "lib.transforms.transforms"),
            ("triangulation", "lib.epipolar.triangulation"),
            ("sed", "lib.epipolar.sed"),
            ("eight_point", "lib.epipolar.eight_point"),
            ("ransac", "lib.ransac.ransac"),
            ("epipolar_ransac", "lib.epipolar.epipolar_ransac"),
            ("ncc", "lib.feature_matching.ncc"),
            ("ssd", "lib.feature_matching.ssd"),
            ("fm_util", "lib.feature_matching.util"),
            ("correlate", "lib.common.correlate"),
            ("harris", "lib.harris.harris_detector"),
            ("gaussian", "lib.blur.gaussian"),
        ]:
            mods[short] = importlib.import_module(name)
        for m in mods.values():
            assert m.__file__.startswith(REFERENCE_ROOT), m.__file__
    finally:
        sys.path.remove(REFERENCE_ROOT)
        # move the reference's modules out of the `lib` namespace
        for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
            sys.modules[_PKG + "." + k] = sys.modules.pop(k)
        sys.modules.update(saved)

    ns = types.SimpleNamespace(**mods)
    # silence the tqdm bar of ransac.py:61 without touching the code
    try:
        import tqdm as _tqdm

        class _Quiet:
            @staticmethod
            def tqdm(it, *a, **k):
                return it

        ns.ransac.tqdm = _Quiet
        ns.matching.tqdm = _Quiet

        class _QuietH(_Quiet):
            @staticmethod
            def trange(n, *a, **k):
                return range(n)

        ns.harris.tqdm = _QuietH
    except Exception:
        pass
    sys.modules[_PKG + ".loaded"] = ns
    return ns
