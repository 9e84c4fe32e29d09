"""Headless two-view structure-from-motion demo: the reference's apps/sfm.py:34-215 without GUI, hydra or the
Middlebury download (SURVEY.md §8(f) N3).  Same stages, same ``lib.*`` imports, same configuration keys:

    Harris corners (:64-71) -> brute-force NCC matching, ratio test + cross-check (:73-87) -> score filter (:107) ->
    RANSAC essential matrix (:110-119) -> relative pose (:133-138) [-> OpenCV cross-check :140-161] ->
    triangulation of the pairs that pass the cheirality vote (:165-186) [-> OpenCV cross-check :188-202]

Every numeric stage runs in libsfm_b200.so on the GPU (no CPU fallback).

    python apps/sfm.py --synthetic 0                      # rendered image pair with known pose
    python apps/sfm.py --image1 a.npy --image2 b.npy --camera-matrix K.npy [--config apps/config/config.yaml]
    python apps/sfm.py --dataset-dir data/temple --index1 170 --index2 172      # Middlebury layout, as the reference

--model auto estimates both the essential matrix and a homography from the filtered matches and keeps the pose of the
one that ORB-SLAM's score ratio picks (structure_from_motion_b200.model_selection), so that planar scenes and
rotation-only pairs get a pose too; --synthetic SEED --planar renders a scene that is one plane.

--refine N polishes the RANSAC winner (both winners with --model auto) by least squares over its inliers, at most N
Levenberg-Marquardt iterations on the device, before the pose; the essential path then runs through the array API
(two_view_arrays) on the same matches and the same global random stream.  The JSON output gains a "refinement" record.
"""
from __future__ import annotations

import argparse
import dataclasses
import functools
import json
import logging
import os
import sys
import time
from typing import List

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from lib.common import feature  # noqa: E402
from lib.data_utils.middlebury_utils import load_camera_k_r_t  # noqa: E402
from lib.epipolar.eight_point import recover_r_t_from_e  # noqa: E402
from lib.epipolar.epipolar_ransac import estimate_essential_mat_with_ransac  # noqa: E402
from lib.epipolar.triangulation import triangulate_points  # noqa: E402
from lib.feature_matching import matching, ncc  # noqa: E402
from lib.harris import harris_detector as harris  # noqa: E402
from lib.ransac.ransac import ErrorAggregationMethod  # noqa: E402
from lib.transforms.transforms import Transform3D  # noqa: E402

DEFAULT_CONFIG = {
    "image_downscale_factor": 1.0,
    "num_harris_corners": 600,
    "ncc_window_size": 9,
    "ratio_test_threshold": 0.7,
    "match_score_threshold": 0.3,
    # homography_inlier_threshold: symmetric transfer error in px^2 (--model auto only; not a key of the reference)
    "ransac": {"sed_inlier_threshold": 1.5e-6, "min_num_extra_inliers": 10, "max_iterations": 2000,
               "homography_inlier_threshold": 4.0},
}


@dataclasses.dataclass
class SfmResult:
    corners_1: List[feature.Feature]
    corners_2: List[feature.Feature]
    matches: List[matching.Match]
    e: np.ndarray
    inlier_feature_pairs: list
    r: np.ndarray
    t: np.ndarray
    inlier_mask: np.ndarray
    cam2_T_cam1: Transform3D
    world_points: np.ndarray
    seconds: dict
    model: str = "essential"          # "homography" when --model auto picked it; e then holds H
    homography_score_ratio: float = None  # S_H / (S_H + S_E) (--model auto)
    rotation_only: bool = False
    refinement: dict = None           # --refine: the report of the refined winner (the chosen one with --model auto)


def load_config(path=None, **overrides):
    cfg = json.loads(json.dumps(DEFAULT_CONFIG))
    if path:
        import yaml

        with open(path) as f:
            loaded = yaml.safe_load(f) or {}
        cfg["ransac"].update(loaded.pop("ransac", {}))
        cfg.update(loaded)
    for k, v in overrides.items():
        if k in cfg["ransac"]:
            cfg["ransac"][k] = v
        else:
            cfg[k] = v
    return cfg


def _create_score_function(image_a, image_b, full_score_function):
    """apps/sfm.py:266-277."""

    def ssd_score(feature_a: feature.Feature, feature_b: feature.Feature) -> float:
        return full_score_function(image_a, image_b, feature_a, feature_b)

    return ssd_score


def _filter_matches(matches: List[matching.Match], score_threshold: float) -> List[matching.Match]:
    """apps/sfm.py:280-296: drop the matches whose score is above the threshold."""
    return [m for m in matches if not (m.match_score > score_threshold)]


def _match_arrays(image_1_corners, image_2_corners, matches):
    pts_a = np.array([[image_1_corners[m.a_index].x, image_1_corners[m.a_index].y] for m in matches],
                     dtype=np.float64).reshape(-1, 2)
    pts_b = np.array([[image_2_corners[m.b_index].x, image_2_corners[m.b_index].y] for m in matches],
                     dtype=np.float64).reshape(-1, 2)
    return pts_a, pts_b


def _report(refinement):
    if refinement is None:
        return None
    return dict(status=refinement.status, iterations=refinement.iterations, rejected=refinement.rejected,
                num=refinement.num, cost_ransac=refinement.cost_ransac, cost_start=refinement.cost_start,
                cost_final=refinement.cost_final)


def _run_selected(image_1_corners, image_2_corners, matches, camera_matrix, cfg, secs, refine=0) -> SfmResult:
    """--model auto: both models on the filtered matches, the pose and points of the one the score ratio picks."""
    from structure_from_motion_b200.model_selection import two_view_select_arrays

    logging.info("Estimating the Essential Matrix and a Homography")
    t0 = time.perf_counter()
    pts_a, pts_b = _match_arrays(image_1_corners, image_2_corners, matches)
    rc = cfg["ransac"]
    sel = two_view_select_arrays(camera_matrix, pts_a, pts_b, rc["sed_inlier_threshold"],
                                 rc["homography_inlier_threshold"], rc["min_num_extra_inliers"],
                                 ErrorAggregationMethod.RMS, rc["max_iterations"], refine_iterations=refine)
    secs["two_view"] = time.perf_counter() - t0
    logging.info("Model: %s (homography score ratio %.3f)", sel.model, sel.scores.ratio_h)
    win = sel.essential if sel.model == "essential" else sel.homography
    model = win.ransac.E if sel.model == "essential" else win.ransac.H
    if win.refinement is not None:
        model = win.refinement.model
    pairs = [(image_1_corners[matches[int(i)].a_index], image_2_corners[matches[int(i)].b_index])
             for i in sel.inlier_indices]
    return SfmResult(image_1_corners, image_2_corners, matches, model, pairs, sel.R, sel.t, np.flatnonzero(sel.passing),
                     Transform3D.from_rmat_t(sel.R, sel.t), sel.points[sel.passing], secs, model=sel.model,
                     homography_score_ratio=sel.scores.ratio_h, rotation_only=sel.rotation_only,
                     refinement=_report(win.refinement))


def _run_refined_essential(image_1_corners, image_2_corners, matches, camera_matrix, cfg, secs, refine) -> SfmResult:
    """--refine with the essential path: RANSAC E (reference sampler on the global random state, as the list API),
    least-squares refinement over its inliers, then the pose vote and triangulation of the refined E."""
    from structure_from_motion_b200.two_view import two_view_arrays

    logging.info("Estimating and refining the Essential Matrix")
    t0 = time.perf_counter()
    pts_a, pts_b = _match_arrays(image_1_corners, image_2_corners, matches)
    rc = cfg["ransac"]
    tv = two_view_arrays(camera_matrix, pts_a, pts_b, rc["sed_inlier_threshold"], rc["min_num_extra_inliers"],
                         ErrorAggregationMethod.RMS, rc["max_iterations"], refine_iterations=refine)
    secs["two_view"] = time.perf_counter() - t0
    logging.info("Refinement: %s after %d iterations, cost %.3e -> %.3e", tv.refinement.status, tv.refinement.iterations,
                 tv.refinement.cost_start, tv.refinement.cost_final)
    pairs = [(image_1_corners[matches[int(i)].a_index], image_2_corners[matches[int(i)].b_index])
             for i in tv.inlier_indices]
    return SfmResult(image_1_corners, image_2_corners, matches, tv.refinement.model, pairs, tv.R, tv.t,
                     np.flatnonzero(tv.passing), Transform3D.from_rmat_t(tv.R, tv.t), tv.points[tv.passing], secs,
                     refinement=_report(tv.refinement))


def run_sfm(image_1_gray: np.ndarray, image_2_gray: np.ndarray, camera_matrix: np.ndarray, cfg=None,
            check_opencv: bool = False, model: str = "essential", refine: int = 0) -> SfmResult:
    """model "essential": the reference's path.  "auto": the essential matrix and a homography, the pose of the one the
    score ratio picks (the OpenCV cross-checks belong to the essential path and are not run).  refine > 0: the winner
    is refined over its inliers before the pose (the essential path then goes through two_view_arrays; the OpenCV
    cross-checks are not run)."""
    cfg = cfg or load_config()
    secs = {}

    def timed(name, t0):
        secs[name] = time.perf_counter() - t0

    logging.info("Extracting features")
    t0 = time.perf_counter()
    image_1_corners = harris.detect_harris_corners(image_1_gray, num_corners=cfg["num_harris_corners"])
    image_2_corners = harris.detect_harris_corners(image_2_gray, num_corners=cfg["num_harris_corners"])
    timed("harris", t0)

    logging.info("Matching features")
    t0 = time.perf_counter()
    ncc_function = functools.partial(ncc.calculate_ncc, window_size=cfg["ncc_window_size"])
    score_function = _create_score_function(image_1_gray, image_2_gray, ncc_function)
    matches = matching.match_brute_force(
        image_1_corners, image_2_corners, score_function,
        validation_strategies={matching.ValidationStrategy.RATIO_TEST, matching.ValidationStrategy.CROSSCHECK},
        ratio_test_threshold=cfg["ratio_test_threshold"])
    matches = _filter_matches(matches, cfg["match_score_threshold"])
    timed("matching", t0)
    if model == "auto":
        return _run_selected(image_1_corners, image_2_corners, matches, camera_matrix, cfg, secs, refine)
    if refine > 0:
        return _run_refined_essential(image_1_corners, image_2_corners, matches, camera_matrix, cfg, secs, refine)

    logging.info("Estimating Essential Matrix")
    t0 = time.perf_counter()
    e, inlier_feature_pairs = estimate_essential_mat_with_ransac(
        camera_matrix, features_a=image_1_corners, features_b=image_2_corners, matches=matches,
        sed_inlier_threshold=cfg["ransac"]["sed_inlier_threshold"], error_aggregation_method=ErrorAggregationMethod.RMS,
        min_num_extra_inliers=cfg["ransac"]["min_num_extra_inliers"], max_iterations=cfg["ransac"]["max_iterations"])
    timed("ransac", t0)
    inlier_features_a = [pair[0] for pair in inlier_feature_pairs]
    inlier_features_b = [pair[1] for pair in inlier_feature_pairs]

    logging.info("Recovering Relative Pose")
    t0 = time.perf_counter()
    r, t, inlier_mask = recover_r_t_from_e(e=e, camera_matrix=camera_matrix, features_a=inlier_features_a,
                                           features_b=inlier_features_b)
    timed("pose", t0)
    if check_opencv:  # apps/sfm.py:140-161
        import cv2 as cv

        _, r_cv, t_cv, _ = cv.recoverPose(e, np.array([[p[0].x, p[0].y] for p in inlier_feature_pairs]),
                                          np.array([[p[1].x, p[1].y] for p in inlier_feature_pairs]), camera_matrix)
        if not np.allclose(r, r_cv, rtol=0.0, atol=1e-5) or not np.allclose(t, np.squeeze(t_cv), rtol=0.0, atol=1e-5):
            raise RuntimeError(f"OpenCV pose estimate\nR:\n{r_cv}\nt:\n{t_cv}\ndiffers from estimated pose\nR:\n{r}\nt:\n{t}")
    cam2_T_cam1 = Transform3D.from_rmat_t(r, t)

    # Only keep matches which passed the cheirality check (apps/sfm.py:167-169).
    inlier_features_a = [inlier_features_a[int(i)] for i in inlier_mask]
    inlier_features_b = [inlier_features_b[int(i)] for i in inlier_mask]

    logging.info("Triangulating points")
    t0 = time.perf_counter()
    world_points = triangulate_points(inlier_features_a, inlier_features_b, intrinsic_camera_matrix=camera_matrix,
                                      cam2_T_cam1=cam2_T_cam1)
    timed("triangulation", t0)
    if check_opencv:  # apps/sfm.py:188-202
        import cv2 as cv

        K_ext = np.hstack((camera_matrix, np.zeros((3, 1))))
        P1 = K_ext @ Transform3D.from_rmat_t(np.eye(3), np.zeros((3,))).Tmat
        P2 = K_ext @ cam2_T_cam1.Tmat
        pts_cv = cv.triangulatePoints(P1, P2, np.array([[f.x, f.y] for f in inlier_features_a]).T,
                                      np.array([[f.x, f.y] for f in inlier_features_b]).T).T
        pts_cv = (pts_cv / pts_cv[:, -1].reshape((-1, 1)))[:, :-1]
        if not np.allclose(world_points, pts_cv, rtol=1e-6, atol=1e-6):
            raise RuntimeError("OpenCV triangulation differs from the estimated points")
    return SfmResult(image_1_corners, image_2_corners, matches, e, inlier_feature_pairs, r, t, np.asarray(inlier_mask),
                     cam2_T_cam1, world_points, secs)


def load_middlebury_pair(dataset_dir, index_1, index_2, downscale_factor=1.0):
    """apps/sfm.py:44-62, 218-234 of the reference: <name>_par.txt + <name><index>.png, OpenCV decode, Lanczos
    downscale, RGB2GRAY; both images must share the intrinsics."""
    import glob

    import cv2 as cv

    pars = glob.glob(os.path.join(dataset_dir, "*_par.txt"))
    if len(pars) != 1:
        raise FileNotFoundError(f"expected exactly one *_par.txt in {dataset_dir}")
    from pathlib import Path

    stem = os.path.basename(pars[0])[:-len("_par.txt")]
    out = []
    for idx in (index_1, index_2):
        k, _ = load_camera_k_r_t(Path(pars[0]), int(idx))
        image = cv.imread(os.path.join(dataset_dir, f"{stem}{int(idx):04d}.png"))
        if image is None:
            raise FileNotFoundError(os.path.join(dataset_dir, f"{stem}{int(idx):04d}.png"))
        size = (int(image.shape[1] / downscale_factor), int(image.shape[0] / downscale_factor))
        image = cv.resize(image, size, interpolation=cv.INTER_LANCZOS4)
        out.append((cv.cvtColor(image, cv.COLOR_RGB2GRAY), k))
    if not np.allclose(out[0][1], out[1][1]):
        raise ValueError("Camera intrinsics params are different for the images, which is currently not supported.")
    return out[0][0], out[1][0], out[0][1]


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--synthetic", type=int, default=None, metavar="SEED", help="render a synthetic image pair")
    ap.add_argument("--image1"), ap.add_argument("--image2"), ap.add_argument("--camera-matrix")
    ap.add_argument("--dataset-dir", help="Middlebury multi-view layout (<name>_par.txt, <name>NNNN.png)")
    ap.add_argument("--index1", type=int, default=170), ap.add_argument("--index2", type=int, default=172)
    ap.add_argument("--config", default=os.path.join(ROOT, "apps", "config", "config.yaml"))
    ap.add_argument("--seed", type=int, default=None, help="random.seed() for the RANSAC sampler")
    ap.add_argument("--check-opencv", action="store_true")
    ap.add_argument("--model", choices=["essential", "auto"], default="essential",
                    help="essential: the essential matrix only; auto: pick between it and a homography")
    ap.add_argument("--planar", action="store_true", help="with --synthetic: render one plane only")
    ap.add_argument("--refine", type=int, default=0, metavar="N",
                    help="refine the winner over its inliers (at most N Levenberg-Marquardt iterations) before the pose")
    args = ap.parse_args(argv)
    if args.refine < 0:
        ap.error("--refine must be >= 0")
    logging.basicConfig(level=logging.INFO, format="%(message)s")
    cfg = load_config(args.config)
    truth = None
    if args.synthetic is not None:
        from structure_from_motion_b200.scenes import make_image_pair

        img1, img2, K, R, t = make_image_pair(args.synthetic, planar=args.planar)
        truth = (R, t)
        cfg["ransac"].update(sed_inlier_threshold=1e-5, min_num_extra_inliers=60)  # integer-pixel corners at f = 520
    elif args.dataset_dir:
        img1, img2, K = load_middlebury_pair(args.dataset_dir, args.index1, args.index2, cfg["image_downscale_factor"])
    else:
        if not (args.image1 and args.image2 and args.camera_matrix):
            ap.error("--synthetic SEED, --dataset-dir DIR or --image1/--image2/--camera-matrix (.npy files) are required")
        img1, img2, K = np.load(args.image1), np.load(args.image2), np.load(args.camera_matrix)
    if args.seed is not None:
        import random

        random.seed(args.seed)
    res = run_sfm(img1, img2, K, cfg, check_opencv=args.check_opencv, model=args.model, refine=args.refine)
    out = dict(corners=[len(res.corners_1), len(res.corners_2)], matches=len(res.matches),
               ransac_inliers=len(res.inlier_feature_pairs), cheirality_inliers=int(len(res.inlier_mask)),
               R=res.r.tolist(), t=res.t.tolist(), seconds=res.seconds)
    if args.model == "auto":
        out.update(model=res.model, homography_score_ratio=res.homography_score_ratio, rotation_only=res.rotation_only)
    if res.refinement is not None:
        out["refinement"] = res.refinement
    if truth is not None:
        R, t = truth
        out["rotation_error_deg"] = float(np.degrees(np.arccos(np.clip((np.trace(res.r.T @ R) - 1) / 2, -1, 1))))
        if not res.rotation_only:
            out["translation_angle_deg"] = float(np.degrees(np.arccos(np.clip(res.t @ t / np.linalg.norm(t) / np.linalg.norm(res.t), -1, 1))))
    print(json.dumps(out))
    return res


if __name__ == "__main__":
    main()
