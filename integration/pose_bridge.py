"""Drop-ins for the pose side of the hot path (SURVEY.md §8b, secondary boundary):

  homography.ransac_essential / estimate_pose_from_matches / match_orb_descriptors /
  estimate_pose_from_orb_with_inliers, robust_pose_estimator.RobustPoseEstimator, and the
  ``cv2.BFMatcher(NORM_HAMMING, crossCheck=True)`` objects that persistent_map and
  keyframe_manager build directly.

The hypothesis loop of ``ransac_essential`` (/root/reference/homography.py:324-339) runs
on the B200: K4 8-point solves, K3 float64 Sampson scoring, winner selection with the
reference's sequential semantics.  ``install()`` rebinds the names inside the reference's
already-imported modules (the reference tree is read-only).
"""
from __future__ import annotations

import logging
import os
import threading
from dataclasses import dataclass
from typing import Sequence

import cv2
import numpy as np

from .feature_pipeline_bridge import (adaptive_ransac_threshold, hamming_match_arrays,
                                      matches_to_points, to_dmatches)

LOGGER = logging.getLogger(__name__)

_ransac = None
_ransac_pid = None
_lock = threading.Lock()

# Reference-stream mode (parity tests, deterministic replays): when set to a callable returning a
# ``numpy.random.Generator``, every RANSAC drop-in called WITHOUT ``rng`` asks it for one — exactly where the
# reference calls ``np.random.default_rng()`` (homography.py:191-192, 315-316) — and draws its minimal samples from
# that generator's ``choice`` stream instead of the device RNG.  None (default) = device RNG, like production.
RNG_FACTORY = None


def _draw_reference_stream(rng, n: int, k: int, max_iter: int):
    """``rng.choice(n, k, replace=False)`` per iteration, in order (homography.py:193 / :325) -> ((max_iter, k) int32,
    the generator state before the first draw)."""
    state = rng.bit_generator.state
    out = np.zeros((max_iter, k), np.int32)
    if n >= k:
        for it in range(max_iter):
            out[it] = rng.choice(n, k, replace=False)
    return out, state


def _rewind_to_reference_state(rng, state, n: int, k: int, draws: int):
    """Leave the caller's generator where the reference's sequential loop leaves it: `draws` iterations consumed
    (it stops at the first hypothesis above 0.8 n, homography.py:210-211 / :338-339)."""
    rng.bit_generator.state = state
    for _ in range(draws):
        rng.choice(n, k, replace=False)


def _device_ransac():
    global _ransac, _ransac_pid
    with _lock:
        if _ransac is None or _ransac_pid != os.getpid():
            from b200slam.frontend import EssentialRansac

            _ransac = EssentialRansac()
            _ransac_pid = os.getpid()
        return _ransac


# --------------------------------------------------------------------------- #
# matching front doors
# --------------------------------------------------------------------------- #

def match_orb_descriptors(desc1, desc2, ratio: float = 0.8):
    """homography.match_orb_descriptors (:9-26): ratio + symmetry, list of (i, j)."""
    if len(desc2) < 2:
        raise ValueError("not enough values to unpack (expected 2, got %d)" % len(desc2))
    qi, ti, _ = hamming_match_arrays(desc1, desc2, cross_check=True, ratio_test=ratio,
                                     combined=True, sort_by_distance=False)
    return [(int(i), int(j)) for i, j in zip(qi, ti)]


class CrossCheckMatcher:
    """Stands in for ``cv2.BFMatcher(cv2.NORM_HAMMING, crossCheck=True)`` where the
    reference builds one directly (persistent_map.py:326-331, keyframe_manager.py:126,141):
    ``match`` returns the cross-checked DMatch list in ascending queryIdx order.  Non-uint8
    descriptors (the float32 / L2 branch) are delegated to OpenCV unchanged."""

    def match(self, desc1, desc2):
        if desc1 is None or desc2 is None or len(desc1) == 0 or len(desc2) == 0:
            return []
        if np.asarray(desc1).dtype != np.uint8:
            return list(cv2.BFMatcher(cv2.NORM_L2, crossCheck=True).match(desc1, desc2))
        return to_dmatches(*hamming_match_arrays(desc1, desc2, cross_check=True, sort_by_distance=False))


# --------------------------------------------------------------------------- #
# RANSAC essential matrix
# --------------------------------------------------------------------------- #

def ransac_essential_batch(src_list, dst_list, K, th=0.01, max_iter: int = 2000, rngs=None, seed: int | None = None):
    """Many independent ``ransac_essential`` problems in one set of launches.
    -> list of (best_h, inlier_index_array) ; best_h = -1 when nothing scored."""
    import torch
    from b200slam import _capi

    _capi.require_cuda()
    R = _device_ransac()
    n_pairs = len(src_list)
    counts_np = np.array([len(s) for s in src_list], np.int32)
    off = np.zeros(n_pairs + 1, np.int32)
    np.cumsum(counts_np, out=off[1:])
    corr = np.zeros((max(int(off[-1]), 1), 4), np.float32)
    for p, (s, d) in enumerate(zip(src_list, dst_list)):
        corr[off[p]:off[p + 1], :2] = np.asarray(s, np.float32).reshape(-1, 2)
        corr[off[p]:off[p + 1], 2:] = np.asarray(d, np.float32).reshape(-1, 2)
    dev = torch.device("cuda", torch.cuda.current_device())
    corr_d = torch.from_numpy(corr).to(dev)
    off_d = torch.from_numpy(off).to(dev)
    cnt_d = torch.from_numpy(counts_np).to(dev)
    samples_d = None
    if rngs is None and RNG_FACTORY is not None:
        rngs = [RNG_FACTORY() for _ in range(n_pairs)]
    states = None
    if rngs is not None:
        smp = np.zeros((n_pairs, max_iter, 8), np.int32)
        states = []
        for p, rng in enumerate(rngs):                               # homography.py:325, same stream
            smp[p], st = _draw_reference_stream(rng, int(counts_np[p]), 8, max_iter)
            states.append(st)
        samples_d = torch.from_numpy(smp).to(dev)
    if seed is None:
        seed = int(np.random.SeedSequence().entropy & (2 ** 63 - 1))
    th = np.broadcast_to(np.asarray(th, np.float64), (n_pairs,))
    th2_d = torch.from_numpy(np.ascontiguousarray(th ** 2)).to(dev)
    E = R.hypotheses(corr_d, off_d, cnt_d, n_pairs, max_iter, samples=samples_d, seed=seed, K=K)
    counts = R.score(corr_d, off_d, cnt_d, n_pairs, E, 0.0, th2_per_pair=th2_d, precision=64, max_m=int(counts_np.max()) if n_pairs else 0)
    best_h, best_c, mask = R.select(counts, corr_d, off_d, cnt_d, n_pairs, E, 0.0, th2_per_pair=th2_d)
    best_h, best_c, mask = best_h.cpu().numpy(), best_c.cpu().numpy(), mask.cpu().numpy()
    if states is not None:
        for p, rng in enumerate(rngs):                               # the early exit consumed best_h + 1 draws only
            n = int(counts_np[p])
            if n >= 8 and best_h[p] >= 0 and best_c[p] > 0.8 * n:
                _rewind_to_reference_state(rng, states[p], n, 8, int(best_h[p]) + 1)
    return [(int(best_h[p]), np.flatnonzero(mask[off[p]:off[p + 1]])) for p in range(n_pairs)]


_hransac = None
_hransac_pid = None


def _device_hransac():
    global _hransac, _hransac_pid
    with _lock:
        if _hransac is None or _hransac_pid != os.getpid():
            from b200slam.frontend import HomographyRansac

            _hransac = HomographyRansac()
            _hransac_pid = os.getpid()
        return _hransac


def ransac_homography_batch(src_list, dst_list, th=3.0, max_iter: int = 2000, rngs=None, seed: int | None = None):
    """Many independent ``ransac_homography`` problems (homography.py:148-216) in one set of
    launches: K5 4-point DLT hypotheses, K6 symmetric transfer error, winner selection.
    -> list of (best_h, inlier_index_array); best_h = -1 when nothing scored."""
    import torch
    from b200slam import _capi

    _capi.require_cuda()
    R = _device_hransac()
    n_pairs = len(src_list)
    counts_np = np.array([len(s) for s in src_list], np.int32)
    off = np.zeros(n_pairs + 1, np.int32)
    np.cumsum(counts_np, out=off[1:])
    corr = np.zeros((max(int(off[-1]), 1), 4), np.float32)
    for p, (s, d) in enumerate(zip(src_list, dst_list)):
        corr[off[p]:off[p + 1], :2] = np.asarray(s, np.float32).reshape(-1, 2)
        corr[off[p]:off[p + 1], 2:] = np.asarray(d, np.float32).reshape(-1, 2)
    dev = torch.device("cuda", torch.cuda.current_device())
    corr_d, off_d, cnt_d = torch.from_numpy(corr).to(dev), torch.from_numpy(off).to(dev), torch.from_numpy(counts_np).to(dev)
    samples_d = None
    if rngs is None and RNG_FACTORY is not None:
        rngs = [RNG_FACTORY() for _ in range(n_pairs)]
    states = None
    if rngs is not None:
        smp = np.zeros((n_pairs, max_iter, 4), np.int32)
        states = []
        for p, rng in enumerate(rngs):                               # homography.py:193, same stream
            smp[p], st = _draw_reference_stream(rng, int(counts_np[p]), 4, max_iter)
            states.append(st)
        samples_d = torch.from_numpy(smp).to(dev)
    if seed is None:
        seed = int(np.random.SeedSequence().entropy & (2 ** 63 - 1))
    th = np.broadcast_to(np.asarray(th, np.float64), (n_pairs,))
    th_d = torch.from_numpy(np.array(th, dtype=np.float64)).to(dev)
    Hm = R.hypotheses(corr_d, off_d, cnt_d, n_pairs, max_iter, samples=samples_d, seed=seed)
    counts = R.score(corr_d, off_d, cnt_d, n_pairs, Hm, 0.0, th_per_pair=th_d)
    best_h, best_c, mask = R.select(counts, corr_d, off_d, cnt_d, n_pairs, Hm, 0.0, th_per_pair=th_d)
    best_h, best_c, mask = best_h.cpu().numpy(), best_c.cpu().numpy(), mask.cpu().numpy()
    if states is not None:
        for p, rng in enumerate(rngs):
            n = int(counts_np[p])
            if n >= 4 and best_h[p] >= 0 and best_c[p] > 0.8 * n:
                _rewind_to_reference_state(rng, states[p], n, 4, int(best_h[p]) + 1)
    return [(int(best_h[p]), np.flatnonzero(mask[off[p]:off[p + 1]])) for p in range(n_pairs)]


def ransac_homography(src, dst, th: float = 3.0, max_iter: int = 2000, rng=None):
    """Drop-in for homography.ransac_homography (:148-216) -> (refined H, inlier indices).
    The hypothesis loop runs on the device; the n-point DLT refit on the winner's inliers
    (:216) is host NumPy, once per call."""
    from b200slam.geometry import dlt_homography_batch

    src, dst = np.asarray(src, dtype=np.float64), np.asarray(dst, dtype=np.float64)
    n = len(src)
    if n < 4:
        raise ValueError("At least four correspondences are required")
    best_h, inl = ransac_homography_batch([src], [dst], th, max_iter, rngs=None if rng is None else [rng])[0]
    if best_h < 0 or inl.size < 4:
        raise RuntimeError("RANSAC failed — too few inliers")
    return dlt_homography_batch(src[inl][None], dst[inl][None])[0], inl


def ransac_essential(src, dst, K, th: float = 0.01, max_iter: int = 2000, rng=None):
    """Drop-in for homography.ransac_essential (:302-345) -> (refined E, inlier indices).

    With ``rng`` the 8-samples are the reference's own stream (``rng.choice(n, 8,
    replace=False)`` per iteration) and the generator is left in the state the reference leaves
    it in (only the iterations up to its early exit consumed); without it (every production
    caller) they are drawn on the device.  All ``max_iter`` hypotheses are scored in one launch
    and the winner is the one the sequential loop would have ended on (strict improvement, early
    exit above 0.8 n)."""
    from b200slam.geometry import eight_point_refit

    src, dst = np.asarray(src), np.asarray(dst)
    n = len(src)
    if n < 8:
        raise ValueError("At least eight correspondences are required")
    best_h, inl = ransac_essential_batch([src], [dst], K, th, max_iter, rngs=None if rng is None else [rng])[0]
    if best_h < 0 or inl.size < 8:
        raise RuntimeError("RANSAC essential matrix failed")
    return eight_point_refit(src[inl], dst[inl], K), inl


def find_essential_mat(points1, points2, K, threshold: float = 1.0, samples: int = 512, seed: int | None = None):
    """Stand-in for the reference's ``cv2.findEssentialMat(pts1, pts2, K, method=cv2.RANSAC,
    threshold=...)`` call sites (slam_viewer.py:195, web_dashboard_server.py:145,
    visual_slam_offline_entry_point.py:51): 5-point RANSAC on the device (K8 minimal solver, the
    float64 Sampson scoring of the 8-point path, the same winner rule).  Like OpenCV it calibrates
    the points with ``K^-1`` and divides the pixel threshold by the mean focal length.  Returns
    ``(E, mask)`` with E in calibrated coordinates (unit Frobenius norm; OpenCV scales differently)
    and mask an (N, 1) uint8 column.  OpenCV's own sampling / termination are not reproduced
    (third-party internals, parity unpinned)."""
    import torch
    from b200slam import _capi

    _capi.require_cuda()
    p1 = np.asarray(points1, np.float64).reshape(-1, 2)
    p2 = np.asarray(points2, np.float64).reshape(-1, 2)
    n = len(p1)
    if n < 5:
        return None, None
    K = np.asarray(K, np.float64).reshape(3, 3)
    Kinv = np.linalg.inv(K)
    a = np.hstack([p1, np.ones((n, 1))]) @ Kinv.T
    b = np.hstack([p2, np.ones((n, 1))]) @ Kinv.T
    corr = np.hstack([a[:, :2] / a[:, 2:], b[:, :2] / b[:, 2:]]).astype(np.float32)
    th = float(threshold) / (0.5 * (K[0, 0] + K[1, 1]))
    R = _device_ransac()
    dev = torch.device("cuda", torch.cuda.current_device())
    corr_d = torch.from_numpy(corr).to(dev)
    off_d = torch.tensor([0, n], dtype=torch.int32, device=dev)
    cnt_d = torch.tensor([n], dtype=torch.int32, device=dev)
    if seed is None:
        seed = int(np.random.SeedSequence().entropy & (2 ** 63 - 1))
    E = R.hypotheses_5pt(corr_d, off_d, cnt_d, 1, samples, seed=seed)
    counts = R.score(corr_d, off_d, cnt_d, 1, E, th * th, precision=64)
    best_h, _, mask = R.select(counts, corr_d, off_d, cnt_d, 1, E, th * th)
    h = int(best_h[0])
    if h < 0:
        return None, None
    return E[0, h].cpu().numpy().reshape(3, 3), mask.cpu().numpy().reshape(-1, 1).astype(np.uint8)


def estimate_poses_batch(src_list, dst_list, K, th=0.01, max_iter: int = 2000):
    """``ransac_essential`` + ``decompose_essential`` (homography.py:302-345, 251-299) for many
    independent correspondence sets, everything on the device: ONE batched RANSAC (K4 + K3h +
    selection), ONE batched n-point refit on the winners' inliers, ONE batched decomposition /
    cheirality vote (K7).  -> list of (R, t, inlier indices), or None where the reference would raise."""
    import torch
    from b200slam.frontend import PoseRecovery

    n_pairs = len(src_list)
    if n_pairs == 0:
        return []
    res = ransac_essential_batch(src_list, dst_list, K, th=th, max_iter=max_iter)
    Ms = np.array([len(s) for s in src_list], np.int32)
    off = np.zeros(n_pairs + 1, np.int32)
    np.cumsum(Ms, out=off[1:])
    corr = np.zeros((max(int(off[-1]), 1), 4), np.float32)
    mask = np.zeros(max(int(off[-1]), 1), np.uint8)
    ok = np.zeros(n_pairs, bool)
    for p, (best_h, inl) in enumerate(res):
        corr[off[p]:off[p + 1], :2] = np.asarray(src_list[p], np.float32).reshape(-1, 2)
        corr[off[p]:off[p + 1], 2:] = np.asarray(dst_list[p], np.float32).reshape(-1, 2)
        if best_h >= 0 and inl.size >= 8:
            mask[off[p] + inl] = 1
            ok[p] = True
    out = [None] * n_pairs
    if not ok.any():
        return out
    dev = torch.device("cuda", torch.cuda.current_device())
    corr_d, off_d, cnt_d, mask_d = (torch.from_numpy(x).to(dev) for x in (corr, off, Ms, mask))
    P = PoseRecovery()
    E, _ = P.refit(corr_d, off_d, cnt_d, n_pairs, mask=mask_d, K=K)
    R, t, _ = P.decompose(E, corr_d, off_d, cnt_d, n_pairs, int(Ms.max()), mask=mask_d, K=K)
    for p in np.flatnonzero(ok):
        out[p] = (R[p], t[p], res[p][1])
    return out


def estimate_pose_from_matches(kp1, kp2, matches, K, ransac_threshold: float = 0.01, min_matches: int = 15):
    """Drop-in for homography.estimate_pose_from_matches (:423-438)."""
    from b200slam.geometry import decompose_essential

    if len(matches) < min_matches:
        raise RuntimeError("too few matches")
    pts1 = np.float32([kp1[m.queryIdx].pt for m in matches])
    pts2 = np.float32([kp2[m.trainIdx].pt for m in matches])
    E, inliers = ransac_essential(pts1, pts2, K, th=ransac_threshold)
    R, t = decompose_essential(E, pts1[inliers], pts2[inliers], K)
    return R, t, inliers, len(matches)


def estimate_pose_from_orb_with_inliers(kp1, des1, kp2, des2, K, ransac_threshold: float = 0.01, min_matches: int = 15):
    """Drop-in for homography.estimate_pose_from_orb_with_inliers (:399-420)."""
    from b200slam.geometry import decompose_essential

    matches = match_orb_descriptors(des1, des2)
    if len(matches) < min_matches:
        raise RuntimeError("too few matches")
    pts1 = np.float32([kp1[i].pt for i, _ in matches])
    pts2 = np.float32([kp2[j].pt for _, j in matches])
    E, inliers = ransac_essential(pts1, pts2, K, th=ransac_threshold)
    R, t = decompose_essential(E, pts1[inliers], pts2[inliers], K)
    return R, t, inliers, len(matches)


# --------------------------------------------------------------------------- #
# robust pose estimator (robust_pose_estimator.py:18-305)
# --------------------------------------------------------------------------- #

@dataclass(frozen=True)
class PoseEstimationDiagnostics:
    method: str
    match_count: int
    inliers: int
    inlier_ratio: float
    median_parallax: float
    cheirality_inliers: int
    cheirality_ratio: float
    score: float


@dataclass(frozen=True)
class PoseEstimate:
    rotation: np.ndarray
    translation: np.ndarray
    inlier_indices: np.ndarray
    diagnostics: PoseEstimationDiagnostics


@dataclass(frozen=True)
class RobustPoseEstimatorConfig:
    """robust_pose_estimator.py:42-70, same defaults and validation."""
    min_matches: int = 20
    min_inliers: int = 30
    base_ransac_threshold: float = 0.01
    min_ransac_threshold: float = 0.005
    max_ransac_threshold: float = 0.02
    min_inlier_ratio: float = 0.25
    homography_bias: float = 0.9
    essential_bias: float = 1.0
    min_parallax: float = 1.0
    min_cheirality_ratio: float = 0.6
    min_cheirality_inliers: int = 12

    def __post_init__(self) -> None:
        if self.min_matches <= 0:
            raise ValueError("min_matches must be positive")
        if self.min_inliers <= 0:
            raise ValueError("min_inliers must be positive")
        if self.min_inlier_ratio <= 0:
            raise ValueError("min_inlier_ratio must be positive")
        if self.min_parallax < 0:
            raise ValueError("min_parallax must be non-negative")
        if self.min_cheirality_ratio <= 0:
            raise ValueError("min_cheirality_ratio must be positive")
        if self.min_cheirality_inliers <= 0:
            raise ValueError("min_cheirality_inliers must be positive")


class PoseEstimationFailure(RuntimeError):
    """robust_pose_estimator.py:73-80."""

    def __init__(self, reason: str, recovery_action: str, metrics: dict) -> None:
        super().__init__(f"{reason} (recovery={recovery_action})")
        self.reason = reason
        self.recovery_action = recovery_action
        self.metrics = metrics


def _normalize_translation(t: np.ndarray) -> np.ndarray:
    if t.ndim != 1 or t.shape[0] != 3:
        raise ValueError("Translation must be a 3D vector")
    norm = float(np.linalg.norm(t))
    if norm == 0.0:
        raise ValueError("Translation norm is zero")
    return t / norm


def _median_parallax(pts1, pts2, inliers) -> float:
    if len(inliers) == 0:
        return 0.0
    return float(np.median(np.linalg.norm(pts2[inliers] - pts1[inliers], axis=1)))


def _cheirality_ratio(pts1, pts2, inliers, R, t, K):
    """robust_pose_estimator.py:269-296 (cv2.triangulatePoints, finite + positive depth in both views)."""
    if len(inliers) == 0:
        return 0.0, 0
    a, b = pts1[inliers].T, pts2[inliers].T
    Pa = K @ np.hstack([np.eye(3), np.zeros((3, 1))])
    Pb = K @ np.hstack([R, t.reshape(3, 1)])
    with np.errstate(all="ignore"):
        hom = cv2.triangulatePoints(Pa, Pb, a, b)
        X = hom[:3] / hom[3]
        da, db = X[2], (R @ X + t.reshape(3, 1))[2]
    valid = np.isfinite(da) & np.isfinite(db)
    if not np.any(valid):
        return 0.0, 0
    count = int(np.sum((da > 0) & (db > 0) & valid))
    return float(count / max(len(inliers), 1)), count


class RobustPoseEstimator:
    """Essential + homography model selection with the reference's stability gates
    (robust_pose_estimator.py:83-251)."""

    def __init__(self, config: RobustPoseEstimatorConfig) -> None:
        self.config = config

    def estimate_pose(self, kp1, kp2, matches, intrinsics: np.ndarray) -> PoseEstimate:
        cfg = self.config
        if intrinsics.shape != (3, 3):
            raise ValueError("Intrinsics must be a 3x3 matrix")
        if len(matches) < cfg.min_matches:
            raise ValueError("Not enough matches for pose estimation")
        if not kp1 or not kp2:
            raise ValueError("Keypoints must be non-empty")
        pts1, pts2 = matches_to_points(kp1, kp2, matches)
        th = adaptive_ransac_threshold(pts1, pts2, cfg.base_ransac_threshold, cfg.min_ransac_threshold,
                                       cfg.max_ransac_threshold)
        cands = [self._estimate_essential(kp1, kp2, matches, pts1, pts2, intrinsics, th),
                 self._estimate_homography(pts1, pts2, intrinsics)]
        best = max(cands, key=lambda c: c.diagnostics.score)
        self._apply_stability_gates(best)
        LOGGER.info("Pose estimation selected %s with %d/%d inliers", best.diagnostics.method,
                    best.diagnostics.inliers, best.diagnostics.match_count)
        return best

    def _estimate_essential(self, kp1, kp2, matches, pts1, pts2, K, th) -> PoseEstimate:
        cfg = self.config
        try:
            R, t, inliers, match_count = estimate_pose_from_matches(kp1, kp2, matches, K, th, cfg.min_matches)
        except RuntimeError as exc:
            LOGGER.exception("Essential matrix pose estimation failed")
            raise RuntimeError("Essential matrix pose estimation failed") from exc
        ratio = float(len(inliers) / max(match_count, 1))
        parallax = _median_parallax(pts1, pts2, inliers)
        ch_ratio, ch_inl = _cheirality_ratio(pts1, pts2, inliers, R, t, K)
        score = cfg.essential_bias * ratio * max(parallax, cfg.min_parallax)
        diag = PoseEstimationDiagnostics("essential", match_count, len(inliers), ratio, parallax, ch_inl, ch_ratio, score)
        return PoseEstimate(R, _normalize_translation(t), inliers, diag)

    def _estimate_homography(self, pts1, pts2, K) -> PoseEstimate:
        from b200slam.geometry import decompose_homography

        cfg = self.config
        try:
            H, inliers = ransac_homography(pts1, pts2)
            R, t = decompose_homography(H, K)
        except (RuntimeError, ValueError) as exc:
            LOGGER.exception("Homography pose estimation failed")
            raise RuntimeError("Homography pose estimation failed") from exc
        ratio = float(len(inliers) / max(len(pts1), 1))
        parallax = float(np.median(np.linalg.norm(pts2 - pts1, axis=1)))
        score = cfg.homography_bias * ratio * max(parallax, cfg.min_parallax)
        diag = PoseEstimationDiagnostics("homography", len(pts1), len(inliers), ratio, parallax, len(inliers), 1.0, score)
        return PoseEstimate(R, _normalize_translation(t), inliers, diag)

    def estimate_pose_batch(self, kp1_list, kp2_list, matches_list, intrinsics: np.ndarray, rngs=None,
                            seed: int | None = None, configs=None) -> list:
        """``estimate_pose`` for many pairs in one pass on the device -> one entry per pair: the PoseEstimate the
        single call returns, or the exception instance it would raise (same type and message; for
        PoseEstimationFailure the same reason, recovery action and metrics).

        The argument checks run on the host: a bad ``intrinsics`` shape fails the whole call; a pair with fewer than
        ``min_matches`` matches, empty keypoints or fewer than eight correspondences gets its ValueError and never
        reaches the device (a batch of such pairs needs no CUDA).  All other pairs go through ONE
        ``b200slam.robust_pose.RobustPose.run``: one upload, one download.

        rngs: optional ``(essential_rng, homography_rng)`` per pair; the samples are drawn from them exactly as the
        reference's loops draw them and each generator is left where the single call leaves it (the homography
        generator untouched when the essential branch raises).  With ``rngs=None`` and ``RNG_FACTORY`` set, two
        generators are requested per pair that reaches RANSAC, in pair order, essential first — the order of
        consecutive single calls whenever no essential branch raises (a single call that raises there never asks
        for its homography generator).  Otherwise the device sampler draws with ``seed`` (random when None).
        configs: optional per-pair RobustPoseEstimatorConfig (default: this estimator's for every pair)."""
        if intrinsics.shape != (3, 3):
            raise ValueError("Intrinsics must be a 3x3 matrix")
        n_pairs = len(matches_list)
        if not (len(kp1_list) == len(kp2_list) == n_pairs):
            raise ValueError("kp1_list, kp2_list and matches_list differ in length")
        cfgs = [self.config] * n_pairs if configs is None else list(configs)
        if len(cfgs) != n_pairs:
            raise ValueError("one config per pair")
        out: list = [None] * n_pairs
        live, pts = [], []
        for p in range(n_pairs):
            kp1, kp2, matches = kp1_list[p], kp2_list[p], matches_list[p]
            if len(matches) < cfgs[p].min_matches:
                out[p] = ValueError("Not enough matches for pose estimation")
            elif not kp1 or not kp2:
                out[p] = ValueError("Keypoints must be non-empty")
            elif len(matches) < 8:                                   # ransac_essential's own check (homography.py:305)
                out[p] = ValueError("At least eight correspondences are required")
            else:
                live.append(p)
                pts.append(matches_to_points(kp1, kp2, matches))
        if not live:
            return out
        from b200slam import _capi

        torch = _capi.require_cuda()
        from b200slam import robust_pose as rp

        max_iter = 2000
        L = len(live)
        counts = np.array([len(a) for a, _ in pts], np.int32)
        off = np.zeros(L + 1, np.int32)
        np.cumsum(counts, out=off[1:])
        rows = int(off[-1])
        if rngs is None and RNG_FACTORY is not None:
            gens = [(RNG_FACTORY(), RNG_FACTORY()) for _ in live]
        elif rngs is not None:
            gens = [tuple(rngs[p]) for p in live]
        else:
            gens = None
        # one host buffer, one upload: corr (float32 bits) | c_off | c_count | samples_e | samples_h
        n_smp = L * max_iter * 12 if gens is not None else 0
        host = np.zeros(rows * 4 + (L + 1) + L + n_smp, np.int32)
        corr = host[:rows * 4].view(np.float32).reshape(rows, 4)
        for i, (a, b) in enumerate(pts):
            corr[off[i]:off[i + 1], :2] = a
            corr[off[i]:off[i + 1], 2:] = b
        host[rows * 4:rows * 4 + L + 1] = off
        host[rows * 4 + L + 1:rows * 4 + 2 * L + 1] = counts
        states = []
        if gens is not None:
            base = rows * 4 + 2 * L + 1
            se = host[base:base + L * max_iter * 8].reshape(L, max_iter, 8)
            sh = host[base + L * max_iter * 8:base + n_smp].reshape(L, max_iter, 4)
            for i, (ge, gh) in enumerate(gens):                     # homography.py:325 and :193, the same streams
                se[i], st_e = _draw_reference_stream(ge, int(counts[i]), 8, max_iter)
                sh[i], st_h = _draw_reference_stream(gh, int(counts[i]), 4, max_iter)
                states.append((st_e, st_h))
        if seed is None:
            seed = int(np.random.SeedSequence().entropy & (2 ** 63 - 1))
        dev = torch.device("cuda", torch.cuda.current_device())
        d = torch.from_numpy(host).to(dev)
        corr_d = d[:rows * 4].view(torch.float32).view(max(rows, 0), 4)
        off_d, cnt_d = d[rows * 4:rows * 4 + L + 1], d[rows * 4 + L + 1:rows * 4 + 2 * L + 1]
        smp_e = smp_h = None
        if gens is not None:
            base = rows * 4 + 2 * L + 1
            smp_e = d[base:base + L * max_iter * 8].view(L, max_iter, 8)
            smp_h = d[base + L * max_iter * 8:base + n_smp].view(L, max_iter, 4)
        if not hasattr(self, "_device"):
            self._device = rp.RobustPose()
        cfg_live = cfgs[0] if configs is None else [cfgs[p] for p in live]
        res = self._device.run(corr_d, off_d, cnt_d, L, intrinsics, cfg_live, samples_e=smp_e, samples_h=smp_h, seed=seed,
                               max_m=int(counts.max()), hypotheses=max_iter)
        packed = res.packed.cpu().numpy()                            # the one download
        recs = rp.decode_results(packed[:L * rp.POSE_RESULT_BYTES])
        mask = packed[L * rp.POSE_RESULT_BYTES:]
        for i, p in enumerate(live):
            r = recs[i]
            out[p] = decode_pose_result(r, np.flatnonzero(mask[off[i]:off[i + 1]]))
            if gens is not None:
                n = int(counts[i])
                (ge, gh), (st_e, st_h) = gens[i], states[i]
                if int(r["e_best_h"]) >= 0 and r["e_inliers"] > 0.8 * n:   # the loop stopped early (homography.py:338)
                    _rewind_to_reference_state(ge, st_e, n, 8, int(r["e_best_h"]) + 1)
                if not _homography_ran(r):
                    _rewind_to_reference_state(gh, st_h, n, 4, 0)
                elif int(r["h_best_h"]) >= 0 and r["h_inliers"] > 0.8 * n:
                    _rewind_to_reference_state(gh, st_h, n, 4, int(r["h_best_h"]) + 1)
        return out

    def _apply_stability_gates(self, est: PoseEstimate) -> None:
        cfg, d = self.config, est.diagnostics
        metrics = {"match_count": float(d.match_count), "inliers": float(d.inliers),
                   "inlier_ratio": float(d.inlier_ratio), "median_parallax": float(d.median_parallax),
                   "cheirality_ratio": float(d.cheirality_ratio), "cheirality_inliers": float(d.cheirality_inliers)}
        if d.inliers < cfg.min_inliers:
            raise PoseEstimationFailure("low_inlier_count", "relocalize", metrics)
        if d.inlier_ratio < cfg.min_inlier_ratio:
            raise PoseEstimationFailure("low_inlier_ratio", "relocalize", metrics)
        if d.median_parallax < cfg.min_parallax:
            raise PoseEstimationFailure("low_parallax", "relocalize", metrics)
        if d.method == "essential":
            if d.cheirality_inliers < cfg.min_cheirality_inliers:
                raise PoseEstimationFailure("cheirality_inliers", "relocalize", metrics)
            if d.cheirality_ratio < cfg.min_cheirality_ratio:
                raise PoseEstimationFailure("cheirality_ratio", "relocalize", metrics)


def _homography_ran(r) -> bool:
    """estimate_pose reaches ransac_homography unless the essential branch raised first."""
    from b200slam import robust_pose as rp

    o = int(r["outcome"])
    if o in (rp.POSE_ERR_MATCHES, rp.POSE_ERR_EIGHT, rp.POSE_ERR_ESSENTIAL):
        return False
    return not (o == rp.POSE_ERR_TRANSLATION and int(r["method"]) == 0)


def decode_pose_result(r, inlier_indices: np.ndarray):
    """One b2s_pose_result (a record of b200slam.robust_pose.POSE_RESULT_DTYPE) -> what estimate_pose returns
    (PoseEstimate) or the exception instance it raises, with the single call's messages.  inlier_indices: the
    selected model's inliers (flatnonzero of the pair's mask)."""
    from b200slam import robust_pose as rp

    o = int(r["outcome"])
    if o == rp.POSE_ERR_MATCHES:
        return ValueError("Not enough matches for pose estimation")
    if o == rp.POSE_ERR_EIGHT:
        return ValueError("At least eight correspondences are required")
    if o == rp.POSE_ERR_ESSENTIAL:
        return RuntimeError("Essential matrix pose estimation failed")
    if o == rp.POSE_ERR_HOMOGRAPHY:
        return RuntimeError("Homography pose estimation failed")
    if o == rp.POSE_ERR_TRANSLATION:
        return ValueError("Translation norm is zero")
    if o not in (rp.POSE_ESTIMATE, rp.POSE_GATE_FAILED):
        raise ValueError(f"unknown pose result outcome {o}")
    diag = PoseEstimationDiagnostics(rp.METHODS[int(r["method"])], int(r["match_count"]), int(r["inliers"]),
                                     float(r["inlier_ratio"]), float(r["median_parallax"]), int(r["cheirality_inliers"]),
                                     float(r["cheirality_ratio"]), float(r["score"]))
    if o == rp.POSE_GATE_FAILED:
        metrics = {"match_count": float(diag.match_count), "inliers": float(diag.inliers),
                   "inlier_ratio": float(diag.inlier_ratio), "median_parallax": float(diag.median_parallax),
                   "cheirality_ratio": float(diag.cheirality_ratio), "cheirality_inliers": float(diag.cheirality_inliers)}
        return PoseEstimationFailure(rp.GATE_REASONS[int(r["gate"])], "relocalize", metrics)
    return PoseEstimate(np.array(r["R"], dtype=np.float64).reshape(3, 3), np.array(r["t"], dtype=np.float64),
                        np.asarray(inlier_indices, dtype=np.int64), diag)


# --------------------------------------------------------------------------- #
# install(): rebind the names inside the reference's modules
# --------------------------------------------------------------------------- #

def install() -> list[str]:
    """Rebind the hot-path names in whichever reference modules are importable
    (``homography``, ``robust_pose_estimator``, ``persistent_map``, ``keyframe_manager``, ``slam_api``,
    ``visual_slam_offline_entry_point``).  Modules that did ``from x import name`` keep their own
    reference to the old object, so every importer is patched by name as well — the result does not
    depend on import order.  Returns the list of ``module.name`` strings patched; names that were looked
    for but could not be patched (module not importable, attribute absent) are in ``install.skipped``."""
    import importlib

    patched, skipped = [], []

    def bind(modname, attr, obj):
        try:
            mod = importlib.import_module(modname)
        except Exception:                                    # module absent or its own deps missing
            skipped.append(f"{modname}.{attr}")
            return
        if hasattr(mod, attr):
            setattr(mod, attr, obj)
            patched.append(f"{modname}.{attr}")
        else:
            skipped.append(f"{modname}.{attr}")

    for name, obj in (("ransac_essential", ransac_essential), ("estimate_pose_from_matches", estimate_pose_from_matches),
                      ("match_orb_descriptors", match_orb_descriptors), ("ransac_homography", ransac_homography),
                      ("estimate_pose_from_orb_with_inliers", estimate_pose_from_orb_with_inliers)):
        bind("homography", name, obj)
    bind("robust_pose_estimator", "estimate_pose_from_matches", estimate_pose_from_matches)
    bind("robust_pose_estimator", "ransac_homography", ransac_homography)
    bind("persistent_map", "estimate_pose_from_matches", estimate_pose_from_matches)
    bind("visual_slam_offline_entry_point", "estimate_pose_from_matches", estimate_pose_from_matches)

    def _build_matcher(desc_a, desc_b=None):                # persistent_map.py:326-331 (called with two arrays, :262)
        return CrossCheckMatcher()

    bind("persistent_map", "_build_matcher", _build_matcher)
    try:                                                    # the batched relocalizer answers with the reference's own result type
        import persistent_map

        from . import relocalization_bridge

        relocalization_bridge.RelocalizationResult = persistent_map.RelocalizationResult
        bind("persistent_map", "MapRelocalizer", relocalization_bridge.BatchedMapRelocalizer)
        bind("slam_api", "MapRelocalizer", relocalization_bridge.BatchedMapRelocalizer)          # slam_api.py:43 binds it by name
        bind("relocalization_demo", "MapRelocalizer", relocalization_bridge.BatchedMapRelocalizer)
        bind("persistent_map", "compute_bow_histogram", relocalization_bridge.compute_bow_histogram)   # K9 (build_snapshot, :110-112)
    except Exception:
        skipped.append("persistent_map.MapRelocalizer")
    try:                                                    # keyframe overlap (keyframe_manager.py:123-155): the reference builds a
        import keyframe_manager                             # cv2.BFMatcher per call unless a matcher= callable was injected

        base = keyframe_manager.KeyframeManager
        if getattr(base, "_b2s_device_matcher", False):     # install() twice: keep the class of the first call
            KeyframeManager = base
        else:
            class KeyframeManager(base):                    # same constructor; matcher=None now means the device cross-check matcher
                _b2s_device_matcher = True

                def __init__(self, *args, **kwargs):
                    super().__init__(*args, **kwargs)
                    if self.matcher is None:
                        self.matcher = CrossCheckMatcher().match

            KeyframeManager.__qualname__ = base.__qualname__
            KeyframeManager.__module__ = base.__module__
        for mod in ("keyframe_manager", "slam_api", "visual_slam_offline_entry_point"):
            bind(mod, "KeyframeManager", KeyframeManager)
    except Exception:
        skipped.append("keyframe_manager.KeyframeManager")
    install.skipped = skipped
    if skipped:
        LOGGER.debug("install(): not patched: %s", ", ".join(skipped))
    return patched


install.skipped = []
