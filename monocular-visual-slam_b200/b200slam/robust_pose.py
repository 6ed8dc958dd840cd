"""Batched RobustPoseEstimator.estimate_pose (robust_pose_estimator.py:89-251) on the device.

Per pair: the adaptive RANSAC threshold from the median displacement, the essential branch (K4 + K3 + selection at
the per-pair threshold, K7 refit + decomposition + cheirality vote), the homography branch (K5 + K6 + selection at
th = 3, n-point DLT refit, decompose_homography), per-branch inlier ratio / median parallax / cheirality / score, model
selection and the five stability gates.  The answer is one fixed-size ``b2s_pose_result`` per pair (include/b2s.h)
plus the selected model's inlier flags in the input's CSR layout; given a record buffer, the decision kernel also
writes every pair's pose record (include/b2s.h: the result record, then the b2s_pose_result).  Everything runs on the
current stream: no host sync, no allocation after the first call of a shape, capturable in a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, fields

import numpy as np

from . import _capi
from ._capi import check, current_stream, ptr

POSE_RESULT_BYTES = 200
ROBUST_POSE_CONFIG_BYTES = 80

# outcome / method / gate codes of b2s_pose_result
POSE_ESTIMATE, POSE_GATE_FAILED, POSE_ERR_MATCHES, POSE_ERR_EIGHT, POSE_ERR_ESSENTIAL, POSE_ERR_HOMOGRAPHY, \
    POSE_ERR_TRANSLATION = range(7)
POSE_EMPTY = -1                   # outcome of a record slot that holds no pair (padding of a sharded gather buffer)
METHODS = ("essential", "homography")
GATE_REASONS = (None, "low_inlier_count", "low_inlier_ratio", "low_parallax", "cheirality_inliers", "cheirality_ratio")

POSE_RESULT_DTYPE = np.dtype([
    ("outcome", "<i4"), ("method", "<i4"), ("gate", "<i4"), ("match_count", "<i4"), ("inliers", "<i4"),
    ("cheirality_inliers", "<i4"), ("e_best_h", "<i4"), ("e_inliers", "<i4"), ("h_best_h", "<i4"), ("h_inliers", "<i4"),
    ("reserved", "<i4", (2,)), ("inlier_ratio", "<f8"), ("median_parallax", "<f8"), ("cheirality_ratio", "<f8"),
    ("score", "<f8"), ("score_essential", "<f8"), ("score_homography", "<f8"), ("threshold", "<f8"),
    ("R", "<f8", (9,)), ("t", "<f8", (3,))])

CONFIG_DTYPE = np.dtype([
    ("min_matches", "<i4"), ("min_inliers", "<i4"), ("min_cheirality_inliers", "<i4"), ("reserved", "<i4"),
    ("base_ransac_threshold", "<f8"), ("min_ransac_threshold", "<f8"), ("max_ransac_threshold", "<f8"),
    ("min_inlier_ratio", "<f8"), ("homography_bias", "<f8"), ("essential_bias", "<f8"), ("min_parallax", "<f8"),
    ("min_cheirality_ratio", "<f8")])

HOMOGRAPHY_THRESHOLD = 3.0        # ransac_homography's default, as _estimate_homography calls it


@dataclass(frozen=True)
class RobustPoseConfig:
    """The fields, defaults and validation of RobustPoseEstimatorConfig (robust_pose_estimator.py:42-70)."""
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

    @staticmethod
    def of(obj) -> "RobustPoseConfig":
        """Any object with the same field names (e.g. the drop-in's RobustPoseEstimatorConfig)."""
        if isinstance(obj, RobustPoseConfig):
            return obj
        return RobustPoseConfig(**{f.name: getattr(obj, f.name) for f in fields(RobustPoseConfig)})


def pack_configs(cfgs) -> np.ndarray:
    """RobustPoseConfig or a sequence of them -> b2s_robust_pose_config records (CONFIG_DTYPE)."""
    seq = [cfgs] if isinstance(cfgs, RobustPoseConfig) else list(cfgs)
    out = np.zeros(len(seq), CONFIG_DTYPE)
    for i, c in enumerate(seq):
        for f in fields(RobustPoseConfig):
            out[i][f.name] = getattr(c, f.name)
    return out


def decode_results(buf) -> np.ndarray:
    """Bytes of n b2s_pose_result structs (uint8 [n, 200] or flat) -> structured array (POSE_RESULT_DTYPE)."""
    a = np.ascontiguousarray(np.asarray(buf, dtype=np.uint8)).reshape(-1)
    if a.size % POSE_RESULT_BYTES:
        raise ValueError("buffer is not a whole number of pose results")
    return a.view(POSE_RESULT_DTYPE)


def homography_seed(seed: int) -> int:
    """Device-sampler seed of the homography branch: a splitmix64 step of the essential seed, so that the 4-sample
    and 8-sample streams (both keyed by (seed, pair, hypothesis)) do not share a state."""
    m = (1 << 64) - 1
    z = (int(seed) + 0x9E3779B97F4A7C15) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    z ^= z >> 31
    return z if z != (int(seed) & m) else z ^ 1


@dataclass
class RobustPoseOutput:
    """Views of RobustPose's buffers (the next run with the same shape overwrites them).  results: uint8
    [n_pairs, 200] b2s_pose_result; mask: uint8 [rows] the selected model's inlier flags; packed: results and mask
    in one buffer (one device->host copy).  The essential branch as Frontend exposes it: E, counts, best_h,
    best_count, inlier_mask (at the adaptive threshold), E_refit, R [n, 9], t [n, 3], votes [n, 4]; th / th2 the
    adaptive thresholds; H_fit [n, 9] the homography refit on the homography winner's inliers."""
    results: "torch.Tensor"
    mask: "torch.Tensor"
    packed: "torch.Tensor"
    th: "torch.Tensor"
    th2: "torch.Tensor"
    E: "torch.Tensor"
    counts: "torch.Tensor"
    best_h: "torch.Tensor"
    best_count: "torch.Tensor"
    inlier_mask: "torch.Tensor"
    E_refit: "torch.Tensor"
    R: "torch.Tensor"
    t: "torch.Tensor"
    votes: "torch.Tensor"
    H_fit: "torch.Tensor"


class RobustPose:
    """The stages of estimate_pose for many pairs, all libb2s kernels on the current stream:
    1. median displacement + adaptive threshold; 2. K4 + K3 + selection at th2_per_pair; 3. K7 refit, decomposition,
    pick + the inlier median; 4. K5 + K6 + selection at th = 3; 5. homography refit; 6. decomposition, selection,
    gates.  Buffers are kept per shape, so repeated runs allocate nothing."""

    def __init__(self):
        self._lib = _capi.load_library()
        self._key = None
        self._buf = None
        self._cfg_host = None
        self._cfg_dev = None

    def _buffers(self, dev, P: int, rows: int, He: int, Hh: int):
        import torch

        key = (str(dev), P, rows, He, Hh)
        if self._key == key:
            return self._buf
        P1, R1 = max(P, 1), max(rows, 1)
        f64, i32, u8 = torch.float64, torch.int32, torch.uint8
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)
        packed = torch.zeros(P1 * POSE_RESULT_BYTES + R1, dtype=u8, device=dev)
        self._buf = dict(
            packed=packed, results=packed[:P1 * POSE_RESULT_BYTES].view(P1, POSE_RESULT_BYTES), mask=packed[P1 * POSE_RESULT_BYTES:],
            th=e(P1, f64), th2=e(P1, f64), med_all=e(P1, torch.float32), med_in=e(P1, torch.float32),
            E=e((P1, max(He, 1), 9), f64), counts_e=e((P1, max(He, 1)), i32), best_h_e=e(P1, i32), best_c_e=e(P1, i32),
            mask_e=torch.zeros(R1, dtype=u8, device=dev), E_refit=e((P1, 9), f64), n_used=e(P1, i32),
            cand=e((P1, 4, 12), f64), votes=e((P1, 4), i32), R=e((P1, 9), f64), t=e((P1, 3), f64),
            Hm=e((P1, max(Hh, 1), 9), f64), counts_h=e((P1, max(Hh, 1)), i32), best_h_h=e(P1, i32), best_c_h=e(P1, i32),
            mask_h=torch.zeros(R1, dtype=u8, device=dev), H_fit=e((P1, 9), f64), h_used=e(P1, i32))
        self._key = key
        return self._buf

    def _configs(self, dev, cfg, n_pairs: int):
        import torch

        if isinstance(cfg, (list, tuple)):
            if len(cfg) != n_pairs:
                raise ValueError("one RobustPoseConfig per pair, or one for all")
            cfgs = [RobustPoseConfig.of(c) for c in cfg]
        else:
            cfgs = RobustPoseConfig.of(cfg)
        host = pack_configs(cfgs)
        if self._cfg_dev is None or self._cfg_dev.device != dev or not np.array_equal(self._cfg_host, host):
            # uploaded when the configuration changes only (the first, eager run of a captured step)
            self._cfg_host = host
            self._cfg_dev = torch.from_numpy(host.view(np.uint8).copy()).to(dev)
        return self._cfg_dev, len(host)

    def run(self, corr, c_off, c_count, n_pairs: int, K, cfg, samples_e=None, samples_h=None, seed: int = 0, *,
            max_m: int, hypotheses: int = 2000, precision: int = 64, mask_stride: int = 0, pair_id0: int = 0,
            records=None, sink_sel=None, before_records=None) -> RobustPoseOutput:
        """corr: device float32 [rows, 4] (x1, y1, x2, y2); c_off / c_count: device int32 CSR of the pairs; K: 3x3
        intrinsics (None = identity); cfg: RobustPoseConfig (or an object with its fields), or one per pair.
        samples_e [n_pairs, H, 8] / samples_h [n_pairs, H, 4]: host-drawn RANSAC samples (device int32), or None =
        the device sampler with `seed` (essential) and homography_seed(seed).  max_m >= every c_count (host-known);
        mask_stride: the compact stride when pairs live at p * stride (the unused tails of the masks are cleared).
        pair_id0: global id of pair 0; both device samplers draw from (seed, pair_id0 + p, h), so a pair draws the same
        samples in whichever batch or shard it is processed.  records (device uint8 [n_pairs, >= pose_record_bytes(S)])
        with sink_sel (the Selection in the compact layout, S = its stride): the decision kernel writes every pair's
        pose record, header pair id pair_id0 + p.  before_records: a callable run on the host immediately before the
        decision kernel is enqueued (ShardedFrontend joins the previous batch's collective there, which reads the buffer
        the kernel writes)."""
        torch = _capi.require_cuda()
        lib, st, P = self._lib, current_stream(), int(n_pairs)
        dev = corr.device
        He = int(samples_e.shape[1]) if samples_e is not None else int(hypotheses)
        Hh = int(samples_h.shape[1]) if samples_h is not None else int(hypotheses)
        b = self._buffers(dev, P, int(corr.shape[0]), He, Hh)
        cfg_d, n_cfg = self._configs(dev, cfg, P)
        Kd = np.eye(3) if K is None else np.asarray(K, dtype=np.float64).reshape(3, 3)
        Kd = np.ascontiguousarray(Kd)
        Kinv = np.ascontiguousarray(np.linalg.inv(Kd))
        c, o, n = ptr(corr), ptr(c_off), ptr(c_count)
        seed64 = C.c_uint64(int(seed) & (2**64 - 1))
        # 1. median displacement of all correspondences -> adaptive threshold
        check(lib.b2s_displacement_median_batched(c, o, n, None, P, ptr(cfg_d), n_cfg, ptr(b["med_all"]), ptr(b["th"]),
                                                  ptr(b["th2"]), st))
        # 2. essential RANSAC at the per-pair threshold
        check(lib.b2s_eight_point_batched(c, o, n, P, He, ptr(samples_e), seed64, None, int(pair_id0), None, ptr(Kd),
                                          ptr(Kinv), ptr(b["E"]), st))
        check(lib.b2s_ransac_score_batched(c, o, n, P, ptr(b["E"]), He, 0.0, ptr(b["th2"]), int(precision), int(max_m),
                                           ptr(b["counts_e"]), st))
        check(lib.b2s_ransac_select(ptr(b["counts_e"]), c, o, n, P, ptr(b["E"]), He, 0.0, ptr(b["th2"]), ptr(b["best_h_e"]),
                                    ptr(b["best_c_e"]), ptr(b["mask_e"]), None, int(mask_stride), st))
        # 3. refit on the inliers, decomposition + cheirality vote, pick; the inlier median
        check(lib.b2s_refit_essential_batched(c, o, n, ptr(b["mask_e"]), P, ptr(Kd), ptr(Kinv), ptr(b["E_refit"]),
                                              ptr(b["n_used"]), st))
        check(lib.b2s_decompose_essential_batched(ptr(b["E_refit"]), c, o, n, ptr(b["mask_e"]), P, int(max_m), ptr(Kd),
                                                  ptr(b["cand"]), ptr(b["votes"]), st))
        check(lib.b2s_pose_pick(ptr(b["cand"]), ptr(b["votes"]), P, ptr(b["R"]), ptr(b["t"]), st))
        check(lib.b2s_displacement_median_batched(c, o, n, ptr(b["mask_e"]), P, None, 0, ptr(b["med_in"]), None, None, st))
        # 4. homography RANSAC at th = 3
        check(lib.b2s_homography_dlt_batched(c, o, n, P, Hh, ptr(samples_h), C.c_uint64(homography_seed(seed)), None,
                                             int(pair_id0), None, ptr(b["Hm"]), st))
        check(lib.b2s_homography_score_batched(c, o, n, P, ptr(b["Hm"]), Hh, HOMOGRAPHY_THRESHOLD, None, ptr(b["counts_h"]), st))
        check(lib.b2s_homography_select(ptr(b["counts_h"]), c, o, n, P, ptr(b["Hm"]), Hh, HOMOGRAPHY_THRESHOLD, None,
                                        ptr(b["best_h_h"]), ptr(b["best_c_h"]), ptr(b["mask_h"]), st))
        # 5. n-point DLT on the homography winner's inliers
        check(lib.b2s_refit_homography_batched(c, o, n, ptr(b["mask_h"]), P, ptr(b["H_fit"]), ptr(b["h_used"]), st))
        # 6. decomposition, diagnostics, selection, gates (+ the pose records)
        sink = None
        if records is not None:
            if sink_sel is None or not sink_sel.stride:
                raise ValueError("pose records need the selection in the compact layout (sink_sel with a stride)")
            sink = _capi.RecordSink(records.data_ptr(), int(records.shape[-1]), sink_sel.out_q.data_ptr(),
                                    sink_sel.out_t.data_ptr(), sink_sel.out_d.data_ptr(), int(sink_sel.stride), int(pair_id0))
        if before_records is not None:
            before_records()
        check(lib.b2s_robust_pose_decide_records(
            o, n, P, ptr(b["best_h_e"]), ptr(b["best_c_e"]), ptr(b["mask_e"]), ptr(b["R"]), ptr(b["t"]), ptr(b["votes"]),
            ptr(b["med_in"]), ptr(b["med_all"]), ptr(b["th"]), ptr(b["best_h_h"]), ptr(b["best_c_h"]), ptr(b["mask_h"]),
            ptr(b["H_fit"]), ptr(Kinv), ptr(cfg_d), n_cfg, ptr(b["results"]), ptr(b["mask"]), int(mask_stride),
            C.byref(sink) if sink is not None else None, st))
        rows = int(corr.shape[0])
        return RobustPoseOutput(
            results=b["results"][:P], mask=b["mask"][:rows], packed=b["packed"][:P * POSE_RESULT_BYTES + rows] if P else b["packed"][:0],
            th=b["th"][:P], th2=b["th2"][:P], E=b["E"][:P, :He], counts=b["counts_e"][:P, :He], best_h=b["best_h_e"][:P],
            best_count=b["best_c_e"][:P], inlier_mask=b["mask_e"][:rows], E_refit=b["E_refit"][:P], R=b["R"][:P],
            t=b["t"][:P], votes=b["votes"][:P], H_fit=b["H_fit"][:P])
