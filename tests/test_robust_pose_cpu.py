"""CPU: the host side of the batched robust pose estimator — the result-struct decoder, the C layouts, the config
dataclass and the drop-in's host-side argument checks (no CUDA needed)."""
import re
from dataclasses import fields
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]

cv2 = pytest.importorskip("cv2")


def _define(name):
    text = (ROOT / "include" / "b2s.h").read_text()
    return int(re.search(rf"#define {name} (\d+)", text).group(1))


def _struct_fields(name):
    text = (ROOT / "include" / "b2s.h").read_text()
    body = re.search(r"typedef struct " + name + r" \{(.*?)\} " + name + ";", text, flags=re.S).group(1)
    out = []
    for line in body.splitlines():
        m = re.match(r"\s*(int32_t|double)\s+(\w+)(?:\[(\d+)\])?;", line)
        if m:
            out.append((m.group(2), m.group(1), int(m.group(3) or 1)))
    return out


def test_struct_layouts_match_the_header():
    from b200slam import robust_pose as rp
    assert rp.POSE_RESULT_DTYPE.itemsize == rp.POSE_RESULT_BYTES == _define("B2S_POSE_RESULT_BYTES")
    assert rp.CONFIG_DTYPE.itemsize == rp.ROBUST_POSE_CONFIG_BYTES == _define("B2S_ROBUST_POSE_CONFIG_BYTES")
    for dt, name in ((rp.POSE_RESULT_DTYPE, "b2s_pose_result"), (rp.CONFIG_DTYPE, "b2s_robust_pose_config")):
        hdr = _struct_fields(name)
        assert [f[0] for f in hdr] == list(dt.names)
        for fname, ctype, count in hdr:
            sub = dt.fields[fname][0]
            base = sub.base if sub.shape else sub
            assert base == np.dtype("<i4" if ctype == "int32_t" else "<f8"), fname
            assert (int(np.prod(sub.shape)) if sub.shape else 1) == count, fname
    for i, n in enumerate(("ESTIMATE", "GATE_FAILED", "ERR_MATCHES", "ERR_EIGHT", "ERR_ESSENTIAL", "ERR_HOMOGRAPHY",
                           "ERR_TRANSLATION")):
        assert _define(f"B2S_POSE_{n}") == i == getattr(rp, f"POSE_{n}")
    for i, reason in enumerate(rp.GATE_REASONS[1:], start=1):
        assert _define(f"B2S_GATE_{reason.upper()}") == i


def test_config_mirrors_the_reference_config():
    from b200slam.robust_pose import RobustPoseConfig
    from integration.pose_bridge import RobustPoseEstimatorConfig
    a, b = fields(RobustPoseConfig), fields(RobustPoseEstimatorConfig)
    assert [(f.name, f.type, f.default) for f in a] == [(f.name, f.type, f.default) for f in b]
    for bad in (dict(min_matches=0), dict(min_inliers=0), dict(min_inlier_ratio=0.0), dict(min_parallax=-1.0),
                dict(min_cheirality_ratio=0.0), dict(min_cheirality_inliers=0)):
        with pytest.raises(ValueError) as e1:
            RobustPoseConfig(**bad)
        with pytest.raises(ValueError) as e2:
            RobustPoseEstimatorConfig(**bad)
        assert str(e1.value) == str(e2.value)
    c = RobustPoseEstimatorConfig(min_matches=7, homography_bias=0.5)
    assert RobustPoseConfig.of(c) == RobustPoseConfig(min_matches=7, homography_bias=0.5)


def test_frontend_config_defaults_to_off():
    from b200slam.frontend import FrontendConfig
    assert FrontendConfig().robust_pose is None


def test_homography_seed_differs_from_the_essential_seed():
    from b200slam.robust_pose import homography_seed
    for s in (0, 1, 1337, 2**63 - 1, 2**64 - 1):
        h = homography_seed(s)
        assert h != s and 0 <= h < 2**64 and homography_seed(s) == h


def _record(**kw):
    from b200slam import robust_pose as rp
    r = np.zeros(1, rp.POSE_RESULT_DTYPE)
    r["e_best_h"] = r["h_best_h"] = -1
    for k, v in kw.items():
        r[k] = v
    return rp.decode_results(r.view(np.uint8))[0]


def test_decoder_builds_the_single_calls_answers():
    from b200slam import robust_pose as rp
    from integration import pose_bridge as pb
    R = np.eye(3).reshape(-1) * 1.0
    est = pb.decode_pose_result(_record(outcome=rp.POSE_ESTIMATE, method=1, match_count=50, inliers=40, cheirality_inliers=40,
                                        inlier_ratio=0.8, median_parallax=np.float64(np.float32(3.7)), cheirality_ratio=1.0,
                                        score=2.664, R=R, t=[0.0, 0.6, 0.8]), np.arange(40))
    assert isinstance(est, pb.PoseEstimate)
    assert est.diagnostics == pb.PoseEstimationDiagnostics("homography", 50, 40, 0.8, float(np.float32(3.7)), 40, 1.0, 2.664)
    assert isinstance(est.diagnostics.match_count, int) and isinstance(est.diagnostics.score, float)
    np.testing.assert_array_equal(est.rotation, np.eye(3))
    np.testing.assert_array_equal(est.translation, [0.0, 0.6, 0.8])
    assert est.inlier_indices.dtype == np.int64
    for gate, reason in enumerate(rp.GATE_REASONS[1:], start=1):
        f = pb.decode_pose_result(_record(outcome=rp.POSE_GATE_FAILED, gate=gate, method=0, match_count=30, inliers=20,
                                          cheirality_inliers=9, inlier_ratio=2 / 3, median_parallax=0.5,
                                          cheirality_ratio=0.45), np.arange(20))
        assert isinstance(f, pb.PoseEstimationFailure) and isinstance(f, RuntimeError)
        assert (f.reason, f.recovery_action) == (reason, "relocalize")
        assert str(f) == f"{reason} (recovery=relocalize)"
        assert f.metrics == {"match_count": 30.0, "inliers": 20.0, "inlier_ratio": 2 / 3, "median_parallax": 0.5,
                             "cheirality_ratio": 0.45, "cheirality_inliers": 9.0}
    cases = {rp.POSE_ERR_MATCHES: (ValueError, "Not enough matches for pose estimation"),
             rp.POSE_ERR_EIGHT: (ValueError, "At least eight correspondences are required"),
             rp.POSE_ERR_ESSENTIAL: (RuntimeError, "Essential matrix pose estimation failed"),
             rp.POSE_ERR_HOMOGRAPHY: (RuntimeError, "Homography pose estimation failed"),
             rp.POSE_ERR_TRANSLATION: (ValueError, "Translation norm is zero")}
    for code, (typ, msg) in cases.items():
        e = pb.decode_pose_result(_record(outcome=code), np.zeros(0, np.int64))
        assert type(e) is typ and str(e) == msg


def test_homography_generator_is_rewound_when_the_essential_branch_raises():
    from b200slam import robust_pose as rp
    from integration import pose_bridge as pb
    assert not pb._homography_ran(_record(outcome=rp.POSE_ERR_ESSENTIAL))
    assert not pb._homography_ran(_record(outcome=rp.POSE_ERR_TRANSLATION, method=0))
    assert pb._homography_ran(_record(outcome=rp.POSE_ERR_TRANSLATION, method=1))
    assert pb._homography_ran(_record(outcome=rp.POSE_ERR_HOMOGRAPHY))
    assert pb._homography_ran(_record(outcome=rp.POSE_GATE_FAILED))


def _pairs(n):
    kp = [cv2.KeyPoint(float(i), float(2 * i), 1.0) for i in range(n)]
    return kp, list(kp), [cv2.DMatch(_queryIdx=i, _trainIdx=i, _distance=0.0) for i in range(n)]


def test_rejected_pairs_need_no_cuda():
    from integration import pose_bridge as pb
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig(min_matches=5))
    a, b, c = _pairs(3), _pairs(6), ([], [], [cv2.DMatch(0, 0, 0.0)] * 5)
    out = est.estimate_pose_batch([a[0], b[0], c[0]], [a[1], b[1], c[1]], [a[2], b[2], c[2]], np.eye(3))
    assert [type(x) for x in out] == [ValueError] * 3
    assert [str(x) for x in out] == ["Not enough matches for pose estimation", "At least eight correspondences are required",
                                     "Keypoints must be non-empty"]
    with pytest.raises(ValueError, match="Intrinsics must be a 3x3 matrix"):
        est.estimate_pose_batch([a[0]], [a[1]], [a[2]], np.eye(4))
    assert est.estimate_pose_batch([], [], [], np.eye(3)) == []


def test_a_pair_for_the_device_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from b200slam import B2SError
    from integration import pose_bridge as pb
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig(min_matches=5))
    a, b = _pairs(3), _pairs(40)
    with pytest.raises(B2SError):
        est.estimate_pose_batch([a[0], b[0]], [a[1], b[1]], [a[2], b[2]], np.eye(3))
