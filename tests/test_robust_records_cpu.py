"""CPU: the pose record layout (include/b2s.h) as the library, the header and the host decoder see it."""
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_pose_record_bytes_is_the_record_plus_256():
    from b200slam import _capi
    from b200slam.frontend import pose_record_bytes, record_bytes
    lib = _capi.load_library()
    for S in (1, 63, 64, 200, 500, 4096):
        assert lib.b2s_pose_record_bytes(S) == lib.b2s_record_bytes(S) + 256
        assert pose_record_bytes(S) == record_bytes(S) + 256
        assert record_bytes(S) % 64 == 0                           # the pose block starts on a 64-byte boundary
    assert pose_record_bytes(500) == 3840 and record_bytes(500) == 3584


def test_pose_block_and_result_layout_match_the_header():
    from b200slam import robust_pose as rp
    text = (ROOT / "include" / "b2s.h").read_text()
    assert int(re.search(r"#define B2S_POSE_BLOCK_BYTES (\d+)", text).group(1)) == 256
    assert int(re.search(r"#define B2S_POSE_RESULT_BYTES (\d+)", text).group(1)) == rp.POSE_RESULT_BYTES == 200
    assert rp.POSE_RESULT_DTYPE.itemsize == 200
    body = re.search(r"typedef struct b2s_pose_result \{(.*?)\} b2s_pose_result;", text, flags=re.S).group(1)
    fields = []
    for m in re.finditer(r"(int32_t|double)\s+([A-Za-z_0-9]+)(?:\[(\d+)\])?;", body):
        fields.append((m.group(2), m.group(1), int(m.group(3) or 1)))
    off = 0
    for name, ctype, n in fields:
        assert name in rp.POSE_RESULT_DTYPE.names, name
        dt, o = rp.POSE_RESULT_DTYPE.fields[name][:2]
        assert o == off, name
        assert dt.itemsize == (4 if ctype == "int32_t" else 8) * n, name
        off += dt.itemsize
    assert off == 200 and list(rp.POSE_RESULT_DTYPE.names) == [f[0] for f in fields]
    # the offsets the header's static_asserts pin
    for name, o in (("inlier_ratio", 48), ("threshold", 96), ("R", 104), ("t", 176)):
        assert rp.POSE_RESULT_DTYPE.fields[name][1] == o


def test_abi_version_is_5_and_agrees_with_the_library():
    from b200slam import _capi
    text = (ROOT / "include" / "b2s.h").read_text()
    assert int(re.search(r"#define B2S_ABI_VERSION (\d+)", text).group(1)) == 5
    assert _capi.ABI_VERSION == 5
    assert _capi.load_library().b2s_abi_version() == 5


def _pose_record(S, *, n, best_h, inliers, pair_id, R, t, q, ti, d, flags, result):
    from b200slam.frontend import pose_record_bytes, record_bytes
    rec = np.zeros(pose_record_bytes(S), np.uint8)
    hdr = np.zeros(16, np.int32)
    hdr[:4] = (n, best_h, inliers, pair_id)
    hdr[4:13] = np.asarray(R, np.float32).reshape(9).view(np.int32)
    hdr[13:16] = np.asarray(t, np.float32).view(np.int32)
    rec[:64] = hdr.view(np.uint8)
    m = max(n, 0)
    body = np.zeros((3, S), np.uint16)
    body[0, :m], body[1, :m], body[2, :m] = q, ti, d
    rec[64:64 + 6 * S] = body.reshape(-1).view(np.uint8)
    rec[64 + 6 * S:64 + 6 * S + m] = flags
    rb = record_bytes(S)
    rec[rb:rb + 200] = result.view(np.uint8)
    return rec


def test_unpack_records_decodes_hand_built_pose_records():
    from b200slam import robust_pose as rp
    from b200slam.frontend import pose_record_bytes, unpack_records
    S = 63
    rng = np.random.default_rng(0)
    ok = np.zeros(1, rp.POSE_RESULT_DTYPE)
    ok["outcome"], ok["method"], ok["match_count"], ok["inliers"] = rp.POSE_ESTIMATE, 1, 40, 31
    ok["e_best_h"], ok["e_inliers"], ok["h_best_h"], ok["h_inliers"] = 17, 29, 5, 31
    ok["inlier_ratio"], ok["median_parallax"], ok["score"], ok["threshold"] = 31 / 40, 3.25, 0.6, 0.01
    R = np.eye(3)[[1, 0, 2]] * np.array([1.0, -1.0, 1.0])
    ok["R"], ok["t"] = R.reshape(1, 9), np.array([[0.6, 0.0, -0.8]])
    flags = (rng.random(40) < 0.8).astype(np.uint8)
    r0 = _pose_record(S, n=40, best_h=5, inliers=31, pair_id=7, R=R, t=ok["t"][0], q=rng.integers(0, 900, 40),
                      ti=rng.integers(0, 900, 40), d=rng.integers(0, 256, 40), flags=flags, result=ok)
    err = np.zeros(1, rp.POSE_RESULT_DTYPE)
    err["outcome"], err["match_count"] = rp.POSE_ERR_MATCHES, 12
    err["e_best_h"] = err["h_best_h"] = err["e_inliers"] = err["h_inliers"] = -1
    r1 = _pose_record(S, n=12, best_h=-1, inliers=0, pair_id=8, R=np.zeros(9), t=np.zeros(3), q=np.arange(12),
                      ti=np.arange(12) + 3, d=np.full(12, 9), flags=np.zeros(12, np.uint8), result=err)
    buf = np.stack([r0, r1])
    for arg in (buf, buf.reshape(-1)):
        u = unpack_records(arg, S, pose=True)
        np.testing.assert_array_equal(u["n_matches"], [40, 12])
        np.testing.assert_array_equal(u["best_h"], [5, -1])
        np.testing.assert_array_equal(u["inliers"], [31, 0])
        np.testing.assert_array_equal(u["pair_id"], [7, 8])
        np.testing.assert_array_equal(u["R"][0], R.astype(np.float32))
        np.testing.assert_array_equal(u["t"][0], np.array([0.6, 0.0, -0.8], np.float32))
        assert not u["R"][1].any() and not u["t"][1].any() and not u["inlier"][1].any()
        np.testing.assert_array_equal(u["inlier"][0, :40], flags)
        assert not u["inlier"][0, 40:].any() and not u["q"][1, 12:].any()
        np.testing.assert_array_equal(u["q"][1, :12], np.arange(12))
        assert u["robust"].dtype == rp.POSE_RESULT_DTYPE and len(u["robust"]) == 2
        assert u["robust"][0].tobytes() == ok.tobytes() and u["robust"][1].tobytes() == err.tobytes()
    assert "robust" not in unpack_records(buf[:, :pose_record_bytes(S) - 256], S)
    with pytest.raises(ValueError):
        unpack_records(buf[:, :pose_record_bytes(S) - 256], S, pose=True)


def test_record_view_exposes_the_pose_block():
    import torch
    from b200slam import robust_pose as rp
    from b200slam.frontend import RecordView
    S = 8
    res = np.zeros(1, rp.POSE_RESULT_DTYPE)
    res["outcome"], res["method"], res["gate"], res["inliers"] = rp.POSE_GATE_FAILED, 0, 3, 4
    rec = _pose_record(S, n=5, best_h=2, inliers=4, pair_id=0, R=np.eye(3), t=np.array([0.0, 0.0, 1.0]), q=np.arange(5),
                       ti=np.arange(5), d=np.arange(5), flags=np.array([1, 1, 0, 1, 1], np.uint8), result=res)
    v = RecordView(torch.from_numpy(rec[None].copy()), S, pose=True)
    assert v["robust"][0].tobytes() == res.tobytes()
    assert int(v["best_count"][0]) == 4 and v["mask"][:5].tolist() == [1, 1, 0, 1, 1]
    plain = RecordView(torch.from_numpy(rec[None, :-256].copy()), S)
    with pytest.raises(KeyError):
        plain["robust"]


def test_empty_slots_of_a_sharded_gather_never_decode_as_an_estimate():
    import torch
    from b200slam import robust_pose as rp
    from b200slam.frontend import FrontendConfig, pose_record_bytes, record_bytes, unpack_records
    from b200slam.sharding import _mark_empty
    S = 200
    rows = torch.zeros((3, pose_record_bytes(S)), dtype=torch.uint8)
    _mark_empty(rows, FrontendConfig(max_matches=S, robust_pose=rp.RobustPoseConfig()))
    u = unpack_records(rows.numpy(), S, pose=True)
    assert (u["pair_id"] == -1).all() and (u["robust"]["outcome"] == rp.POSE_EMPTY).all()
    assert not u["n_matches"].any() and not u["inlier"].any()
    plain = torch.zeros((2, record_bytes(S)), dtype=torch.uint8)
    _mark_empty(plain, FrontendConfig(max_matches=S))
    u = unpack_records(plain.numpy(), S)
    assert (u["pair_id"] == -1).all() and int(plain[:, 16:].sum()) == 0


def test_record_view_repeats_the_overflow_error():
    import torch
    from b200slam import _capi
    from b200slam.frontend import RecordView, record_bytes
    rec = np.zeros((1, record_bytes(8)), np.uint8)
    rec[0, :4] = np.array([-1], np.int32).view(np.uint8)          # n_matches = -1: a pair overflowed the stride
    v = RecordView(torch.from_numpy(rec), 8)
    for _ in range(2):
        with pytest.raises(_capi.B2SError):
            v["count"]
