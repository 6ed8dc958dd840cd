"""GPU: pose records — the robust pose answer (b2s_pose_result + the selected model's flags) carried in the result
records that leave the GPU, from every front door and keyed by the global pair id.  Every comparison is byte-equal."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
S = 500


def _rcfg():
    from b200slam.robust_pose import RobustPoseConfig
    # K = I scenes in normalised coordinates: th = 3 makes every correspondence a homography inlier, so a pair with
    # outliers selects the homography (0.9 > its essential inlier ratio) and an outlier-free pair the essential model;
    # 20-match pairs fail the inlier-count gate, 6-match pairs raise "fewer than eight", 3-match pairs "min_matches"
    return RobustPoseConfig(min_matches=5, min_parallax=0.0)


def _scene_pairs(n_pairs, seed=0):
    """Descriptor pairs whose cross-checked matches are known correspondences: (qs, ts, kq, kt).  Kinds by position:
    outlier-free 300-match pairs, 35 %-outlier 300-match pairs, 20-, 6- and 3-match pairs (the tiny ones last)."""
    rng = np.random.default_rng(seed)
    tail = ["gate"] * 6 + ["eight"] * 3 + ["few"] * 3
    kinds = (["clean", "outliers"] * n_pairs)[:max(0, n_pairs - len(tail))] + tail
    kinds = kinds[:n_pairs]
    qs, ts, kq, kt = [], [], [], []
    for kind in kinds:
        n = {"clean": 300, "outliers": 300, "gate": 20, "eight": 6, "few": 3}[kind]
        extra = 200 if n >= 20 else 10
        P = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 12, n)], 1)
        a = rng.uniform(-0.05, 0.05, 3)
        cx, sx, cy, sy, cz, sz = np.cos(a[0]), np.sin(a[0]), np.cos(a[1]), np.sin(a[1]), np.cos(a[2]), np.sin(a[2])
        R = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]]) @ \
            np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        t = rng.uniform(-0.5, 0.5, 3) + np.array([0.3, 0.0, 0.0])
        c2 = P @ R.T + t
        p1 = P[:, :2] / P[:, 2:] + rng.normal(0, 5e-4, (n, 2))
        p2 = c2[:, :2] / c2[:, 2:] + rng.normal(0, 5e-4, (n, 2))
        if kind == "outliers":
            k = int(0.35 * n)
            idx = rng.permutation(n)[:k]
            p2[idx] = rng.uniform(p2.min(0), p2.max(0), (k, 2))
        q = rng.integers(0, 256, (n + extra, 32), dtype=np.uint8)
        tr = rng.integers(0, 256, (n + extra, 32), dtype=np.uint8)
        bits = np.unpackbits(q[:n], axis=1)
        bits ^= (rng.random(bits.shape) < 0.03).astype(np.uint8)
        tr[:n] = np.packbits(bits, axis=1)
        a1 = np.vstack([p1, rng.uniform(-0.6, 0.6, (extra, 2))]).astype(np.float32)
        a2 = np.vstack([p2, rng.uniform(-0.6, 0.6, (extra, 2))]).astype(np.float32)
        perm = rng.permutation(n + extra)
        qs.append(q), ts.append(tr[perm]), kq.append(a1), kt.append(a2[perm])
    return qs, ts, kq, kt


def _fe(**kw):
    from b200slam.frontend import Frontend, FrontendConfig
    return Frontend(FrontendConfig(max_matches=S, robust_pose=_rcfg(), seed=2024, **kw))


def _host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().copy()


@pytest.mark.parametrize("scale", [1.0, 700.0], ids=["normalised_K_I", "pixel_scale_K"])
def test_records_equal_the_result_arrays(scale):
    """scale 700: the same scenes at pixel scale with their intrinsics K = diag(700, 700, 1)."""
    import torch
    from b200slam import _capi
    from b200slam import robust_pose as rp
    from b200slam.frontend import PairBatch, pack_records, pose_record_bytes, record_bytes, unpack_records
    qs, ts, kq, kt = _scene_pairs(32, seed=1)
    K = None if scale == 1.0 else np.diag([scale, scale, 1.0])
    kq, kt = [k * np.float32(scale) for k in kq], [k * np.float32(scale) for k in kt]
    b = PairBatch.from_host(qs, ts, kq, kt)
    P, rb = b.n_pairs, record_bytes(S)
    lib = _capi.load_library()
    fe = _fe()
    fe.run(b, K=K)                                                      # warm-up: lazy init, buffers of the shape
    n0 = lib.b2s_launch_count()
    plain = fe.run(b, K=K)
    n1 = lib.b2s_launch_count()
    want_res, want_mask = _host(plain.robust), _host(plain.robust_mask)
    rec = torch.full((P, pose_record_bytes(S)), 0xAB, dtype=torch.uint8, device="cuda")
    res = fe.run(b, K=K, records=rec, pair_id0=0)
    n2 = lib.b2s_launch_count()
    assert n2 - n1 == n1 - n0                                           # the records cost no launch
    assert res.records is rec
    got_rec, got_res, got_mask = _host(rec), _host(res.robust), _host(res.robust_mask)
    np.testing.assert_array_equal(got_res, want_res)                    # records change nothing else
    np.testing.assert_array_equal(got_mask, want_mask)
    r = rp.decode_results(got_res)
    cnt = _host(res.sel.count)
    # the pose block is the result, then 56 zero bytes
    np.testing.assert_array_equal(got_rec[:, rb:rb + 200], got_res.reshape(P, 200))
    assert not got_rec[:, rb + 200:].any()
    # q / t / d as pack_records writes them for the same selection
    ref = torch.zeros((P, rb), dtype=torch.uint8, device="cuda")
    pack_records(ref, res.sel, n_records=P)
    ref = _host(ref)
    np.testing.assert_array_equal(got_rec[:, 64:64 + 6 * S], ref[:, 64:64 + 6 * S])
    # flags: robust_mask in the compact layout, zero tail; the padding up to the pose block is zero
    np.testing.assert_array_equal(got_rec[:, 64 + 6 * S:64 + 7 * S], want_mask.reshape(P, S))
    assert not got_rec[:, 64 + 7 * S:rb].any()
    # header
    u = unpack_records(got_rec, S, pose=True)
    np.testing.assert_array_equal(u["n_matches"], cnt)
    answer = np.isin(r["outcome"], [rp.POSE_ESTIMATE, rp.POSE_GATE_FAILED])
    np.testing.assert_array_equal(u["best_h"], np.where(answer, np.where(r["method"] == 1, r["h_best_h"], r["e_best_h"]), -1))
    np.testing.assert_array_equal(u["inliers"], r["inliers"])
    np.testing.assert_array_equal(u["pair_id"], np.arange(P))
    np.testing.assert_array_equal(u["R"].reshape(P, 9), r["R"].astype(np.float32))
    np.testing.assert_array_equal(u["t"], r["t"].astype(np.float32))
    assert u["robust"].tobytes() == got_res.tobytes()
    for p in range(P):
        assert not u["inlier"][p, max(cnt[p], 0):].any()
        if not answer[p]:
            assert not u["R"][p].any() and not u["t"][p].any() and not u["inlier"][p].any()
    # the batch covers every kind of answer.  At pixel scale the 300- and 20-match pairs end in the essential branch's
    # RuntimeError: the reference's essential path (K^T F K applied to pixel points, thresholds in point units) is only
    # self-consistent for K = I, and the records must carry that answer as faithfully as any other
    kinds = {(int(o), int(m)) for o, m in zip(r["outcome"], r["method"])}
    assert (rp.POSE_ERR_MATCHES, 0) in kinds and (rp.POSE_ERR_EIGHT, 0) in kinds, kinds
    if K is None:
        assert any(o == rp.POSE_GATE_FAILED for o, _ in kinds), kinds
        assert (rp.POSE_ESTIMATE, 0) in kinds and any(m == 1 and o in (0, 1) for o, m in kinds), kinds
    else:
        assert (rp.POSE_ERR_ESSENTIAL, 0) in kinds, kinds
    # a narrower buffer is refused before anything is launched; the C ABI refuses a narrow sink too
    with pytest.raises(_capi.B2SError):
        fe.run(b, K=K, records=torch.zeros((P, pose_record_bytes(S) - 16), dtype=torch.uint8, device="cuda"))
    with pytest.raises(_capi.B2SError):
        fe.run(b, K=K, records=torch.zeros((P, record_bytes(S)), dtype=torch.uint8, device="cuda"))
    narrow = torch.zeros((P, record_bytes(S)), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="b2s_pose_record_bytes"):
        fe.robust.run(res.sel.corr, res.sel.c_off, res.sel.count, P, K, _rcfg(), seed=2024, max_m=S, mask_stride=S,
                      records=narrow, sink_sel=res.sel)


def test_refusals_kept():
    from b200slam.frontend import PairBatch
    qs, ts, kq, kt = _scene_pairs(4, seed=2)
    b = PairBatch.from_host(qs, ts, kq, kt)
    for kw in (dict(winner_only=True), dict(scoring="tc")):
        with pytest.raises(ValueError):
            _fe(**kw).run(b)


@pytest.mark.parametrize("k", [0, 1, 13, 36, 37])
def test_a_pair_answers_the_same_in_any_batch_position(k):
    """[0, k) with pair_id0 = 0 and [k, 37) with pair_id0 = k answer what the whole batch answers: both samplers are
    keyed by the global pair id."""
    import torch
    from b200slam import robust_pose as rp
    from b200slam.frontend import PairBatch, pose_record_bytes
    qs, ts, kq, kt = _scene_pairs(37, seed=3)
    fe = _fe()
    whole = torch.zeros((37, pose_record_bytes(S)), dtype=torch.uint8, device="cuda")
    rw = fe.run(PairBatch.from_host(qs, ts, kq, kt), records=whole)
    w_res, w_mask, w_rec = _host(rw.robust), _host(rw.robust_mask).reshape(37, S), _host(whole)
    parts_res, parts_mask, parts_rec = [], [], []
    for lo, hi in ((0, k), (k, 37)):
        if hi == lo:
            continue
        rec = torch.zeros((hi - lo, pose_record_bytes(S)), dtype=torch.uint8, device="cuda")
        r = _fe().run(PairBatch.from_host(qs[lo:hi], ts[lo:hi], kq[lo:hi], kt[lo:hi]), records=rec, pair_id0=lo)
        parts_res.append(_host(r.robust)), parts_mask.append(_host(r.robust_mask).reshape(hi - lo, S)), parts_rec.append(_host(rec))
    np.testing.assert_array_equal(np.concatenate(parts_res), w_res)      # includes the E / H winners (e_best_h, h_best_h)
    np.testing.assert_array_equal(np.concatenate(parts_mask), w_mask)
    np.testing.assert_array_equal(np.concatenate(parts_rec), w_rec)
    r = rp.decode_results(w_res)
    assert (r["h_best_h"] >= 0).sum() >= 20                              # the homography sampler ran on most pairs


def test_homography_sampler_is_keyed_by_the_global_pair_id():
    import torch
    from b200slam.frontend import HomographyRansac
    rng = np.random.default_rng(4)
    counts = rng.integers(4, 400, 37).astype(np.int32)
    off = np.zeros(38, np.int32)
    np.cumsum(counts, out=off[1:])
    corr = torch.from_numpy(rng.uniform(-1, 1, (int(off[-1]), 4)).astype(np.float32)).cuda()
    o, c = torch.from_numpy(off).cuda(), torch.from_numpy(counts).cuda()
    R = HomographyRansac()
    H0, s0 = R.hypotheses(corr, o, c, 37, 64, seed=7, return_samples=True)
    H0, s0 = _host(H0), _host(s0)
    for k in (1, 13, 36):
        Hk, sk = R.hypotheses(corr, o[k:], c[k:], 37 - k, 64, seed=7, return_samples=True, pair_id0=k)
        np.testing.assert_array_equal(_host(sk), s0[k:])
        np.testing.assert_array_equal(_host(Hk), H0[k:])
    rev = np.arange(36, -1, -1)
    ids = torch.from_numpy(rev.astype(np.int32)).cuda()
    o_r = torch.from_numpy(off[:-1][rev].copy()).cuda()
    c_r = torch.from_numpy(counts[rev].copy()).cuda()
    Hr, sr = R.hypotheses(corr, o_r, c_r, 37, 64, seed=7, return_samples=True, pair_ids=ids, pair_id0=1000)
    np.testing.assert_array_equal(_host(sr), s0[rev])
    np.testing.assert_array_equal(_host(Hr), H0[rev])


def _sequence(F=9, N=700, seed=11):
    from b200slam.synthetic import tracking_sequence
    desc, kp = tracking_sequence(F, N, seed=seed)
    return desc, kp * np.float32(700), np.diag([700.0, 700.0, 1.0])        # pixel-like scale with its K


def _seq_cfg():
    from b200slam.frontend import FrontendConfig
    from b200slam.robust_pose import RobustPoseConfig
    return FrontendConfig(max_matches=S, robust_pose=RobustPoseConfig(min_parallax=0.5), seed=2024)


def test_sequence_tracker_and_pipelines_carry_the_answer():
    import torch
    from b200slam.frontend import Frontend, SequencePipeline, SequenceTracker, pose_record_bytes, sequence_batch
    desc, kp, K = _sequence()
    F, N = desc.shape[:2]
    counts = np.full(F, N, np.int32)
    counts[3] = 640                                                     # ragged frame sizes
    cfg = _seq_cfg()
    rec = torch.zeros((F - 1, pose_record_bytes(S)), dtype=torch.uint8, device="cuda")
    b = sequence_batch(torch.from_numpy(desc.reshape(-1, 32)).cuda(), torch.from_numpy(kp.reshape(-1, 2)).cuda(), counts, 0, F - 1, N)
    ref_res = Frontend(cfg).run(b, K=K, records=rec)
    want = _host(rec)
    dh = torch.from_numpy(desc.reshape(-1, 32)).pin_memory()
    kh = torch.from_numpy(kp.reshape(-1, 2)).pin_memory()
    for chunks in (1, 4):
        for graph in (False, True):
            tr = SequenceTracker(F, N, cfg, chunks=chunks, use_graph=graph, K=K)
            assert tr.rec_bytes == pose_record_bytes(S)
            for _ in range(3):                                          # eager, capture, replay
                tr.rec_host.zero_()
                v = tr.run(dh, kh, counts)
                torch.cuda.synchronize()
                np.testing.assert_array_equal(v.records.numpy(), want, err_msg=f"chunks={chunks} graph={graph}")
            assert v["robust"].tobytes() == _host(ref_res.robust).tobytes()
    for schedule in ("interleaved", "serial"):
        pl = SequencePipeline(F, N, cfg, depth=3, schedule=schedule, K=K)
        slots = [pl.submit(dh, kh, counts) for _ in range(6)]           # two steps per slot
        for s in slots:
            v = pl.result(s)
            np.testing.assert_array_equal(v.records.numpy(), want, err_msg=schedule)
        np.testing.assert_array_equal(v["mask"].numpy(), _host(ref_res.robust_mask))
    # the decoded answer against the drop-in on the same correspondences (same positions: same device draws)
    cv2 = pytest.importorskip("cv2")
    from integration import pose_bridge as pb
    cnt, corr = _host(ref_res.sel.count), _host(ref_res.sel.corr)
    kps = []
    for p in range(F - 1):
        c = corr[p * S:p * S + cnt[p]]
        kps.append(([cv2.KeyPoint(float(x), float(y), 1.0) for x, y in c[:, :2]],
                    [cv2.KeyPoint(float(x), float(y), 1.0) for x, y in c[:, 2:]],
                    [cv2.DMatch(_queryIdx=j, _trainIdx=j, _distance=0.0) for j in range(len(c))]))
    assert (cnt >= 20).all()
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig(min_parallax=0.5))
    got = est.estimate_pose_batch([k[0] for k in kps], [k[1] for k in kps], [k[2] for k in kps], K, seed=2024)
    mask = v["mask"].numpy().reshape(F - 1, S)
    assert len(got) >= 8
    for p in range(F - 1):
        mine = pb.decode_pose_result(v["robust"][p], np.flatnonzero(mask[p, :cnt[p]]))
        assert type(mine) is type(got[p]), (p, mine, got[p])
        if isinstance(mine, pb.PoseEstimate):
            np.testing.assert_array_equal(mine.rotation, got[p].rotation)
            np.testing.assert_array_equal(mine.translation, got[p].translation)
            np.testing.assert_array_equal(np.asarray(mine.inlier_indices), np.asarray(got[p].inlier_indices))
            assert mine.diagnostics == got[p].diagnostics
        elif isinstance(mine, pb.PoseEstimationFailure):
            assert (mine.reason, mine.metrics) == (got[p].reason, got[p].metrics)
        else:
            assert str(mine) == str(got[p])


def test_pair_pipeline_carries_the_answer():
    import torch
    from b200slam.frontend import FrontendConfig, PairBatch, PairPipeline, pose_record_bytes
    qs, ts, kq, kt = _scene_pairs(24, seed=5)
    rec = torch.zeros((24, pose_record_bytes(S)), dtype=torch.uint8, device="cuda")
    _fe().run(PairBatch.from_host(qs, ts, kq, kt), records=rec)
    want = _host(rec)
    pp = PairPipeline(24, 600, 600, FrontendConfig(max_matches=S, robust_pose=_rcfg(), seed=2024), depth=2)
    staged = pp.stage_host(qs, ts, kq, kt)
    slots = [pp.submit(staged) for _ in range(4)]
    for s in slots:
        v = pp.result(s)
        np.testing.assert_array_equal(v.records.numpy(), want)
    assert v["robust"].tobytes() == want[:, -256:-56].tobytes()


def test_sharded_frontend_world1_and_lanes():
    import torch
    from b200slam.frontend import Frontend, FrontendConfig, PairBatch, pose_record_bytes
    from b200slam.sharding import ShardedFrontend
    cfg = FrontendConfig(max_matches=S, robust_pose=_rcfg(), seed=2024, hypotheses=512)
    sets = [_scene_pairs(14, seed=20 + j) for j in range(5)]
    bl = [PairBatch.from_host(*s) for s in sets]
    want = []
    for b in bl:
        rec = torch.zeros((14, pose_record_bytes(S)), dtype=torch.uint8, device="cuda")
        Frontend(cfg).run(b, records=rec)
        want.append(_host(rec))
    # one launch set, captured and replayed
    sf = ShardedFrontend(cfg, 14)
    assert sf.rec_bytes == pose_record_bytes(S)
    sf.capture(bl[0])
    sf.gather.buf.zero_()
    sf.replay()
    sf.flush()
    np.testing.assert_array_equal(_host(sf.records()[0]), want[0])
    sf.close()
    # five launch sets over 3 lanes equal 1 lane, eagerly and replayed
    got = {}
    for lanes in (1, 3):
        sf = ShardedFrontend(cfg, 14, sets_per_gather=5, lanes=lanes)
        for b in bl:
            sf.step(b)
        sf.flush()
        eager = _host(sf.records())
        sf.capture(bl)
        sf.gather.buf.zero_()
        for _ in range(2):
            sf.replay()
        sf.flush()
        np.testing.assert_array_equal(_host(sf.records()), eager)
        got[lanes] = eager
        sf.close()
    np.testing.assert_array_equal(got[1], got[3])
    np.testing.assert_array_equal(got[1], np.stack(want))


@pytest.mark.parametrize("config", [2, 3])
def test_two_gpus_equal_one_gpu_robust(config, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out1, out2 = tmp_path / "w1.npz", tmp_path / "w2.npz"
    env = dict(os.environ, PYTHONPATH=f"{ROOT}{os.pathsep}{ROOT / 'monocular-visual-slam_b200'}")
    tool = str(ROOT / "tools" / "sharded_check.py")
    r1 = subprocess.run([sys.executable, tool, "--robust", "--config", str(config), "--out", str(out1)], env=env,
                        capture_output=True, text=True, timeout=300)
    assert r1.returncode == 0, r1.stderr[-3000:]
    r2 = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                         "127.0.0.1", "--master-port", "29521", tool, "--robust", "--config", str(config), "--out", str(out2)],
                        env=env, capture_output=True, text=True, timeout=300)
    assert r2.returncode == 0, r2.stderr[-3000:]
    a, b = np.load(out1), np.load(out2)
    assert set(a.files) == set(b.files) and any(k.endswith("robust") for k in a.files)
    for k in a.files:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    info = json.loads(r2.stdout.strip().splitlines()[-1])
    assert info["world"] == 2 and info["robust"]
