"""GPU: batched RobustPoseEstimator.estimate_pose (b200slam.robust_pose, pose_bridge.estimate_pose_batch).

The batch must answer what the single call answers: the seven reference scenes of tests/golden/pose_golden.npz in one
call (either order), about fifty seeded scenes against single estimate_pose calls with the same generators, the new
kernels against NumPy, and Frontend(robust_pose=...) against the drop-in on the same correspondences, eager and in a
CUDA graph."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

KITTI_K = np.array([[718.856, 0.0, 607.1928], [0.0, 718.856, 185.2157], [0.0, 0.0, 1.0]])


def _kp_matches(p1, p2):
    kp1 = [cv2.KeyPoint(float(x), float(y), 1.0) for x, y in p1]
    kp2 = [cv2.KeyPoint(float(x), float(y), 1.0) for x, y in p2]
    return kp1, kp2, [cv2.DMatch(_queryIdx=j, _trainIdx=j, _distance=0.0) for j in range(len(kp1))]


@pytest.fixture(scope="module")
def pg(golden_dir):
    return np.load(golden_dir / "pose_golden.npz")


def _golden_cfg(pb, pg, name):
    kw = {str(k): float(v) for k, v in zip(pg[f"{name}/cfg_keys"], pg[f"{name}/cfg_vals"])}
    for k in ("min_matches", "min_inliers", "min_cheirality_inliers"):
        if k in kw:
            kw[k] = int(kw[k])
    return pb.RobustPoseEstimatorConfig(**kw)


def _check_golden(pb, pg, name, got):
    outcome = str(pg[f"{name}/outcome"])
    if outcome == "failure":
        assert isinstance(got, pb.PoseEstimationFailure), (name, got)
        assert got.reason == str(pg[f"{name}/reason"]) and got.recovery_action == "relocalize"
        want = dict(zip((str(k) for k in pg[f"{name}/metric_keys"]), pg[f"{name}/metric_vals"]))
        assert set(got.metrics) == set(want)
        for k, v in want.items():
            assert got.metrics[k] == pytest.approx(v, rel=1e-9, abs=1e-12), (name, k)
    elif outcome == "estimate":
        assert isinstance(got, pb.PoseEstimate), (name, got)
        d = got.diagnostics
        assert d.method == str(pg[f"{name}/method"])
        np.testing.assert_array_equal(np.asarray(got.inlier_indices), pg[f"{name}/inlier_indices"])
        want = pg[f"{name}/diag"]
        assert (d.match_count, d.inliers, d.cheirality_inliers) == (int(want[0]), int(want[1]), int(want[4]))
        assert d.inlier_ratio == pytest.approx(want[2], rel=1e-12)
        assert d.median_parallax == pytest.approx(want[3], rel=1e-9)
        assert d.cheirality_ratio == pytest.approx(want[5], rel=1e-12)
        assert d.score == pytest.approx(want[6], rel=1e-9)
        np.testing.assert_allclose(got.rotation, pg[f"{name}/R"], atol=1e-7)
        np.testing.assert_allclose(got.translation, pg[f"{name}/t"], atol=1e-7)
    else:
        assert type(got).__name__ == str(pg[f"{name}/error_type"])


@pytest.mark.parametrize("order", ["forward", "reverse"])
def test_golden_scenes_in_one_batch(pg, order):
    from integration import pose_bridge as pb
    names = [str(n) for n in pg["names"]]
    if order == "reverse":
        names = names[::-1]
    kp1s, kp2s, ms, cfgs, rngs = [], [], [], [], []
    for name in names:
        kp1, kp2, m = _kp_matches(pg[f"{name}/pts1"], pg[f"{name}/pts2"])
        kp1s.append(kp1), kp2s.append(kp2), ms.append(m)
        cfgs.append(_golden_cfg(pb, pg, name))
        s0 = int(pg[f"{name}/seed0"])
        rngs.append((np.random.default_rng(s0), np.random.default_rng(s0 + 1)))
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig())
    got = est.estimate_pose_batch(kp1s, kp2s, ms, np.eye(3), rngs=rngs, configs=cfgs)
    assert len(got) == len(names)
    for name, g in zip(names, got):
        _check_golden(pb, pg, name, g)


# ---- batch == single on seeded scenes ------------------------------------------------------------------------

def _rot(ax, ay, az):
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def _scene(i):
    """(pts1, pts2, K, config kwargs) of seeded scene i: kinds general / planar / low parallax, outliers 0-60 %,
    counts 8-1200 plus tiny ones, K = I or KITTI."""
    rng = np.random.default_rng(5000 + i)
    kind = ("general", "planar", "lowpar")[i % 3]
    K = KITTI_K if (i // 3) % 2 else np.eye(3)
    sizes = (8, 12, 25, 40, 60, 100, 150, 200, 300, 500, 800, 1200)
    n = sizes[(i * 5) % len(sizes)]
    if i % 12 == 0:                   # K = I, general motion, no outliers: the scenes that end in an essential estimate
        n = (300, 500, 200, 800)[i // 12]
    kw = {}
    if i in (44, 45):                 # below min_matches
        n = 15
    if i in (46, 47):                 # fewer than eight with a small min_matches
        n, kw = 6, dict(min_matches=5)
    out_rate = (0.0, 0.1, 0.2, 0.3, 0.45, 0.6)[i % 6]
    if kind == "planar":
        X = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), np.zeros(n)], 1)
        P = X + np.array([0, 0, 6.0]) + X[:, :1] * np.array([0, 0, 0.2])
    else:
        P = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 12, n)], 1)
    if kind == "lowpar":
        R, t = _rot(0.0005, 0.001, 0.0), np.array([0.002, 0.0, 0.001])
    else:
        R, t = _rot(*rng.uniform(-0.05, 0.05, 3)), rng.uniform(-0.5, 0.5, 3) + np.array([0.3, 0, 0])
    c2 = P @ R.T + t
    h1 = P @ K.T
    h2 = c2 @ K.T
    p1 = h1[:, :2] / h1[:, 2:]
    p2 = h2[:, :2] / h2[:, 2:]
    noise = 0.5 if K is KITTI_K else 5e-4
    p1 = p1 + rng.normal(0, noise, p1.shape)
    p2 = p2 + rng.normal(0, noise, p2.shape)
    k = int(out_rate * n)
    if k:
        idx = rng.permutation(n)[:k]
        lo, hi = p2.min(0), p2.max(0)
        p2[idx] = rng.uniform(lo, hi, (k, 2))
    if i % 4 == 0:
        kw.setdefault("min_parallax", 0.0)
    if i % 5 == 1:
        kw["min_inliers"] = 8
    return p1.astype(np.float32), p2.astype(np.float32), K, kw


class _Recorder:
    def __init__(self, seeds):
        self.seeds, self.made = list(seeds), []

    def __call__(self):
        g = np.random.default_rng(self.seeds[len(self.made)])
        self.made.append(g)
        return g


def _same(pb, a, b):
    """a: single-call outcome, b: batch entry."""
    if isinstance(a, Exception):
        assert type(b) is type(a), (a, b)
        assert str(b) == str(a)
        if isinstance(a, pb.PoseEstimationFailure):
            assert (b.reason, b.recovery_action) == (a.reason, a.recovery_action)
            assert set(b.metrics) == set(a.metrics)
            for k in a.metrics:
                assert b.metrics[k] == pytest.approx(a.metrics[k], rel=1e-12, abs=1e-15), k
        return
    assert isinstance(b, pb.PoseEstimate), b
    da, db = a.diagnostics, b.diagnostics
    assert db.method == da.method
    np.testing.assert_array_equal(np.asarray(b.inlier_indices), np.asarray(a.inlier_indices))
    assert (db.match_count, db.inliers, db.cheirality_inliers) == (da.match_count, da.inliers, da.cheirality_inliers)
    assert db.median_parallax == da.median_parallax                       # the float32 median, bit for bit
    assert db.inlier_ratio == pytest.approx(da.inlier_ratio, rel=1e-12)
    assert db.cheirality_ratio == pytest.approx(da.cheirality_ratio, rel=1e-12)
    assert db.score == pytest.approx(da.score, rel=1e-12)
    np.testing.assert_allclose(b.rotation, a.rotation, atol=1e-7)
    np.testing.assert_allclose(b.translation, a.translation, atol=1e-7)


def test_batch_equals_single_calls():
    from integration import pose_bridge as pb
    scenes = [_scene(i) for i in range(48)]
    kinds = set()
    for K in (np.eye(3), KITTI_K):
        idx = [i for i, s in enumerate(scenes) if (s[2] is KITTI_K) == (K is KITTI_K)]
        cfgs = [pb.RobustPoseEstimatorConfig(**scenes[i][3]) for i in idx]
        kps = [_kp_matches(scenes[i][0], scenes[i][1]) for i in idx]
        singles, gens_single = [], []
        for j, i in enumerate(idx):
            rec = _Recorder([900 + 2 * i, 901 + 2 * i])
            pb.RNG_FACTORY = rec
            try:
                singles.append(pb.RobustPoseEstimator(cfgs[j]).estimate_pose(*kps[j], K))
            except Exception as e:                                          # noqa: BLE001 — the outcome under test
                singles.append(e)
            finally:
                pb.RNG_FACTORY = None
            gens_single.append(rec.made)
        rngs = [(np.random.default_rng(900 + 2 * i), np.random.default_rng(901 + 2 * i)) for i in idx]
        got = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig()).estimate_pose_batch(
            [k[0] for k in kps], [k[1] for k in kps], [k[2] for k in kps], K, rngs=rngs, configs=cfgs)
        for j, i in enumerate(idx):
            _same(pb, singles[j], got[j])
            kinds.add(type(got[j]).__name__ + ("/" + got[j].diagnostics.method if isinstance(got[j], pb.PoseEstimate) else ""))
            # generators end where the single call leaves them (a generator it never asked for: untouched)
            for g_b, k, seed in ((rngs[j][0], 0, 900 + 2 * i), (rngs[j][1], 1, 901 + 2 * i)):
                ref = gens_single[j][k] if k < len(gens_single[j]) else np.random.default_rng(seed)
                assert g_b.bit_generator.state == ref.bit_generator.state, (i, k)
            if isinstance(got[j], pb.PoseEstimate) and got[j].diagnostics.method == "essential":
                p1, p2 = scenes[i][0], scenes[i][1]
                _, cnt = pb._cheirality_ratio(p1, p2, got[j].inlier_indices, got[j].rotation, got[j].translation, K)
                assert cnt == got[j].diagnostics.cheirality_inliers, i
    # the scene set exercises estimates, gate failures and rejected pairs
    assert "PoseEstimate/essential" in kinds and "ValueError" in kinds and "PoseEstimationFailure" in kinds, kinds


def test_device_sampler_and_rng_factory_paths():
    """seed= draws on the device (deterministic for a seed); RNG_FACTORY hands out two generators per pair that
    reaches RANSAC, essential first."""
    from integration import pose_bridge as pb
    scenes = [_scene(i) for i in (3, 6, 9, 46)]
    kps = [_kp_matches(s[0], s[1]) for s in scenes]
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig(min_matches=5, min_parallax=0.0))
    args = ([k[0] for k in kps], [k[1] for k in kps], [k[2] for k in kps], np.eye(3))
    a = est.estimate_pose_batch(*args, seed=11)
    b = est.estimate_pose_batch(*args, seed=11)
    for x, y in zip(a, b):
        _same(pb, x, y)
    rec = _Recorder(range(100, 200))
    pb.RNG_FACTORY = rec
    try:
        est.estimate_pose_batch(*args)
    finally:
        pb.RNG_FACTORY = None
    assert len(rec.made) == 2 * 3                          # scene 46 has six matches: rejected before RANSAC


# ---- the kernels alone ------------------------------------------------------------------------------------------

def _median_call(corr, counts, mask=None, cfg=None):
    import torch
    from b200slam import _capi
    from b200slam import robust_pose as rp
    lib = _capi.load_library()
    off = np.zeros(len(counts) + 1, np.int32)
    np.cumsum(counts, out=off[1:])
    dev = torch.device("cuda")
    c = torch.from_numpy(np.ascontiguousarray(corr, np.float32).reshape(-1, 4) if len(corr) else np.zeros((1, 4), np.float32)).to(dev)
    o, n = torch.from_numpy(off).to(dev), torch.from_numpy(np.asarray(counts, np.int32)).to(dev)
    m = None if mask is None else torch.from_numpy(np.asarray(mask, np.uint8) if len(mask) else np.zeros(1, np.uint8)).to(dev)
    P = len(counts)
    med = torch.empty(P, dtype=torch.float32, device=dev)
    th = torch.empty(P, dtype=torch.float64, device=dev)
    th2 = torch.empty(P, dtype=torch.float64, device=dev)
    cfg_d = None if cfg is None else torch.from_numpy(rp.pack_configs(cfg).view(np.uint8).copy()).to(dev)
    _capi.check(lib.b2s_displacement_median_batched(_capi.ptr(c), _capi.ptr(o), _capi.ptr(n), _capi.ptr(m), P, _capi.ptr(cfg_d), 1,
                                                    _capi.ptr(med), _capi.ptr(th), _capi.ptr(th2), _capi.current_stream()))
    return med.cpu().numpy(), th.cpu().numpy(), th2.cpu().numpy(), off


def test_median_and_threshold_are_bit_exact():
    from b200slam.robust_pose import RobustPoseConfig
    from integration.feature_pipeline_bridge import adaptive_ransac_threshold
    rng = np.random.default_rng(3)
    counts = [0, 1, 2, 3, 4, 5, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 4096, 10000]
    blocks, masks = [], []
    for k, n in enumerate(counts):
        p1 = rng.uniform(0, 1200, (n, 2)).astype(np.float32)
        if k % 3 == 0:                                                   # heavy ties: few distinct displacements
            d = rng.integers(0, 4, (n, 2)).astype(np.float32) * np.float32(0.5)
        elif k % 3 == 1:                                                 # zero displacements mixed in
            d = rng.normal(0, 20, (n, 2)).astype(np.float32)
            d[rng.random(n) < 0.3] = 0
        else:
            d = rng.normal(0, 30, (n, 2)).astype(np.float32)
        p2 = (p1 + d).astype(np.float32)
        blocks.append(np.hstack([p1, p2]))
        mk = (rng.random(n) < 0.5).astype(np.uint8)
        if k == 5:
            mk[:] = 0                                                    # an empty mask
        masks.append(mk)
    corr = np.concatenate(blocks)
    for cfg in (RobustPoseConfig(), RobustPoseConfig(base_ransac_threshold=0.7, min_ransac_threshold=0.2, max_ransac_threshold=1.3)):
        med, th, th2, off = _median_call(corr, counts, cfg=cfg)
        for p, n in enumerate(counts):
            b = blocks[p]
            want = np.float32(np.median(np.linalg.norm(b[:, 2:] - b[:, :2], axis=1))) if n else np.float32(0.0)
            assert med[p].view(np.uint32) == want.view(np.uint32), (n, med[p], want)
            w = adaptive_ransac_threshold(b[:, :2], b[:, 2:], cfg.base_ransac_threshold, cfg.min_ransac_threshold,
                                          cfg.max_ransac_threshold)
            assert th[p] == w and th2[p] == w * w, (n, th[p], w)
    med, _, _, _ = _median_call(corr, counts, mask=np.concatenate(masks))
    for p, n in enumerate(counts):
        b, sel = blocks[p], np.flatnonzero(masks[p])
        want = np.float32(np.median(np.linalg.norm(b[sel, 2:] - b[sel, :2], axis=1))) if sel.size else np.float32(0.0)
        assert med[p].view(np.uint32) == want.view(np.uint32), (n, med[p], want)


def test_homography_refit_matches_numpy():
    import torch
    from b200slam import _capi, geometry
    rng = np.random.default_rng(8)
    counts = np.array([4, 5, 9, 40, 200, 500, 1200, 3000, 3], np.int32)
    blocks, masks = [], []
    for n in counts:
        X = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), np.full(n, 5.0)], 1)
        R, t = _rot(*rng.uniform(-0.1, 0.1, 3)), rng.uniform(-0.6, 0.6, 3)
        h1, h2 = X @ KITTI_K.T, (X @ R.T + t) @ KITTI_K.T
        p1 = h1[:, :2] / h1[:, 2:] + rng.normal(0, 0.4, (n, 2))
        p2 = h2[:, :2] / h2[:, 2:] + rng.normal(0, 0.4, (n, 2))
        blocks.append(np.hstack([p1, p2]).astype(np.float32))
        mk = (rng.random(n) < 0.7).astype(np.uint8)
        mk[:4] = 1
        masks.append(mk)
    off = np.zeros(len(counts) + 1, np.int32)
    np.cumsum(counts, out=off[1:])
    dev = torch.device("cuda")
    c = torch.from_numpy(np.concatenate(blocks)).to(dev)
    o, n_d = torch.from_numpy(off).to(dev), torch.from_numpy(counts).to(dev)
    m = torch.from_numpy(np.concatenate(masks)).to(dev)
    H = torch.empty((len(counts), 9), dtype=torch.float64, device=dev)
    used = torch.empty(len(counts), dtype=torch.int32, device=dev)
    lib = _capi.load_library()
    _capi.check(lib.b2s_refit_homography_batched(_capi.ptr(c), _capi.ptr(o), _capi.ptr(n_d), _capi.ptr(m), len(counts),
                                                 _capi.ptr(H), _capi.ptr(used), _capi.current_stream()))
    Hd, used = H.cpu().numpy().reshape(-1, 3, 3), used.cpu().numpy()
    for p, n in enumerate(counts):
        sel = np.flatnonzero(masks[p])
        assert used[p] == sel.size
        if sel.size < 4:
            assert not Hd[p].any()
            continue
        b = blocks[p][sel].astype(np.float64)
        want = geometry.dlt_homography_batch(b[None, :, :2], b[None, :, 2:])[0]
        np.testing.assert_allclose(Hd[p], want, rtol=1e-9, atol=1e-9 * np.abs(want).max())


def test_homography_decomposition_matches_numpy():
    """The decision kernel alone, fed a homography winner that must be selected: its (R, t) is decompose_homography's
    (polar factor of [r1 r2 r1 x r2]) for arbitrary H and K."""
    import torch
    from b200slam import _capi, geometry
    from b200slam import robust_pose as rp
    rng = np.random.default_rng(9)
    P, M = 64, 40
    Hs = np.empty((P, 3, 3))
    for p in range(P):
        X = rng.normal(0, 1, (3, 3))
        Hs[p] = np.eye(3) + (0.3 if p % 2 else 2.0) * X
        Hs[p] /= Hs[p, 2, 2]
    dev = torch.device("cuda")
    i32 = lambda a: torch.from_numpy(np.asarray(a, np.int32)).to(dev)
    f64 = lambda a: torch.from_numpy(np.asarray(a, np.float64)).to(dev)
    off, cnt = i32(np.arange(P + 1) * M), i32(np.full(P, M))
    ones = torch.ones(P * M, dtype=torch.uint8, device=dev)
    med = torch.full((P,), 5.0, dtype=torch.float32, device=dev)
    cfg = rp.RobustPoseConfig(min_matches=8, min_inliers=8, homography_bias=10.0, min_parallax=0.0)
    cfg_d = torch.from_numpy(rp.pack_configs(cfg).view(np.uint8).copy()).to(dev)
    res = torch.empty((P, rp.POSE_RESULT_BYTES), dtype=torch.uint8, device=dev)
    out_mask = torch.empty(P * M, dtype=torch.uint8, device=dev)
    e_R, e_t = f64(np.tile(np.eye(3).reshape(1, 9), (P, 1))), f64(np.tile([1.0, 0.0, 0.0], (P, 1)))
    keep = [off, cnt, ones, med, cfg_d, res, out_mask, e_R, e_t]
    for K in (np.eye(3), KITTI_K):
        Kinv = np.ascontiguousarray(np.linalg.inv(K))
        args = [off, cnt, i32(np.zeros(P)), i32(np.full(P, 20)), ones, e_R, e_t, i32(np.tile([20, 0, 0, 0], (P, 1))), med, med,
                f64(np.full(P, 0.01)), i32(np.zeros(P)), i32(np.full(P, M)), ones, f64(Hs.reshape(P, 9))]
        keep += args
        _capi.check(_capi.load_library().b2s_robust_pose_decide(
            *[_capi.ptr(a) for a in args[:2]], P, *[_capi.ptr(a) for a in args[2:]], _capi.ptr(Kinv), _capi.ptr(cfg_d), 1,
            _capi.ptr(res), _capi.ptr(out_mask), 0, _capi.current_stream()))
        r = rp.decode_results(res.cpu().numpy())
        for p in range(P):
            assert r[p]["outcome"] == rp.POSE_ESTIMATE and r[p]["method"] == 1, r[p]
            R, t = geometry.decompose_homography(Hs[p], K)
            np.testing.assert_allclose(r[p]["R"].reshape(3, 3), R, atol=1e-10)
            np.testing.assert_allclose(r[p]["t"], t / np.linalg.norm(t), atol=1e-10)
            assert r[p]["score_homography"] == 10.0 * 1.0 * 5.0


# ---- Frontend(robust_pose=...) -------------------------------------------------------------------------------------

def test_frontend_robust_pose_matches_the_dropin_eager_and_graph():
    import torch
    from b200slam import synthetic
    from b200slam.frontend import Frontend, FrontendConfig, PairBatch
    from b200slam.robust_pose import RobustPoseConfig
    from integration import pose_bridge as pb
    qs, ts, kq, kt = synthetic.tracking_pairs(32, n_desc=1000, seed=77)
    kq = [k * np.float32(700) for k in kq]                 # pixel-like scale so the parallax gates are exercised
    kt = [k * np.float32(700) for k in kt]
    rcfg = RobustPoseConfig(min_parallax=0.5)
    K = np.diag([700.0, 700.0, 1.0])
    fe = Frontend(FrontendConfig(max_matches=500, robust_pose=rcfg, seed=2024))
    b = PairBatch.from_host(qs, ts, kq, kt)
    r1 = fe.run(b, K=K)
    a1 = (r1.robust.cpu().numpy().copy(), r1.robust_mask.cpu().numpy().copy())
    r2 = fe.run(b, K=K)
    np.testing.assert_array_equal(r2.robust.cpu().numpy(), a1[0])
    np.testing.assert_array_equal(r2.robust_mask.cpu().numpy(), a1[1])
    # the drop-in on the correspondences the selection handed over
    cnt = r1.sel.count.cpu().numpy()
    corr = r1.sel.corr.cpu().numpy()
    stride = r1.sel.stride
    assert (cnt >= rcfg.min_matches).all()
    kps = [_kp_matches(corr[p * stride:p * stride + cnt[p], :2], corr[p * stride:p * stride + cnt[p], 2:]) for p in range(32)]
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig(min_parallax=0.5))
    got = est.estimate_pose_batch([k[0] for k in kps], [k[1] for k in kps], [k[2] for k in kps], K, seed=2024)
    from b200slam.robust_pose import decode_results
    rec = decode_results(a1[0])
    dropin = decode_results(est._device._buf["results"][:32].cpu().numpy())     # the drop-in's last device answer
    np.testing.assert_array_equal(rec.view(np.uint8), dropin.view(np.uint8))          # byte for byte
    for p in range(32):
        want = pb.decode_pose_result(rec[p], np.flatnonzero(a1[1][p * stride:p * stride + cnt[p]]))
        _same(pb, want, got[p])
        if isinstance(want, pb.PoseEstimate):
            np.testing.assert_array_equal(want.rotation, got[p].rotation)
            np.testing.assert_array_equal(want.translation, got[p].translation)
        assert not a1[1][p * stride + cnt[p]:(p + 1) * stride].any()
    # captured in a CUDA graph and replayed
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rg = fe.run(b, K=K)
    fe.robust._buf["packed"].zero_()
    g.replay()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(rg.robust.cpu().numpy(), a1[0])
    np.testing.assert_array_equal(rg.robust_mask.cpu().numpy(), a1[1])
