"""K5 / K6 (RANSAC homography, next-row #3) against fixtures produced by the unmodified
reference (tests/golden/make_homography_golden.py) and the NumPy oracle."""
import numpy as np
import pytest

from oracle import homography_oracle as hom

pytestmark = pytest.mark.gpu
FLIP_TOL = 1e-3          # north-star tolerance: <= 0.1 % of correspondences may flip at the threshold


@pytest.fixture(scope="module")
def hgold(golden_dir):
    return np.load(golden_dir / "homography_golden.npz")


@pytest.fixture(scope="module")
def R():
    from b200slam.frontend import HomographyRansac
    return HomographyRansac()


def _dev(src, dst):
    import torch
    corr = torch.from_numpy(np.hstack([src, dst]).astype(np.float32)).cuda()
    off = torch.tensor([0, len(src)], dtype=torch.int32, device="cuda")
    cnt = torch.tensor([len(src)], dtype=torch.int32, device="cuda")
    return corr, off, cnt


def test_dlt_hypotheses_and_scores_match_reference(hgold, R):
    import torch
    for name in hgold["names"]:
        src, dst, th = hgold[f"{name}/src"], hgold[f"{name}/dst"], float(hgold[f"{name}/th"])
        samples, Hs, masks, valid = hgold[f"{name}/samples"], hgold[f"{name}/H"], hgold[f"{name}/masks"], hgold[f"{name}/valid"]
        corr, off, cnt = _dev(src, dst)
        Hm = R.hypotheses(corr, off, cnt, 1, len(samples), samples=torch.from_numpy(samples.astype(np.int32)).cuda()[None])
        Hd = Hm[0].cpu().numpy().reshape(-1, 3, 3)
        scale = np.abs(Hs[valid]).max(axis=(1, 2), keepdims=True)
        np.testing.assert_allclose(Hd[valid] / scale, Hs[valid] / scale, atol=1e-8, err_msg=name)   # H[2][2] = 1 fixes sign and scale
        # identical hypotheses (the reference's own H) -> identical inlier counts
        Href = torch.from_numpy(np.nan_to_num(Hs).reshape(1, -1, 9).copy()).cuda()
        counts = R.score(corr, off, cnt, 1, Href, th).cpu().numpy()[0]
        np.testing.assert_array_equal(counts[valid], masks[valid].sum(1), err_msg=name)
        # device hypotheses: counts equal the high-precision reference's on the same hypotheses outside the band
        c_dev = R.score(corr, off, cnt, 1, Hm, th).cpu().numpy()[0]
        ref, band = hom.classify(Hd, src, dst, th)
        n_band = hom.check_counts(c_dev, ref, band, name)
        print(f"{name}: band cases excused {n_band}")
        assert n_band == 0, name
        best_h, best_c, mask = R.select(torch.from_numpy(counts[None].astype(np.int32)).cuda(), corr, off, cnt, 1, Href, th)
        full = np.where(valid, masks.sum(1), 0)
        want = hom.select_hypothesis(np.where(valid, counts, 0), len(src))
        if valid.all():
            assert int(best_h[0]) == hom.select_hypothesis(counts, len(src)) == want
            np.testing.assert_array_equal(mask.cpu().numpy().astype(bool), masks[want])
            assert int(best_c[0]) == full[want]


def test_ransac_homography_dropin_matches_reference_runs(hgold):
    from integration.pose_bridge import ransac_homography
    agree = 0
    for name in hgold["names"]:
        src, dst, th = hgold[f"{name}/src"], hgold[f"{name}/dst"], float(hgold[f"{name}/th"])
        seed = 100 + int(np.flatnonzero(hgold["names"] == name)[0]) + 1
        H, inl = ransac_homography(src, dst, th=th, max_iter=len(hgold[f"{name}/samples"]), rng=np.random.default_rng(seed))
        if np.array_equal(inl, hgold[f"{name}/run_inliers"]):
            agree += 1
            np.testing.assert_allclose(H, hgold[f"{name}/run_H"], rtol=1e-6, atol=1e-6, err_msg=name)
        else:                                   # a flip at the threshold may move the early exit: inlier sets still nearly equal
            a, b = set(inl.tolist()), set(hgold[f"{name}/run_inliers"].tolist())
            assert len(a ^ b) <= max(2, FLIP_TOL * len(src) * 5), name
    assert agree >= len(hgold["names"]) - 1


def test_device_sampler_ragged_and_degenerate(R):
    import torch
    rng = np.random.default_rng(9)
    Ms = [0, 3, 4, 50, 300]
    stride = 320
    corr = torch.zeros((len(Ms) * stride, 4), dtype=torch.float32, device="cuda")
    srcs = []
    for p, m in enumerate(Ms):
        s = rng.uniform(0, 640, (m, 2)).astype(np.float32)
        d = (s * 1.01 + 3.0 + rng.normal(0, 0.3, s.shape)).astype(np.float32)
        srcs.append((s, d))
        if m:
            corr[p * stride:p * stride + m] = torch.from_numpy(np.hstack([s, d])).cuda()
    c_off = (torch.arange(len(Ms) + 1, dtype=torch.int32, device="cuda") * stride).contiguous()
    c_cnt = torch.tensor(Ms, dtype=torch.int32, device="cuda")
    Hm, smp = R.hypotheses(corr, c_off, c_cnt, len(Ms), 200, seed=77, return_samples=True)
    Hm2 = R.hypotheses(corr, c_off, c_cnt, len(Ms), 200, seed=77)
    assert torch.equal(torch.nan_to_num(Hm), torch.nan_to_num(Hm2))                           # deterministic in the seed
    smp = smp.cpu().numpy()
    counts = R.score(corr, c_off, c_cnt, len(Ms), Hm, 3.0)
    best_h, best_c, mask = R.select(counts, corr, c_off, c_cnt, len(Ms), Hm, 3.0)
    counts, best_h, best_c = counts.cpu().numpy(), best_h.cpu().numpy(), best_c.cpu().numpy()
    for p, m in enumerate(Ms):
        if m < 4:
            assert (Hm[p].cpu().numpy() == 0).all() and best_h[p] == -1 and best_c[p] == 0
            continue
        assert all(len(set(r)) == 4 and 0 <= min(r) and max(r) < m for r in smp[p])
        s, d = srcs[p]
        ref, band = hom.classify(Hm[p].cpu().numpy().reshape(-1, 3, 3), s, d, 3.0)
        n_band = hom.check_counts(counts[p], ref, band, f"M={m}")
        print(f"M={m}: band cases excused {n_band}")
        assert n_band == 0
        assert best_c[p] >= 0.9 * m                                                            # the planted similarity is found
