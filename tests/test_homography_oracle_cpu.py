"""CPU: the high-precision transfer-error reference and the band classifier of oracle/homography_oracle.py, which the
homography parity tests (tests/test_gpu_homography_parity.py) measure K6 and the selection kernel against."""
import numpy as np

from oracle import homography_oracle as hom


def _translation(tx, ty):
    return np.array([[1.0, 0.0, tx], [0.0, 1.0, ty], [0.0, 0.0, 1.0]])


def test_exact_cases_give_exactly_representable_errors():
    # translation (3, 4), destination offset (1.5, 2): each direction is off by 2.5, the sum is 5.0
    src = np.array([[0.5, 1.0], [10.0, -7.5], [1023.5, 640.0]], np.float32)
    dst = (src + np.float32([3 + 1.5, 4 + 2])).astype(np.float32)
    e = hom.transfer_error_hp(_translation(3, 4), src, dst)
    assert (e == 5.0).all(), e
    # integer scale 2 plus a translation: forward off by |o| = 2.5, backward by |o| / 2 = 1.25
    H2 = np.array([[2.0, 0.0, 1.0], [0.0, 2.0, -3.0], [0.0, 0.0, 1.0]])
    dst2 = (src * 2 + np.float32([1 + 1.5, -3 + 2])).astype(np.float32)
    e2 = hom.transfer_error_hp(H2, src, dst2)
    assert (e2 == 3.75).all(), e2
    # float64 agrees on these, so the float64 screen never hides them
    np.testing.assert_array_equal(hom.transfer_error(H2, src, dst2), e2)
    # at th = e the point is an outlier, just above it an inlier; neither decision is excused
    for th, want in ((5.0, False), (np.nextafter(5.0, np.inf), True)):
        mask, band = hom.classify(_translation(3, 4)[None], src, dst, th)
        assert (mask == want).all() and band.sum() == 3       # e == th exactly: inside the band by definition
    mask, band = hom.classify(_translation(3, 4)[None], src, dst, 5.001)
    assert mask.all() and not band.any()


def test_undefined_errors_are_nan_and_outliers():
    src = np.array([[2.0, 1.0], [3.0, 1.0]], np.float32)
    dst = np.array([[1.0, 1.0], [2.0, 2.0]], np.float32)
    assert np.isnan(hom.transfer_error_hp(np.zeros((3, 3)), src, dst)).all()
    rank2 = np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0], [5.0, 7.0, 9.0]])
    assert np.isnan(hom.transfer_error_hp(rank2, src, dst)).all()
    w0 = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [1.0, 0.0, -2.0]])       # sends x = 2 to w = 0
    e = hom.transfer_error_hp(w0, src, dst)
    assert np.isnan(e[0]) and np.isfinite(e[1])
    for th in (np.inf, 3.0, 0.0, -1.0):
        for H in (np.zeros((3, 3)), rank2):
            mask, band = hom.classify(H[None], src, dst, th)
            assert not mask.any() and not band.any()
        mask, band = hom.classify(w0[None], src, dst, th)
        assert not mask[0, 0] and not band.any()
        assert mask[0, 1] == (th == np.inf or e[1] < th)


def _random_case(rng, M, scale):
    src = rng.uniform(0, scale, (M, 2))
    A = np.eye(3) + rng.normal(0, 0.05, (3, 3))
    A[:2, 2] = rng.normal(0, 0.05 * scale, 2)
    A[2, :2] /= scale
    A /= A[2, 2]
    h = np.hstack([src, np.ones((M, 1))]) @ A.T
    dst = h[:, :2] / h[:, 2:] + rng.normal(0, 0.0004 * scale, (M, 2))
    out = rng.random(M) < 0.3
    dst[out] = rng.uniform(0, scale, (out.sum(), 2))
    return A, src.astype(np.float32), dst.astype(np.float32)


def test_hp_agrees_with_float64_on_random_cases():
    rng = np.random.default_rng(1)
    for scale in (1240.0, 1.0):
        for _ in range(4):
            A, src, dst = _random_case(rng, 200, scale)
            e_hp, e64 = hom.transfer_error_hp(A, src, dst), hom.transfer_error(A, src, dst)
            # relative to the coordinates' magnitude: float64 cancels in the differences p - u
            np.testing.assert_allclose(e_hp, e64, rtol=1e-13, atol=1e-13 * scale)


def test_classifier_matches_float64_and_reports_a_planted_off_by_one():
    rng = np.random.default_rng(2)
    A, src, dst = _random_case(rng, 3000, 1240.0)
    Hs = np.stack([A, A + rng.normal(0, 1e-4, (3, 3)), A * 3.0, _translation(2.0, -1.0)])
    th = 3.0
    mask, band = hom.classify(Hs, src, dst, th)
    assert band.sum() == 0                                  # random, well-conditioned data: no rounding-band cases
    want = np.stack([hom.transfer_error(H, src, dst) < th for H in Hs])
    np.testing.assert_array_equal(mask, want)
    counts = mask.sum(1)
    assert counts[0] > 1000
    assert hom.check_counts(counts, mask, band) == 0
    for delta in (+1, -1):                                  # a kernel that miscounts by one correspondence
        bad = counts.copy()
        bad[0] += delta
        try:
            hom.check_counts(bad, mask, band)
        except AssertionError:
            continue
        raise AssertionError(f"an off-by-one of {delta:+d} passed the classifier")
    # a threshold placed on one evaluation's exact error: that evaluation, and only it, is a band case
    e = hom.transfer_error_hp(Hs[0], src[1023:1024], dst[1023:1024])[0]
    mask2, band2 = hom.classify(Hs[:1], src, dst, float(e))
    assert band2.sum() == 1 and band2[0, 1023]
    excused = mask2.sum() - 1 if mask2[0, 1023] else mask2.sum() + 1      # the other decision on that evaluation
    assert hom.check_counts([excused], mask2, band2) == 1
