"""GPU: the homography RANSAC kernels (K5 DLT hypotheses, K6 transfer-error scoring, winner selection) against the
high-precision reference of oracle/homography_oracle.py, at the shapes and values where such kernels go wrong: the
1024-correspondence chunk edges of K6, hypothesis counts that leave dead lanes, per-pair and scalar thresholds,
thresholds exactly on an error, singular and overflowing hypotheses, the early-exit and tie rules of the selection,
and the robust-pose branch that chains them.

A device decision may differ from the reference only inside the rounding band (homography_oracle.classify); every
test asserts and prints how many band cases it excused."""
import numpy as np
import pytest

from oracle import homography_oracle as hom

pytestmark = pytest.mark.gpu

SENTINEL = 0xAB


@pytest.fixture(scope="module")
def R():
    from b200slam.frontend import HomographyRansac
    return HomographyRansac()


def _true_h(rng, scale):
    """A well-conditioned homography for coordinates in [0, scale] (pixel) or [-1, 1] (scale = 1, normalised)."""
    A = np.eye(3) + rng.normal(0, 0.04, (3, 3))
    A[:2, 2] = rng.normal(0, 0.03 * scale, 2)
    A[2, :2] /= scale
    return A / A[2, 2]


def _pair(rng, M, scale, out_rate, keep=()):
    """(src, dst) float32 of M correspondences of a random homography with `out_rate` outliers (never at `keep`)."""
    lo = 0.0 if scale > 1 else -1.0
    A = _true_h(rng, scale)
    src = rng.uniform(lo, scale, (M, 2))
    h = np.hstack([src, np.ones((M, 1))]) @ A.T
    dst = h[:, :2] / h[:, 2:] + rng.normal(0, 4e-4 * scale, (M, 2))
    out = rng.random(M) < out_rate
    out[[k for k in keep if 0 <= k < M]] = False
    dst[out] = rng.uniform(lo, scale, (int(out.sum()), 2))
    return src.astype(np.float32), dst.astype(np.float32), A


def _perturbed(rng, A, n, scale):
    """n hypotheses around A, from exact to far off (relative perturbations 1e-6 .. 1e-1)."""
    out = np.empty((n, 3, 3))
    for k in range(n):
        D = np.eye(3) + rng.normal(0, 10 ** rng.uniform(-6, -1), (3, 3))
        D[:2, 2] *= scale
        D[2, :2] /= scale
        out[k] = A @ D
        out[k] /= out[k, 2, 2]
    out[0] = A
    return out


class _Batch:
    """Pairs laid out with a gap of `gap` rows after each (the gaps must never be written); host and device copies."""

    def __init__(self, blocks, counts=None, gap=8):
        import torch
        self.blocks = blocks
        n = [len(s) for s, _ in blocks]
        self.counts = np.array(n if counts is None else counts, np.int32)
        self.off = np.zeros(len(blocks) + 1, np.int32)
        for p, m in enumerate(n):
            self.off[p + 1] = self.off[p] + m + gap
        corr = np.full((max(int(self.off[-1]), 1), 4), 7.0, np.float32)
        for p, (s, d) in enumerate(blocks):
            corr[self.off[p]:self.off[p] + len(s)] = np.hstack([s, d])
        self.P = len(blocks)
        dev = torch.device("cuda")
        self.corr = torch.from_numpy(corr).to(dev)
        self.off_d = torch.from_numpy(self.off).to(dev)
        self.cnt_d = torch.from_numpy(self.counts).to(dev)

    def args(self):
        return self.corr, self.off_d, self.cnt_d, self.P


def _f64(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


def _i32(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.int32)).cuda()


def _select_raw(b, counts, Hm, th, th_pp=None):
    """b2s_homography_select into sentinel-filled outputs, so rows it must not write can be checked."""
    import torch
    from b200slam import _capi
    H = int(Hm.shape[1])
    mask = torch.full((b.corr.shape[0],), SENTINEL, dtype=torch.uint8, device="cuda")
    best_h = torch.full((b.P,), -7, dtype=torch.int32, device="cuda")
    best_c = torch.full((b.P,), -7, dtype=torch.int32, device="cuda")
    p = _capi.ptr
    _capi.check(_capi.load_library().b2s_homography_select(
        p(counts), p(b.corr), p(b.off_d), p(b.cnt_d), b.P, p(Hm), H, float(th), p(th_pp), p(best_h), p(best_c), p(mask),
        _capi.current_stream()))
    return best_h.cpu().numpy(), best_c.cpu().numpy(), mask.cpu().numpy()


def _check_untouched(b, mask):
    """Every row outside [off, off + max(count, 0)) keeps the sentinel."""
    written = np.zeros(len(mask), bool)
    for p in range(b.P):
        written[b.off[p]:b.off[p] + max(int(b.counts[p]), 0)] = True
    assert (mask[~written] == SENTINEL).all(), np.flatnonzero(mask[~written] != SENTINEL)[:5]


def _ill_conditioned_only(Hs, band):
    """Band cases of device-drawn hypotheses are excused only where H is near-singular (2-norm condition > 1e8): a
    nearly collinear 4-point sample gives such an H, and its back-projection error is then rounding-dominated."""
    hs = np.flatnonzero(band.any(1))
    well = [h for h in hs if np.linalg.cond(Hs[h]) < 1e8]
    assert not well, f"band cases on well-conditioned hypotheses {well[:5]}"
    return int(band.sum())


# ---- 1. K6 on ragged counts in one batch ---------------------------------------------------------------------------

K6_COUNTS = [0, 1, 3, 4, 5, 127, 128, 129, 1023, 1024, 1025, 2047, 2048, 2049, 3000, 10000]
# (count, correspondence index, hypothesis) whose exact error becomes that pair's threshold: the last element of a chunk
K6_ON_ERROR = {1024: (1023, 129), 1025: (1023, 0), 2048: (2047, 0), 2049: (2047, 129), 3000: (2999, 0), 10000: (9999, 129)}


@pytest.mark.parametrize("H", [130, 257])
def test_k6_ragged_chunks_equal_the_reference(R, H):
    rng = np.random.default_rng(600 + H)
    blocks, Hs, ths, scales = [], [], [], []
    for i, M in enumerate(K6_COUNTS):
        scale = 1240.0 if i % 2 == 0 else 1.0
        src, dst, A = _pair(rng, M, scale, out_rate=0.6 * (i % 4) / 3, keep=(1023, 2047, M - 1))
        blocks.append((src, dst))
        Hs.append(_perturbed(rng, A, H, scale))
        scales.append(scale)
        if M in K6_ON_ERROR:
            m, h = K6_ON_ERROR[M]
            ths.append(float(hom.transfer_error_hp(Hs[-1][h], src[m:m + 1], dst[m:m + 1])[0]))
        else:
            ths.append(float(rng.uniform(1.0, 5.0) * (1.0 if scale > 1 else 1e-3)))
    # a pair with a negative count (the overflow flag): rows exist, but nothing may be read or written for it
    src, dst, A = _pair(rng, 50, 1240.0, 0.0)
    blocks.append((src, dst))
    Hs.append(_perturbed(rng, A, H, 1240.0))
    ths.append(3.0)
    counts_in = K6_COUNTS + [-5]
    b = _Batch(blocks, counts_in)
    Hm = _f64(np.stack(Hs).reshape(b.P, H, 9))
    th_pp = _f64(ths)
    counts = R.score(*b.args(), Hm, 0.0, th_per_pair=th_pp).cpu().numpy()
    best_h, best_c, mask = _select_raw(b, R.score(*b.args(), Hm, 0.0, th_per_pair=th_pp), Hm, 0.0, th_pp)
    _check_untouched(b, mask)
    band_total, forced = 0, 0
    for p, M in enumerate(counts_in):
        if M <= 0:
            assert (counts[p] == 0).all() and best_h[p] == -1 and best_c[p] == 0, (M, best_h[p], best_c[p])
            continue
        src, dst = blocks[p]
        ref, band = hom.classify(Hs[p], src, dst, ths[p])
        n_band = hom.check_counts(counts[p], ref, band, f"M={M}")
        band_total += n_band
        if M in K6_ON_ERROR:
            m, h = K6_ON_ERROR[M]
            assert band[h, m]                                    # the threshold sits on this evaluation's error
            forced += 1
        w = int(best_h[p])
        assert w == hom.select_hypothesis(counts[p], M)
        if n_band == 0:
            assert w == hom.select_hypothesis(ref.sum(1), M)
        if w < 0:
            assert best_c[p] == 0 and not mask[b.off[p]:b.off[p] + M].any()
            continue
        mk = mask[b.off[p]:b.off[p] + M]
        assert best_c[p] == counts[p, w] == mk.sum(), (M, w, best_c[p], counts[p, w], mk.sum())
        np.testing.assert_array_equal((mk == 1)[~band[w]], ref[w][~band[w]], err_msg=f"M={M}")
    # the negative-count pair also gets all-zero hypotheses from K5
    Hd = R.hypotheses(*b.args(), H, seed=5).cpu().numpy()
    assert not Hd[-1].any()
    # the scalar-threshold path equals the per-pair path when the thresholds are equal
    for t0 in (3.0, 2e-3, ths[10]):
        a = R.score(*b.args(), Hm, t0).cpu().numpy()
        c = R.score(*b.args(), Hm, 0.0, th_per_pair=_f64(np.full(b.P, t0))).cpu().numpy()
        np.testing.assert_array_equal(a, c)
        bh_a, bc_a, mk_a = _select_raw(b, _i32(a), Hm, t0)
        bh_c, bc_c, mk_c = _select_raw(b, _i32(c), Hm, 0.0, _f64(np.full(b.P, t0)))
        np.testing.assert_array_equal(bh_a, bh_c), np.testing.assert_array_equal(bc_a, bc_c)
        np.testing.assert_array_equal(mk_a, mk_c)
    print(f"H={H}: band cases excused {band_total} ({forced} forced by thresholds on an error, "
          f"{band_total - forced} on random data)")
    assert forced == len(K6_ON_ERROR)
    assert band_total - forced == 0


# ---- 2. thresholds exactly on an exactly representable error --------------------------------------------------------

def _exact_pair(rng, M, Hx, off, far):
    """Integer / half-integer source points; dst = H src exactly (error 0), + off at the probe positions (error e),
    + far elsewhere (a large exact error). Returns src, dst and the exact error of every correspondence."""
    src = (rng.integers(-400, 400, (M, 2)) * 0.5).astype(np.float64)
    dst = (np.hstack([src, np.ones((M, 1))]) @ Hx.T)[:, :2]
    kind = rng.integers(0, 2, M)                                   # 0: exact, 1: far
    probes = sorted({0, 1023, 1024, M - 1} & set(range(M)))
    kind[probes] = 2
    dst = dst + np.where(kind[:, None] == 1, far, 0.0) + np.where(kind[:, None] == 2, off, 0.0)
    return src.astype(np.float32), dst.astype(np.float32), kind, probes


def test_thresholds_on_exact_errors(R):
    rng = np.random.default_rng(7)
    cases = []   # (H, exact error of an offset point, of a far point)
    cases.append((np.array([[1.0, 0, 3], [0, 1, 4], [0, 0, 1]]), 5.0, 1000.0))     # 2.5 + 2.5; 500 + 500
    cases.append((np.array([[2.0, 0, 1], [0, 2, -3], [0, 0, 1]]), 3.75, 750.0))    # 2.5 + 1.25; 500 + 250
    blocks, errs, Hs = [], [], []
    for Hx, e, fe in cases:
        for M in (2049, 1025, 1024):
            src, dst, kind, probes = _exact_pair(rng, M, Hx, np.array([1.5, 2.0]), np.array([300.0, 400.0]))
            err = np.choose(kind, [0.0, fe, e])
            np.testing.assert_array_equal(hom.transfer_error_hp(Hx, src[probes], dst[probes]), e)
            blocks.append((src, dst))
            errs.append(err)
            Hs.append(np.stack([np.zeros((3, 3)), Hx, Hx]))
    b = _Batch(blocks)
    Hm = _f64(np.stack(Hs).reshape(b.P, 3, 9))
    for t in (3.75, 5.0):
        for th in (t, np.nextafter(t, np.inf)):
            want = [int((err < th).sum()) for err in errs]
            for th_pp in (None, _f64(np.full(b.P, th))):
                counts = R.score(*b.args(), Hm, th if th_pp is None else 0.0, th_per_pair=th_pp)
                c = counts.cpu().numpy()
                assert (c[:, 0] == 0).all()
                np.testing.assert_array_equal(c[:, 1], want, err_msg=f"th={th!r}")
                np.testing.assert_array_equal(c[:, 2], want, err_msg=f"th={th!r}")
                best_h, best_c, mask = _select_raw(b, counts, Hm, th if th_pp is None else 0.0, th_pp)
                _check_untouched(b, mask)
                for p, err in enumerate(errs):
                    assert best_h[p] == 1 and best_c[p] == want[p]
                    np.testing.assert_array_equal(mask[b.off[p]:b.off[p] + len(err)], (err < th).astype(np.uint8))
    print("exact-threshold cases: band cases excused 0 (the errors are exact)")


# ---- 3. degenerate hypotheses and thresholds ------------------------------------------------------------------------

def test_degenerate_hypotheses_and_thresholds(R):
    rng = np.random.default_rng(11)
    M = 1100
    src, dst, A = _pair(rng, M, 1240.0, 0.3)
    x0 = 321.0
    src[0, 0] = src[1024, 0] = np.float32(x0)                       # two points the w0 hypothesis sends to w = 0
    Hs = np.stack([
        np.zeros((3, 3)),
        np.array([[1.0, 2, 3], [4, 5, 6], [5, 7, 9]]),               # rank 2 (row 3 = row 1 + row 2), det exactly 0
        np.array([[1.0, 0, 0], [0, 1, 0], [1, 0, -x0]]),             # w = x - x0 = 0 exactly at x = x0
        A * 1e100, A * 1e-100, A, -A])
    ths = [np.inf, 0.0, -1.0, 3.0, 1e-300]
    b = _Batch([(src, dst)] * len(ths))
    Hm = _f64(np.broadcast_to(Hs.reshape(1, -1, 9), (b.P, len(Hs), 9)))
    counts = R.score(*b.args(), Hm, 0.0, th_per_pair=_f64(ths)).cpu().numpy()
    best_h, best_c, mask = _select_raw(b, _i32(counts), Hm, 0.0, _f64(ths))
    _check_untouched(b, mask)
    band_total = 0
    for p, th in enumerate(ths):
        ref, band = hom.classify(Hs, src, dst, th)
        band_total += hom.check_counts(counts[p], ref, band, f"th={th}")
        assert counts[p, 0] == counts[p, 1] == 0                     # zero and singular H: never an inlier
        assert not ref[2, 0] and not ref[2, 1024]                    # w = 0: an outlier even at th = inf
        if th <= 0:
            assert not counts[p].any() and best_h[p] == -1 and best_c[p] == 0
        if th == np.inf:
            assert counts[p, 3] == counts[p, 4] == counts[p, 5] == counts[p, 6] == M
            assert counts[p, 2] <= M - 2
        assert counts[p, 3] == counts[p, 4] == counts[p, 5] == counts[p, 6]    # scale and sign do not matter
        w = int(best_h[p])
        assert w == hom.select_hypothesis(counts[p], M)
        mk = mask[b.off[p]:b.off[p] + M]
        if w >= 0:
            np.testing.assert_array_equal(mk == 1, ref[w])
            assert best_c[p] == counts[p, w] == mk.sum()
        else:
            assert not mk.any()
    print(f"degenerate hypotheses: band cases excused {band_total}")
    assert band_total == 0


# ---- 4. selection on hand-built counts ------------------------------------------------------------------------------

def _select_case(R, Ms, count_rows, seed):
    """Pairs of real correspondences with the given counts; every hypothesis is the pair's true H, so the mask of any
    winner is that H's reference mask."""
    rng = np.random.default_rng(seed)
    blocks, As = [], []
    for M in Ms:
        s, d, A = _pair(rng, M, 1240.0, 0.3)
        blocks.append((s, d))
        As.append(A)
    H = len(count_rows[0])
    b = _Batch(blocks)
    Hm = _f64(np.stack([np.broadcast_to(A.reshape(1, 9), (H, 9)) for A in As]))
    best_h, best_c, mask = _select_raw(b, _i32(np.array(count_rows)), Hm, 3.0)
    _check_untouched(b, mask)
    band_total = 0
    for p, M in enumerate(Ms):
        w = int(best_h[p])
        assert w == hom.select_hypothesis(count_rows[p], M), (p, w)
        mk = mask[b.off[p]:b.off[p] + M]
        if w < 0:
            assert best_c[p] == 0 and not mk.any()
            continue
        ref, band = hom.classify(As[p][None], *blocks[p], 3.0)
        band_total += int(band.sum())
        np.testing.assert_array_equal((mk == 1)[~band[0]], ref[0][~band[0]])
        assert best_c[p] == mk.sum()
    return best_h, band_total


def test_selection_rules(R):
    rows5 = [
        [3, 9, 10, 0, 0],       # M = 10: the first count above 0.8 M (h = 1) beats the later, larger one
        [8, 9, 7, 0, 0],        # M = 10: 8 == 0.8 M does not stop; 9 does
        [4, 5, 1, 0, 0],        # M = 5: 4 == 0.8 M does not stop
        [2, 7, 3, 7, 7],        # ties at the maximum: the lowest h
        [0, 0, 0, 0, 0],        # nothing scored: -1, count 0, zeroed mask
        [0, 6, 9, 9, 1],        # M = 10: 9 > 8 at h = 2 stops, h = 3 ties it
    ]
    best, band5 = _select_case(R, [10, 10, 5, 100, 40, 10], rows5, 1)
    assert best.tolist() == [1, 1, 1, 1, -1, 2]
    best, band1 = _select_case(R, [10, 10], [[5], [0]], 2)               # H = 1
    assert best.tolist() == [0, -1]
    rows257 = np.zeros((4, 257), np.int64)
    rows257[0, 256] = 3                                                  # the only count, beyond the 256-thread stride
    rows257[1, 255] = rows257[1, 256] = 4                                # tie across the stride: 255
    rows257[2, 0] = 5
    rows257[2, 256] = 6                                                  # a later maximum at h = 256
    rows257[3, 1] = rows257[3, 256] = 90                                 # M = 100: both above 0.8 M, first wins
    best, band257 = _select_case(R, [100, 100, 100, 100], rows257.tolist(), 3)
    assert best.tolist() == [256, 255, 256, 1]
    print(f"selection: band cases excused {band5 + band1 + band257}")
    assert band5 + band1 + band257 == 0


# ---- 5. K5 against dlt_homography on device-drawn samples ------------------------------------------------------------

def _normalised_system(src, dst):
    """The normalised 8x9 DLT system of dlt_homography and its transforms."""
    sn, Ts = hom.normalise_points(src)
    dn, Td = hom.normalise_points(dst)
    x, y, u, v = sn[:, 0], sn[:, 1], dn[:, 0], dn[:, 1]
    z, o = np.zeros_like(x), np.ones_like(x)
    r1 = np.stack([-x, -y, -o, z, z, z, u * x, u * y, u], axis=1)
    r2 = np.stack([z, z, z, -x, -y, -o, v * x, v * y, v], axis=1)
    return np.stack([r1, r2], axis=1).reshape(-1, 9), Ts, Td


def test_k5_matches_dlt_on_device_samples(R):
    rng = np.random.default_rng(21)
    Ms = [0, 3, 4, 5, 50, 1100, 3000]
    H = 256
    blocks = []
    for i, M in enumerate(Ms):
        s, d, _ = _pair(rng, M, 1240.0 if i % 2 else 1.0, 0.3)
        blocks.append((s, d))
    b = _Batch(blocks)
    Hm, smp = R.hypotheses(*b.args(), H, seed=1234, return_samples=True)
    Hd, smp = Hm.cpu().numpy().reshape(b.P, H, 3, 3), smp.cpu().numpy()
    eps = np.finfo(np.float64).eps
    checked, skipped, worst = 0, 0, 0.0
    for p, M in enumerate(Ms):
        if M < 4:
            assert not Hd[p].any()
            continue
        s, d = (a.astype(np.float64) for a in blocks[p])
        for h in range(H):
            idx = smp[p, h]
            assert len(set(idx.tolist())) == 4 and idx.min() >= 0 and idx.max() < M
            A, Ts, Td = _normalised_system(s[idx], d[idx])
            sv = np.linalg.svd(A, compute_uv=False)
            cond = sv[0] / sv[7]                                         # largest over smallest non-zero
            if not (cond < 1e8) or not np.isfinite(Hd[p, h]).all():
                skipped += 1
                continue
            want = hom.dlt_homography(s[idx], d[idx])
            # compare in the normalised space the null vector lives in: T_dst H T_src^-1, unit norm, sign fixed
            n_d, n_r = Td @ Hd[p, h] @ np.linalg.inv(Ts), Td @ want @ np.linalg.inv(Ts)
            n_d, n_r = n_d / np.linalg.norm(n_d), n_r / np.linalg.norm(n_r)
            n_d *= np.sign(np.vdot(n_d, n_r))
            err = np.abs(n_d - n_r).max()
            worst = max(worst, err / (eps * cond))
            assert err <= 256 * eps * cond, (p, h, err, cond)
            checked += 1
    print(f"K5: {checked} hypotheses checked, {skipped} near-degenerate samples skipped, worst error "
          f"{worst:.1f} eps * cond")
    assert skipped <= 0.01 * checked
    # host samples: coincident points, out-of-range indices and M < 4 give a hypothesis that scores 0 and never wins
    s, d, _ = _pair(rng, 50, 1240.0, 0.0)
    s[10:14] = s[10]
    d[10:14] = d[10]                                                     # four distinct indices, one coordinate
    bh = _Batch([(s, d), (s, d), (s[:3], d[:3])])
    bad = [[10, 11, 12, 13], [0, 1, 2, 50], [-1, 1, 2, 3], [0, 1, 2, 2**30]]
    samples = np.zeros((3, 5, 4), np.int32)
    samples[0, :4] = bad
    samples[0, 4] = [1, 2, 3, 4]                                         # pair 0: h = 4 is a good sample
    samples[1, :4] = bad
    samples[1, 4] = bad[0]                                               # pair 1: nothing good
    samples[2, :] = [0, 1, 2, 0]                                         # M < 4
    Hm = R.hypotheses(*bh.args(), 5, samples=_i32(samples))
    counts = R.score(*bh.args(), Hm, 3.0)
    best_h, best_c, _ = _select_raw(bh, counts, Hm, 3.0)
    c, Hn = counts.cpu().numpy(), Hm.cpu().numpy()
    assert not Hn[0, 1:4].any() and not Hn[1, 1:4].any() and not Hn[2].any()   # out of range / M < 4: zero H
    assert not np.isfinite(Hn[0, 0]).all() or not Hn[0, 0].any()               # coincident: no finite model
    assert (c[0, :4] == 0).all() and (c[1] == 0).all() and (c[2] == 0).all(), c
    assert c[0, 4] > 0 and best_h.tolist() == [4, -1, -1] and best_c[1] == best_c[2] == 0


# ---- 6. the robust-pose shape ----------------------------------------------------------------------------------------

def test_robust_pose_shape_with_device_sampler(R):
    P, H, M = 296, 2000, 500
    rng = np.random.default_rng(31)
    blocks = [_pair(rng, M, 1240.0, (0.0, 0.2, 0.4, 0.6)[p % 4])[:2] for p in range(P)]
    b = _Batch(blocks, gap=0)
    Hm = R.hypotheses(*b.args(), H, seed=99)
    counts = R.score(*b.args(), Hm, 3.0)
    best_h, best_c, mask = _select_raw(b, counts, Hm, 3.0)
    counts, Hd = counts.cpu().numpy(), Hm.cpu().numpy().reshape(P, H, 3, 3)
    band_full, band_win = 0, 0
    full = set(np.random.default_rng(32).choice(P, 8, replace=False).tolist())
    for p in range(P):
        src, dst = blocks[p]
        w = int(best_h[p])
        assert w == hom.select_hypothesis(counts[p], M) and w >= 0
        mk = mask[b.off[p]:b.off[p] + M]
        assert best_c[p] == counts[p, w] == mk.sum()
        if p in full:                                                    # every hypothesis against the reference
            ref, band = hom.classify(Hd[p], src, dst, 3.0)
            hom.check_counts(counts[p], ref, band, f"pair {p}")
            band_full += _ill_conditioned_only(Hd[p], band)
            if not band.any():
                assert w == hom.select_hypothesis(ref.sum(1), M)
            ref, band = ref[w:w + 1], band[w:w + 1]
        else:                                                            # the winner against the reference
            ref, band = hom.classify(Hd[p, w], src, dst, 3.0)
        band_win += _ill_conditioned_only(Hd[p, w:w + 1], band)
        np.testing.assert_array_equal((mk == 1)[~band[0]], ref[0][~band[0]], err_msg=f"pair {p}")
    print(f"robust-pose shape: band cases excused {band_full} (all hypotheses of {len(full)} pairs), "
          f"{band_win} (winners of {P} pairs)")
    assert band_full <= 4 and band_win == 0


# ---- 7. the batched robust-pose homography branch against the reference ---------------------------------------------

KITTI_K = np.array([[718.856, 0.0, 607.1928], [0.0, 718.856, 185.2157], [0.0, 0.0, 1.0]])


def _pose_scene(rng, i, M):
    """Pixel-scale two-view correspondences (KITTI intrinsics): planar or general structure, 0-60 % outliers."""
    planar = i % 2 == 0
    if planar:
        X = np.stack([rng.uniform(-2, 2, M), rng.uniform(-1.5, 1.5, M), np.zeros(M)], 1)
        Pw = X + np.array([0, 0, 6.0]) + X[:, :1] * np.array([0, 0, 0.2])
    else:
        Pw = np.stack([rng.uniform(-2, 2, M), rng.uniform(-1.5, 1.5, M), rng.uniform(4, 12, M)], 1)
    ax, ay, az = rng.uniform(-0.05, 0.05, 3)
    Rx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
    Ry = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
    Rz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
    Rm = Rz @ Ry @ Rx
    t = rng.uniform(-0.5, 0.5, 3) + np.array([0.3, 0, 0])
    h1, h2 = Pw @ KITTI_K.T, (Pw @ Rm.T + t) @ KITTI_K.T
    p1 = h1[:, :2] / h1[:, 2:] + rng.normal(0, 0.5, (M, 2))
    p2 = h2[:, :2] / h2[:, 2:] + rng.normal(0, 0.5, (M, 2))
    k = int((0.0, 0.15, 0.3, 0.45, 0.6)[i % 5] * M)
    if k:
        idx = rng.permutation(M)[:k]
        p2[idx] = rng.uniform(p2.min(0), p2.max(0), (k, 2))
    return p1.astype(np.float32), p2.astype(np.float32)


def test_robust_pose_homography_branch_against_the_reference():
    import torch
    from b200slam import robust_pose as rp
    Ms = [8, 12, 30, 60, 100, 250, 400, 700, 1000, 1023, 1024, 1025, 1100, 1500, 2000, 2047, 2048, 2049, 2100, 2500,
          3000, 1300, 900, 500]
    Hh = 400
    rng = np.random.default_rng(41)
    blocks, smp = [], np.zeros((len(Ms), Hh, 4), np.int32)
    for i, M in enumerate(Ms):
        blocks.append(_pose_scene(rng, i, M))
        smp[i] = hom.draw_samples(np.random.default_rng(4100 + i), M, Hh)
    b = _Batch(blocks, gap=0)
    # per-pair configurations: a large homography bias on every third scene so that the homography model is selected
    cfgs = [rp.RobustPoseConfig(min_parallax=0.0, homography_bias=10.0 if i % 3 == 0 else 0.9) for i in range(len(Ms))]
    est = rp.RobustPose()
    out = est.run(b.corr, b.off_d, b.cnt_d, b.P, KITTI_K, cfgs, samples_h=_i32(smp), seed=3, max_m=max(Ms), hypotheses=256)
    torch.cuda.synchronize()
    res = rp.decode_results(out.results.cpu().numpy())
    out_mask, H_fit = out.mask.cpu().numpy(), out.H_fit.cpu().numpy().reshape(-1, 3, 3)
    bh, bc = est._buf["best_h_h"][:b.P].cpu().numpy(), est._buf["best_c_h"][:b.P].cpu().numpy()
    counts, Hd = est._buf["counts_h"][:b.P].cpu().numpy(), est._buf["Hm"][:b.P].cpu().numpy().reshape(b.P, Hh, 3, 3)
    band_total, n_skip_decide, n_h = 0, 0, 0
    for p, M in enumerate(Ms):
        src, dst = blocks[p]
        ref, band = hom.classify(Hd[p], src, dst, rp.HOMOGRAPHY_THRESHOLD)
        hom.check_counts(counts[p], ref, band, f"scene {p} (M={M})")
        band_total += _ill_conditioned_only(Hd[p], band)
        want_h = hom.select_hypothesis(ref.sum(1), M)
        assert want_h >= 0 and bh[p] == want_h, (p, M, bh[p], want_h)
        assert bc[p] == ref[want_h].sum()
        # the hypothesis itself is dlt_homography's on the same four host-drawn indices
        s64, d64 = src.astype(np.float64), dst.astype(np.float64)
        want_H = hom.dlt_homography(s64[smp[p, want_h]], d64[smp[p, want_h]])
        np.testing.assert_allclose(Hd[p, want_h], want_H, rtol=1e-7, atol=1e-7 * np.abs(want_H).max())
        if res[p]["h_best_h"] == -1:                     # stopped before the homography branch is decided
            n_skip_decide += 1
        else:
            assert (res[p]["h_best_h"], res[p]["h_inliers"]) == (want_h, ref[want_h].sum())
        inl = np.flatnonzero(ref[want_h]) if want_h >= 0 else np.zeros(0, np.int64)
        if inl.size >= 4:
            want_fit = hom.dlt_homography(s64[inl], d64[inl])
            np.testing.assert_allclose(H_fit[p], want_fit, rtol=1e-9, atol=1e-9 * np.abs(want_fit).max())
        else:
            assert not H_fit[p].any()
        if res[p]["outcome"] in (rp.POSE_ESTIMATE, rp.POSE_GATE_FAILED) and res[p]["method"] == 1:
            n_h += 1
            np.testing.assert_array_equal(out_mask[b.off[p]:b.off[p] + M] == 1, ref[want_h])
    print(f"robust pose: band cases excused {band_total}; {n_skip_decide} scenes read from the branch buffers, "
          f"{n_h} scenes select the homography")
    assert band_total <= 4
    assert n_skip_decide >= 1 and n_h >= 1
