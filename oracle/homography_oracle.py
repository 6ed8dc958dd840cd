"""CPU oracle — RANSAC homography hypothesis generation / scoring.  TEST INFRASTRUCTURE ONLY.

NumPy restatement of /root/reference/homography.py:118-216 (Hartley normalisation, 4-point /
n-point DLT, symmetric transfer error, sequential best / early-exit selection).  float64
throughout, like the reference.  Nothing in the product imports this module.
"""
from __future__ import annotations

import numpy as np


def normalise_points(pts):
    """homography.py:118-125."""
    pts = np.asarray(pts, dtype=np.float64)
    c = pts.mean(axis=0)
    diffs = pts - c
    with np.errstate(divide="ignore", invalid="ignore"):
        rms = np.sqrt((diffs ** 2).sum(axis=1).mean())
        s = np.sqrt(2) / rms
    T = np.array([[s, 0, -s * c[0]], [0, s, -s * c[1]], [0, 0, 1]])
    pts_h = np.hstack([pts, np.ones((len(pts), 1))])
    return (T @ pts_h.T).T[:, :2], T


def dlt_homography(src, dst) -> np.ndarray:
    """homography.py:131-142: normalised DLT, null vector = last right-singular vector,
    de-normalised, scaled so that H[2, 2] = 1."""
    src_n, T_src = normalise_points(src)
    dst_n, T_dst = normalise_points(dst)
    x, y, u, v = src_n[:, 0], src_n[:, 1], dst_n[:, 0], dst_n[:, 1]
    z, o = np.zeros_like(x), np.ones_like(x)
    r1 = np.stack([-x, -y, -o, z, z, z, u * x, u * y, u], axis=1)
    r2 = np.stack([z, z, z, -x, -y, -o, v * x, v * y, v], axis=1)
    A = np.stack([r1, r2], axis=1).reshape(-1, 9)
    _, _, Vt = np.linalg.svd(A)
    Hn = Vt[-1].reshape(3, 3)
    H = np.linalg.inv(T_dst) @ Hn @ T_src
    return H / H[2, 2]


def transfer_error(H, src, dst) -> np.ndarray:
    """Symmetric transfer error of homography.py:199-205 (sum of the two Euclidean norms)."""
    src, dst = np.asarray(src, dtype=np.float64), np.asarray(dst, dtype=np.float64)
    n = len(src)
    src_h, dst_h = np.hstack([src, np.ones((n, 1))]), np.hstack([dst, np.ones((n, 1))])
    with np.errstate(all="ignore"):
        pf = (H @ src_h.T).T
        pf = pf[:, :2] / pf[:, 2, None]
        pb = (np.linalg.inv(H) @ dst_h.T).T
        pb = pb[:, :2] / pb[:, 2, None]
        return np.linalg.norm(pf - dst, axis=1) + np.linalg.norm(pb - src, axis=1)


def score_hypotheses(Hs, src, dst, th: float):
    """Inlier masks (n_hyp, M) and counts for every homography (NaN error -> outlier)."""
    Hs = np.asarray(Hs, dtype=np.float64).reshape(-1, 3, 3)
    masks = np.zeros((len(Hs), len(src)), dtype=bool)
    for h, H in enumerate(Hs):
        try:
            with np.errstate(all="ignore"):
                masks[h] = transfer_error(H, src, dst) < th
        except np.linalg.LinAlgError:
            pass                                   # singular H: the reference would raise here; the device scores it as no inliers
    return masks, masks.sum(axis=1).astype(np.int64)


HP_DIGITS = 60              # working precision of transfer_error_hp (decimal digits)
BAND_TAU = 2.0 ** -40       # half-width of the rounding band, relative to the per-evaluation scale B
HP_SCREEN = 1e-6            # evaluations with |e64 - th| <= HP_SCREEN * B are re-evaluated in high precision


def _mp_transfer(H, src, dst):
    """mpmath symmetric transfer errors (list of mpf, nan where undefined) of one H over the given points.
    Inputs are taken exactly: the float64 entries of H and the coordinates as given (float32 -> exact float)."""
    import mpmath

    with mpmath.workdps(HP_DIGITS):
        h = [mpmath.mpf(float(v)) for v in np.asarray(H, dtype=np.float64).reshape(9)]
        c = [h[4] * h[8] - h[5] * h[7], h[5] * h[6] - h[3] * h[8], h[3] * h[7] - h[4] * h[6]]
        det = h[0] * c[0] + h[1] * c[1] + h[2] * c[2]
        n = len(src)
        if det == 0:
            return [mpmath.mpf("nan")] * n
        # adjugate / det in the same precision (never np.linalg.inv's float64 result)
        g = [c[0], h[2] * h[7] - h[1] * h[8], h[1] * h[5] - h[2] * h[4],
             c[1], h[0] * h[8] - h[2] * h[6], h[2] * h[3] - h[0] * h[5],
             c[2], h[1] * h[6] - h[0] * h[7], h[0] * h[4] - h[1] * h[3]]
        g = [v / det for v in g]
        out = []
        for (x, y), (u, v) in zip(np.asarray(src, dtype=np.float64), np.asarray(dst, dtype=np.float64)):
            x, y, u, v = mpmath.mpf(float(x)), mpmath.mpf(float(y)), mpmath.mpf(float(u)), mpmath.mpf(float(v))
            pw = h[6] * x + h[7] * y + h[8]
            qw = g[6] * u + g[7] * v + g[8]
            if pw == 0 or qw == 0:
                out.append(mpmath.mpf("nan"))
                continue
            px, py = (h[0] * x + h[1] * y + h[2]) / pw, (h[3] * x + h[4] * y + h[5]) / pw
            qx, qy = (g[0] * u + g[1] * v + g[2]) / qw, (g[3] * u + g[4] * v + g[5]) / qw
            out.append(mpmath.sqrt((px - u) ** 2 + (py - v) ** 2) + mpmath.sqrt((qx - x) ** 2 + (qy - y) ** 2))
        return out


def transfer_error_hp(H, src, dst) -> np.ndarray:
    """transfer_error in HP_DIGITS-digit arithmetic from the exact inputs, rounded once to float64 at the end.
    nan where H is singular or a point maps to w = 0 (an outlier, as in score_hypotheses)."""
    return np.array([float(e) for e in _mp_transfer(H, src, dst)], dtype=np.float64).reshape(len(src))


def _adj_abs(Hs):
    """Adjugates of (n, 3, 3) H, and the sums of the absolute values of the two products forming each entry."""
    h = Hs.reshape(-1, 9)
    pairs = (((4, 8), (5, 7)), ((2, 7), (1, 8)), ((1, 5), (2, 4)),
             ((5, 6), (3, 8)), ((0, 8), (2, 6)), ((2, 3), (0, 5)),
             ((3, 7), (4, 6)), ((1, 6), (0, 7)), ((0, 4), (1, 3)))
    adj = np.stack([h[:, a] * h[:, b] - h[:, c] * h[:, d] for (a, b), (c, d) in pairs], 1).reshape(-1, 3, 3)
    aab = np.stack([np.abs(h[:, a] * h[:, b]) + np.abs(h[:, c] * h[:, d]) for (a, b), (c, d) in pairs], 1).reshape(-1, 3, 3)
    return adj, aab


def _project_bound(A, Aabs, P):
    """Projections of points P (M, 2) through (n, 3, 3) A -> (proj (n, M, 2), w (n, M), condition (n, M)).
    condition bounds |d proj| / eps for componentwise relative perturbations of A's entries and of the products:
    (|A| |p|)_0 + (|A| |p|)_1 + (|proj_x| + |proj_y|) (|A| |p|)_2, over |w|."""
    Ph = np.hstack([P, np.ones((len(P), 1))])
    num = np.einsum("nij,mj->nmi", A, Ph)
    mag = np.einsum("nij,mj->nmi", Aabs, np.abs(Ph))
    w = num[..., 2]
    proj = num[..., :2] / w[..., None]
    cond = (mag[..., 0] + mag[..., 1] + np.abs(proj).sum(-1) * mag[..., 2]) / np.abs(w)
    return proj, w, cond, mag[..., 2]


def classify(Hs, src, dst, th: float, hyp_block: int = 256):
    """Reference inlier decisions (transfer error < th) for every (hypothesis, correspondence), and the rounding band.

    Two stages: every evaluation in vectorised float64, then the ones whose float64 error lies within
    HP_SCREEN * B of th (or whose float64 evaluation is non-finite, or whose denominators are within rounding of
    zero) again in HP_DIGITS-digit arithmetic. Returns (mask, band), both bool (n_hyp, M): mask is the
    high-precision decision; band marks the evaluations a correct float64 kernel may decide either way:
      * |e* - th| <= BAND_TAU * B, with the per-evaluation scale
            B = max(1, |x|, |y|, |u|, |v|, |Hx|, |H^-1 u|) + C_f + C_b,
        C_f / C_b the componentwise condition numbers of the forward / backward projections (_project_bound; the
        backward one is taken over the adjugate, because the 1 / det factor of the inverse cancels in the ratio).
        A kernel that evaluates the reference's formulas in float64 with any order of fma / mul / add makes an
        absolute error of at most a small multiple (< 100) of eps * B in e; BAND_TAU = 2^-40 = 4096 eps leaves
        a wide margin above that while keeping the band ~1e-8 px wide on pixel-scale data (expected hits on random
        data: 0). Near-singular H makes C_b large, so such evaluations are honestly reported as band cases.
      * the high-precision error is finite but float64 overflows, or the exact denominator is 0 while float64
        rounding left it non-zero (either way rounding decides).
    th <= 0 has no inliers and no band (the error is a sum of square roots, >= 0 in any rounding); non-finite
    errors are outliers at every th, th = +inf included."""
    Hs = np.asarray(Hs, dtype=np.float64).reshape(-1, 3, 3)
    src = np.asarray(src, dtype=np.float64).reshape(-1, 2)
    dst = np.asarray(dst, dtype=np.float64).reshape(-1, 2)
    n, M = len(Hs), len(src)
    mask = np.zeros((n, M), dtype=bool)
    band = np.zeros((n, M), dtype=bool)
    if M == 0 or n == 0 or not th > 0:
        return mask, band
    eps_screen = HP_SCREEN
    ptmax = np.maximum(np.abs(src).max(1), np.abs(dst).max(1))
    for b0 in range(0, n, hyp_block):
        A = Hs[b0:b0 + hyp_block]
        adj, aab = _adj_abs(A)
        with np.errstate(all="ignore"):
            pf, wf, cf, wf_mag = _project_bound(A, np.abs(A), src)
            pb, wb, cb, wb_mag = _project_bound(adj, aab, dst)
            h = A.reshape(-1, 9)
            det = h[:, 0] * adj[:, 0, 0] + h[:, 1] * adj[:, 1, 0] + h[:, 2] * adj[:, 2, 0]
            det_mag = np.abs(h[:, 0] * adj[:, 0, 0]) + np.abs(h[:, 1] * adj[:, 1, 0]) + np.abs(h[:, 2] * adj[:, 2, 0])
            e64 = np.linalg.norm(pf - dst[None], axis=2) + np.linalg.norm(pb - src[None], axis=2)
            e64[det == 0] = np.nan                                    # singular: no inverse, as the device's 1 / det
            B = np.fmax(np.fmax(1.0, ptmax[None]), np.fmax(np.abs(pf).max(2), np.abs(pb).max(2)))
            B = B + np.nan_to_num(cf, nan=0.0) + np.nan_to_num(cb, nan=0.0)
            fin = np.isfinite(e64)
            mask[b0:b0 + len(A)] = fin & (e64 < th)
            near = ~fin | (np.abs(wf) <= eps_screen * wf_mag) | (np.abs(wb) <= eps_screen * wb_mag)
            if np.isfinite(th):
                near |= np.abs(e64 - th) <= eps_screen * B
            near |= ~np.isfinite(B)
            near |= (np.abs(det) <= eps_screen * det_mag)[:, None]    # singular within rounding
        for hl in np.flatnonzero(near.any(1)):
            hg = b0 + hl
            idx = np.flatnonzero(near[hl])
            ehp = _mp_transfer(Hs[hg], src[idx], dst[idx])
            for k, m in enumerate(idx):
                e = ehp[k]
                if e != e:                                            # nan: undefined, an outlier
                    mask[hg, m] = False
                    band[hg, m] = bool(fin[hl, m])
                    continue
                mask[hg, m] = bool(e < th)
                if not fin[hl, m] or not np.isfinite(B[hl, m]):
                    band[hg, m] = True
                elif np.isfinite(th):
                    band[hg, m] = bool(abs(float(e - th)) <= BAND_TAU * B[hl, m])
    return mask, band


def check_counts(dev_counts, ref_mask, band, label=""):
    """Device counts (n_hyp,) against a reference (mask, band) pair: equal outside the band, i.e.
    count_ref - (band & ref inlier) <= count_dev <= count_ref + (band & ref outlier). Returns the band size."""
    dev_counts = np.asarray(dev_counts, dtype=np.int64).reshape(-1)
    lo = (ref_mask & ~band).sum(1)
    hi = (ref_mask | band).sum(1)
    bad = np.flatnonzero((dev_counts < lo) | (dev_counts > hi))
    assert bad.size == 0, (f"{label}: {bad.size} hypotheses differ from the reference outside the band, first h={bad[0]}: "
                           f"device {dev_counts[bad[0]]}, reference {ref_mask[bad[0]].sum()} (band {band[bad[0]].sum()})")
    return int(band.sum())


def select_hypothesis(counts, n: int) -> int:
    """homography.py:207-211: strictly-more-inliers update, break above 0.8 n; -1 if nothing scored."""
    best, best_count = -1, 0
    for h, c in enumerate(np.asarray(counts)):
        if c > best_count:
            best, best_count = h, int(c)
            if c > 0.8 * n:
                break
    return best


def draw_samples(rng: np.random.Generator, n: int, max_iter: int) -> np.ndarray:
    """The index stream of ransac_homography (homography.py:193)."""
    return np.stack([rng.choice(n, 4, replace=False) for _ in range(max_iter)])


def ransac_homography(src, dst, th: float = 3.0, max_iter: int = 2000, rng=None):
    """homography.py:148-216 -> (refined H, inlier indices)."""
    src, dst = np.asarray(src, dtype=np.float64), np.asarray(dst, dtype=np.float64)
    n = len(src)
    if n < 4:
        raise ValueError("At least four correspondences are required")
    if rng is None:
        rng = np.random.default_rng()
    best_H, best_inliers = None, np.array([], dtype=int)
    for _ in range(max_iter):
        idx = rng.choice(n, 4, replace=False)
        H = dlt_homography(src[idx], dst[idx])
        inliers = np.flatnonzero(transfer_error(H, src, dst) < th)
        if inliers.size > best_inliers.size:
            best_H, best_inliers = H, inliers
            if inliers.size > 0.8 * n:
                break
    if best_H is None or best_inliers.size < 4:
        raise RuntimeError("RANSAC failed — too few inliers")
    return dlt_homography(src[best_inliers], dst[best_inliers]), best_inliers
