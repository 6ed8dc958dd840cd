"""GPU parity — Hamming kNN-2 / column-min / selection through the C ABI, bit-exact
against the golden vectors (cv2.BFMatcher 4.13 + the reference's own matchers) and the
CPU oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import hamming_oracle as ho


@pytest.fixture(scope="module")
def hg(golden_dir):
    return np.load(golden_dir / "hamming_golden.npz")


@pytest.fixture(scope="module")
def matcher():
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher
    return HammingMatcher(variant=_capi.VARIANT_POPC)          # K1; the i8 variants have their own fixture below


def _pad(a):
    return a if a.shape[1] == 32 else np.concatenate([a, np.zeros((len(a), 32 - a.shape[1]), np.uint8)], 1)


def test_knn2_keys_match_cv2_golden(hg, matcher):
    names = list(hg["names"])
    qs = [hg[f"{n}/q"] for n in names]
    ts = [hg[f"{n}/t"] for n in names]
    out = matcher.knn2_pairs(qs, ts)            # all 45 cases as ONE batched launch (ragged sizes)
    for name, (fb, fs, bb) in zip(names, out):
        idx, dist = hg[f"{name}/knn_idx"], hg[f"{name}/knn_dist"]
        kf = min(2, len(hg[f"{name}/t"]))
        np.testing.assert_array_equal(fb & ho.IDX_MASK, idx[:, 0], err_msg=name)
        np.testing.assert_array_equal(fb >> ho.IDX_BITS, dist[:, 0], err_msg=name)
        if kf == 2:
            np.testing.assert_array_equal(fs & ho.IDX_MASK, idx[:, 1], err_msg=name)
            np.testing.assert_array_equal(fs >> ho.IDX_BITS, dist[:, 1], err_msg=name)
        else:
            assert (fs == ho.NONE_KEY).all(), name
        b, s, bw = ho.packed_keys(hg[f"{name}/q"], hg[f"{name}/t"])
        np.testing.assert_array_equal(bb, bw, err_msg=name)


@pytest.mark.parametrize("csa", [0, 1, 2, 3])
@pytest.mark.parametrize("rows,warps", [(2, 4), (2, 8), (4, 4), (4, 8)])
def test_every_kernel_configuration_is_bit_exact(hg, csa, rows, warps):
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher
    lib = _capi.load_library()
    _capi.check(lib.b2s_hamming_set_config(csa, rows, warps))
    try:
        m = HammingMatcher(variant=0)
        names = ["noisy_1944x2000", "tie_w2_127x129", "orb_real_0", "duplicates_70x70", "tie_w32_300x257"]
        out = m.knn2_pairs([hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names])
        for n, (fb, fs, bb) in zip(names, out):
            b, s, bw = ho.packed_keys(hg[f"{n}/q"], hg[f"{n}/t"])
            np.testing.assert_array_equal(fb, b, err_msg=n)
            np.testing.assert_array_equal(fs, s, err_msg=n)
            np.testing.assert_array_equal(bb, bw, err_msg=n)
    finally:
        _capi.check(lib.b2s_hamming_set_config(2, 2, 4))


@pytest.mark.parametrize("t_split", [1, 2, 3, 7, 0])
def test_train_split_merge_is_exact(hg, t_split):
    from b200slam.frontend import HammingMatcher
    m = HammingMatcher(variant=0, t_split=t_split)
    for n in ("noisy_2000x2000", "noisy_640x33", "tie_w1_300x257"):
        (fb, fs, bb), = m.knn2_pairs([hg[f"{n}/q"]], [hg[f"{n}/t"]])
        b, s, bw = ho.packed_keys(hg[f"{n}/q"], hg[f"{n}/t"])
        np.testing.assert_array_equal(fb, b, err_msg=n)
        np.testing.assert_array_equal(fs, s, err_msg=n)
        np.testing.assert_array_equal(bb, bw, err_msg=n)


def test_cross_check_equals_cv2(hg, matcher):
    names = list(hg["names"])
    out = matcher.match_pairs([hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names],
                              use_ratio=False, use_cross=True, sort_by_distance=False)
    for n, (qi, ti, d) in zip(names, out):
        np.testing.assert_array_equal(qi, hg[f"{n}/cc_q"], err_msg=n)
        np.testing.assert_array_equal(ti, hg[f"{n}/cc_t"], err_msg=n)
        np.testing.assert_array_equal(d, hg[f"{n}/cc_d"], err_msg=n)


def test_pipeline_match_equals_reference(hg, matcher):
    names = list(hg["names"])
    qs, ts = [hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names]
    checked = 0
    for cross in (True, False):
        for ratio in (0.6, 0.75, 0.8, 1.0):
            for mm in (None, 1, 500):
                if cross and ratio != 0.8:
                    continue
                out = matcher.match_pairs(qs, ts, use_ratio=not cross, use_cross=cross, ratio=ratio,
                                          sort_by_distance=True, max_matches=mm)
                for n, (qi, ti, d) in zip(names, out):
                    key = f"{n}/pipe_c{int(cross)}_r{ratio}_m{mm}"
                    np.testing.assert_array_equal(qi, hg[key + "_q"], err_msg=key)
                    np.testing.assert_array_equal(ti, hg[key + "_t"], err_msg=key)
                    np.testing.assert_array_equal(d, hg[key + "_d"], err_msg=key)
                    checked += 1
    assert checked > 500


def test_combined_mode_equals_match_orb_descriptors(hg, matcher):
    names = [n for n in hg["names"] if f"{n}/mod_r0.8" in hg]
    for ratio in (0.8, 0.6, 1.0):
        out = matcher.match_pairs([hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names],
                                  use_ratio=True, use_cross=True, ratio=ratio, sort_by_distance=False)
        for n, (qi, ti, d) in zip(names, out):
            got = np.stack([qi, ti], 1).reshape(-1, 2)
            np.testing.assert_array_equal(got, hg[f"{n}/mod_r{ratio}"], err_msg=f"{n} r={ratio}")


def test_randomised_ragged_batches_against_oracle(matcher):
    rng = np.random.default_rng(11)
    for trial in range(4):
        sizes = [(int(rng.integers(1, 700)), int(rng.integers(1, 700))) for _ in range(12)] + [(0, 5), (5, 0), (513, 129)]
        qs = [rng.integers(0, 4 if trial % 2 else 256, (a, 32), dtype=np.uint8) for a, _ in sizes]
        ts = [rng.integers(0, 4 if trial % 2 else 256, (b, 32), dtype=np.uint8) for _, b in sizes]
        out = matcher.knn2_pairs(qs, ts)
        for (q, t), (fb, fs, bb) in zip(zip(qs, ts), out):
            b, s, bw = ho.packed_keys(q, t)
            np.testing.assert_array_equal(fb, b)
            np.testing.assert_array_equal(fs, s)
            np.testing.assert_array_equal(bb, bw)
        sel = matcher.match_pairs(qs, ts, use_ratio=True, use_cross=True, ratio=0.9, max_matches=50)
        for (q, t), (qi, ti, d) in zip(zip(qs, ts), sel):
            if len(q) == 0 or len(t) == 0:
                assert len(qi) == 0
                continue
            e = ho.select_matches(*ho.packed_keys(q, t), use_ratio=True, use_cross=True, ratio=0.9, max_matches=50)
            np.testing.assert_array_equal(qi, e[0])
            np.testing.assert_array_equal(ti, e[1])
            np.testing.assert_array_equal(d, e[2])


def test_full_size_properties_10k(matcher):
    """BASELINE config #4 size (10k x 10k): checked through size-independent properties
    plus the oracle on a row subset."""
    rng = np.random.default_rng(4096)
    n = 10_000
    q = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    perm = rng.permutation(n)
    bits = np.unpackbits(q[perm], axis=1)
    bits ^= (rng.random(bits.shape) < 0.08).astype(np.uint8)
    t = np.packbits(bits, axis=1)
    (fb, fs, bb), = matcher.knn2_pairs([q], [t])
    assert (fb <= fs).all()                                           # top-2 ordered
    # symmetry: swapping the roles swaps forward and backward minima
    (fb2, fs2, bb2), = matcher.knn2_pairs([t], [q])
    np.testing.assert_array_equal(bb, fb2)
    np.testing.assert_array_equal(bb2, fb)
    # the planted permutation is recovered (noise 8% << random-pair distance 128)
    inv = np.empty(n, np.int64)
    inv[perm] = np.arange(n)
    assert ((fb & ho.IDX_MASK) == inv).mean() > 0.999
    rows = rng.choice(n, 200, replace=False)
    D = ho.hamming_matrix(q[rows], t)
    kf = (D.astype(np.uint32) << ho.IDX_BITS) | np.arange(n, dtype=np.uint32)[None]
    part = np.sort(kf, axis=1)[:, :2]
    np.testing.assert_array_equal(fb[rows], part[:, 0])
    np.testing.assert_array_equal(fs[rows], part[:, 1])
    # identical sets: every row matches itself at distance 0 (tests/test_keyframe_manager.py:30-37)
    (fb3, _, bb3), = matcher.knn2_pairs([q], [q])
    np.testing.assert_array_equal(fb3, np.arange(n, dtype=np.uint32))
    np.testing.assert_array_equal(bb3, np.arange(n, dtype=np.uint32))


def test_shared_train_block_via_src_rows(matcher):
    """Relocalization layout: many query blocks against ONE shared train block."""
    import torch
    from b200slam.frontend import PairBatch
    rng = np.random.default_rng(3)
    cur = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    kfs = [rng.integers(0, 256, (int(rng.integers(50, 400)), 32), dtype=np.uint8) for _ in range(6)]
    b = PairBatch.from_host(kfs, [cur] * 6)
    b.t_desc = torch.from_numpy(cur).cuda()               # one copy of the train block
    b.t_src = torch.zeros(6, dtype=torch.int32, device="cuda")
    k = matcher.knn2(b)
    fb = k.fwd_best.cpu().numpy().view(np.uint32)
    bb = k.bwd_best.cpu().numpy().view(np.uint32)
    for p, kf in enumerate(kfs):
        e = ho.packed_keys(kf, cur)
        np.testing.assert_array_equal(fb[b.q_off_host[p]:b.q_off_host[p + 1]], e[0])
        np.testing.assert_array_equal(bb[b.t_off_host[p]:b.t_off_host[p + 1]], e[2])


def test_bad_arguments_raise(matcher):
    with pytest.raises(ValueError):
        matcher.knn2_pairs([np.zeros((3, 32), np.float32)], [np.zeros((3, 32), np.uint8)])
    with pytest.raises(ValueError):
        matcher.knn2_pairs([np.zeros((3, 64), np.uint8)], [np.zeros((3, 64), np.uint8)])


# ---- K2: tcgen05 kind::i8 variant, same contract, same bit-exact bar -------------------

@pytest.fixture(scope="module", params=["two_products", "single_product"])
def matcher_i8(request):
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher
    return HammingMatcher(variant=_capi.VARIANT_I8MMA if request.param == "two_products" else _capi.VARIANT_I8MMA1)


def test_i8_variant_golden_bit_exact(hg, matcher_i8):
    names = list(hg["names"])
    out = matcher_i8.knn2_pairs([hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names])
    for n, (fb, fs, bb) in zip(names, out):
        b, s, bw = ho.packed_keys(_pad(hg[f"{n}/q"]), _pad(hg[f"{n}/t"]))
        np.testing.assert_array_equal(fb, b, err_msg=n)
        np.testing.assert_array_equal(fs, s, err_msg=n)
        np.testing.assert_array_equal(bb, bw, err_msg=n)


def test_i8_variant_ragged_and_large(matcher_i8, matcher):
    rng = np.random.default_rng(21)
    sizes = [(int(rng.integers(1, 900)), int(rng.integers(1, 900))) for _ in range(10)] + [(0, 7), (7, 0), (128, 128), (129, 127), (256, 300), (257, 1), (1, 257), (384, 385), (2000, 2000), (1944, 2000)]
    for alphabet in (256, 4):
        qs = [rng.integers(0, alphabet, (a, 32), dtype=np.uint8) for a, _ in sizes]
        ts = [rng.integers(0, alphabet, (b, 32), dtype=np.uint8) for _, b in sizes]
        got = matcher_i8.knn2_pairs(qs, ts)
        want = matcher.knn2_pairs(qs, ts)          # K1, itself pinned to the oracle above
        for (fb, fs, bb), (wb, ws, wbb), sz in zip(got, want, sizes):
            np.testing.assert_array_equal(fb, wb, err_msg=str(sz))
            np.testing.assert_array_equal(fs, ws, err_msg=str(sz))
            np.testing.assert_array_equal(bb, wbb, err_msg=str(sz))
    q, t = qs[-2], ts[-2]
    b, s, bw = ho.packed_keys(q, t)
    np.testing.assert_array_equal(got[-2][0], b)
    np.testing.assert_array_equal(got[-2][2], bw)


def test_i8_variant_pipeline_front_doors(hg, matcher_i8):
    names = ["noisy_2000x2000", "orb_real_0", "duplicates_70x70", "identical_50"]
    qs, ts = [hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names]
    out = matcher_i8.match_pairs(qs, ts, use_ratio=False, use_cross=True, sort_by_distance=True, max_matches=500)
    for n, (qi, ti, d) in zip(names, out):
        key = f"{n}/pipe_c1_r0.8_m500"
        np.testing.assert_array_equal(qi, hg[key + "_q"], err_msg=key)
        np.testing.assert_array_equal(ti, hg[key + "_t"], err_msg=key)
        np.testing.assert_array_equal(d, hg[key + "_d"], err_msg=key)


def test_shared_block_path_equals_per_pair_expansion():
    """b2s_hamming_knn2_shared (every frame expanded once, pairs address the tiles) against the
    per-pair expansion and against the POPC kernel on a ragged frame sequence: tile-edge sizes, a
    one-row frame and an empty frame."""
    import dataclasses
    import torch
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher, sequence_batch
    rng = np.random.default_rng(77)
    N = 320
    counts = np.array([300, 1, 128, 0, 257, 129, 320, 127], np.int32)
    F = len(counts)
    desc = rng.integers(0, 4, (F * N, 32), dtype=np.uint8)          # tie-heavy
    desc[2 * N:2 * N + 64] = desc[:64]                               # duplicates across frames
    dev = torch.from_numpy(desc).cuda()
    kp = torch.zeros((F * N, 2), dtype=torch.float32, device="cuda")
    b = sequence_batch(dev, kp, counts, 0, F - 1, N)
    assert b.shared is not None and b.shared.n_blocks == F
    shared = HammingMatcher(variant=_capi.VARIANT_I8MMA1).knn2(b)
    plain = HammingMatcher(variant=_capi.VARIANT_I8MMA1).knn2(dataclasses.replace(b, shared=None))
    popc = HammingMatcher(variant=_capi.VARIANT_POPC).knn2(b)
    for name in ("fwd_best", "fwd_second", "bwd_best"):
        a, c, d = (getattr(x, name).cpu().numpy() for x in (shared, plain, popc))
        assert np.array_equal(a, c), name
        assert np.array_equal(a, d), name
    # and against the oracle, pair by pair
    fb, fs, bw = (getattr(shared, n).cpu().numpy().view(np.uint32) for n in ("fwd_best", "fwd_second", "bwd_best"))
    for p in range(F - 1):
        q = desc[p * N:p * N + counts[p]]
        t = desc[(p + 1) * N:(p + 1) * N + counts[p + 1]]
        rb, rs, rw = ho.packed_keys(q, t)
        qo, to = int(b.q_off_host[p]), int(b.t_off_host[p])
        assert np.array_equal(fb[qo:qo + len(q)], rb) and np.array_equal(fs[qo:qo + len(q)], rs), p
        assert np.array_equal(bw[to:to + len(t)], rw), p


# ---- K2s work decomposition: 2 query sub-tiles per item x train-axis split ----------

def _plan(lib):
    import ctypes as C
    v = [C.c_int(0) for _ in range(3)]
    lib.b2s_hamming_last_plan(*[C.byref(x) for x in v])
    return tuple(x.value for x in v)


@pytest.mark.parametrize("t_split", [0, 1, 2, 3, 4, 5, 6, 7, 8, 11, 16, 64])
def test_k2s_decompositions_are_bit_exact(hg, t_split):
    """Every train-split plan of the single-product kernel gives the POPC kernel's / the oracle's keys:
    golden tie-heavy cases, ragged batches with empty sides and tile-edge sizes, and a lone 2000 x 2000
    pair (the drop-in call: 8 work items without the split)."""
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher
    lib = _capi.load_library()
    m = HammingMatcher(variant=_capi.VARIANT_I8MMA1, t_split=t_split)
    k1 = HammingMatcher(variant=_capi.VARIANT_POPC)
    names = ["noisy_2000x2000", "tie_w2_127x129", "orb_real_0", "duplicates_70x70", "tie_w32_300x257", "noisy_640x33"]
    rng = np.random.default_rng(5 + t_split)
    sizes = [(int(rng.integers(1, 1200)), int(rng.integers(1, 1200))) for _ in range(6)] + [(0, 9), (9, 0), (513, 129), (1, 1025), (1025, 1)]
    qs = [_pad(hg[f"{n}/q"]) for n in names] + [rng.integers(0, 4, (a, 32), dtype=np.uint8) for a, _ in sizes]
    ts = [_pad(hg[f"{n}/t"]) for n in names] + [rng.integers(0, 4, (b, 32), dtype=np.uint8) for _, b in sizes]
    got, want = m.knn2_pairs(qs, ts), k1.knn2_pairs(qs, ts)
    subs, ts_used, _ = _plan(lib)
    assert subs == 2
    if t_split > 0:
        assert ts_used == min(t_split, (max(len(t) for t in ts) + 127) // 128)
    for i, ((fb, fs, bb), (wb, ws, wbb)) in enumerate(zip(got, want)):
        np.testing.assert_array_equal(fb, wb, err_msg=str(i))
        np.testing.assert_array_equal(fs, ws, err_msg=str(i))
        np.testing.assert_array_equal(bb, wbb, err_msg=str(i))
    # one lone pair, against the oracle
    (fb, fs, bb), = m.knn2_pairs([qs[0]], [ts[0]])
    b, s, bw = ho.packed_keys(qs[0], ts[0])
    np.testing.assert_array_equal(fb, b)
    np.testing.assert_array_equal(fs, s)
    np.testing.assert_array_equal(bb, bw)
    if t_split == 0:
        assert _plan(lib)[1] > 1, "a lone pair must be split along the train axis"


@pytest.mark.parametrize("t_split", [0, 1, 3, 7])
def test_k2s_shared_blocks_with_split(t_split):
    """The shared-block entry (frames expanded once) with and without a train split, ragged frame sequence."""
    import torch
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher, sequence_batch
    lib = _capi.load_library()
    rng = np.random.default_rng(78)
    N = 700
    counts = np.array([700, 1, 128, 0, 513, 129, 640, 127, 512], np.int32)
    F = len(counts)
    desc = rng.integers(0, 4, (F * N, 32), dtype=np.uint8)
    dev = torch.from_numpy(desc).cuda()
    kp = torch.zeros((F * N, 2), dtype=torch.float32, device="cuda")
    b = sequence_batch(dev, kp, counts, 0, F - 1, N)
    got = HammingMatcher(variant=_capi.VARIANT_I8MMA1, t_split=t_split).knn2(b)
    assert _plan(lib)[0] == 2
    popc = HammingMatcher(variant=_capi.VARIANT_POPC).knn2(b)
    for name in ("fwd_best", "fwd_second", "bwd_best"):
        assert np.array_equal(getattr(got, name).cpu().numpy(), getattr(popc, name).cpu().numpy()), name


@pytest.mark.parametrize("t_split", [0, 3])
def test_k2s_best_only_variant(hg, t_split):
    """B2S_HAMMING_BEST_ONLY (cross-check-only matching: BFMatcher(crossCheck=True).match never reads the second
    neighbour): fwd_best and bwd_best are those of the full kernel / the oracle, fwd_second is all "none", and the
    cross-check front door returns cv2's matches — per-pair and shared-block entries, with and without a train split."""
    import torch
    from b200slam import _capi
    from b200slam.frontend import HammingMatcher, PairBatch, sequence_batch
    names = list(hg["names"])
    qs, ts = [_pad(hg[f"{n}/q"]) for n in names], [_pad(hg[f"{n}/t"]) for n in names]
    m = HammingMatcher(variant=_capi.VARIANT_I8MMA1, t_split=t_split)
    b = PairBatch.from_host(qs, ts)
    full, best = m.knn2(b), m.knn2(b, need_second=False)
    assert torch.equal(full.fwd_best, best.fwd_best) and torch.equal(full.bwd_best, best.bwd_best)
    assert bool((best.fwd_second == -1).all())                       # 0xFFFFFFFF = "none"
    out = m.match_pairs([hg[f"{n}/q"] for n in names], [hg[f"{n}/t"] for n in names], use_ratio=False, use_cross=True, sort_by_distance=False)
    for n, (qi, ti, d) in zip(names, out):
        np.testing.assert_array_equal(qi, hg[f"{n}/cc_q"], err_msg=n)
        np.testing.assert_array_equal(ti, hg[f"{n}/cc_t"], err_msg=n)
        np.testing.assert_array_equal(d, hg[f"{n}/cc_d"], err_msg=n)
    rng = np.random.default_rng(79)
    N, counts = 700, np.array([700, 1, 128, 0, 513, 129, 640], np.int32)
    desc = torch.from_numpy(rng.integers(0, 4, (len(counts) * N, 32), dtype=np.uint8)).cuda()
    sb = sequence_batch(desc, torch.zeros((len(counts) * N, 2), dtype=torch.float32, device="cuda"), counts, 0, len(counts) - 1, N)
    full, best = m.knn2(sb), m.knn2(sb, need_second=False)
    assert torch.equal(full.fwd_best, best.fwd_best) and torch.equal(full.bwd_best, best.bwd_best)
    assert bool((best.fwd_second == -1).all())
