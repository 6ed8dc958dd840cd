"""Batched device API over libb2s: Hamming kNN-2 -> selection -> 8-point hypotheses ->
Sampson scoring -> winner + inlier mask, for many frame pairs per launch.

This is the measured API (bench.py); the reference-shaped single-pair interfaces in
``integration/`` are thin veneers over it.  Tensors are only containers for device
memory; every computation is a libb2s kernel on torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Sequence

import numpy as np

from . import _capi
from ._capi import DESC_BYTES, IDX_BITS, IDX_MASK, NONE_KEY, check, current_stream, ptr


def ratio_lut(ratio: float) -> np.ndarray:
    """keep iff d1 < lut[d2]  ==  float(d1) < ratio * float(d2) in float64
    (feature_pipeline.py.bak:90, homography.py:16)."""
    return np.array([math.ceil(float(ratio) * float(d)) for d in range(257)], dtype=np.int32)


def _prep_desc(d) -> np.ndarray:
    """Validate one descriptor block; narrower rows are zero-padded to 32 bytes (padding
    both sides with zeros leaves every Hamming distance unchanged)."""
    a = np.asarray(d)
    if a.ndim != 2 or a.dtype != np.uint8:
        raise ValueError("descriptors must be a (N, W) uint8 array for the Hamming matcher")
    if a.shape[1] > DESC_BYTES:
        raise ValueError(f"descriptor width {a.shape[1]} > {DESC_BYTES} bytes is not supported")
    if a.shape[1] < DESC_BYTES:
        a = np.concatenate([a, np.zeros((a.shape[0], DESC_BYTES - a.shape[1]), np.uint8)], axis=1)
    return np.ascontiguousarray(a)


@dataclass
class SharedBlocks:
    """Block structure of a batch whose pairs share descriptor blocks (b2s_hamming_knn2_shared):
    block b = `rows[b]` descriptor rows starting at row `row0[b]` of the one descriptor buffer; its
    tensor-core operand tiles start at tile `tile0[b]`; pair p's query / train side is the block
    whose first tile is `q_xtile[p]` / `t_xtile[p]`.  Device int32 tensors + host sizes."""
    row0: "torch.Tensor"
    rows: "torch.Tensor"
    tile0: "torch.Tensor"
    q_xtile: "torch.Tensor"
    t_xtile: "torch.Tensor"
    n_blocks: int
    total_tiles: int
    max_rows: int

    @staticmethod
    def build(row0: np.ndarray, rows: np.ndarray, q_blk: np.ndarray, t_blk: np.ndarray, device) -> "SharedBlocks":
        import torch

        row0 = np.asarray(row0, np.int32)
        rows = np.asarray(rows, np.int32)
        tiles = (rows.astype(np.int64) + 127) // 128
        tile0 = np.zeros(len(rows) + 1, np.int32)
        np.cumsum(tiles, out=tile0[1:])
        nb, npairs = len(rows), len(q_blk)
        pack = torch.from_numpy(np.concatenate([row0, rows, tile0[:-1], tile0[np.asarray(q_blk)], tile0[np.asarray(t_blk)]]).astype(np.int32)).to(device)
        return SharedBlocks(pack[:nb], pack[nb:2 * nb], pack[2 * nb:3 * nb], pack[3 * nb:3 * nb + npairs],
                            pack[3 * nb + npairs:], nb, int(tile0[-1]), int(rows.max()) if nb else 0)


@dataclass
class PairBatch:
    """Device-resident CSR batch of (query, train) descriptor sets."""
    q_desc: "torch.Tensor"
    t_desc: "torch.Tensor"
    q_off: "torch.Tensor"
    t_off: "torch.Tensor"
    q_off_host: np.ndarray
    t_off_host: np.ndarray
    kp_q: "torch.Tensor | None" = None
    kp_t: "torch.Tensor | None" = None
    q_src: "torch.Tensor | None" = None
    t_src: "torch.Tensor | None" = None
    shared: "SharedBlocks | None" = None   # pairs share descriptor blocks (frames): expand each block once

    @property
    def n_pairs(self) -> int:
        return len(self.q_off_host) - 1

    @property
    def total_nq(self) -> int:
        return int(self.q_off_host[-1])

    @property
    def total_nt(self) -> int:
        return int(self.t_off_host[-1])

    @property
    def max_nq(self) -> int:
        return int(np.diff(self.q_off_host).max()) if self.n_pairs else 0

    @property
    def max_nt(self) -> int:
        return int(np.diff(self.t_off_host).max()) if self.n_pairs else 0

    @staticmethod
    def from_host(q_list: Sequence[np.ndarray], t_list: Sequence[np.ndarray],
                  kpq_list: Sequence[np.ndarray] | None = None,
                  kpt_list: Sequence[np.ndarray] | None = None, device=None) -> "PairBatch":
        torch = _capi.require_cuda()
        if len(q_list) != len(t_list):
            raise ValueError("q_list and t_list differ in length")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        q = [_prep_desc(x) for x in q_list]
        t = [_prep_desc(x) for x in t_list]
        q_off = np.zeros(len(q) + 1, np.int32)
        t_off = np.zeros(len(t) + 1, np.int32)
        np.cumsum([len(x) for x in q], out=q_off[1:])
        np.cumsum([len(x) for x in t], out=t_off[1:])
        empty = np.zeros((0, DESC_BYTES), np.uint8)

        def up(arrs, dtype, width):
            cat = np.concatenate(arrs, axis=0) if arrs else np.zeros((0, width), dtype)
            if cat.shape[0] == 0:
                return torch.zeros((1, width), dtype=getattr(torch, np.dtype(dtype).name), device=dev)[:0]
            return torch.from_numpy(np.ascontiguousarray(cat)).pin_memory().to(dev, non_blocking=True)

        kp_q = kp_t = None
        if kpq_list is not None and kpt_list is not None:
            kq = [np.asarray(k, np.float32).reshape(-1, 2) for k in kpq_list]
            kt = [np.asarray(k, np.float32).reshape(-1, 2) for k in kpt_list]
            for a, b in zip(kq, q):
                if len(a) != len(b):
                    raise ValueError("keypoints / descriptors length mismatch (query)")
            for a, b in zip(kt, t):
                if len(a) != len(b):
                    raise ValueError("keypoints / descriptors length mismatch (train)")
            kp_q, kp_t = up(kq, np.float32, 2), up(kt, np.float32, 2)
        return PairBatch(
            q_desc=up(q or [empty], np.uint8, DESC_BYTES), t_desc=up(t or [empty], np.uint8, DESC_BYTES),
            q_off=torch.from_numpy(q_off).to(dev), t_off=torch.from_numpy(t_off).to(dev),
            q_off_host=q_off, t_off_host=t_off, kp_q=kp_q, kp_t=kp_t)


def sequence_batch(desc_dev, kp_dev, counts: np.ndarray, first_pair: int, n_pairs: int, frame_rows: int) -> PairBatch:
    """Consecutive-frame pairs (frame k, frame k+1) over frames that were uploaded ONCE:
    descriptors/keypoints of frame f start at row f*frame_rows of desc_dev / kp_dev; pair p
    matches frame first_pair+p (query) against frame first_pair+p+1 (train) through the
    q_src/t_src row indirection, so no descriptor is copied or stored twice."""
    torch = _capi.require_cuda()
    dev = desc_dev.device
    nq = counts[first_pair:first_pair + n_pairs].astype(np.int32)
    nt = counts[first_pair + 1:first_pair + n_pairs + 1].astype(np.int32)
    q_off = np.zeros(n_pairs + 1, np.int32)
    t_off = np.zeros(n_pairs + 1, np.int32)
    np.cumsum(nq, out=q_off[1:])
    np.cumsum(nt, out=t_off[1:])
    q_src = (np.arange(first_pair, first_pair + n_pairs, dtype=np.int64) * frame_rows).astype(np.int32)
    t_src = q_src + np.int32(frame_rows)
    pack = torch.from_numpy(np.concatenate([q_off, t_off, q_src, t_src])).to(dev)
    n1 = n_pairs + 1
    # frames first_pair .. first_pair + n_pairs are the blocks; pair p = (block p, block p + 1)
    frames = np.arange(first_pair, first_pair + n_pairs + 1, dtype=np.int64)
    shared = SharedBlocks.build((frames * frame_rows).astype(np.int32), counts[first_pair:first_pair + n_pairs + 1],
                                np.arange(n_pairs), np.arange(1, n_pairs + 1), dev)
    return PairBatch(q_desc=desc_dev, t_desc=desc_dev, q_off=pack[:n1], t_off=pack[n1:2 * n1],
                     q_off_host=q_off, t_off_host=t_off, kp_q=kp_dev, kp_t=kp_dev,
                     q_src=pack[2 * n1:2 * n1 + n_pairs], t_src=pack[2 * n1 + n_pairs:], shared=shared)


@dataclass
class Keys:
    fwd_best: "torch.Tensor"
    fwd_second: "torch.Tensor"
    bwd_best: "torch.Tensor"


@dataclass
class Selection:
    """Selected matches.  Pair p's entries live at [c_off[p], c_off[p] + count[p]) of
    out_q / out_t / out_d / corr: CSR over the query rows (stride 0) or the compact layout
    p * stride (stride = max_matches) that keeps device->host copies small."""
    out_q: "torch.Tensor"
    out_t: "torch.Tensor"
    out_d: "torch.Tensor"
    count: "torch.Tensor"
    corr: "torch.Tensor | None"
    c_off: "torch.Tensor"
    stride: int = 0
    total: "torch.Tensor | None" = None    # matches per pair before truncation to max_matches (with_total=True)


class HammingMatcher:
    """K1/K2 + selection.  Mirrors cv2.BFMatcher(NORM_HAMMING) knnMatch/match semantics
    (feature_pipeline.py.bak:68,82,84) on batches."""

    def __init__(self, variant: int = _capi.VARIANT_I8MMA1, t_split: int = 0):
        self.variant = variant
        self.t_split = t_split
        self._lib = _capi.load_library()
        self._ws = None
        self._coff = {}

    def knn2(self, b: PairBatch, need_second: bool = True) -> Keys:
        """need_second=False (cross-check-only matching, the reference's default matcher): the tensor-core kernel
        skips the per-row second neighbour — fwd_second is all "none" — and runs ~15 % faster."""
        torch = _capi.require_cuda()
        dev = b.q_desc.device
        nq, nt = b.total_nq, b.total_nt
        fb = torch.empty(max(nq, 1), dtype=torch.int32, device=dev)
        fs = torch.empty(max(nq, 1), dtype=torch.int32, device=dev)
        bb = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
        ws_ptr, ws_bytes = None, 0
        sh = b.shared
        if sh is not None and self.variant == _capi.VARIANT_I8MMA1 and nq > 0 and nt > 0 and b.q_desc.data_ptr() == b.t_desc.data_ptr():
            # pairs share descriptor blocks (frames): every block is expanded once
            ws_bytes = int(self._lib.b2s_hamming_shared_workspace_bytes(sh.total_tiles, b.n_pairs, nq, b.max_nq, b.max_nt, self.t_split))
            if self._ws is None or self._ws.numel() < ws_bytes or self._ws.device != dev:
                self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            check(self._lib.b2s_hamming_knn2_shared(
                ptr(b.q_desc), ptr(sh.row0), ptr(sh.rows), ptr(sh.tile0), sh.n_blocks, sh.total_tiles, sh.max_rows,
                ptr(sh.q_xtile), ptr(sh.t_xtile), ptr(b.q_off), ptr(b.t_off), b.n_pairs, nq, nt, b.max_nq, b.max_nt,
                ptr(fb), ptr(fs), ptr(bb), self.t_split, int(need_second), self._ws.data_ptr(), ws_bytes, current_stream()))
            return Keys(fb[:nq], fs[:nq], bb[:nt])
        if nq > 0 and (self.variant != _capi.VARIANT_POPC or self.t_split != 1):
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            if self.variant == _capi.VARIANT_POPC:
                want = self.t_split if self.t_split > 1 else max(1, min(64, (4 * sms) // max(1, b.n_pairs)))
            else:
                want = self.t_split          # tensor-core kernels: 0 = the library's own plan
            ws_bytes = int(self._lib.b2s_hamming_workspace_bytes_v(self.variant, b.n_pairs, nq, b.max_nq, b.max_nt, want))
            if ws_bytes:
                if self._ws is None or self._ws.numel() < ws_bytes or self._ws.device != dev:
                    self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                ws_ptr = self._ws.data_ptr()
        check(self._lib.b2s_hamming_knn2_batched(
            ptr(b.q_desc), ptr(b.t_desc), ptr(b.q_off), ptr(b.t_off), ptr(b.q_src), ptr(b.t_src),
            b.n_pairs, nq, nt, b.max_nq, b.max_nt, ptr(fb), ptr(fs), ptr(bb),
            self.variant | (0 if need_second else _capi.HAMMING_BEST_ONLY), self.t_split, ws_ptr, ws_bytes, current_stream()))
        return Keys(fb[:nq], fs[:nq], bb[:nt])

    def select(self, b: PairBatch, k: Keys, *, use_ratio: bool, use_cross: bool, ratio: float = 0.8,
               sort_by_distance: bool = True, max_matches: int | None = None,
               with_corr: bool = False, compact: bool = False, with_total: bool = False) -> Selection:
        torch = _capi.require_cuda()
        dev = b.q_desc.device
        nq = b.total_nq
        stride = int(max_matches) if (compact and max_matches) else 0
        rows = b.n_pairs * stride if stride else nq
        oq = torch.empty(max(rows, 1), dtype=torch.int32, device=dev)
        ot = torch.empty(max(rows, 1), dtype=torch.int32, device=dev)
        od = torch.empty(max(rows, 1), dtype=torch.int32, device=dev)
        cnt = torch.empty(max(b.n_pairs, 1), dtype=torch.int32, device=dev)      # the kernel writes every pair's count
        total = torch.empty(max(b.n_pairs, 1), dtype=torch.int32, device=dev) if with_total else None
        corr = None
        if with_corr:
            if b.kp_q is None or b.kp_t is None:
                raise ValueError("with_corr needs keypoint coordinates in the batch")
            corr = torch.empty((max(rows, 1), 4), dtype=torch.float32, device=dev)
        if stride:
            key = (str(dev), b.n_pairs, stride)
            if key not in self._coff:
                self._coff[key] = (torch.arange(b.n_pairs + 1, dtype=torch.int32, device=dev) * stride).contiguous()
            c_off = self._coff[key]
        else:
            c_off = b.q_off
        lut = ratio_lut(ratio) if use_ratio else None
        check(self._lib.b2s_select_matches(
            ptr(k.fwd_best), ptr(k.fwd_second), ptr(k.bwd_best), ptr(b.q_off), ptr(b.t_off),
            b.n_pairs, b.max_nq, int(use_ratio), int(use_cross), ptr(lut), int(sort_by_distance),
            int(max_matches or 0), ptr(b.kp_q) if with_corr else None, ptr(b.kp_t) if with_corr else None,
            ptr(b.q_src) if with_corr else None, ptr(b.t_src) if with_corr else None, stride,
            ptr(oq), ptr(ot), ptr(od), ptr(corr), ptr(cnt), ptr(total), current_stream()))
        return Selection(oq[:rows], ot[:rows], od[:rows], cnt[:b.n_pairs], None if corr is None else corr[:rows],
                         c_off, stride, None if total is None else total[:b.n_pairs])

    # ---- host convenience: numpy in, numpy out (includes H2D / D2H) -------------------
    def match_pairs(self, q_list, t_list, *, use_ratio: bool, use_cross: bool, ratio: float = 0.8,
                    sort_by_distance: bool = True, max_matches: int | None = None):
        """-> list of (queryIdx, trainIdx, distance) int32 arrays, one per pair."""
        torch = _capi.require_cuda()
        b = PairBatch.from_host(q_list, t_list)
        if b.n_pairs == 0:
            return []
        if b.max_nq > _capi.SELECT_MAX_QUERIES:
            raise ValueError(f"more than {_capi.SELECT_MAX_QUERIES} query descriptors in one pair")
        keys = self.knn2(b, need_second=bool(use_ratio))
        sel = self.select(b, keys, use_ratio=use_ratio, use_cross=use_cross, ratio=ratio,
                          sort_by_distance=sort_by_distance, max_matches=max_matches)
        packed = torch.stack([sel.out_q, sel.out_t, sel.out_d]).cpu().numpy()
        cnt = sel.count.cpu().numpy()
        out = []
        for p in range(b.n_pairs):
            o, c = int(b.q_off_host[p]), int(cnt[p])
            if c < 0:
                raise _capi.B2SError("select kernel: pair larger than the declared maximum")
            out.append((packed[0, o:o + c].copy(), packed[1, o:o + c].copy(), packed[2, o:o + c].copy()))
        return out

    def knn2_pairs(self, q_list, t_list):
        """-> list of (fwd_best, fwd_second, bwd_best) uint32 packed-key arrays per pair."""
        b = PairBatch.from_host(q_list, t_list)
        if b.n_pairs == 0:
            return []
        k = self.knn2(b)
        fb = k.fwd_best.cpu().numpy().view(np.uint32)
        fs = k.fwd_second.cpu().numpy().view(np.uint32)
        bb = k.bwd_best.cpu().numpy().view(np.uint32)
        return [(fb[b.q_off_host[p]:b.q_off_host[p + 1]], fs[b.q_off_host[p]:b.q_off_host[p + 1]],
                 bb[b.t_off_host[p]:b.t_off_host[p + 1]]) for p in range(b.n_pairs)]


class EssentialRansac:
    """K4 + K3 + winner selection (homography.py:302-345 batched)."""

    def __init__(self):
        self._lib = _capi.load_library()

    @staticmethod
    def _k_args(K):
        if K is None:
            return None, None, None
        Kd = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(3, 3))
        Kinv = np.ascontiguousarray(np.linalg.inv(Kd))          # homography.py:228
        return Kd, Kinv, (Kd, Kinv)

    def hypotheses(self, corr, c_off, c_count, n_pairs: int, H: int, *, samples=None, seed: int = 0,
                   K=None, return_samples: bool = False, pair_ids=None, pair_id0: int = 0):
        """pair_ids (device int32 [n_pairs]) / pair_id0: the pairs' GLOBAL ids; the device sample stream is keyed
        by (seed, id, h), so sharded and single-GPU runs draw the same samples for the same pair."""
        torch = _capi.require_cuda()
        E = torch.empty((max(n_pairs, 1), max(H, 1), 9), dtype=torch.float64, device=corr.device)
        s_out = torch.empty((max(n_pairs, 1), max(H, 1), 8), dtype=torch.int32, device=corr.device) if return_samples else None
        Kd, Kinv, _keep = self._k_args(K)
        check(self._lib.b2s_eight_point_batched(
            ptr(corr), ptr(c_off), ptr(c_count), n_pairs, H, ptr(samples), C.c_uint64(seed & (2**64 - 1)),
            ptr(pair_ids), int(pair_id0), ptr(s_out), ptr(Kd), ptr(Kinv), ptr(E), current_stream()))
        E = E[:n_pairs, :H]
        return (E, s_out[:n_pairs, :H]) if return_samples else E

    def hypotheses_5pt(self, corr, c_off, c_count, n_pairs: int, S: int, *, samples=None, seed: int = 0, return_counts: bool = False):
        """K8: 5-point minimal solver on CALIBRATED correspondences: S samples per pair, up to 10
        real solutions each -> E [n_pairs, 10 S, 9] (unused slots zero), ready for score()."""
        torch = _capi.require_cuda()
        E = torch.empty((max(n_pairs, 1), max(S, 1), 10, 9), dtype=torch.float64, device=corr.device)
        ns = torch.empty((max(n_pairs, 1), max(S, 1)), dtype=torch.int32, device=corr.device)
        check(self._lib.b2s_five_point_batched(ptr(corr), ptr(c_off), ptr(c_count), n_pairs, S, ptr(samples),
                                               C.c_uint64(seed & (2**64 - 1)), None, ptr(E), ptr(ns), current_stream()))
        E = E[:n_pairs, :S].reshape(n_pairs, S * 10, 9)
        return (E, ns[:n_pairs, :S]) if return_counts else E

    def score_tc(self, corr, c_off, c_count, n_pairs: int, E, th2: float, max_m: int, th2_per_pair=None, debug: bool = False):
        """K3t: the counts of score(precision=64) from the tensor cores (csrc/ransac_tc.cu).
        max_m >= every count.  debug=True also returns (num, den, band): the raw float32
        accumulators [pair, H, max_m] and the number of float64 re-evaluations."""
        torch = _capi.require_cuda()
        H = E.shape[1]
        dev = corr.device
        counts = torch.empty((max(n_pairs, 1), max(H, 1)), dtype=torch.int32, device=dev)
        need = int(self._lib.b2s_ransac_score_tc_workspace_bytes(n_pairs, H, int(max_m)))
        if getattr(self, "_tc_ws", None) is None or self._tc_ws.numel() < need or self._tc_ws.device != dev:
            self._tc_ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
        num = den = band = None
        if debug:
            num = torch.zeros((n_pairs, H, int(max_m)), dtype=torch.float32, device=dev)
            den = torch.zeros_like(num)
            band = torch.zeros(2, dtype=torch.int32, device=dev)
        check(self._lib.b2s_ransac_score_tc(
            ptr(corr), ptr(c_off), ptr(c_count), n_pairs, int(max_m), ptr(E), H, float(th2), ptr(th2_per_pair),
            ptr(counts), self._tc_ws.data_ptr(), need, ptr(num), ptr(den), int(max_m), ptr(band), current_stream()))
        counts = counts[:n_pairs, :H]
        return (counts, num, den, band) if debug else counts

    def score(self, corr, c_off, c_count, n_pairs: int, E, th2: float, th2_per_pair=None, precision: int = 64, max_m: int = 0):
        """max_m: host-known bound on the correspondences of a pair (0 = unknown); lets a batch of few
        pairs with thousands of correspondences each (BASELINE config #4) be cut along the correspondences too."""
        torch = _capi.require_cuda()
        H = E.shape[1]
        counts = torch.empty((max(n_pairs, 1), max(H, 1)), dtype=torch.int32, device=corr.device)
        check(self._lib.b2s_ransac_score_batched(
            ptr(corr), ptr(c_off), ptr(c_count), n_pairs, ptr(E), H, float(th2), ptr(th2_per_pair),
            precision, int(max_m), ptr(counts), current_stream()))
        return counts[:n_pairs, :H]

    @staticmethod
    def _sink(sink):
        """sink = (records tensor [n_pairs, record_bytes], Selection, pair_id0) or None -> (ctypes struct or None, mask_stride)."""
        if sink is None:
            return None, 0
        rec, sel, pid0 = sink
        st = _capi.RecordSink(rec.data_ptr(), int(rec.shape[-1]), sel.out_q.data_ptr(), sel.out_t.data_ptr(), sel.out_d.data_ptr(),
                              int(sel.stride), int(pid0))
        return st, int(sel.stride)

    def winner(self, corr, c_off, c_count, n_pairs: int, E, th2: float, th2_per_pair=None, return_counts: bool = False, sink=None):
        """Winner-only scoring (b2s_ransac_winner_batched): best_h / best_count / inlier mask identical to
        score(precision=64) + select, but hypotheses that can neither exceed 0.8 M nor reach the largest complete count
        are abandoned after the first ~3/8 of the correspondences.  return_counts: also (counts [pair, H] — complete
        for finished hypotheses, lower bounds for abandoned ones — and the number finished per pair)."""
        torch = _capi.require_cuda()
        H, dev = E.shape[1], corr.device
        best_h = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=dev)
        best_c = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=dev)
        st, mstride = self._sink(sink)
        mask = (torch.empty if mstride else torch.zeros)(max(corr.shape[0], 1), dtype=torch.uint8, device=dev)
        need = int(self._lib.b2s_ransac_winner_workspace_bytes(n_pairs, H))
        if getattr(self, "_win_ws", None) is None or self._win_ws.numel() < need or self._win_ws.device != dev:
            self._win_ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
        counts = torch.empty((max(n_pairs, 1), max(H, 1)), dtype=torch.int32, device=dev) if return_counts else None
        nfin = torch.zeros(max(n_pairs, 1), dtype=torch.int32, device=dev) if return_counts else None
        check(self._lib.b2s_ransac_winner_batched(
            ptr(corr), ptr(c_off), ptr(c_count), n_pairs, ptr(E), H, float(th2), ptr(th2_per_pair), ptr(best_h), ptr(best_c),
            ptr(mask), self._win_ws.data_ptr(), need, ptr(counts), ptr(nfin), C.byref(st) if st is not None else None, mstride,
            current_stream()))
        out = (best_h[:n_pairs], best_c[:n_pairs], mask[:corr.shape[0]])
        return out + (counts[:n_pairs, :H], nfin[:n_pairs]) if return_counts else out

    def select(self, counts, corr, c_off, c_count, n_pairs: int, E, th2: float, th2_per_pair=None, sink=None):
        """sink = (records, Selection, pair_id0): the winner kernel also writes every pair's result record and clears
        the unused tail of the inlier mask (no zero-fill, no separate record kernel)."""
        torch = _capi.require_cuda()
        H = E.shape[1]
        best_h = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=corr.device)
        best_c = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=corr.device)
        st, mstride = self._sink(sink)
        mask = (torch.empty if mstride else torch.zeros)(max(corr.shape[0], 1), dtype=torch.uint8, device=corr.device)
        check(self._lib.b2s_ransac_select(
            ptr(counts), ptr(corr), ptr(c_off), ptr(c_count), n_pairs, ptr(E), H, float(th2),
            ptr(th2_per_pair), ptr(best_h), ptr(best_c), ptr(mask), C.byref(st) if st is not None else None, mstride,
            current_stream()))
        return best_h[:n_pairs], best_c[:n_pairs], mask[:corr.shape[0]]


# ---- result records (csrc/records.cu): ONE fixed-size record per pair is what leaves the GPU ------------
RECORD_HEADER_BYTES = 64


def record_bytes(max_matches: int) -> int:
    return int(_capi.load_library().b2s_record_bytes(int(max_matches)))


def pose_record_bytes(max_matches: int) -> int:
    """Bytes of a pose record (include/b2s.h): a result record of record_bytes(max_matches) bytes, then the pair's
    b2s_pose_result (200 bytes) and 56 zero bytes.  What a step with FrontendConfig.robust_pose writes per pair."""
    return int(_capi.load_library().b2s_pose_record_bytes(int(max_matches)))


def step_record_bytes(cfg) -> int:
    """Record bytes per pair of a step run with `cfg` (FrontendConfig): pose records when cfg.robust_pose is set."""
    return pose_record_bytes(cfg.max_matches) if cfg.robust_pose is not None else record_bytes(cfg.max_matches)


def pack_records(records, sel: Selection, best_h=None, best_count=None, mask=None, R=None, t=None, *, n_records: int,
                 pair_id0: int = 0, pair_ids=None, src_pair=None, count_total=None):
    """Write one record per pair into `records` (device uint8 [n_records, record_bytes(sel.stride)], e.g. this
    rank's slice of the all-gather buffer) on the current stream: header (n_matches, best_h, inliers, pair id,
    R | t as float32) + stride x (queryIdx u16, trainIdx u16, distance u16, inlier u8)."""
    if not sel.stride:
        raise ValueError("records need the compact selection layout (max_matches / stride)")
    check(_capi.load_library().b2s_pack_records(
        ptr(sel.count), ptr(count_total), ptr(best_h), ptr(best_count), ptr(sel.out_q), ptr(sel.out_t), ptr(sel.out_d),
        ptr(mask), ptr(R), ptr(t), ptr(pair_ids), ptr(src_pair), int(n_records), int(sel.stride), int(pair_id0),
        records.data_ptr(), int(records.shape[-1]) if records.ndim > 1 else record_bytes(sel.stride), current_stream()))
    return records


def unpack_records(buf, stride: int, pose: bool = False):
    """Host view of a record buffer (NumPy uint8 [n, record_bytes]) -> dict of arrays: n_matches, best_h,
    inliers, pair_id (int32 [n]); R float32 [n, 3, 3]; t float32 [n, 3]; q, t_idx, d (uint16 [n, stride]);
    inlier (uint8 [n, stride]).  Entries past n_matches are zero.  pose=True: pose records (pose_record_bytes), and
    "robust" holds every pair's b2s_pose_result (robust_pose.POSE_RESULT_DTYPE [n]); best_h / inliers / R / t / inlier
    are then those of the selected model."""
    a = np.ascontiguousarray(np.asarray(buf, dtype=np.uint8))
    if a.ndim == 1:
        a = a.reshape(-1, pose_record_bytes(stride) if pose else record_bytes(stride))
    n = a.shape[0]
    hdr = a[:, :64].copy().view(np.int32).reshape(n, 16)
    body = a[:, 64:64 + 6 * stride].copy().view(np.uint16).reshape(n, 3, stride)
    out = {"n_matches": hdr[:, 0], "best_h": hdr[:, 1], "inliers": hdr[:, 2], "pair_id": hdr[:, 3],
           "R": hdr[:, 4:13].copy().view(np.float32).reshape(n, 3, 3), "t": hdr[:, 13:16].copy().view(np.float32).reshape(n, 3),
           "q": body[:, 0], "t_idx": body[:, 1], "d": body[:, 2], "inlier": a[:, 64 + 6 * stride:64 + 7 * stride]}
    if pose:
        from .robust_pose import POSE_RESULT_BYTES, decode_results

        rb = record_bytes(stride)
        if a.shape[1] < pose_record_bytes(stride):
            raise ValueError(f"pose records of stride {stride} are {pose_record_bytes(stride)} bytes, got {a.shape[1]}")
        out["robust"] = decode_results(a[:, rb:rb + POSE_RESULT_BYTES].copy())
    return out


def rank_pairs(score, k: int, *, ids=None, sel_count=None, stride: int = 0, with_ids: bool = False):
    """The k (<= 32) pairs with the largest score, ties to the lower id then position, on the device
    (persistent_map.py:236-242).  -> (top_idx [k], c_off [k], c_count [k]) int32 device tensors."""
    torch = _capi.require_cuda()
    dev = score.device
    out = torch.empty((4, max(k, 1)), dtype=torch.int32, device=dev)
    check(_capi.load_library().b2s_rank_pairs(ptr(score), ptr(ids), ptr(sel_count), int(score.numel()), int(k), int(stride),
                                             ptr(out[0]), ptr(out[3]), ptr(out[1]), ptr(out[2]), current_stream()))
    if with_ids:
        return out[0, :k], out[1, :k], out[2, :k], out[3, :k]
    return out[0, :k], out[1, :k], out[2, :k]


class PoseRecovery:
    """K7: decompose_essential (homography.py:251-299) for many pairs in two launches — the
    four (R, t) candidates per E and the DLT cheirality vote over the pair's inliers."""

    def __init__(self):
        self._lib = _capi.load_library()

    def refit(self, corr, c_off, c_count, n_pairs: int, mask=None, K=None):
        """n-point E on each pair's inliers (homography.py:344) -> (E [n_pairs, 9] float64 device, n_used device)."""
        torch = _capi.require_cuda()
        E = torch.empty((max(n_pairs, 1), 9), dtype=torch.float64, device=corr.device)
        used = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=corr.device)
        Kd = Kinv = None
        if K is not None:
            Kd = np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(3, 3))
            Kinv = np.ascontiguousarray(np.linalg.inv(Kd))
        check(self._lib.b2s_refit_essential_batched(ptr(corr), ptr(c_off), ptr(c_count), ptr(mask), n_pairs, ptr(Kd), ptr(Kinv),
                                                    ptr(E), ptr(used), current_stream()))
        return E[:n_pairs], used[:n_pairs]

    def recover(self, corr, c_off, c_count, n_pairs: int, max_m: int, mask=None, K=None):
        """refit + decompose + pick, all on the current stream, nothing copied to the host:
        -> (E [n,9], R [n,9], t [n,3], votes [n,4]) device tensors."""
        torch = _capi.require_cuda()
        dev = corr.device
        E, _ = self.refit(corr, c_off, c_count, n_pairs, mask=mask, K=K)
        cand = torch.empty((max(n_pairs, 1), 4, 12), dtype=torch.float64, device=dev)
        votes = torch.empty((max(n_pairs, 1), 4), dtype=torch.int32, device=dev)
        R = torch.empty((max(n_pairs, 1), 9), dtype=torch.float64, device=dev)
        t = torch.empty((max(n_pairs, 1), 3), dtype=torch.float64, device=dev)
        Kd = None if K is None else np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(3, 3))
        check(self._lib.b2s_decompose_essential_batched(ptr(E), ptr(corr), ptr(c_off), ptr(c_count), ptr(mask), n_pairs, int(max_m),
                                                        ptr(Kd), ptr(cand), ptr(votes), current_stream()))
        check(self._lib.b2s_pose_pick(ptr(cand), ptr(votes), n_pairs, ptr(R), ptr(t), current_stream()))
        return E, R[:n_pairs], t[:n_pairs], votes[:n_pairs]

    def decompose(self, E, corr, c_off, c_count, n_pairs: int, max_m: int, mask=None, K=None):
        """E: [n_pairs, 9] float64 device; -> (R [n_pairs,3,3], t [n_pairs,3], votes [n_pairs,4]) as
        NumPy arrays; first maximum of the votes wins (homography.py:296-298)."""
        torch = _capi.require_cuda()
        dev = corr.device
        cand = torch.empty((max(n_pairs, 1), 4, 12), dtype=torch.float64, device=dev)
        votes = torch.empty((max(n_pairs, 1), 4), dtype=torch.int32, device=dev)
        Kd = None if K is None else np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(3, 3))
        check(self._lib.b2s_decompose_essential_batched(ptr(E), ptr(corr), ptr(c_off), ptr(c_count), ptr(mask), n_pairs, int(max_m),
                                                        ptr(Kd), ptr(cand), ptr(votes), current_stream()))
        c, v = cand[:n_pairs].cpu().numpy(), votes[:n_pairs].cpu().numpy()
        win = np.argmax(v, axis=1)
        sel = c[np.arange(n_pairs), win]
        return sel[:, :9].reshape(-1, 3, 3), sel[:, 9:], v


class HomographyRansac:
    """K5 + K6 + winner selection (homography.py:148-216 batched): 4-point normalised DLT
    hypotheses, symmetric transfer error, the reference's sequential selection rule."""

    def __init__(self):
        self._lib = _capi.load_library()

    def hypotheses(self, corr, c_off, c_count, n_pairs: int, H: int, *, samples=None, seed: int = 0, return_samples: bool = False,
                   pair_ids=None, pair_id0: int = 0):
        """pair_ids (device int32 [n_pairs]) / pair_id0: the pairs' GLOBAL ids, as in EssentialRansac.hypotheses: the
        device 4-sample stream is keyed by (seed, id, h), so a pair draws the same samples in any batch position."""
        torch = _capi.require_cuda()
        Hm = torch.empty((max(n_pairs, 1), max(H, 1), 9), dtype=torch.float64, device=corr.device)
        s_out = torch.empty((max(n_pairs, 1), max(H, 1), 4), dtype=torch.int32, device=corr.device) if return_samples else None
        check(self._lib.b2s_homography_dlt_batched(ptr(corr), ptr(c_off), ptr(c_count), n_pairs, H, ptr(samples),
                                                   C.c_uint64(seed & (2**64 - 1)), ptr(pair_ids), int(pair_id0), ptr(s_out),
                                                   ptr(Hm), current_stream()))
        Hm = Hm[:n_pairs, :H]
        return (Hm, s_out[:n_pairs, :H]) if return_samples else Hm

    def score(self, corr, c_off, c_count, n_pairs: int, Hm, th: float, th_per_pair=None):
        torch = _capi.require_cuda()
        H = Hm.shape[1]
        counts = torch.empty((max(n_pairs, 1), max(H, 1)), dtype=torch.int32, device=corr.device)
        check(self._lib.b2s_homography_score_batched(ptr(corr), ptr(c_off), ptr(c_count), n_pairs, ptr(Hm), H, float(th),
                                                     ptr(th_per_pair), ptr(counts), current_stream()))
        return counts[:n_pairs, :H]

    def select(self, counts, corr, c_off, c_count, n_pairs: int, Hm, th: float, th_per_pair=None):
        torch = _capi.require_cuda()
        H = Hm.shape[1]
        best_h = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=corr.device)
        best_c = torch.empty(max(n_pairs, 1), dtype=torch.int32, device=corr.device)
        mask = torch.zeros(max(corr.shape[0], 1), dtype=torch.uint8, device=corr.device)
        check(self._lib.b2s_homography_select(ptr(counts), ptr(corr), ptr(c_off), ptr(c_count), n_pairs, ptr(Hm), H, float(th),
                                              ptr(th_per_pair), ptr(best_h), ptr(best_c), ptr(mask), current_stream()))
        return best_h[:n_pairs], best_c[:n_pairs], mask[:corr.shape[0]]


class BowIndex:
    """K9 — bag-of-words candidate ranking on the device (csrc/bow.cu): the step in front of the
    relocalizer's matching.  ``histograms`` = compute_bow_histogram (persistent_map.py:82-96) /
    BoWDatabase._compute_hist (loop_closure.py:36-48) for a whole batch of frames in one launch;
    ``scores`` = cosine_similarity([hist], hists)[0] (persistent_map.py:235, loop_closure.py:63)."""

    def __init__(self, vocab: np.ndarray):
        torch = _capi.require_cuda()
        self.lib = _capi.load_library()
        v = np.ascontiguousarray(vocab, dtype=np.float32)
        if v.ndim != 2 or v.shape[0] == 0:
            raise ValueError("BoW vocabulary must be a non-empty 2D array")
        if v.shape[1] != DESC_BYTES:
            raise ValueError(f"the device BoW path takes {DESC_BYTES}-dimensional (ORB) vocabularies")
        self.k = int(v.shape[0])
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.vocab = torch.from_numpy(v).to(self.dev)
        self.map_hists = None

    def histograms(self, desc, f_off, n_frames: int, max_n: int, return_words: bool = False):
        """desc: device uint8 [total, 32]; f_off: device int32 [n_frames + 1] -> hist float32 [n_frames, k]."""
        import torch

        hist = torch.empty((n_frames, self.k), dtype=torch.float32, device=self.dev)
        counts = torch.empty((n_frames, self.k), dtype=torch.int32, device=self.dev)
        words = torch.empty((int(desc.shape[0]),), dtype=torch.int32, device=self.dev) if return_words else None
        check(self.lib.b2s_bow_histogram_batched(ptr(desc), ptr(f_off), n_frames, max_n, ptr(self.vocab), self.k,
                                                 ptr(words), ptr(counts), ptr(hist), current_stream()))
        return (hist, words) if return_words else hist

    def histograms_host(self, desc_list: Sequence[np.ndarray], return_words: bool = False):
        """Host lists of (N_i, 32) uint8 blocks -> NumPy [n, k] float32 (one upload, one launch)."""
        import torch

        blocks = [np.ascontiguousarray(d, dtype=np.uint8).reshape(-1, DESC_BYTES) if d is not None and len(d) else
                  np.zeros((0, DESC_BYTES), np.uint8) for d in desc_list]
        n = len(blocks)
        if n == 0:
            return np.zeros((0, self.k), np.float32)
        off = np.zeros(n + 1, np.int32)
        off[1:] = np.cumsum([len(b) for b in blocks])
        allb = np.concatenate(blocks) if off[-1] else np.zeros((1, DESC_BYTES), np.uint8)
        desc = torch.from_numpy(allb).to(self.dev)
        out = self.histograms(desc, torch.from_numpy(off).to(self.dev), n, int(max(len(b) for b in blocks)), return_words)
        if return_words:
            return out[0].cpu().numpy(), out[1].cpu().numpy()[: off[-1]]
        return out.cpu().numpy()

    def upload_map(self, hists):
        """Map histograms [n, k] -> a device float32 tensor the CALLER keeps (one vocabulary object may
        serve several maps: old and new snapshot, two relocalizers)."""
        import torch

        h = hists if hasattr(hists, "data_ptr") else torch.from_numpy(np.ascontiguousarray(hists, dtype=np.float32))
        if h.ndim != 2 or h.shape[1] != self.k:
            raise ValueError("map histograms must be [n, k]")
        return h.to(self.dev, dtype=torch.float32).contiguous()

    def set_map(self, hists):
        """Convenience for a single-map owner of this object: keep the histograms here."""
        self.map_hists = self.upload_map(hists)

    def scores(self, hist_q, map_hists=None):
        """hist_q: device float32 [k] (or host array) -> device float32 [n] cosine scores against
        `map_hists` (device tensor from upload_map; default: the one given to set_map)."""
        import torch

        hists = self.map_hists if map_hists is None else map_hists
        if hists is None:
            raise ValueError("set_map() first, or pass map_hists")
        q = hist_q if hasattr(hist_q, "data_ptr") else torch.from_numpy(np.ascontiguousarray(hist_q, dtype=np.float32))
        q = q.to(self.dev, dtype=torch.float32).contiguous().reshape(-1)
        if q.numel() != self.k:
            raise ValueError("query histogram must have k entries")
        n = int(hists.shape[0])
        out = torch.empty((n,), dtype=torch.float32, device=self.dev)
        check(self.lib.b2s_bow_cosine(ptr(q), ptr(hists), n, self.k, ptr(out), current_stream()))
        return out


@dataclass
class FrontendConfig:
    """One pass of the hot path.  Defaults = configs/pipeline/kitti_default.json + the
    north-star's combined matcher (kNN-2 + Lowe ratio + cross-check)."""
    use_ratio: bool = True
    use_cross: bool = True
    ratio: float = 0.8
    max_matches: int | None = 500
    hypotheses: int = 2000
    threshold: float = 0.01
    precision: int = 64
    seed: int = 1337
    with_pose: bool = False    # also refit E on the winner's inliers and recover (R, t) on the device (K7)
    scoring: str = "cuda"      # "cuda": K3h on the CUDA cores (default, 0.30 ms per 296-pair step); "tc": K3t tensor-core
                               # scoring (0.35 ms).  Same counts.
    winner_only: bool = False  # True: same winner / inlier mask, but hypotheses that cannot win are abandoned early
                               # (EssentialRansac.winner); FrontendResult.counts is then None
    robust_pose: "RobustPoseConfig | None" = None   # set: RobustPoseEstimator.estimate_pose for every pair (robust_pose.py):
                               # the essential RANSAC runs at the adaptive per-pair threshold, the homography branch,
                               # model selection and gates follow; FrontendResult.robust / robust_mask hold the answer


@dataclass
class FrontendResult:
    keys: Keys
    sel: Selection
    E: "torch.Tensor"
    counts: "torch.Tensor"
    best_h: "torch.Tensor"
    best_count: "torch.Tensor"
    inlier_mask: "torch.Tensor"
    E_refit: "torch.Tensor | None" = None
    R: "torch.Tensor | None" = None
    t: "torch.Tensor | None" = None
    votes: "torch.Tensor | None" = None
    records: "torch.Tensor | None" = None
    robust: "torch.Tensor | None" = None        # uint8 [n_pairs, 200] b2s_pose_result (robust_pose.decode_results)
    robust_mask: "torch.Tensor | None" = None   # the selected model's inlier flags, layout of inlier_mask


class Frontend:
    """match -> select -> hypotheses -> score -> winner, all on the current stream."""

    def __init__(self, cfg: FrontendConfig | None = None, variant: int = _capi.VARIANT_I8MMA1, t_split: int = 0):
        self.cfg = cfg or FrontendConfig()
        self.matcher = HammingMatcher(variant=variant, t_split=t_split)
        self.ransac = EssentialRansac()
        self.pose = None
        self.robust = None
        self.launches_per_run = 0

    def score(self, sel: Selection, b: PairBatch, E):
        c = self.cfg
        th2 = c.threshold ** 2
        if c.scoring == "tc" and c.precision == 64:
            return self.ransac.score_tc(sel.corr, sel.c_off, sel.count, b.n_pairs, E, th2, max_m=sel.stride or b.max_nq)
        return self.ransac.score(sel.corr, sel.c_off, sel.count, b.n_pairs, E, th2, precision=c.precision,
                                 max_m=sel.stride or b.max_nq)

    def run(self, b: PairBatch, K=None, samples=None, records=None, pair_id0: int = 0,
            after_select=None, before_records=None) -> FrontendResult:
        """records: optional device uint8 [n_pairs, record_bytes(max_matches)] — e.g. this rank's slice of the
        all-gather buffer, or the staging buffer of the step's one device->host copy; the last kernel of the
        step writes every pair's result record into it (pair ids pair_id0 + p).  With cfg.robust_pose the records are
        pose records (pose_record_bytes(max_matches) wide, written by the decision kernel), and pair_id0 also keys both
        RANSAC samplers, so that a pair's answer does not depend on its batch position.
        after_select / before_records: optional callables run (on the current stream) after the selection kernel and
        before the record kernel — where ShardedFrontend starts and joins the collective of the PREVIOUS batch, so
        that it overlaps the multi-wave RANSAC kernels and never the persistent one-CTA-per-SM Hamming kernel."""
        c = self.cfg
        if c.robust_pose is not None:
            if c.winner_only or c.scoring == "tc":
                raise ValueError("robust_pose scores with the CUDA-core kernel (scoring='cuda', winner_only=False)")
            if records is not None:
                if not c.max_matches:
                    raise ValueError("records need the compact selection layout (max_matches)")
                need = pose_record_bytes(c.max_matches)
                if records.ndim != 2 or records.shape[0] < b.n_pairs or records.shape[-1] < need:
                    raise _capi.B2SError(f"robust_pose writes pose records: need [{b.n_pairs}, >= {need}] bytes "
                                         f"(pose_record_bytes({c.max_matches})), got {tuple(records.shape)}")
        keys = self.matcher.knn2(b, need_second=bool(c.use_ratio))
        sel = self.matcher.select(b, keys, use_ratio=c.use_ratio, use_cross=c.use_cross, ratio=c.ratio,
                                  sort_by_distance=True, max_matches=c.max_matches, with_corr=True,
                                  compact=True)
        if after_select is not None:
            after_select()
        if c.robust_pose is not None:
            if self.robust is None:
                from .robust_pose import RobustPose

                self.robust = RobustPose()
            out = self.robust.run(sel.corr, sel.c_off, sel.count, b.n_pairs, K, c.robust_pose, samples_e=samples, seed=c.seed,
                                  max_m=sel.stride or b.max_nq, hypotheses=c.hypotheses, precision=c.precision,
                                  mask_stride=sel.stride, pair_id0=pair_id0, records=records, sink_sel=sel,
                                  before_records=before_records)
            return FrontendResult(keys, sel, out.E, out.counts, out.best_h, out.best_count, out.inlier_mask,
                                  E_refit=out.E_refit, R=out.R, t=out.t, votes=out.votes, records=records, robust=out.results,
                                  robust_mask=out.mask)
        E = self.ransac.hypotheses(sel.corr, sel.c_off, sel.count, b.n_pairs, c.hypotheses,
                                   samples=samples, seed=c.seed, K=K, pair_id0=pair_id0)
        th2 = c.threshold ** 2
        # without pose recovery the winner kernel itself writes the records (with it, R | t arrive later: pack kernel below)
        fused = records is not None and not c.with_pose and sel.stride and before_records is None
        sink = (records, sel, pair_id0) if fused else None
        if c.winner_only:
            counts = None
            best_h, best_c, mask = self.ransac.winner(sel.corr, sel.c_off, sel.count, b.n_pairs, E, th2, sink=sink)
        else:
            counts = self.score(sel, b, E)
            best_h, best_c, mask = self.ransac.select(counts, sel.corr, sel.c_off, sel.count, b.n_pairs, E, th2, sink=sink)
        res = FrontendResult(keys, sel, E, counts, best_h, best_c, mask)
        if c.with_pose:      # next-row #2: refit on the winner's inliers + decomposition / cheirality vote (K7)
            if self.pose is None:
                self.pose = PoseRecovery()
            res.E_refit, res.R, res.t, res.votes = self.pose.recover(sel.corr, sel.c_off, sel.count, b.n_pairs,
                                                                      sel.stride or b.max_nq, mask=mask, K=K)
        if before_records is not None:
            before_records()
        if records is not None:
            if not fused:
                pack_records(records, sel, best_h, best_c, mask, res.R, res.t, n_records=b.n_pairs, pair_id0=pair_id0)
            res.records = records
        return res


class RecordView(dict):
    """The result of a step as the arrays the reference hands back, unpacked lazily from the ONE pinned record
    buffer the step downloaded: count, best_h, best_count (per pair), out_q / out_t / out_d / mask (compact,
    stride = max_matches), R [P, 3, 3], t [P, 3] (float32; zero unless the step ran with_pose).  pose=True (a step with
    FrontendConfig.robust_pose): also "robust", every pair's b2s_pose_result (robust_pose.POSE_RESULT_DTYPE [P]);
    best_h / best_count / mask / R / t are then those of the selected model."""

    def __init__(self, host_records, stride: int, pose: bool = False):
        super().__init__()
        self.records, self.stride, self.pose = host_records, stride, bool(pose)

    def _fill(self):
        import torch

        u = unpack_records(self.records.numpy(), self.stride, pose=self.pose)
        if (u["n_matches"] < 0).any():     # the selection kernel's overflow flag (a pair larger than the declared maximum / stride)
            raise _capi.B2SError("select kernel: a pair did not fit the declared maximum rows / record stride (count = -1)")
        flat = lambda a: torch.from_numpy(np.ascontiguousarray(a).reshape(-1))
        dict.update(self, {"count": torch.from_numpy(u["n_matches"].copy()), "best_h": torch.from_numpy(u["best_h"].copy()),
                           "best_count": torch.from_numpy(u["inliers"].copy()), "pair_id": torch.from_numpy(u["pair_id"].copy()),
                           "out_q": flat(u["q"].astype(np.int32)), "out_t": flat(u["t_idx"].astype(np.int32)),
                           "out_d": flat(u["d"].astype(np.int32)), "mask": flat(u["inlier"].copy()),
                           "R": torch.from_numpy(u["R"].copy()), "t": torch.from_numpy(u["t"].copy())})
        if self.pose:
            dict.__setitem__(self, "robust", u["robust"])

    def __missing__(self, key):
        if not getattr(self, "_filled", False):
            self._fill()                    # raises (and raises again on the next lookup) for an overflowed pair
            self._filled = True
            if dict.__contains__(self, key):
                return dict.__getitem__(self, key)
        raise KeyError(key)


class SequenceTracker:
    """End-to-end tracking of ONE frame sequence from HOST buffers, in `chunks` pieces so that the upload of
    chunk c+1 and the download of chunk c-1 overlap the kernels of chunk c (three streams).

    Frames (descriptors uint8 [F, N, 32], keypoints float32 [F, N, 2], pinned) are uploaded once each; every
    chunk ends with the record kernel and ONE device->host copy of its records (it was seven copies per chunk).
    ``run`` returns a RecordView over the pinned record buffer.  For several steps in flight use SequencePipeline.
    K: 3x3 intrinsics of the keypoints (None = identity), passed to every Frontend.run — robust pose at pixel scale
    needs them (adaptive threshold units, cheirality, decompose_homography).
    """

    def __init__(self, n_frames: int, frame_rows: int, cfg: FrontendConfig, variant: int = _capi.VARIANT_I8MMA1,
                 chunks: int = 4, device=None, use_graph: bool = False, K=None):
        torch = _capi.require_cuda()
        if not cfg.max_matches:
            raise ValueError("SequenceTracker needs max_matches (compact output stride)")
        self.torch, self.cfg = torch, cfg
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.F, self.N = n_frames, frame_rows
        self.n_pairs = n_frames - 1
        self.fe = Frontend(cfg, variant=variant)
        self.desc = torch.empty((n_frames * frame_rows, DESC_BYTES), dtype=torch.uint8, device=self.dev)
        self.kp = torch.empty((n_frames * frame_rows, 2), dtype=torch.float32, device=self.dev)
        chunks = max(1, min(chunks, self.n_pairs))
        self.bounds = [(self.n_pairs * c // chunks, self.n_pairs * (c + 1) // chunks) for c in range(chunks)]
        self.s_up, self.s_down = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
        self.K, self.pose = K, cfg.robust_pose is not None
        self.rec_bytes = step_record_bytes(cfg)
        self.rec_dev = torch.empty((self.n_pairs, self.rec_bytes), dtype=torch.uint8, device=self.dev)
        self.rec_host = torch.empty((self.n_pairs, self.rec_bytes), dtype=torch.uint8).pin_memory()
        self.out = RecordView(self.rec_host, cfg.max_matches, self.pose)
        self._batches = None
        self.h2d_bytes = int(self.F * frame_rows * (DESC_BYTES + 8))
        self.d2h_bytes = int(self.rec_host.numel())
        self.use_graph = use_graph
        self._graph, self._graph_key, self._eager_key = None, None, None

    def run(self, desc_host, kp_host, counts: np.ndarray):
        """desc_host: pinned uint8 [F*N, 32]; kp_host: pinned float32 [F*N, 2]; counts: rows used per frame."""
        self.out = RecordView(self.rec_host, self.cfg.max_matches, self.pose)
        if not self.use_graph:
            return self._run_eager(desc_host, kp_host, counts)
        key = (desc_host.data_ptr(), kp_host.data_ptr(), np.asarray(counts).tobytes())
        if self._graph is not None and self._graph_key == key:
            self._graph.replay()
            return self.out
        if self._eager_key != key:                                 # first call: eager (also warms every lazy init)
            self._eager_key = key
            return self._run_eager(desc_host, kp_host, counts)
        torch = self.torch
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._run_eager(desc_host, kp_host, counts)
        self._graph, self._graph_key = g, key
        g.replay()
        return self.out

    def _run_eager(self, desc_host, kp_host, counts: np.ndarray):
        torch, N = self.torch, self.N
        if self._batches is None or not np.array_equal(self._counts, counts):
            self._counts = np.array(counts, copy=True)
            self._batches = [sequence_batch(self.desc, self.kp, self._counts, lo, hi - lo, N) for lo, hi in self.bounds]
        main = torch.cuda.current_stream()
        self.s_up.wait_stream(main)
        ups, keep = [], []
        with torch.cuda.stream(self.s_up):
            for c, (lo, hi) in enumerate(self.bounds):
                f0 = lo if c == 0 else lo + 1                      # frame `lo` came with the previous chunk
                r0, r1 = f0 * N, (hi + 1) * N
                self.desc[r0:r1].copy_(desc_host[r0:r1], non_blocking=True)
                self.kp[r0:r1].copy_(kp_host[r0:r1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.s_up)
                ups.append(ev)
        for c, (lo, hi) in enumerate(self.bounds):
            main.wait_event(ups[c])
            res = self.fe.run(self._batches[c], K=self.K, records=self.rec_dev[lo:hi], pair_id0=lo)
            done = torch.cuda.Event()
            done.record(main)
            keep.append(res)
            with torch.cuda.stream(self.s_down):
                self.s_down.wait_event(done)
                self.rec_host[lo:hi].copy_(self.rec_dev[lo:hi], non_blocking=True)      # the chunk's ONE download
        main.wait_stream(self.s_down)
        self._keep = keep                                          # device tensors stay alive until the next run
        return self.out


class SequencePipeline:
    """End-to-end consecutive-frame tracking from pinned host buffers with `depth` steps in flight — the
    library's throughput front door (bench.py's ``e2e`` is ``submit`` x K + ``result``).

    A step = upload of the F frames (descriptors + keypoints), the hot-path kernels on the F-1 consecutive
    pairs, the record kernel, and ONE device->host copy of the records (``record_bytes(max_matches)`` per pair).

    schedule = "interleaved" (default): every slot has its own stream, device / pinned buffers and Frontend
      (workspace); a step is four operations on that stream — two uploads, ONE CUDA graph with every kernel of
      the step, one download.  Steps of different slots overlap freely: the upload of step s+1 and the download of
      step s-1 run under the kernels of step s, and so may the first / last kernels of neighbouring steps, which
      hides the gaps between back-to-back graph launches (measured: 437k against 427k pairs/s).
    schedule = "serial": three streams (uploads, kernels, downloads); copies overlap, but the kernels of all steps
      run on ONE stream and never interleave; accepts different host buffers on every call without re-capture.

    submit() is asynchronous and returns the slot; result(slot) waits for that slot's download and returns a
    RecordView over its pinned record buffer (valid until the slot is submitted again).  With cfg.robust_pose the
    records are pose records (pose_record_bytes per pair) and the view has "robust".  K: 3x3 intrinsics of the
    keypoints (None = identity), passed to every Frontend.run."""

    def __init__(self, n_frames: int, frame_rows: int, cfg: FrontendConfig, variant: int = _capi.VARIANT_I8MMA1,
                 depth: int = 3, device=None, use_graph: bool = True, schedule: str = "interleaved", after_compute=None,
                 K=None):
        torch = _capi.require_cuda()
        if not cfg.max_matches:
            raise ValueError("SequencePipeline needs max_matches (compact output stride)")
        if schedule not in ("interleaved", "serial"):
            raise ValueError("schedule must be 'interleaved' or 'serial'")
        self.torch, self.cfg, self.schedule = torch, cfg, schedule
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.F, self.N, self.n_pairs = n_frames, frame_rows, n_frames - 1
        self.depth = max(1, depth)
        self.after_compute = after_compute       # optional callable(slot dict) enqueued after the kernels (e.g. a collective)
        shared_fe = Frontend(cfg, variant=variant) if schedule == "serial" else None   # one stream: one workspace serves every slot
        self.s_up, self.s_compute, self.s_down = (torch.cuda.Stream(self.dev) for _ in range(3))
        P = self.n_pairs
        self.K = K
        self.rec_bytes = step_record_bytes(cfg)
        self.slots = []
        for _ in range(self.depth):
            self.slots.append({
                "desc": torch.empty((n_frames * frame_rows, DESC_BYTES), dtype=torch.uint8, device=self.dev),
                "kp": torch.empty((n_frames * frame_rows, 2), dtype=torch.float32, device=self.dev),
                "rec_dev": torch.empty((P, self.rec_bytes), dtype=torch.uint8, device=self.dev),
                "rec_host": torch.empty((P, self.rec_bytes), dtype=torch.uint8).pin_memory(),
                "fe": shared_fe or Frontend(cfg, variant=variant),
                "stream": torch.cuda.Stream(self.dev) if schedule == "interleaved" else None,
                "uploaded": torch.cuda.Event(), "computed": torch.cuda.Event(), "downloaded": torch.cuda.Event(),
                "used": False, "batch": None, "graph": None, "res": None})
        self.fe = self.slots[0]["fe"]
        self.h2d_bytes = int(self.F * frame_rows * (DESC_BYTES + 8))
        self.d2h_bytes = int(P * self.rec_bytes)
        self.use_graph = use_graph
        self._counts = None
        self._next = 0

    # ---- shared -----------------------------------------------------------------------------------------
    def _run_kernels(self, sl):
        sl["res"] = sl["fe"].run(sl["batch"], K=self.K, records=sl["rec_dev"], pair_id0=0)

    def _after(self, sl):
        # A collective hook runs EAGERLY behind the slot's graph, never inside it: graphs of different slots replay on
        # different streams with no mutual order, and two ranks must issue a communicator's collectives in the same
        # order — torch's process group serialises eager calls on its own stream in program order, a graph node does not.
        if self.after_compute is not None:
            self.after_compute(sl)

    def _prepare(self, counts: np.ndarray):
        """(Re)build the per-slot batches (and, for the serial schedule, the kernel graphs) for this frame-size vector."""
        torch = self.torch
        self._counts = np.array(counts, copy=True)
        torch.cuda.synchronize()
        for sl in self.slots:
            sl["batch"] = sequence_batch(sl["desc"], sl["kp"], self._counts, 0, self.n_pairs, self.N)
            sl["graph"], sl["used"] = None, False
            st = sl["stream"] or self.s_compute
            with torch.cuda.stream(st):
                self._run_kernels(sl)                                     # eager once: lazy init, workspace
                self._after(sl)
            st.synchronize()
            if self.use_graph and self.schedule == "serial":
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self.s_compute):
                    self._run_kernels(sl)
                sl["graph"] = g
        torch.cuda.synchronize()

    def submit(self, desc_host, kp_host, counts: np.ndarray) -> int:
        """desc_host: pinned uint8 [F*N, 32]; kp_host: pinned float32 [F*N, 2]; counts: rows used per frame."""
        if self._counts is None or not np.array_equal(self._counts, counts):
            self._prepare(counts)
        i = self._next % self.depth
        self._next += 1
        sl = self.slots[i]
        if self.schedule == "serial":
            self._submit_serial(sl, desc_host, kp_host)
        else:
            self._submit_interleaved(sl, desc_host, kp_host)
        sl["used"] = True
        return i

    # ---- interleaved: the slot's stream carries upload -> kernel graph -> download ------------------------
    def _submit_interleaved(self, sl, desc_host, kp_host):
        torch = self.torch
        st = sl["stream"]
        if self.use_graph and sl["graph"] is None:
            st.synchronize()
            g = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(g, stream=st):
                    self._run_kernels(sl)
                sl["graph"] = g
            except Exception:                                  # e.g. a collective hook the NCCL build cannot capture
                torch.cuda.synchronize()
                self.use_graph = False
        with torch.cuda.stream(st):
            sl["desc"].copy_(desc_host, non_blocking=True)     # any pinned host buffers: the copies are not part of the graph
            sl["kp"].copy_(kp_host, non_blocking=True)
            if sl["graph"] is not None:
                sl["graph"].replay()
            else:
                self._run_kernels(sl)
            self._after(sl)
            sl["rec_host"].copy_(sl["rec_dev"], non_blocking=True)      # the step's ONE download
            sl["downloaded"].record(st)

    # ---- serial: copies overlap, kernels on one stream ---------------------------------------------------
    def _submit_serial(self, sl, desc_host, kp_host):
        torch = self.torch
        if sl["used"]:
            self.s_up.wait_event(sl["computed"])            # the slot's device inputs are free again
        with torch.cuda.stream(self.s_up):
            sl["desc"].copy_(desc_host, non_blocking=True)
            sl["kp"].copy_(kp_host, non_blocking=True)
            sl["uploaded"].record(self.s_up)
        self.s_compute.wait_event(sl["uploaded"])
        if sl["used"]:
            self.s_compute.wait_event(sl["downloaded"])     # the slot's device results have been read
        with torch.cuda.stream(self.s_compute):
            if sl["graph"] is not None:
                sl["graph"].replay()
            else:
                self._run_kernels(sl)
            self._after(sl)
            sl["computed"].record(self.s_compute)
        self.s_down.wait_event(sl["computed"])
        with torch.cuda.stream(self.s_down):
            sl["rec_host"].copy_(sl["rec_dev"], non_blocking=True)      # the step's ONE download
            sl["downloaded"].record(self.s_down)

    def result(self, slot: int):
        sl = self.slots[slot]
        sl["downloaded"].synchronize()
        return RecordView(sl["rec_host"], self.cfg.max_matches, self.cfg.robust_pose is not None)

    def streams(self):
        if self.schedule == "interleaved":
            return tuple(sl["stream"] for sl in self.slots)
        return (self.s_up, self.s_compute, self.s_down)


class PairPipeline:
    """SequencePipeline's sibling for batches of INDEPENDENT pairs (loop-closure candidates, BASELINE config #3;
    high-density pairs, config #4): `depth` steps in flight, each on its own stream — upload of the pairs'
    descriptors and keypoints from pinned host memory, ONE CUDA graph with every kernel of the step, ONE download of
    the result records.  Pair p's query / train rows live at p * rows_q / p * rows_t of the slot's device buffers
    (fixed stride, so the copies are four contiguous transfers); the per-pair row counts may be ragged.  With
    cfg.robust_pose the records are pose records; K: 3x3 intrinsics of the keypoints (None = identity)."""

    def __init__(self, n_pairs: int, rows_q: int, rows_t: int, cfg: FrontendConfig, variant: int = _capi.VARIANT_I8MMA1,
                 depth: int = 2, device=None, use_graph: bool = True, after_compute=None, K=None):
        torch = _capi.require_cuda()
        if not cfg.max_matches:
            raise ValueError("PairPipeline needs max_matches (record stride)")
        self.torch, self.cfg = torch, cfg
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.P, self.rq, self.rt, self.depth = int(n_pairs), int(rows_q), int(rows_t), max(1, depth)
        self.after_compute, self.use_graph, self.K = after_compute, use_graph, K
        self.rec_bytes = step_record_bytes(cfg)
        P = self.P
        self.slots = []
        for _ in range(self.depth):
            self.slots.append({
                "q": torch.empty((P * self.rq, DESC_BYTES), dtype=torch.uint8, device=self.dev),
                "t": torch.empty((P * self.rt, DESC_BYTES), dtype=torch.uint8, device=self.dev),
                "kq": torch.empty((P * self.rq, 2), dtype=torch.float32, device=self.dev),
                "kt": torch.empty((P * self.rt, 2), dtype=torch.float32, device=self.dev),
                "rec_dev": torch.empty((P, self.rec_bytes), dtype=torch.uint8, device=self.dev),
                "rec_host": torch.empty((P, self.rec_bytes), dtype=torch.uint8).pin_memory(),
                "fe": Frontend(cfg, variant=variant), "stream": torch.cuda.Stream(self.dev), "downloaded": torch.cuda.Event(),
                "batch": None, "graph": None, "key": None, "res": None})
        self.h2d_bytes = int(P * (self.rq + self.rt) * (DESC_BYTES + 8))
        self.d2h_bytes = int(P * self.rec_bytes)
        self._next = 0

    def stage_host(self, qs, ts, kq, kt):
        """Host lists of per-pair arrays -> pinned, fixed-stride staging buffers (done once per batch by the caller;
        a real caller writes its frames straight into such buffers)."""
        torch, P = self.torch, self.P
        if not (len(qs) == len(ts) == len(kq) == len(kt) == P):
            raise ValueError("stage_host: need exactly n_pairs entries")
        q = np.zeros((P, self.rq, DESC_BYTES), np.uint8)
        t = np.zeros((P, self.rt, DESC_BYTES), np.uint8)
        a = np.zeros((P, self.rq, 2), np.float32)
        b = np.zeros((P, self.rt, 2), np.float32)
        nq, nt = np.zeros(P, np.int32), np.zeros(P, np.int32)
        for p in range(P):
            nq[p], nt[p] = len(qs[p]), len(ts[p])
            if nq[p] > self.rq or nt[p] > self.rt:
                raise ValueError("pair larger than the pipeline's row stride")
            q[p, :nq[p]], t[p, :nt[p]] = _prep_desc(qs[p]), _prep_desc(ts[p])
            a[p, :nq[p]], b[p, :nt[p]] = np.asarray(kq[p], np.float32).reshape(-1, 2), np.asarray(kt[p], np.float32).reshape(-1, 2)
        pin = lambda x, w: torch.from_numpy(x.reshape(-1, w)).pin_memory()
        return {"q": pin(q, DESC_BYTES), "t": pin(t, DESC_BYTES), "kq": pin(a, 2), "kt": pin(b, 2), "nq": nq, "nt": nt}

    def _batch(self, sl, nq, nt):
        torch, P = self.torch, self.P
        q_off, t_off = np.zeros(P + 1, np.int32), np.zeros(P + 1, np.int32)
        np.cumsum(nq, out=q_off[1:])
        np.cumsum(nt, out=t_off[1:])
        q_src = (np.arange(P, dtype=np.int64) * self.rq).astype(np.int32)
        t_src = (np.arange(P, dtype=np.int64) * self.rt).astype(np.int32)
        pack = torch.from_numpy(np.concatenate([q_off, t_off, q_src, t_src])).to(self.dev)
        return PairBatch(q_desc=sl["q"], t_desc=sl["t"], q_off=pack[:P + 1], t_off=pack[P + 1:2 * P + 2], q_off_host=q_off, t_off_host=t_off,
                         kp_q=sl["kq"], kp_t=sl["kt"], q_src=pack[2 * P + 2:3 * P + 2], t_src=pack[3 * P + 2:])

    def _run_kernels(self, sl):
        sl["res"] = sl["fe"].run(sl["batch"], K=self.K, records=sl["rec_dev"], pair_id0=0)

    def submit(self, staged) -> int:
        torch = self.torch
        i = self._next % self.depth
        self._next += 1
        sl = self.slots[i]
        st = sl["stream"]
        key = (staged["nq"].tobytes(), staged["nt"].tobytes())
        if sl["key"] != key:                                   # new row counts: new CSR tables, new graph
            st.synchronize()
            sl["batch"], sl["key"], sl["graph"] = self._batch(sl, staged["nq"], staged["nt"]), key, None
            with torch.cuda.stream(st):
                for k in ("q", "t", "kq", "kt"):
                    sl[k].copy_(staged[k], non_blocking=True)
                self._run_kernels(sl)                          # eager once: lazy init, workspace
            st.synchronize()
            if self.use_graph:
                g = torch.cuda.CUDAGraph()
                try:
                    with torch.cuda.graph(g, stream=st):
                        self._run_kernels(sl)
                    sl["graph"] = g
                except Exception:
                    torch.cuda.synchronize()
                    self.use_graph = False
        with torch.cuda.stream(st):
            for k in ("q", "t", "kq", "kt"):
                sl[k].copy_(staged[k], non_blocking=True)
            if sl["graph"] is not None:
                sl["graph"].replay()
            else:
                self._run_kernels(sl)
            if self.after_compute is not None:                 # eager, behind the graph (see SequencePipeline._after)
                self.after_compute(sl)
            sl["rec_host"].copy_(sl["rec_dev"], non_blocking=True)
            sl["downloaded"].record(st)
        return i

    def result(self, slot: int):
        sl = self.slots[slot]
        sl["downloaded"].synchronize()
        return RecordView(sl["rec_host"], self.cfg.max_matches, self.cfg.robust_pose is not None)

    def streams(self):
        return tuple(sl["stream"] for sl in self.slots)


class MapSweep:
    """BASELINE config #5 on one GPU: one query frame against EVERY keyframe of a persistent map (the loop of
    MapRelocalizer.relocalize, persistent_map.py:244-309, without the BoW cut to max_candidates), the map's
    descriptors and keypoints resident on the device.  Per query: ONE Hamming launch over all keyframes (pair p =
    keyframe p as the query side, the current frame as the train side, like the reference's
    ``matcher.match(kf.descriptors, descriptors)``, :266; every block expanded once), the cross-check selection
    sorted by distance with the top `max_matches` kept (:270) and the untruncated match count, the ranking of the
    keyframes by that count on the device, geometric verification (RANSAC E + refit + decomposition) of the best
    `top` only (mirrors max_candidates, :242), and `top` candidate records."""

    def __init__(self, kf_desc, kf_kp, frame_ids, cfg: FrontendConfig, *, top: int = 5, max_query_rows: int = 2048,
                 device=None, variant: int = _capi.VARIANT_I8MMA1):
        torch = _capi.require_cuda()
        if not cfg.max_matches:
            raise ValueError("MapSweep needs max_matches (compact output stride)")
        self.cfg, self.top = cfg, int(top)
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n_kf = len(kf_desc)
        sizes = np.array([len(d) for d in kf_desc], np.int64)
        self.off = np.zeros(self.n_kf + 1, np.int32)
        np.cumsum(sizes, out=self.off[1:])
        self.q_row0, self.max_query_rows = int(self.off[-1]), int(max_query_rows)
        rows = self.q_row0 + self.max_query_rows
        self.desc = torch.zeros((rows, DESC_BYTES), dtype=torch.uint8, device=self.dev)
        self.kp = torch.zeros((rows, 2), dtype=torch.float32, device=self.dev)
        if self.n_kf:
            self.desc[: self.q_row0].copy_(torch.from_numpy(np.concatenate([_prep_desc(d) for d in kf_desc], axis=0)))
            self.kp[: self.q_row0].copy_(torch.from_numpy(np.concatenate([np.asarray(k, np.float32).reshape(-1, 2) for k in kf_kp], axis=0)))
        self.frame_ids = torch.from_numpy(np.asarray(frame_ids, np.int32).copy()).to(self.dev)
        self.max_kf_rows = int(sizes.max()) if self.n_kf else 0
        self.matcher, self.ransac, self.pose = HammingMatcher(variant=variant), EssentialRansac(), PoseRecovery()
        self._batches = {}
        self.nq = 0
        self.last = None

    def query_desc_slot(self):
        return self.desc[self.q_row0:]

    def query_kp_slot(self):
        return self.kp[self.q_row0:]

    def set_query_rows(self, n: int):
        if not 0 < n <= self.max_query_rows:
            raise ValueError("query frame does not fit the slot")
        self.nq = int(n)

    def set_query(self, desc_dev, kp_dev):
        n = int(desc_dev.shape[0])
        self.set_query_rows(n)
        self.desc[self.q_row0:self.q_row0 + n].copy_(desc_dev, non_blocking=True)
        self.kp[self.q_row0:self.q_row0 + n].copy_(kp_dev.reshape(-1, 2), non_blocking=True)

    def _batch(self, n: int) -> PairBatch:
        if n not in self._batches:
            torch, K = _capi.require_cuda(), self.n_kf
            t_off = (np.arange(K + 1, dtype=np.int64) * n).astype(np.int32)
            shared = SharedBlocks.build(np.concatenate([self.off[:-1], [self.q_row0]]), np.concatenate([np.diff(self.off), [n]]),
                                        np.arange(K), np.full(K, K), self.dev)
            pack = torch.from_numpy(np.concatenate([self.off, t_off, self.off[:-1], np.full(K, self.q_row0, np.int32)]).astype(np.int32)).to(self.dev)
            self._batches[n] = PairBatch(q_desc=self.desc, t_desc=self.desc, q_off=pack[:K + 1], t_off=pack[K + 1:2 * K + 2],
                                         q_off_host=self.off, t_off_host=t_off, kp_q=self.kp, kp_t=self.kp,
                                         q_src=pack[2 * K + 2:3 * K + 2], t_src=pack[3 * K + 2:], shared=shared)
        return self._batches[n]

    def run(self, records=None, counts_out=None):
        """All launches on the current stream, nothing touches the host.  records: device uint8 [top, record_bytes];
        counts_out: device int32 [n_kf] (per-keyframe cross-check match counts).  -> dict of device tensors."""
        torch = _capi.require_cuda()
        c, S, k = self.cfg, self.cfg.max_matches, min(self.top, max(self.n_kf, 1))
        b = self._batch(self.nq)
        keys = self.matcher.knn2(b, need_second=False)          # cross-check only (persistent_map.py:266): no second neighbour
        sel = self.matcher.select(b, keys, use_ratio=False, use_cross=True, sort_by_distance=True, max_matches=S,
                                  with_corr=True, compact=True, with_total=True)
        top_idx, c_off, c_cnt, top_id = rank_pairs(sel.total, k, ids=self.frame_ids, sel_count=sel.count, stride=S, with_ids=True)
        E = self.ransac.hypotheses(sel.corr, c_off, c_cnt, k, c.hypotheses, seed=c.seed, pair_ids=top_id)   # keyed by frame id: sharding-independent
        th2 = c.threshold ** 2
        counts = self.ransac.score(sel.corr, c_off, c_cnt, k, E, th2, precision=c.precision, max_m=S)
        best_h, best_c, mask = self.ransac.select(counts, sel.corr, c_off, c_cnt, k, E, th2)
        E_refit, R, t, votes = self.pose.recover(sel.corr, c_off, c_cnt, k, S, mask=mask)
        if records is not None:
            pack_records(records, sel, best_h, best_c, mask, R, t, n_records=k, pair_ids=self.frame_ids, src_pair=top_idx,
                         count_total=sel.total)
        if counts_out is not None:
            counts_out.copy_(sel.total, non_blocking=True)
        self.last = {"keys": keys, "sel": sel, "top_idx": top_idx, "c_off": c_off, "c_count": c_cnt, "best_h": best_h,
                     "best_count": best_c, "mask": mask, "R": R, "t": t, "E": E, "counts": counts}
        return self.last


def pipe_microbench(which: str, iters: int = 2000, ctas_per_sm: int = 8, repeats: int = 5):
    """Measured instruction rate of one SM pipe: (thread-instructions/s, per clk per SM
    at the reported max clock).  Roofline denominator for the POPC kernel (SURVEY §8d)."""
    torch = _capi.require_cuda()
    lib = _capi.load_library()
    sink = torch.zeros(4, dtype=torch.int32, device="cuda")
    ops = C.c_double(0.0)
    best = float("inf")
    for r in range(repeats + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib.b2s_pipe_microbench(_capi.PIPE_IDS[which], iters, ctas_per_sm, C.byref(ops), ptr(sink), current_stream()))
        e1.record()
        e1.synchronize()
        if r:
            best = min(best, e0.elapsed_time(e1) * 1e-3)
    return ops.value / best


def mma_microbench(iters: int = 4000, repeats: int = 3):
    """Measured dense tcgen05.mma kind::i8 rate (int8 op/s, 2 per MAC): every SM issues
    M128.N128.K32 MMAs from shared memory back to back.  Roofline denominator of K2/K2s."""
    torch = _capi.require_cuda()
    lib = _capi.load_library()
    macs = C.c_double(0.0)
    best = float("inf")
    for r in range(repeats + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib.b2s_mma_microbench(iters, 128, C.byref(macs), current_stream()))
        e1.record()
        e1.synchronize()
        if r:
            best = min(best, e0.elapsed_time(e1) * 1e-3)
    return 2.0 * macs.value / best


def unpack_keys(k: np.ndarray):
    k = np.asarray(k, np.uint32)
    return (k >> np.uint32(IDX_BITS)).astype(np.int64), (k & np.uint32(IDX_MASK)).astype(np.int64), k >= np.uint32(0x80000000)
