"""Multi-GPU path: frame pairs are independent, so ranks take contiguous blocks of the pair batch (or of the
map's keyframes) and the only collective is ONE all-gather of fixed-size result records (SURVEY.md §8e).
One process per B200 (torchrun), NCCL over NVLink; the same classes run over gloo on CPU tensors (tests).

* ``shard_bounds``        who owns what.
* ``RecordGather``        the persistent all-gather buffer: every rank's last kernel writes its records straight
                          into its own slice (``local``), ``all_gather()`` is the in-place collective.
* ``ShardedFrontend``     match -> select -> RANSAC -> pose -> records on this rank's pairs + the gather, captured
                          as ONE CUDA graph (the NCCL all-gather is a node of it): BASELINE configs #2 / #3.
* ``ShardedSweep``        relocalization sweep (config #5): the map's keyframes sharded by id and resident on each
                          GPU, the query broadcast once, every rank verifies its local top-k, the gathered
                          candidates hold the global top-k.
"""
from __future__ import annotations

import numpy as np

RECORD_WIDTH = 4  # legacy int32 record: (n_matches, best_h, inlier_count, pair_id)


def shard_bounds(n_items: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [lo, hi) of rank `rank`; sizes differ by at most one."""
    if world <= 0 or not 0 <= rank < world:
        raise ValueError("bad rank/world")
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_capacity(n_items: int, world: int) -> int:
    return -(-n_items // world) if world > 0 else n_items


def pack_records(pair_ids, n_matches, best_h, inlier_count):
    """-> (n_local, RECORD_WIDTH) int32 array (the small legacy record; the full record is csrc/records.cu)."""
    return np.stack([np.asarray(n_matches, np.int32), np.asarray(best_h, np.int32),
                     np.asarray(inlier_count, np.int32), np.asarray(pair_ids, np.int32)], axis=1)


def gather_records(local, n_items: int, group=None):
    """All-gather per-pair result records (torch tensor, (n_local, W), on the backend's device) from every rank;
    returns the (n_items, W) tensor ordered by pair id.  One fixed-size collective (shards padded to the largest)."""
    import torch.distributed as dist

    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return local
    g = RecordGather(n_items, int(local.shape[1]), dtype=local.dtype, device=local.device, group=group, pad_value=-1)
    g.local[: local.shape[0]] = local
    g.all_gather()
    return g.ordered()


def shutdown_process_group(timeout_s: float = 20.0):
    """Destroy the default process group at the end of a run.  CUDA graphs that captured NCCL collectives must be
    released BEFORE their communicator is destroyed (ncclCommDestroy waits for them forever otherwise — measured: a
    15-minute hang): the caller drops its ShardedFrontend / ShardedSweep objects first, this collects what is left,
    and a timer ends the process normally if the teardown still does not return."""
    import gc
    import os
    import sys
    import threading

    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    dist.barrier()
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    t = threading.Timer(timeout_s, lambda: os._exit(0))
    t.daemon = True
    t.start()
    dist.destroy_process_group()
    t.cancel()


class RecordGather:
    """Persistent gather buffer [world, cap, width]: ``local`` (this rank's [cap, width] slice) is where the last
    kernel of a step writes; ``all_gather()`` completes the other slices in place (NCCL recognises
    sendbuff == recvbuff + rank * count and moves nothing locally).  ``ordered()`` drops the padding."""

    def __init__(self, n_items: int, width: int, *, dtype=None, device=None, group=None, pad_value=0):
        import torch
        import torch.distributed as dist

        self.group = group
        self.dist_on = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if self.dist_on else 1
        self.rank = dist.get_rank(group) if self.dist_on else 0
        self.n_items, self.width = int(n_items), int(width)
        self.cap = shard_capacity(self.n_items, self.world)
        self.lo, self.hi = shard_bounds(self.n_items, self.rank, self.world)
        self.buf = torch.full((self.world, self.cap, self.width), pad_value, dtype=dtype or torch.uint8, device=device)
        self.local = self.buf[self.rank]

    @property
    def n_local(self) -> int:
        return self.hi - self.lo

    def all_gather(self, async_op: bool = False):
        """Enqueue the collective behind the current stream's work (capturable into a CUDA graph with NCCL).
        async_op=True returns the work handle instead of making the current stream wait for the collective: the
        caller's next kernels then overlap it, and `handle.wait()` orders whatever reads or rewrites the buffer."""
        if self.world > 1:
            import torch.distributed as dist

            return dist.all_gather_into_tensor(self.buf.view(-1), self.local.reshape(-1), group=self.group, async_op=async_op)
        return None

    def ordered(self):
        """[n_items, width] in pair order (a copy; padding rows of short shards dropped)."""
        import torch

        if self.cap * self.world == self.n_items:
            return self.buf.reshape(self.n_items, self.width)
        parts = []
        for r in range(self.world):
            lo, hi = shard_bounds(self.n_items, r, self.world)
            parts.append(self.buf[r, : hi - lo])
        return torch.cat(parts, dim=0)


def _mark_empty(rows, cfg):
    """Records [n, record_bytes] that hold no pair (padding slots of a short shard): pair id -1, and in pose records
    outcome -1 (robust_pose.POSE_EMPTY), so that an empty slot never decodes as an estimate."""
    from .frontend import record_bytes

    rows[:, 12:16] = 0xFF                                              # int32 header[3] = -1
    if cfg.robust_pose is not None:
        o = record_bytes(cfg.max_matches)                              # the pose block: b2s_pose_result.outcome
        rows[:, o:o + 4] = 0xFF


DEFAULT_LANES = 3    # measured on the metric's step (tools/lanes_ab.py): 1 lane 473.5 k pairs/s, 2 lanes 488.7 k, 3 lanes 494.8 k


class ShardedFrontend:
    """The hot path on this rank's block of a global pair batch + the gather of every rank's result records.

    ``n_pairs_global`` pairs are split with ``shard_bounds``; the caller builds the PairBatch of ITS pairs
    (``self.lo .. self.hi``).  ``step(batch)`` runs match -> select -> hypotheses -> score -> winner (-> refit ->
    decomposition when cfg.with_pose) and the record kernel writes this rank's records into the send buffer.
    A batch may be processed as ``sets_per_gather`` launch sets (sub-batches that keep every kernel's grid at a few
    waves); its records leave in ONE ``all_gather_into_tensor``.

    ``pipelined=True`` (default): the collective of batch k is issued inside the first launch set of batch k + 1 —
    started after that set's selection kernel, joined before its record kernel — so it runs under the multi-wave
    RANSAC kernels (8-point, scoring, winner) and is off the critical path; ``flush()`` gathers the last batch, and
    ``records()`` is then complete.  ``pipelined=False``: the collective follows the batch's last launch set on the
    same stream.  Measured at 8 GPUs against 1 GPU on the same box (profiles/r02_scale.md): a collective per launch set
    0.912, the same overlapped with the next set's kernels 0.938 (the NCCL kernel takes SMs away from the persistent
    one-CTA-per-SM Hamming kernel that follows it, whose late CTAs then finish late), one collective per batch 0.969,
    pipelined under the RANSAC kernels: see that file.

    ``lanes`` (default 3): the launch sets of a batch alternate between that many streams, see __init__.

    ``capture(batches)`` records a whole batch — collective included — into ONE CUDA graph (``replay()``); if the
    NCCL build cannot be captured the kernels are replayed and the collective is issued eagerly (``gather_in_graph``
    says which).  ``records()`` -> device uint8 [sets_per_gather, n_pairs_global, record_bytes]."""

    def __init__(self, cfg, n_pairs_global: int, *, variant=None, group=None, device=None, sets_per_gather: int = 1,
                 pipelined: bool = True, lanes: int | None = None):
        import os

        from . import _capi
        from .frontend import Frontend, step_record_bytes

        torch = _capi.require_cuda()
        if not cfg.max_matches:
            raise ValueError("ShardedFrontend needs max_matches (record stride)")
        self.cfg = cfg            # cfg.with_pose decides whether the records carry R | t (else zeros); cfg.robust_pose: pose records
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        # lanes: the launch sets of a batch alternate between `lanes` streams (each with its own Frontend = its own
        # workspaces), so the tail of one set's kernels, its one-CTA-per-pair selection / winner kernels and the gaps
        # between dependent launches are filled with the other set's work.  Lane 0 is the caller's stream; the side
        # lanes fork from it at their first launch set of a batch and join it behind the last (also under capture).
        self.lanes = max(1, min(int(os.environ.get("B2S_LANES", 0)) or (DEFAULT_LANES if lanes is None else int(lanes)), max(1, int(sets_per_gather))))
        self.fes = [Frontend(self.cfg, variant=_capi.VARIANT_I8MMA1 if variant is None else variant) for _ in range(self.lanes)]
        self.fe = self.fes[0]
        self._side = [torch.cuda.Stream(device=self.dev) for _ in range(self.lanes - 1)]
        self.rec_bytes = step_record_bytes(cfg)      # pose records when cfg.robust_pose is set
        self.sets = max(1, int(sets_per_gather))
        self.n_pairs_global = int(n_pairs_global)
        self.world, self.group = _world(group), group
        self.cap = shard_capacity(self.n_pairs_global, self.world)
        # send = this rank's records of the batch in progress [sets * cap][record]; recv = every rank's records of
        # the last gathered batch [world][sets * cap][record]
        self.gather = RecordGather(self.world * self.sets * self.cap, self.rec_bytes, dtype=torch.uint8, device=self.dev, group=group)
        self.rank = self.gather.rank
        _mark_empty(self.gather.buf.view(-1, self.rec_bytes), cfg)     # padding slots: pair id -1
        self.pipelined = bool(pipelined) and os.environ.get("B2S_GATHER", "pipelined") != "sync"
        if self.pipelined and self.world > 1:
            self.send = torch.zeros((self.sets * self.cap, self.rec_bytes), dtype=torch.uint8, device=self.dev)
            _mark_empty(self.send, cfg)
        else:
            self.send = self.gather.local               # in-place: the send slice of the gather buffer itself
        self.lo, self.hi = shard_bounds(self.n_pairs_global, self.rank, self.world)
        self._work, self._k, self._pending, self._kernels_only = None, 0, False, False
        self._held = []
        self._graph, self.res = None, None
        self.gather_in_graph = False

    # ---- the collective ------------------------------------------------------------------------------------
    def _start_gather(self):
        if self.world > 1:
            import torch.distributed as dist

            self._work = dist.all_gather_into_tensor(self.gather.buf.view(-1), self.send.reshape(-1), group=self.group, async_op=True)

    def _join_gather(self):
        if self._work is not None:
            self._work.wait()
            self._work = None

    def step(self, batch, K=None):
        if batch.n_pairs != self.hi - self.lo:
            raise ValueError(f"rank {self.rank} owns pairs [{self.lo}, {self.hi}) but the batch has {batch.n_pairs}")
        j = self._k % self.sets
        self._k += 1
        rows = self.send[j * self.cap: j * self.cap + batch.n_pairs]
        first = j == 0 and self.pipelined and self.world > 1 and self._pending and not self._kernels_only
        lane = j % self.lanes
        if lane == 0:
            # pipelined: the previous batch's records (still in `send`) leave while this set's RANSAC kernels run; the
            # record kernel of this set, which overwrites the first rows of `send`, waits for the collective
            self.res = self.fes[0].run(batch, K=K, records=rows, pair_id0=self.lo,
                                       after_select=self._start_gather if first else None,
                                       before_records=self._join_gather if first else None)
        else:
            import torch

            side = self._side[lane - 1]
            if j < self.lanes:                      # fork: behind everything the caller's stream holds so far — set 0
                side.wait_stream(torch.cuda.current_stream(self.dev))   # included, i.e. behind the join of the collective that reads `send`
            with torch.cuda.stream(side):
                self.res = self.fes[lane].run(batch, K=K, records=rows, pair_id0=self.lo)
            # the caller's stream is ordered behind this lane only at the batch's join: keep the inputs alive until
            # then, so that memory the caller frees early is not handed out again while the lane still reads it
            self._held.append((batch, K))
        if j == self.sets - 1:                      # the batch's last launch set
            if self.lanes > 1:
                import torch

                for side in self._side[:min(self.lanes, self.sets) - 1]:
                    torch.cuda.current_stream(self.dev).wait_stream(side)
                self._held.clear()
            if self._kernels_only:
                pass
            elif self.pipelined and self.world > 1:
                self._pending = True                # gathered inside the next batch (or by flush())
            else:
                self.gather.all_gather()
        return self.res

    def flush(self):
        """Gather the last batch's records (pipelined mode) and order the current stream behind the collective."""
        if self._pending:
            self._start_gather()
            self._pending = False
        self._join_gather()

    wait = flush

    def capture(self, batches, K=None, collective_in_graph: bool = True):
        """One eager pass (lazy init, workspaces, NCCL warm-up), then the capture of step(b) for every b of `batches`
        (one PairBatch or a list of sets_per_gather launch sets = one batch).  In pipelined mode the graph holds the
        collective of the PREVIOUS replay's batch (steady state: one collective per replay); call flush() after the
        last replay."""
        import torch

        batches = batches if isinstance(batches, (list, tuple)) else [batches]
        if len(batches) != self.sets:
            raise ValueError("capture: pass exactly sets_per_gather launch sets (one batch)")

        def body():
            for b in batches:
                self.step(b, K)
        self._k = 0
        body()
        self.flush()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        self.gather_in_graph = False
        if collective_in_graph and self.world > 1:
            self._k, self._pending = 0, self.pipelined
            try:
                with torch.cuda.graph(g):
                    body()
                self.gather_in_graph = True
            except Exception:                      # NCCL / torch build that cannot capture the collective
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                self._work = None
        if not self.gather_in_graph:
            with torch.cuda.graph(g):
                self._k, self._kernels_only = 0, True          # step() then issues no collective
                try:
                    body()
                finally:
                    self._kernels_only = False
        self._k = 0
        self._pending = self.pipelined and self.world > 1     # the eager pass left a complete batch in `send`
        self._graph = g
        torch.cuda.synchronize()
        return self.gather_in_graph

    def replay(self):
        self._graph.replay()
        if self.world > 1:
            if not self.gather_in_graph:
                self._start_gather()                # eager, behind the graph
                self._join_gather()
                self._pending = False
            elif self.pipelined:
                self._pending = True                # this replay's batch is gathered by the next replay, or by flush()
        return self.res

    def records(self):
        """[sets_per_gather, n_pairs_global, record_bytes] in pair order (padding rows of short shards dropped); in
        pipelined mode call flush() first."""
        import torch

        v = self.gather.buf.view(self.world, self.sets, self.cap, self.rec_bytes)
        parts = []
        for r in range(self.world):
            lo, hi = shard_bounds(self.n_pairs_global, r, self.world)
            parts.append(v[r, :, : hi - lo])
        return torch.cat(parts, dim=1)

    def close(self):
        """Release the captured graph (it holds the NCCL all-gather node: see shutdown_process_group)."""
        self._work = None
        self._graph = None


def _dist_on(group=None) -> bool:
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized()


def _world(group=None) -> int:
    import torch.distributed as dist

    return dist.get_world_size(group) if _dist_on(group) else 1


class ShardedSweep:
    """BASELINE config #5 on N GPUs: keyframes sharded by id (contiguous blocks), each shard resident on its GPU
    (``MapSweep``), the query frame broadcast from rank 0, every rank cross-check-matches the query against
    ITS keyframes, verifies its local top-k geometrically and contributes k candidate records + its per-keyframe
    match counts to ONE all-gather.  The global top-k by match count is among the world x k gathered candidates."""

    def __init__(self, kf_desc, kf_kp, frame_ids, cfg, *, top: int = 5, max_query_rows: int = 2048, group=None, device=None,
                 n_keyframes_global: int | None = None):
        """kf_desc / kf_kp / frame_ids: THIS rank's keyframes (lists of (n_i, 32) uint8 / (n_i, 2) float32, ids)."""
        from . import _capi
        from .frontend import MapSweep, record_bytes

        torch = _capi.require_cuda()
        import torch.distributed as dist

        self.group = group
        self.dist_on = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if self.dist_on else 1
        self.rank = dist.get_rank(group) if self.dist_on else 0
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.sweep = MapSweep(kf_desc, kf_kp, frame_ids, cfg, top=top, max_query_rows=max_query_rows, device=self.dev)
        self.top, self.stride = top, cfg.max_matches
        self.n_global = n_keyframes_global if n_keyframes_global is not None else len(kf_desc) * self.world
        self.cap = shard_capacity(self.n_global, self.world)
        rb = record_bytes(cfg.max_matches)
        self.slot_bytes = top * rb + ((4 * self.cap + 63) // 64) * 64          # k candidate records | per-keyframe counts
        self.gather = RecordGather(self.world, self.slot_bytes, dtype=torch.uint8, device=self.dev, group=group)
        slot = self.gather.local[0]
        self.cand = slot[: top * rb].view(top, rb)
        self.counts = slot[top * rb: top * rb + 4 * self.cap].view(torch.int32)
        self.counts.fill_(-1)
        self._graph = None

    def query(self, q_desc_dev=None, q_kp_dev=None, n_rows: int | None = None):
        """Rank 0 passes the query frame (device uint8 [n, 32], float32 [n, 2]); the others pass None."""
        import torch
        import torch.distributed as dist

        sw = self.sweep
        if self.rank == 0 and q_desc_dev is not None:
            sw.set_query(q_desc_dev, q_kp_dev)
        if self.world > 1:                          # the 64 KB + 16 KB query, once
            dist.broadcast(sw.query_desc_slot(), src=0, group=self.group)
            dist.broadcast(sw.query_kp_slot(), src=0, group=self.group)
        sw.run(records=self.cand, counts_out=self.counts[: sw.n_kf])
        self.gather.all_gather()
        return self.gather.buf

    def capture(self):
        import torch

        self.query()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g):
                self.query()
            self._graph = g
        except Exception:
            torch.cuda.synchronize()
            self._graph = None
        return self._graph is not None

    def replay(self):
        if self._graph is not None:
            self._graph.replay()
        else:
            self.query()

    def close(self):
        self._graph = None

    def result_host(self):
        """-> (per-keyframe match counts in global keyframe order, the global top-k candidates as a dict of arrays
        sorted by (-count, frame id))."""
        from .frontend import unpack_records

        buf = self.gather.buf.cpu().numpy().reshape(self.world, self.slot_bytes)
        rb = (self.slot_bytes - ((4 * self.cap + 63) // 64) * 64) // self.top
        counts, cands = [], []
        for r in range(self.world):
            lo, hi = shard_bounds(self.n_global, r, self.world)
            counts.append(buf[r, self.top * rb: self.top * rb + 4 * self.cap].copy().view(np.int32)[: hi - lo])
            cands.append(buf[r, : self.top * rb].reshape(self.top, rb))
        rec = unpack_records(np.concatenate(cands, axis=0), self.stride)
        ok = np.flatnonzero(rec["pair_id"] >= 0)
        order = ok[np.lexsort((rec["pair_id"][ok], -rec["n_matches"][ok]))][: self.top]
        return np.concatenate(counts), {k: v[order] for k, v in rec.items()}
