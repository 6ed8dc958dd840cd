"""A/B of the K2s work decompositions (GPU): kernel-only time (library events) and clk per 128x128 tile pair
for train-axis splits, on the BASELINE shapes.
Usage: python tools/k2s_plans.py"""
import ctypes as C
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "monocular-visual-slam_b200")]
import numpy as np
import torch

from b200slam import _capi
from b200slam.frontend import HammingMatcher, PairBatch, sequence_batch

lib = _capi.load_library()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def kernel_ms(m, batch, reps=8):
    for _ in range(2):
        m.knn2(batch)
    torch.cuda.synchronize()
    lib.b2s_hamming_kernel_timing(1, None)
    ks, calls = [], []
    for _ in range(reps):
        flush.fill_(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); m.knn2(batch); e1.record(); torch.cuda.synchronize()
        v = C.c_float(0.0)
        lib.b2s_hamming_kernel_timing(-1, C.byref(v))
        ks.append(v.value); calls.append(e0.elapsed_time(e1))
    lib.b2s_hamming_kernel_timing(0, None)
    return float(np.median(ks)), float(np.median(calls))


def graph_call_ms(m, batch, reps=20):
    """Whole knn2 call (memsets, expansion, kernel, merge) replayed back to back from ONE CUDA graph:
    no host launch gaps, which dominate the eager timing of 10-40 us calls."""
    m.knn2(batch)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            m.knn2(batch)
    g.replay()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        flush.fill_(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    return best


def plan():
    v = [C.c_int(0) for _ in range(3)]
    lib.b2s_hamming_last_plan(*[C.byref(x) for x in v])
    return tuple(x.value for x in v)


def report(name, batch, nq, nt, pairs, splits=(0,)):
    tile_pairs = pairs * ((nq + 127) // 128) * ((nt + 127) // 128)
    ops = 2.0 * 256 * nq * nt * pairs
    for ts in splits:
        m = HammingMatcher(variant=_capi.VARIANT_I8MMA1, t_split=ts)
        k, call = kernel_ms(m, batch)
        subs, tsu, grid = plan()
        gcall = graph_call_ms(m, batch)
        print(f"{name:28s} t_split {ts:2d} -> plan subs {subs} t_split {tsu:2d} grid {grid:3d}: kernel(events, eager) {k:.4f} ms "
              f"call(eager) {call:.4f} ms  call(graph x20) {gcall:.4f} ms = {ops / (gcall * 1e-3) / 1e15:.3f} POP/s whole call", flush=True)


rng = np.random.default_rng(0)
# configs[1]: 296 consecutive pairs over 297 frames (shared blocks)
F, N = 297, 2000
desc = torch.from_numpy(rng.integers(0, 256, (F * N, 32), dtype=np.uint8)).cuda()
kp = torch.zeros((F * N, 2), dtype=torch.float32, device="cuda")
report("config2 296 x 2000^2 shared", sequence_batch(desc, kp, np.full(F, N, np.int32), 0, F - 1, N), N, N, F - 1)
# config 3: 256 independent pairs
qs = [rng.integers(0, 256, (N, 32), dtype=np.uint8) for _ in range(256)]
ts_ = [rng.integers(0, 256, (N, 32), dtype=np.uint8) for _ in range(256)]
report("config3 256 x 2000^2", PairBatch.from_host(qs, ts_), N, N, 256)
# config 4: one 10k x 10k pair
q = rng.integers(0, 256, (10000, 32), dtype=np.uint8)
t = rng.integers(0, 256, (10000, 32), dtype=np.uint8)
report("config4 1 x 10000^2", PairBatch.from_host([q], [t]), 10000, 10000, 1, splits=(1, 0, 3, 7, 11, 14, 20))
# the drop-in call: one 2000 x 2000 pair
report("single 2000^2", PairBatch.from_host([qs[0]], [ts_[0]]), N, N, 1, splits=(1, 0, 8, 16))
