"""World-size-independence check of the sharded library paths (run plain for world 1, or under torchrun):
writes the gathered result records of a small config #3 batch (pair-sharded ShardedFrontend) or a small
config #5 sweep (keyframe-sharded ShardedSweep) to --out on rank 0.  tests/test_gpu_records.py compares the
world-1 and world-2 files bit for bit.  --robust (configs 2 and 3): the step runs RobustPoseEstimator.estimate_pose
for every pair (FrontendConfig.robust_pose) and the gathered records are pose records; the output then also holds
every pair's b2s_pose_result bytes ("robust"); tests/test_gpu_robust_records.py compares those files."""
import argparse
import faulthandler
import json
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "monocular-visual-slam_b200")]
import numpy as np
import torch
import torch.distributed as dist

from b200slam.frontend import FrontendConfig, PairBatch, unpack_records
from b200slam.robust_pose import RobustPoseConfig
from b200slam.sharding import ShardedFrontend, ShardedSweep, shard_bounds
from b200slam.synthetic import tracking_pairs

faulthandler.dump_traceback_later(int(os.environ.get("B2S_WATCHDOG_S", "120")), exit=True)   # a stuck collective must not hang the box
ap = argparse.ArgumentParser()
ap.add_argument("--config", type=int, default=3)
ap.add_argument("--out", required=True)
ap.add_argument("--no-graph-collective", action="store_true", help="keep the collective out of the CUDA graph (diagnostics)")
ap.add_argument("--robust", action="store_true", help="configs 2 / 3 with robust_pose=RobustPoseConfig(): pose records")
a = ap.parse_args()
if a.robust and a.config not in (2, 3):
    ap.error("--robust applies to the pair-sharded configs 2 and 3")
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
S = 200
cfg = FrontendConfig(hypotheses=256, max_matches=S, threshold=0.01, seed=99, with_pose=not a.robust,
                     robust_pose=RobustPoseConfig() if a.robust else None)


def unpack(rec):
    u = unpack_records(rec, S, pose=a.robust)
    if a.robust:
        u["robust"] = u["robust"].view(np.uint8).reshape(len(rec), -1)     # raw bytes: compared bit for bit
    return u


out = {}
in_graph = None
sf = sw = None
if a.config == 3:
    n = 21                                                     # not divisible by 2: exercises the padded shard
    qs, ts, kq, kt = tracking_pairs(n, 500, seed=5, keep=0.4, ragged=True)
    sf = ShardedFrontend(cfg, n)
    lo, hi = sf.lo, sf.hi
    batch = PairBatch.from_host(qs[lo:hi], ts[lo:hi], kq[lo:hi], kt[lo:hi])
    print(f"[rank {rank}] eager step ok, capturing", file=sys.stderr, flush=True)
    in_graph = sf.capture(batch, collective_in_graph=not a.no_graph_collective)
    print(f"[rank {rank}] captured, collective_in_graph={in_graph}", file=sys.stderr, flush=True)
    for _ in range(2):
        sf.replay()
    sf.flush()
    torch.cuda.synchronize()
    u = unpack(sf.records()[0].cpu().numpy())
    out = {k: v for k, v in u.items()}
elif a.config == 2:
    # a batch of 5 launch sets (alternating over the stream lanes), ONE pipelined collective per batch
    n, sets = 21, 5
    sf = ShardedFrontend(cfg, n, sets_per_gather=sets)
    lo, hi = sf.lo, sf.hi
    bl = []
    for j in range(sets):
        qs, ts, kq, kt = tracking_pairs(n, 500, seed=50 + j, keep=0.4, ragged=True)
        bl.append(PairBatch.from_host(qs[lo:hi], ts[lo:hi], kq[lo:hi], kt[lo:hi]))
    in_graph = sf.capture(bl, collective_in_graph=not a.no_graph_collective)
    print(f"[rank {rank}] captured, collective_in_graph={in_graph}, lanes={sf.lanes}", file=sys.stderr, flush=True)
    for _ in range(3):
        sf.replay()
    sf.flush()
    torch.cuda.synchronize()
    rec = sf.records().cpu().numpy()
    for j in range(sets):
        for k, v in unpack(rec[j]).items():
            out[f"set{j}/{k}"] = v
    out["n_matches"], out["inliers"], out["pair_id"] = out["set0/n_matches"], out["set0/inliers"], out["set0/pair_id"]
else:
    rng = np.random.default_rng(9)
    n_kf = 31
    kf_desc = [rng.integers(0, 256, (int(rng.integers(250, 401)), 32), dtype=np.uint8) for _ in range(n_kf)]
    kf_kp = [rng.uniform(-0.5, 0.5, (len(d), 2)).astype(np.float32) for d in kf_desc]
    ids = (np.arange(n_kf) * 2 + 3).astype(np.int32)
    # the query re-observes keyframes 4 (strongly) and 20 (weakly)
    nq = 400
    q_desc = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    q_kp = rng.uniform(-0.5, 0.5, (nq, 2)).astype(np.float32)
    for kf, rows in ((4, 220), (20, 120)):
        m = min(rows, len(kf_desc[kf]))
        P = np.stack([rng.uniform(-6, 6, m), rng.uniform(-2, 2, m), rng.uniform(6, 30, m)], axis=1)
        kf_kp[kf][:m] = (P[:, :2] / P[:, 2:]).astype(np.float32)
        P2 = P + np.array([0.2, 0.0, -0.8])
        bits = np.unpackbits(kf_desc[kf][:m], axis=1)
        bits ^= (rng.random(bits.shape) < 0.05).astype(np.uint8)
        sl = slice(0, m) if kf == 4 else slice(nq - m, nq)
        q_desc[sl] = np.packbits(bits, axis=1)
        q_kp[sl] = (P2[:, :2] / P2[:, 2:]).astype(np.float32)
    lo, hi = shard_bounds(n_kf, rank, world)
    sw = ShardedSweep(kf_desc[lo:hi], kf_kp[lo:hi], ids[lo:hi], cfg, top=5, max_query_rows=512, n_keyframes_global=n_kf)
    sw.sweep.set_query_rows(nq)
    if rank == 0:
        sw.query(torch.from_numpy(q_desc).cuda(), torch.from_numpy(q_kp).cuda(), n_rows=nq)
    else:
        sw.query(n_rows=nq)
    print(f"[rank {rank}] eager query ok, capturing", file=sys.stderr, flush=True)
    in_graph = sw.capture() if not a.no_graph_collective else False
    print(f"[rank {rank}] captured={in_graph}", file=sys.stderr, flush=True)
    sw.replay()
    torch.cuda.synchronize()
    counts, cand = sw.result_host()
    out = dict(cand, counts=counts)
if rank == 0:
    np.savez(a.out, **out)
    print(json.dumps({"world": world, "config": a.config, "robust": a.robust, "collective_in_graph": in_graph,
                      "summary": {k: np.asarray(v).reshape(-1)[:5].tolist() for k, v in out.items() if k in ("n_matches", "inliers", "pair_id", "counts")}}))
sf = sw = None          # graphs that captured the collective go before their communicator
if world > 1:
    from b200slam.sharding import shutdown_process_group
    shutdown_process_group()
