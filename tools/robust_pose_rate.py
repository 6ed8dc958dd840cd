#!/usr/bin/env python
"""Rate of the batched robust pose estimator on the 296-pair tracking launch set (BASELINE config #2 shape:
2000 x 2000 descriptors per pair, 500 matches, 2000 hypotheses for each of E and H).

  1. Step time, CUDA-graph replay timed with CUDA events, L2 overwritten (256 MB memset) before every replay:
     Frontend(with_pose=True) against Frontend(robust_pose=...).
  2. Per-kernel device time of the robust step from torch.profiler (a separate, eager run, L2 overwritten before
     every step): median/threshold, K5, K6, homography selection, homography refit, decision.
  3. Host wall clock of RobustPoseEstimator.estimate_pose_batch on the 296 selected correspondence sets against a
     loop of 296 single estimate_pose calls (device sampler in both).

    python tools/robust_pose_rate.py --out robust_pose_rate.json [--pairs 296] [--reps 30]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "monocular-visual-slam_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

KERNELS = {"median_threshold": "displacement_median_kernel", "K5_homography_dlt": "homography_dlt_kernel",
           "K6_homography_score": "homography_score_kernel", "H_select": "homography_select_kernel",
           "H_refit": "refit_homography_kernel", "select_gates": "robust_pose_decide_kernel"}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                      # noqa: BLE001 — informational only
        import torch
        return {"name": torch.cuda.get_device_name(0), "error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=296)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--singles", type=int, default=296)
    ap.add_argument("--out", required=True, help="where the JSON result is written")
    a = ap.parse_args()

    import cv2
    import torch
    from b200slam import _capi, synthetic
    from b200slam.frontend import Frontend, FrontendConfig, PairBatch
    from b200slam.robust_pose import RobustPoseConfig, decode_results
    from integration import pose_bridge as pb

    _capi.require_cuda()
    torch.cuda.set_device(0)
    qs, ts, kq, kt = synthetic.tracking_pairs(a.pairs, n_desc=2000, seed=1234)
    b = PairBatch.from_host(qs, ts, kq, kt)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rcfg = RobustPoseConfig()

    def graph_time(fe):
        fe.run(b)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fe.run(b)
        g.replay()
        torch.cuda.synchronize()
        out = []
        for _ in range(a.reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            e1.synchronize()
            out.append(e0.elapsed_time(e1))
        return out

    fe_pose = Frontend(FrontendConfig(max_matches=500, hypotheses=2000, with_pose=True))
    fe_rob = Frontend(FrontendConfig(max_matches=500, hypotheses=2000, robust_pose=rcfg))
    t_pose, t_rob = [], []
    for _ in range(2):                                   # alternate the two variants
        t_pose += graph_time(fe_pose)
        t_rob += graph_time(fe_rob)

    # per-kernel device time of the robust step
    from torch.profiler import ProfilerActivity, profile
    steps = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            flush.zero_()
            fe_rob.run(b)
        torch.cuda.synchronize()
    per_kernel = {}
    for ev in prof.key_averages():
        per_kernel[ev.key] = getattr(ev, "device_time_total", 0) / 1000.0 / steps   # ms per step
    stages = {}
    for k, needle in KERNELS.items():
        hits = [v for name, v in per_kernel.items() if needle in name]
        stages[k] = round(sum(hits), 4) if hits else None
    top = sorted(((v, k) for k, v in per_kernel.items() if "Memset" not in k and "fill" not in k.lower()), reverse=True)[:12]

    # estimate_pose_batch against single calls on the selected correspondences
    res = fe_rob.run(b)
    cnt = res.sel.count.cpu().numpy()
    corr = res.sel.corr.cpu().numpy()
    stride = res.sel.stride
    kps = []
    for p in range(a.pairs):
        c = corr[p * stride:p * stride + cnt[p]]
        k1 = [cv2.KeyPoint(float(x), float(y), 1.0) for x, y in c[:, :2]]
        k2 = [cv2.KeyPoint(float(x), float(y), 1.0) for x, y in c[:, 2:]]
        kps.append((k1, k2, [cv2.DMatch(_queryIdx=j, _trainIdx=j, _distance=0.0) for j in range(len(k1))]))
    est = pb.RobustPoseEstimator(pb.RobustPoseEstimatorConfig())
    K = np.eye(3)
    args = ([k[0] for k in kps], [k[1] for k in kps], [k[2] for k in kps], K)
    est.estimate_pose_batch(*args, seed=1)
    t_batch = []
    for r in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = est.estimate_pose_batch(*args, seed=1)
        t_batch.append((time.perf_counter() - t0) * 1000)
    n_single = min(a.singles, a.pairs)
    try:                                              # warm the single path's lazily built objects
        est.estimate_pose(*kps[0], K)
    except Exception:                                 # noqa: BLE001
        pass
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for p in range(n_single):
        try:
            est.estimate_pose(*kps[p], K)
        except Exception:                             # noqa: BLE001 — gate failures are answers too
            pass
    t_single = (time.perf_counter() - t0) * 1000
    outcomes = {}
    for g in got:
        key = type(g).__name__ + ("/" + g.diagnostics.method if isinstance(g, pb.PoseEstimate) else
                                  "/" + g.reason if isinstance(g, pb.PoseEstimationFailure) else "")
        outcomes[key] = outcomes.get(key, 0) + 1
    rec = decode_results(res.robust.cpu().numpy())

    out = {
        "gpu": gpu_info(),
        "shape": {"pairs": a.pairs, "descriptors": 2000, "max_matches": 500, "hypotheses_E": 2000, "hypotheses_H": 2000,
                  "matches_mean": float(cnt.mean())},
        "step_ms": {"with_pose": {"median": float(np.median(t_pose)), "min": float(np.min(t_pose)), "n": len(t_pose)},
                    "robust_pose": {"median": float(np.median(t_rob)), "min": float(np.min(t_rob)), "n": len(t_rob)},
                    "timing": "CUDA-graph replay between CUDA events, 256 MB memset before every replay (L2 overwritten)"},
        "robust_stage_ms": stages,
        "robust_top_kernels_ms": [[k, round(v, 4)] for v, k in top],
        "dropin_wall_ms": {"estimate_pose_batch_median": float(np.median(t_batch)), "single_loop": t_single,
                           "single_calls": n_single, "pairs": a.pairs,
                           "single_loop_per_pair": t_single / n_single},
        "outcomes": outcomes,
        "frontend_methods": {"essential": int(((rec["outcome"] <= 1) & (rec["method"] == 0)).sum()),
                             "homography": int(((rec["outcome"] <= 1) & (rec["method"] == 1)).sum())},
    }
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(out, indent=1))
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
