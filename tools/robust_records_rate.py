#!/usr/bin/env python
"""Rate of the robust pose step when its answer leaves the GPU in the result records (pose records, include/b2s.h).

  1. The 296-pair robust launch set (BASELINE config #2 shape: 2000 x 2000 descriptors per pair, 500 matches, 2000
     hypotheses for each of E and H) with and without records: CUDA-graph replay between CUDA events, L2 overwritten
     (256 MB memset) before every replay, the two variants alternated.
  2. SequencePipeline(schedule="interleaved") end to end at the config #2 shape (297 frames x 2000 descriptors,
     S = 500, depth 3): every step uploads its frames from pinned host memory, runs the kernels as one CUDA graph and
     downloads its records in one copy; with robust_pose (pose records) and without (the plain essential step),
     alternated in the same process.  pairs/s over K steps between CUDA events; bytes down per step.

The device name and power limit are read in the same run.

    python tools/robust_records_rate.py --out profiles/r04_robust_records.json [--reps 30] [--steps 40] [--rounds 3]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "monocular-visual-slam_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        info.update(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as exc:                      # noqa: BLE001 — informational only
        info["error"] = str(exc)
    return info


def stats(ms):
    return {"median": float(np.median(ms)), "min": float(np.min(ms)), "max": float(np.max(ms)), "n": len(ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=296)
    ap.add_argument("--reps", type=int, default=30, help="graph replays per variant and round (step timing)")
    ap.add_argument("--steps", type=int, default=40, help="pipeline steps per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the variants")
    ap.add_argument("--out", required=True, help="where the JSON result is written")
    a = ap.parse_args()

    import torch
    from b200slam import _capi, synthetic
    from b200slam.frontend import Frontend, FrontendConfig, PairBatch, SequencePipeline, pose_record_bytes
    from b200slam.robust_pose import RobustPoseConfig, decode_results

    _capi.require_cuda()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # normalised keypoints with K = I: the reference's essential path is only self-consistent there, so the estimator
    # gives real answers (at pixel scale nearly every pair ends in the essential branch's error); min_parallax = 0
    # because normalised displacements are far below the default 1.0 gate
    K = None
    rcfg = RobustPoseConfig(min_parallax=0.0)
    S, H, N, P = 500, 2000, 2000, a.pairs

    # ---- 1. the robust launch set with and without records -----------------------------------------------
    qs, ts, kq, kt = synthetic.tracking_pairs(P, n_desc=N, seed=1234)
    b = PairBatch.from_host(qs, ts, kq, kt)
    rec = torch.zeros((P, pose_record_bytes(S)), dtype=torch.uint8, device=dev)
    graphs = {}
    for name, records in (("without_records", None), ("with_records", rec)):
        fe = Frontend(FrontendConfig(max_matches=S, hypotheses=H, robust_pose=rcfg))
        fe.run(b, K=K, records=records)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            res = fe.run(b, K=K, records=records)
        g.replay()
        torch.cuda.synchronize()
        graphs[name] = (g, fe, res)
    same = (graphs["with_records"][2].robust.cpu().numpy().tobytes() == graphs["without_records"][2].robust.cpu().numpy().tobytes())
    step_ms = {k: [] for k in graphs}
    for _ in range(a.rounds):
        for name, (g, _, _) in graphs.items():
            for _ in range(a.reps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g.replay()
                e1.record()
                e1.synchronize()
                step_ms[name].append(e0.elapsed_time(e1))
    r = decode_results(graphs["with_records"][2].robust.cpu().numpy())
    outcomes = {"estimate_essential": int(((r["outcome"] == 0) & (r["method"] == 0)).sum()),
                "estimate_homography": int(((r["outcome"] == 0) & (r["method"] == 1)).sum()),
                "gate_failed": int((r["outcome"] == 1).sum()), "error": int((r["outcome"] >= 2).sum())}
    del graphs

    # ---- 2. SequencePipeline end to end, robust against plain, alternated -------------------------------------
    F = P + 1
    desc, kp = synthetic.tracking_sequence(F, N, seed=77)
    d_host = torch.from_numpy(desc.reshape(-1, 32)).pin_memory()
    k_host = torch.from_numpy(kp.reshape(-1, 2)).pin_memory()
    counts = np.full(F, N, np.int32)
    pipes = {"robust_pose": SequencePipeline(F, N, FrontendConfig(max_matches=S, hypotheses=H, robust_pose=rcfg), depth=3,
                                             schedule="interleaved", K=K),
             "plain": SequencePipeline(F, N, FrontendConfig(max_matches=S, hypotheses=H), depth=3, schedule="interleaved", K=K)}

    def timed(pipe, steps):
        main = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for st in pipe.streams():
            st.wait_event(e0)
        for _ in range(steps):
            pipe.submit(d_host, k_host, counts)
        for st in pipe.streams():
            main.wait_stream(st)
        e1.record(main)
        e1.synchronize()
        return e0.elapsed_time(e1)

    for pipe in pipes.values():                               # warm-up: batches, graphs of every slot
        timed(pipe, 6)
    e2e = {k: [] for k in pipes}
    for _ in range(a.rounds):
        for name, pipe in pipes.items():
            ms = timed(pipe, a.steps)
            e2e[name].append(P * a.steps / (ms * 1e-3))
    view = pipes["robust_pose"].result(0)
    robust_view = view["robust"]

    out = {
        "gpu": gpu_info(),
        "shape": {"pairs": P, "descriptors": N, "max_matches": S, "hypotheses_E": H, "hypotheses_H": H,
                  "keypoints": "synthetic tracking data, normalised coordinates, K = I",
                  "robust_config": "RobustPoseConfig(min_parallax=0.0)"},
        "robust_step_ms": {**{k: stats(v) for k, v in step_ms.items()},
                           "timing": "CUDA-graph replay between CUDA events, 256 MB memset before every replay (L2 "
                                     "overwritten); the two variants alternated", "results_identical": bool(same),
                           "outcomes": outcomes},
        "sequence_pipeline": {
            "schedule": "interleaved", "depth": 3, "frames": F, "steps_per_window": a.steps, "windows": a.rounds,
            "pairs_per_s": {k: {"per_window": [round(x, 1) for x in v], "median": float(np.median(v))} for k, v in e2e.items()},
            "bytes_down_per_step": {k: int(p.d2h_bytes) for k, p in pipes.items()},
            "record_bytes": {k: int(p.rec_bytes) for k, p in pipes.items()},
            "bytes_up_per_step": int(pipes["plain"].h2d_bytes),
            "robust_outcomes_last_step": {"estimate": int((robust_view["outcome"] == 0).sum()),
                                          "gate_failed": int((robust_view["outcome"] == 1).sum()),
                                          "error": int((robust_view["outcome"] >= 2).sum())},
            "timing": "one CUDA event pair around K submits (uploads, graph replays, downloads all inside)"},
    }
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(out, indent=1))
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
