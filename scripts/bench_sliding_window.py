"""Sliding-window inference over whole scans (csrc/windows.cu, LSSD3D.predict_scans), measured for two cases:
  C3: the 1ch 96^3 model on 1ch 192x224x192 scans, overlap 0.5 (36 windows per scan);
  C2: the 2ch 128^3 model on 2ch 256^3 scans, overlap 0.5 (27 windows per scan).

    python scripts/bench_sliding_window.py [--out profiles/r04_sliding_window.json] [--scans 8] [--rounds 3]

Per case, with the GPU's name and power limit read in the same run, the four measurements below are taken in
--rounds alternating rounds (median, min and max reported):
  1. predict_scans scans/s and ms per step (one scan per step, device-resident fp32 scans, host sync included);
  2. ssd3d_window_gather alone (CUDA events over 20 launches) with its algorithmic bytes and its rate;
  3. ssd3d_merge_windows alone on the step's own per-window detections (CUDA events over 50 launches);
  4. the same window batch through predict_step from a resident bf16 tensor: the network + per-window detect
     floor that the gather and the merge add to.
Random weights (synthetic.random_state_dict) on synthetic volumes; the network's time does not depend on them.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CASES = {"C3": dict(channels=1, window=(96, 96, 96), scan=(192, 224, 192)),
         "C2": dict(channels=2, window=(128, 128, 128), scan=(256, 256, 256))}
OVERLAP = 0.5


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else "unavailable"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "unavailable"
    return info


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def summary(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "runs": v}


def run_case(name, cfg, n_scans, rounds):
    from mslesions3d_b200 import ops, synthetic
    from mslesions3d_b200.data import window_origins
    from mslesions3d_b200.ssd3d import LSSD3D
    c, window, scan = cfg["channels"], cfg["window"], cfg["scan"]
    m = LSSD3D(n_classes=2, input_channels=c, input_size=window)
    m.load_state_dict(synthetic.random_state_dict(c, n_classes=2, seed=1))
    m = m.cuda().eval()
    nd, nh, nw, _ = window_origins(scan, window, OVERLAP)
    t_count = nd * nh * nw
    scans = torch.cat([torch.from_numpy(synthetic.make_batch(1, c, scan, first_idx=i)) for i in range(n_scans)]).cuda()
    win = ops.window_gather(scans[:1], window, OVERLAP)
    with torch.no_grad():
        m.predict_scans(scans, OVERLAP)                      # capture + warm-up of both plan slots
        m.predict_step({"img": win})
        plan = m._plan_for(scans[:1], 0, True, OVERLAP)
        wo = plan.out
        ws = torch.empty_like(plan.merge_ws)
        out = {"scans_per_s": [], "ms_per_step": [], "gather_ms": [], "merge_ms": [], "predict_step_windows_ms": []}
        for _ in range(rounds):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                m.predict_scans(scans, OVERLAP)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / (3 * n_scans)
            out["scans_per_s"].append(1.0 / dt)
            out["ms_per_step"].append(dt * 1e3)
            out["gather_ms"].append(event_ms(lambda: ops.window_gather(scans[:1], window, OVERLAP, out=win), 20))
            out["merge_ms"].append(event_ms(lambda: ops.merge_windows(
                wo.boxes, wo.scores, wo.labels, wo.count, 1, scan, window, OVERLAP, 2, m.min_score, m.max_overlap,
                m.top_k, offset=plan.offset, workspace=ws), 50))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(10):
                m.predict_step({"img": win})
            torch.cuda.synchronize()
            out["predict_step_windows_ms"].append((time.perf_counter() - t0) / 10 * 1e3)
    # bytes the gather has to move: read each scan voxel the windows cover (fp32), write every window voxel (bf16)
    read_b = 4 * c * scan[0] * scan[1] * scan[2]
    write_b = 2 * c * t_count * window[0] * window[1] * window[2]
    res = {k: summary(v) for k, v in out.items()}
    res["windows_per_scan"] = t_count
    res["gather_bytes"] = {"read_scan": read_b, "write_windows": write_b}
    res["gather_GB_per_s"] = (read_b + write_b) / (res["gather_ms"]["median"] * 1e-3) / 1e9
    res["gather_share_of_step"] = res["gather_ms"]["median"] / res["ms_per_step"]["median"]
    res["merge_share_of_step"] = res["merge_ms"]["median"] / res["ms_per_step"]["median"]
    res["config"] = {"channels": c, "window": window, "scan": scan, "overlap": OVERLAP, "n_classes": 2,
                     "min_score": m.min_score, "top_k": m.top_k, "scans_timed": n_scans}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_sliding_window.json"))
    ap.add_argument("--scans", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sliding_window.py measures the GPU; no CUDA device found")
    res = {"gpu": gpu_info()}
    for name, cfg in CASES.items():
        res[name] = run_case(name, cfg, args.scans, args.rounds)
        print(name, json.dumps({k: res[name][k] for k in ("scans_per_s", "ms_per_step", "gather_ms", "merge_ms",
                                                          "predict_step_windows_ms")}), flush=True)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
