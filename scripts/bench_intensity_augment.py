"""MR intensity augmentation (ssd3d_augment_intensity_batch, Augment.bias_prob / gamma_prob / noise_prob) measured at
C3: 1ch 96^3 output, batch 16, fp32 sources of 96^3 (1024 volumes, 3.6 GB, larger than L2).

    python scripts/bench_intensity_augment.py [--out profiles/r07_intensity_augment.json]

Reports, with the GPU's name and power limit read in the same run:
  1. the pass alone (its two launches between a pair of CUDA events, on the batch ssd3d_augment_batch has just
     written, as in the training step; median and mean over 200 batches) with gamma, the bias field and the noise
     each on its own and all three together (probability 1), alternating over 3 rounds in one process;
  2. fit_epoch ms per step with bench_data_pipeline.py's full set plus the MR set (probabilities 0.5), against the
     full set alone, alternating (3 rounds);
  3. the per-kernel split of one MR epoch from torch.profiler (a separate pass, after the timings).
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from bench_data_pipeline import BATCH, COPY_PEAK, N_DATA, SIZE, epoch_leg, gpu_info, make_dataset, model  # noqa: E402

STRENGTH = dict(bias_coefficient=0.5, gamma_log_range=0.3, noise_std=0.1)
PASSES = {"gamma": dict(gamma_prob=1.0), "bias": dict(bias_prob=1.0), "noise": dict(noise_prob=1.0),
          "all_three": dict(bias_prob=1.0, gamma_prob=1.0, noise_prob=1.0)}


def pass_us(ds, aug, iters=200):
    """The pass's device time per batch: each of ``iters`` batches is written by ssd3d_augment_batch (outside the
    events), then the pass runs between two events."""
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import epoch_order
    order = epoch_order(len(ds), 0, aug.seed).cuda()
    state = torch.tensor([aug.seed, 0, 0, 0, 1, 0, 0, 0], dtype=torch.int64, device="cuda")
    out = (torch.empty((BATCH, 1, *SIZE), dtype=torch.bfloat16, device="cuda"),
           torch.empty((BATCH, *SIZE), dtype=torch.uint8, device="cuda"),
           torch.empty((BATCH, 16), dtype=torch.int32, device="cuda"))
    rec = torch.empty((BATCH, 27), dtype=torch.int32, device="cuda")
    ws = torch.empty((ops.augment_intensity_workspace_bytes(BATCH, 1, *SIZE),), dtype=torch.uint8, device="cuda")

    def batch():
        ops.augment_batch(ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, BATCH, SIZE, aug.pos_ratio,
                          aug.flip_prob, aug.rot90_prob, aug.rot90_axes, aug.scale, aug.shift, out=out)

    def run():
        ops.augment_intensity_batch(out[0], state, BATCH, aug.bias_prob, aug.bias_coefficient, aug.gamma_prob,
                                    aug.gamma_log_range, aug.noise_prob, aug.noise_std, out_record=rec, workspace=ws)
    for _ in range(5):
        batch()
        run()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for e0, e1 in ev:
        batch()
        e0.record()
        run()
        e1.record()
    torch.cuda.synchronize()
    t = [e0.elapsed_time(e1) * 1000.0 for e0, e1 in ev]
    return statistics.median(t), statistics.fmean(t)


def passes(ds, base, rounds=3):
    legs = {name: dataclasses.replace(base, **kw, **STRENGTH) for name, kw in PASSES.items()}
    med = {name: [] for name in legs}
    mean = {name: [] for name in legs}
    for _ in range(rounds):
        for name, aug in legs.items():
            m, a = pass_us(ds, aug)
            med[name].append(m)
            mean[name].append(a)
    nbytes = BATCH * SIZE[0] * SIZE[1] * SIZE[2] * 2 * 2               # bf16 batch read and written once
    res = {"rounds_median_us": med, "rounds_mean_us": mean,
           "median_us": {name: statistics.median(v) for name, v in med.items()},
           "algorithmic_bytes": nbytes, "copy_peak_floor_us": nbytes / COPY_PEAK * 1e6, "batches_per_round": 200,
           "augment": {name: repr(aug) for name, aug in legs.items()}}
    return res


def kernel_split(ds, aug):
    """torch.profiler over one epoch of the captured step: CUDA time per kernel family, per step."""
    from torch.profiler import ProfilerActivity, profile
    m = model("cuda")
    m.fit_epoch(ds, BATCH, aug, epoch=0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.fit_epoch(ds, BATCH, aug, epoch=1)
        torch.cuda.synchronize()
    n = -(-len(ds) // BATCH)
    fam = {"intensity_slot_kernel": 0.0, "intensity_voxel_kernel": 0.0, "augment_kernel": 0.0,
           "gt_extraction (cc_*)": 0.0, "gt_pack_kernel": 0.0, "all kernels": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if ev.key.startswith("cuda") or "Memcpy" in ev.key or "Memset" in ev.key or not t:
            continue
        fam["all kernels"] += t
        for k in ("intensity_slot_kernel", "intensity_voxel_kernel", "gt_pack_kernel"):
            if k in ev.key:
                fam[k] += t
        if "augment_kernel<" in ev.key:
            fam["augment_kernel"] += t
        elif "cc_" in ev.key:
            fam["gt_extraction (cc_*)"] += t
    return {k + "_us_per_step": v / n for k, v in fam.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_intensity_augment.json"))
    ap.add_argument("--data", type=int, default=N_DATA)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_intensity_augment needs a CUDA device")
    from mslesions3d_b200 import _lib
    from mslesions3d_b200.data import Augment
    _lib.load()
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "config": {"volume": list(SIZE), "channels": 1, "batch": BATCH, "data_set": args.data}}
    full = Augment(pos_ratio=0.5, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1, seed=1)
    ds = make_dataset(args.data, SIZE)
    res["pass_96"] = passes(ds, full)
    mr = dataclasses.replace(full, bias_prob=0.5, gamma_prob=0.5, noise_prob=0.5, **STRENGTH)
    for r in range(3):                                                   # alternating: the spread of the comparison
        res["fit_epoch_full_set_%d" % r] = epoch_leg(ds, full)
        res["fit_epoch_full_set_mr_%d" % r] = epoch_leg(ds, mr)
    res["kernel_split_full_set_mr"] = kernel_split(ds, mr)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
