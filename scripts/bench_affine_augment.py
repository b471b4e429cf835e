"""Rotation / zoom augmentation (ssd3d_augment_affine_batch, Augment.affine_prob) measured at C3: 1ch 96^3 output,
batch 16, fp32 sources of 96^3 (1024 volumes, 3.6 GB, larger than L2) and 128^3 (64 volumes).

    python scripts/bench_affine_augment.py [--out profiles/r05_affine_augment.json] [--loss-steps 300]

Reports, with the GPU's name and power limit read in the same run:
  1. the affine kernel's time (CUDA events over 200 launches) with every augmentation of
     bench_data_pipeline.py's full set plus affine_prob = 1, rotate_range = 0.26 rad and zoom_range = 0.1 per axis,
     its algorithmic bytes and its share of the copy-peak floor (as bench_data_pipeline.py counts them: one
     source read per output voxel, although trilinear taps read up to eight);
  2. the affine kernel with affine_prob = 0 against ssd3d_augment_batch on the same affine-free workload,
     alternating over 3 rounds in one process (median): which of the two kernels an affine-free epoch should run;
  3. fit_epoch ms per step with the affine, with the full set and with Augment(), in the same process;
  4. the per-kernel split of one affine epoch from torch.profiler (a separate pass, after the timings);
  5. the first --loss-steps losses with the affine on (recorded, not asserted).
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

from bench_data_pipeline import (BATCH, COPY_PEAK, N_DATA, SIZE, epoch_leg, event_ms, gpu_info,  # noqa: E402
                                 loss_curve, make_dataset, model)


def launcher(ds, aug, affine):
    """A closure that launches one batch (the affine kernel or ssd3d_augment_batch) into fixed outputs."""
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import epoch_order
    order = epoch_order(len(ds), 0, aug.seed).cuda()
    state = torch.tensor([aug.seed, 0, 0, 0, 1, 0, 0, 0], dtype=torch.int64, device="cuda")
    out = (torch.empty((BATCH, 1, *SIZE), dtype=torch.bfloat16, device="cuda"),
           torch.empty((BATCH, *SIZE), dtype=torch.uint8, device="cuda"),
           torch.empty((BATCH, 32 if affine else 16), dtype=torch.int32, device="cuda"))
    args = (ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, BATCH, SIZE, aug.pos_ratio, aug.flip_prob,
            aug.rot90_prob, aug.rot90_axes, aug.scale, aug.shift)
    if affine:
        return lambda: ops.augment_affine_batch(*args, aug.affine_prob, aug.rotate_range, aug.zoom_range, out=out)
    return lambda: ops.augment_batch(*args, out=out)


def kernel_time(ds, aug, affine, iters=200):
    run = launcher(ds, aug, affine)
    for _ in range(5):
        run()
    torch.cuda.synchronize()
    ms = event_ms(run, iters)
    vox = BATCH * SIZE[0] * SIZE[1] * SIZE[2]
    nbytes = vox * (ds.images.element_size() + 1 + 2 + 1)      # image read, mask read, bf16 write, mask write
    floor_us = nbytes / COPY_PEAK * 1e6
    return {"us": ms * 1000.0, "launches": iters, "algorithmic_bytes": nbytes, "copy_peak_floor_us": floor_us,
            "fraction_of_floor": floor_us / (ms * 1000.0), "source": list(ds.shape), "augment": repr(aug)}


def alternate(ds, aug, rounds=3, iters=200):
    """ssd3d_augment_batch and the affine kernel with affine_prob = 0 on the same workload, alternating."""
    old, new = launcher(ds, aug, False), launcher(ds, dataclasses.replace(aug, affine_prob=0.0), True)
    for run in (old, new):
        for _ in range(5):
            run()
    torch.cuda.synchronize()
    t_old, t_new = [], []
    for _ in range(rounds):
        t_old.append(event_ms(old, iters) * 1000.0)
        t_new.append(event_ms(new, iters) * 1000.0)
    return {"augment_batch_us": t_old, "affine_kernel_prob0_us": t_new,
            "median_augment_batch_us": statistics.median(t_old),
            "median_affine_kernel_prob0_us": statistics.median(t_new), "launches_per_round": iters,
            "source": list(ds.shape), "augment": repr(aug)}


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
    fam = {"augment_affine_kernel": 0.0, "augment_kernel": 0.0, "gt_extraction (cc_*)": 0.0, "gt_pack_kernel": 0.0,
           "all kernels": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if ev.key.startswith("cuda") or "Memcpy" in ev.key or "Memset" in ev.key or not t:
            continue
        fam["all kernels"] += t
        for k in ("augment_affine_kernel", "augment_kernel", "gt_pack_kernel"):
            if k + "<" in ev.key or ev.key.endswith(k) or (k + "(") in ev.key:
                fam[k] += t
                break
        else:
            if "cc_" in ev.key:
                fam["gt_extraction (cc_*)"] += t
    return {k + "_us_per_step": v / n for k, v in fam.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_affine_augment.json"))
    ap.add_argument("--loss-steps", type=int, default=300)
    ap.add_argument("--data", type=int, default=N_DATA)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_affine_augment needs a CUDA device")
    from mslesions3d_b200 import _lib
    from mslesions3d_b200.data import Augment
    _lib.load()
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "config": {"volume": list(SIZE), "channels": 1, "batch": BATCH, "data_set": args.data,
                                         "copy_peak_Bps": COPY_PEAK}}
    full = Augment(pos_ratio=0.5, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1, seed=1)
    affine = dataclasses.replace(full, affine_prob=1.0, rotate_range=(0.26,) * 3, zoom_range=(0.1,) * 3)
    ds96 = make_dataset(args.data, SIZE)
    res["affine_96"] = kernel_time(ds96, affine, True)
    res["prob0_vs_augment_batch_96"] = alternate(ds96, full)
    ds128 = make_dataset(64, (128, 128, 128), seed=1)
    res["affine_128_crop"] = kernel_time(ds128, affine, True)
    res["prob0_vs_augment_batch_128_crop"] = alternate(ds128, full)
    del ds128
    res["fit_epoch_identity"] = epoch_leg(ds96, Augment())
    res["fit_epoch_full_set"] = epoch_leg(ds96, full)
    res["fit_epoch_affine"] = epoch_leg(ds96, affine)
    res["fit_epoch_full_set_again"] = epoch_leg(ds96, full)           # the spread of the comparison
    res["kernel_split_affine"] = kernel_split(ds96, affine)
    res["loss_curve_affine"] = loss_curve(ds96, affine, args.loss_steps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "loss_curve_affine"}, indent=1))


if __name__ == "__main__":
    main()
