"""Elastic deformation (ssd3d_augment_elastic_batch, Augment.elastic_prob) measured at C3: 1ch 96^3 output, batch 16,
fp32 sources of 96^3 (1024 volumes, 3.6 GB, larger than L2) and 128^3 (64 volumes).

    python scripts/bench_elastic_augment.py [--out profiles/r06_elastic_augment.json]

Reports, with the GPU's name and power limit read in the same run:
  1. per source size, four kernels on bench_data_pipeline.py's full set, alternating over 3 rounds of 200 launches
     in one process (CUDA events, median): the elastic kernel (elastic_prob = 1, 7 control points and 4 voxels of
     displacement per axis) with the affine (affine_prob = 1, rotate_range = 0.26 rad, zoom_range = 0.1) and
     without it, the affine kernel with that affine, and ssd3d_augment_batch;
  2. fit_epoch ms per step with the full set plus the field (elastic_prob = 1, the same field), against the full
     set alone, alternating (2 rounds);
  3. the per-kernel split of one elastic epoch from torch.profiler (a separate pass, after the timings).
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

from bench_data_pipeline import BATCH, N_DATA, SIZE, epoch_leg, event_ms, gpu_info, make_dataset, model  # noqa: E402


def launcher(ds, aug, kind):
    """A closure that launches one batch of ``kind`` ("elastic", "affine" or "batch") into fixed outputs."""
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import epoch_order
    order = epoch_order(len(ds), 0, aug.seed).cuda()
    state = torch.tensor([aug.seed, 0, 0, 0, 1, 0, 0, 0], dtype=torch.int64, device="cuda")
    out = (torch.empty((BATCH, 1, *SIZE), dtype=torch.bfloat16, device="cuda"),
           torch.empty((BATCH, *SIZE), dtype=torch.uint8, device="cuda"),
           torch.empty((BATCH, {"elastic": 33, "affine": 32, "batch": 16}[kind]), dtype=torch.int32, device="cuda"))
    args = (ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, BATCH, SIZE, aug.pos_ratio, aug.flip_prob,
            aug.rot90_prob, aug.rot90_axes, aug.scale, aug.shift)
    if kind == "elastic":
        return lambda: ops.augment_elastic_batch(*args, aug.affine_prob, aug.rotate_range, aug.zoom_range,
                                                 aug.elastic_prob, aug.elastic_points, aug.elastic_magnitude, out=out)
    if kind == "affine":
        return lambda: ops.augment_affine_batch(*args, aug.affine_prob, aug.rotate_range, aug.zoom_range, out=out)
    return lambda: ops.augment_batch(*args, out=out)


def kernels(ds, legs, rounds=3, iters=200):
    """{name: (kind, Augment)} timed round-robin, ``rounds`` times ``iters`` launches each."""
    runs = {name: launcher(ds, aug, kind) for name, (kind, aug) in legs.items()}
    for run in runs.values():
        for _ in range(5):
            run()
    torch.cuda.synchronize()
    times = {name: [] for name in runs}
    for _ in range(rounds):
        for name, run in runs.items():
            times[name].append(event_ms(run, iters) * 1000.0)
    res = {name + "_us": t for name, t in times.items()}
    res.update({"median_" + name + "_us": statistics.median(t) for name, t in times.items()})
    res.update({"launches_per_round": iters, "source": list(ds.shape),
                "augment": {name: repr(aug) for name, (_, aug) in legs.items()}})
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
    fam = {"augment_elastic (augment_affine_kernel<T, true>)": 0.0, "gt_extraction (cc_*)": 0.0,
           "gt_pack_kernel": 0.0, "all kernels": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if ev.key.startswith("cuda") or "Memcpy" in ev.key or "Memset" in ev.key or not t:
            continue
        fam["all kernels"] += t
        if "augment_affine_kernel<" in ev.key and ", true>" in ev.key:
            fam["augment_elastic (augment_affine_kernel<T, true>)"] += t
        elif "gt_pack_kernel" in ev.key:
            fam["gt_pack_kernel"] += t
        elif "cc_" in ev.key:
            fam["gt_extraction (cc_*)"] += t
    return {k + "_us_per_step": v / n for k, v in fam.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_elastic_augment.json"))
    ap.add_argument("--data", type=int, default=N_DATA)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_elastic_augment needs a CUDA device")
    from mslesions3d_b200 import _lib
    from mslesions3d_b200.data import Augment
    _lib.load()
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "config": {"volume": list(SIZE), "channels": 1, "batch": BATCH, "data_set": args.data}}
    full = Augment(pos_ratio=0.5, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1, seed=1)
    affine = dataclasses.replace(full, affine_prob=1.0, rotate_range=(0.26,) * 3, zoom_range=(0.1,) * 3)
    field = dict(elastic_prob=1.0, elastic_points=(7, 7, 7), elastic_magnitude=(4.0, 4.0, 4.0))
    legs = {"elastic_with_affine": ("elastic", dataclasses.replace(affine, **field)),
            "elastic_without_affine": ("elastic", dataclasses.replace(full, **field)),
            "affine_kernel": ("affine", affine), "augment_batch": ("batch", full)}
    ds96 = make_dataset(args.data, SIZE)
    res["kernels_96"] = kernels(ds96, legs)
    ds128 = make_dataset(64, (128, 128, 128), seed=1)
    res["kernels_128_crop"] = kernels(ds128, legs)
    del ds128
    elastic_full = dataclasses.replace(full, **field)
    for r in range(2):                                                   # alternating: the spread of the comparison
        res["fit_epoch_full_set_%d" % r] = epoch_leg(ds96, full)
        res["fit_epoch_full_set_elastic_%d" % r] = epoch_leg(ds96, elastic_full)
    res["kernel_split_full_set_elastic"] = kernel_split(ds96, elastic_full)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
