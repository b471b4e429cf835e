"""Training from a device-resident data set (csrc/augment.cu, data.py, LSSD3D.fit_epoch), measured at C3: 1ch 96^3
volumes, batch 16, a data set of 1024 volumes from ops.generate_volumes.

    python scripts/bench_data_pipeline.py [--out profiles/r03_data_pipeline.json] [--loss-steps 300]

Reports, with the GPU's name and power limit read in the same run:
  1. ssd3d_augment_batch time (CUDA events over 200 launches) with its algorithmic bytes and its share of the
     copy-peak floor, for a 96^3 source (all augmentations on, rot90 in the H-W plane so that W moves) and a 128^3
     source cropped to 96^3; the sources are larger than L2 (3.6 GB / 0.5 GB), slots draw different subjects;
  2. GT extraction + pack time on the augmented masks (same method);
  3. fit_epoch ms per step with Augment() and with every augmentation on, and the host-staged fit_step loop
     exactly as bench.py's training leg runs it (3 rotating device-resident batches), in the same process;
  4. kernel launches per step of each;
  5. the loss of the first --loss-steps steps with every augmentation on (recorded, not asserted);
  and the per-kernel split of one augmented epoch from torch.profiler (a separate pass, after the timings).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

COPY_PEAK = 7.7e12       # B/s, HBM3e of one B200 (data sheet); a floor, not a measured rate
SIZE, BATCH, N_DATA = (96, 96, 96), 16, 1024


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


def make_dataset(n, size, seed=0):
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import DeviceDataset
    parts_img, parts_mask = [], []
    for i in range(0, n, 128):
        raw, mask, _, _ = ops.generate_volumes(min(128, n - i), 1, size, i, seed, (1, 5), (6, 14))
        parts_img.append(raw)
        parts_mask.append(mask)
    return DeviceDataset.from_arrays(torch.cat(parts_img), torch.cat(parts_mask))


def augment_kernel(ds, aug, iters=200):
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import epoch_order
    order = epoch_order(len(ds), 0, aug.seed).cuda()
    state = torch.tensor([aug.seed, 0, 0, 0, 1, 0, 0, 0], dtype=torch.int64, device="cuda")
    out = (torch.empty((BATCH, 1, *SIZE), dtype=torch.bfloat16, device="cuda"),
           torch.empty((BATCH, *SIZE), dtype=torch.uint8, device="cuda"),
           torch.empty((BATCH, 16), dtype=torch.int32, device="cuda"))

    def run():
        ops.augment_batch(ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, BATCH, SIZE, aug.pos_ratio,
                          aug.flip_prob, aug.rot90_prob, aug.rot90_axes, aug.scale, aug.shift, out=out)
    for _ in range(5):
        run()
    torch.cuda.synchronize()
    ms = event_ms(run, iters)
    vox = BATCH * SIZE[0] * SIZE[1] * SIZE[2]
    nbytes = vox * (ds.images.element_size() + 1 + 2 + 1)      # image read, mask read, bf16 write, mask write
    floor_us = nbytes / COPY_PEAK * 1e6
    return {"us": ms * 1000.0, "algorithmic_bytes": nbytes, "copy_peak_floor_us": floor_us,
            "fraction_of_floor": floor_us / (ms * 1000.0), "source": list(ds.shape), "augment": repr(aug)}, out[1]


def gt_extract_pack(masks, per_volume=64, iters=200):
    from mslesions3d_b200 import _lib, ops
    n = masks.shape[0]
    gt_out = (torch.empty((n, per_volume, 6), dtype=torch.float32, device="cuda"),
              torch.empty((n, per_volume), dtype=torch.int64, device="cuda"),
              torch.empty((2, n), dtype=torch.int32, device="cuda"))
    ws = torch.empty((_lib.load().ssd3d_gt_boxes_workspace_bytes(n, *SIZE, per_volume),), dtype=torch.uint8,
                     device="cuda")
    packed = (torch.empty((n * per_volume, 6), device="cuda"), torch.empty((n * per_volume,), dtype=torch.int64,
                                                                            device="cuda"),
              torch.empty((n + 1,), dtype=torch.int32, device="cuda"))
    status = torch.zeros((2,), dtype=torch.int32, device="cuda")

    def extract():
        ops.gt_boxes_padded(masks, 0, per_volume, out=gt_out, workspace=ws)

    def both():
        extract()
        ops.gt_pack(*gt_out, per_volume, out=packed, status=status)
    for _ in range(5):
        both()
    torch.cuda.synchronize()
    return {"extract_us": event_ms(extract, iters) * 1000.0, "extract_and_pack_us": event_ms(both, iters) * 1000.0,
            "overflowing_batches": int(status[1].item())}


def model(dev):
    from mslesions3d_b200 import synthetic
    from mslesions3d_b200.ssd3d import LSSD3D
    m = LSSD3D(n_classes=2, input_channels=1, input_size=SIZE, threshold=[0.1, 0.2], lr=1e-4)
    m.load_state_dict(synthetic.random_state_dict(1, seed=0))
    return m.to(dev).train()


def epoch_leg(ds, aug, epochs=3):
    from mslesions3d_b200 import ops
    m = model("cuda")
    m.fit_epoch(ds, BATCH, aug, epoch=0)                      # capture + one epoch of warm-up
    torch.cuda.synchronize()
    plan = [p for k, p in m.train_engine().plans.items() if k[0] == "epoch"][0]
    steps = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for ep in range(1, 1 + epochs):
        losses, _ = m.fit_epoch(ds, BATCH, aug, epoch=ep)
        steps += losses.shape[0]
    e1.record()
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) * 1000.0
    ms = e0.elapsed_time(e1)
    return {"ms_per_step": ms / steps, "host_ms_per_step": host / steps, "steps": steps,
            "volumes_per_s": BATCH * steps / (ms / 1000.0), "launches_per_step": plan.n_kernels,
            "skipped_steps": m.fit_skipped_steps(), "augment": repr(aug)}


def host_staged_leg(steps=192):
    """bench.py's training leg: fit_step over 3 rotating device-resident fp32 batches from synthetic.make_batch."""
    from mslesions3d_b200 import ops, synthetic
    dev = torch.device("cuda")
    m = model(dev)
    batches = []
    for r in range(3):
        x, b, l = synthetic.make_batch(BATCH, 1, SIZE, first_idx=r * BATCH, with_boxes=True)
        batches.append({"img": torch.from_numpy(x).to(dev), "boxes": [torch.from_numpy(v).to(dev) for v in b],
                        "labels": [torch.from_numpy(v).to(dev) for v in l]})
    for i in range(3):
        m.fit_step(batches[i % 3])
    torch.cuda.synchronize()
    ops.LAUNCHES[0] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(steps):
        m.fit_step(batches[i % 3])
    e1.record()
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) * 1000.0
    ms = e0.elapsed_time(e1)
    return {"ms_per_step": ms / steps, "host_ms_per_step": host / steps, "steps": steps,
            "volumes_per_s": BATCH * steps / (ms / 1000.0), "launches_per_step": ops.LAUNCHES[0] / steps}


def loss_curve(ds, aug, n_steps):
    m = model("cuda")
    out, ep = [], 0
    while len(out) < n_steps:
        losses, _ = m.fit_epoch(ds, BATCH, aug, epoch=ep)
        out.extend([[float(a), float(b)] for a, b in losses.cpu().tolist()])
        ep += 1
    return {"losses_conf_loc": out[:n_steps], "skipped_steps": m.fit_skipped_steps(), "augment": repr(aug)}


def kernel_split(ds, aug, steps=32):
    """torch.profiler over ``steps`` replays of the augmented epoch step: CUDA time per kernel family."""
    from torch.profiler import ProfilerActivity, profile
    m = model("cuda")
    m.fit_epoch(ds, BATCH, aug, epoch=0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.fit_epoch(ds, BATCH, aug, epoch=1)
        torch.cuda.synchronize()
    n = -(-len(ds) // BATCH)
    fam = {"augment_kernel": 0.0, "gt_extraction (cc_*)": 0.0, "gt_pack_kernel": 0.0, "all kernels": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if ev.key.startswith("cuda") or "Memcpy" in ev.key or "Memset" in ev.key or not t:
            continue
        fam["all kernels"] += t
        if "augment_kernel" in ev.key:
            fam["augment_kernel"] += t
        elif "cc_" in ev.key:
            fam["gt_extraction (cc_*)"] += t
        elif "gt_pack_kernel" in ev.key:
            fam["gt_pack_kernel"] += t
    return {k + "_us_per_step": v / n for k, v in fam.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_data_pipeline.json"))
    ap.add_argument("--loss-steps", type=int, default=300)
    ap.add_argument("--data", type=int, default=N_DATA)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_data_pipeline needs a CUDA device")
    from mslesions3d_b200 import _lib
    from mslesions3d_b200.data import Augment
    _lib.load()
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "config": {"volume": list(SIZE), "channels": 1, "batch": BATCH, "data_set": args.data,
                                         "copy_peak_Bps": COPY_PEAK}}
    ds96 = make_dataset(args.data, SIZE)
    full = Augment(pos_ratio=0.5, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1, seed=1)
    res["augment_96"], masks = augment_kernel(ds96, full)
    ds128 = make_dataset(64, (128, 128, 128), seed=1)
    res["augment_128_crop"], _ = augment_kernel(ds128, full)
    del ds128
    res["gt_extract_pack"] = gt_extract_pack(masks)
    res["host_staged_fit_step"] = host_staged_leg()
    res["fit_epoch_identity"] = epoch_leg(ds96, Augment())
    res["fit_epoch_all_augment"] = epoch_leg(ds96, full)
    res["host_staged_fit_step_again"] = host_staged_leg()          # the spread of the comparison
    res["loss_curve_all_augment"] = loss_curve(ds96, full, args.loss_steps)
    res["kernel_split_all_augment"] = kernel_split(ds96, full)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    brief = {k: v for k, v in res.items() if k != "loss_curve_all_augment"}
    print(json.dumps(brief, indent=1))


if __name__ == "__main__":
    main()
