#!/usr/bin/env python
"""Profiling driver for ncu: the C2 inference step (2ch 128^3, batch 8) launched kernel by kernel (no CUDA graph),
and optionally the C3 training step, with the region of interest inside an NVTX range "prof".

    python scripts/prof_kernels.py [--train] [--steps 2]
    ncu --set full --clock-control none --import-source on --nvtx --nvtx-include "prof/" -o gpurun_out/prof \
        python scripts/prof_kernels.py

Numbers printed under a profiler are never bench values; this only feeds profiles/*.json summaries."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--train", action="store_true")
    ap.add_argument("--steps", type=int, default=2)
    args = ap.parse_args()
    from mslesions3d_b200 import _lib, synthetic
    from mslesions3d_b200.ssd3d import LSSD3D
    _lib.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    if not args.train:
        sd = synthetic.random_state_dict(2, seed=0)
        model = LSSD3D(n_classes=2, input_channels=2, input_size=(128, 128, 128))
        model.load_state_dict(sd)
        model = model.to(dev).eval()
        model.use_cuda_graph = False
        xs = [torch.from_numpy(synthetic.make_batch(8, 2, (128, 128, 128), first_idx=8 * i)).to(torch.bfloat16).to(dev)
              for i in range(2)]
        with torch.no_grad():
            for i in range(3):
                model.predict_step({"img": xs[i % 2]}, 0)
            torch.cuda.synchronize()
            torch.cuda.nvtx.range_push("prof")
            for i in range(args.steps):
                model.predict_step({"img": xs[i % 2]}, 0)
            torch.cuda.synchronize()
            torch.cuda.nvtx.range_pop()
    else:
        sd = synthetic.random_state_dict(1, seed=0)
        model = LSSD3D(n_classes=2, input_channels=1, input_size=(96, 96, 96), threshold=[0.1, 0.2], lr=1e-4)
        model.load_state_dict(sd)
        model = model.to(dev).train()
        model.use_cuda_graph = False
        x, b, l = synthetic.make_batch(16, 1, (96, 96, 96), with_boxes=True)
        batch = {"img": torch.from_numpy(x).to(dev), "boxes": [torch.from_numpy(v).to(dev) for v in b],
                 "labels": [torch.from_numpy(v).to(dev) for v in l]}
        for _ in range(3):
            model.fit_step(batch)
        torch.cuda.synchronize()
        torch.cuda.nvtx.range_push("prof")
        for _ in range(args.steps):
            model.fit_step(batch)
        torch.cuda.synchronize()
        torch.cuda.nvtx.range_pop()
    print("done")


if __name__ == "__main__":
    main()
