#!/usr/bin/env python
"""Benchmark of the SSD3D hot path: volumes/sec for forward + decode + NMS (= ``LSSD3D.predict_step``).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): SSD3D-MobileNet inference on synthetic 2-channel 128^3 cube-lesion
volumes (generate_artificial_dataset.py distribution), batch 8 per GPU, bf16 activations, random-init
weights with randomised BN statistics.  One step = one predict_step over one batch.  With N > 1 every rank
runs the same per-GPU batch (independent volumes, no data-path collective): weak scaling.

The single JSON line printed by rank 0 carries
  value        whole-job volumes/s with the input batches already resident in HBM (device-timed, max over ranks).
               Exactly K steps inside ONE event pair, taken from the middle of one pipelined pass: W warm-up
               batches fill the pipeline before it, the batches still in flight after it drain outside it
               (``timed_steps``, ``timed_region_ms``); ms_per_step = region / K.  Nothing stretches the region:
               at about 0.18 ms per step (B200, 1000 W power limit) a small K gives a window of a few ms and
               a number that carries clock and scheduler noise; K of a few hundred (>= 50 ms) gives a stable one
  e2e          the same through the public streaming API (LSSD3D.predict_batches, the analogue of the
               reference's Trainer.predict loop) from PINNED HOST buffers: H2D of every batch and D2H of its
               detections inside the timed region.  Headline: bf16 host batches (the stem rounds fp32 inputs
               to bf16 on load, so the detections are bit-identical); ``e2e.fp32_host`` is the same from the
               fp32 batches the reference's loader yields (twice the bytes); ``e2e.h2d_ceiling_gbs`` is a bare
               pinned->device copy loop of the same buffers on all ranks at once (no compute): the host fabric
  roofline     the dominant kernel timed alone with CUDA events, algorithmic bytes / time vs the measured
               HBM peak of MEASURED_PEAKS.json
  cpu_baseline the reference's CPU path on a bounded sample of the same workload (see --impl reference)
  extras.train (every N) BASELINE.json configs[2]: LSSD3D.fit_step (forward + IoU matching + MultiBox loss +
               backward + NCCL all-reduce of the flat gradient + Adam), 1ch 96^3, batch 16 per GPU
  extras.nms_any_length (N = 1) greedy 3-D NMS over 2.5 M score-sorted candidates (configs[3]/[4])
``--impl reference`` times the UNMODIFIED reference (``oracle/_ref``, staged by ``oracle/make_ref.py``;
``kind: "reference"``) -- LSSD3D.forward + detect_objects on the host CPU, best thread count of a sweep --
or, where the staged files are missing, the oracle port (``kind: "port"``); rank 0 only.

``--dump-outputs DIR`` writes what the last timed step handed back (rank 0's detections for its batch of 8
volumes, concatenated in volume order) as float32 ``.npy`` files: ``boxes`` (n, 6), ``labels`` (n,), ``scores``
(n,) and ``counts`` (8,), the number of detections per volume.  Inputs and weights are seeded, so two builds
run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

if any(a in ("reference", "--impl=reference") for a in sys.argv[1:]):
    # the reference decides its device from torch.cuda.is_available() at import (ssd3d.py:23): its CPU path is
    # what this arm times, so the process never sees a GPU
    os.environ["CUDA_VISIBLE_DEVICES"] = ""

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "SSD3D volumes/sec (fwd+decode+NMS)"
UNIT = "volumes/s"
WORKLOAD = "SSD3D-MobileNet inference, 2ch 128^3 synthetic cube-lesion volumes, batch 8 per GPU, bf16"
CHANNELS, SIZE, BATCH = 2, (128, 128, 128), 8
MIN_SCORE, MAX_OVERLAP, TOP_K = 0.5, 0.5, 100
N_ROTATE = 4   # distinct resident input batches: 4 x 67 MB > 126 MB of L2
MIN_REGION_MS = 50.0
TRAIN_CHANNELS, TRAIN_SIZE, TRAIN_BATCH = 1, (96, 96, 96), 16


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(*names):
    """dram read + write bytes per launch from the first committed ncu --set full summary found (profiles/)."""
    for name in names:
        try:
            rows = json.load(open(os.path.join(ROOT, "profiles", name)))
            vals = []
            for r in rows:
                rd, wr = r["dram__bytes_read.sum"].split(), r["dram__bytes_write.sum"].split()
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                vals.append(float(rd[0]) * scale[rd[1]] + float(wr[0]) * scale[wr[1]])
            if vals:
                return float(np.mean(vals)), "profiles/" + name
        except Exception:
            continue
    return None, None


# ------------------------------------------------------------------------------------------------------
# clocks sampled DURING the timed regions (started before the warm-up, so a short region still has samples)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []        # (wall time, csv line)
        self.windows = []      # (t0, t1) wall-clock windows of the timed regions

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "10"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

        def parse(rows):
            sm, mx, reasons = [], [], set()
            for _, line in rows:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 6:
                    continue
                try:
                    sm.append(float(parts[0]))
                    mx.append(float(parts[1]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[2:6]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons

        # nvidia-smi's own sampling lags the wall clock by up to a period: widen the windows by 30 ms
        inside = [r for r in self.lines if any(t0 - 0.03 <= r[0] <= t1 + 0.03 for t0, t1 in self.windows)]
        sm, mx, reasons = parse(inside)
        scope = "timed regions"
        if not sm:                      # region shorter than nvidia-smi's period: everything since the warm-up
            sm, mx, reasons = parse(self.lines)
            scope = "whole run incl. warm-up"
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "scope": scope, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------
# the reference arm: the unmodified reference (oracle/_ref) or the oracle port on the host CPU
# ------------------------------------------------------------------------------------------------------
def make_inputs(n_batches: int, rank: int):
    """Host fp32 batches (n_batches, BATCH, C, D, H, W) of normalised synthetic volumes."""
    from mslesions3d_b200 import synthetic
    out = []
    for b in range(n_batches):
        out.append(synthetic.make_batch(BATCH, CHANNELS, SIZE, first_idx=(rank * n_batches + b) * BATCH))
    return out


class CpuReference:
    """forward + detect_objects per volume (batch 1, fp32) on the host: the unmodified reference's
    ``LSSD3D.predict_step`` (ssd3d.py:692-702) when its sources are staged, else the oracle restatement."""

    def __init__(self):
        from oracle import ssd3d_oracle as O
        from oracle import ref_shim
        self.O = O
        self.sd = O.random_state_dict(CHANNELS, seed=0)
        self.kind = "port"
        self.model = None
        if ref_shim.reference_available() and not torch.cuda.is_available():
            try:
                ssd3d = ref_shim.load_reference()[0]
                torch.manual_seed(0)
                m = ssd3d.LSSD3D(n_classes=2, input_channels=CHANNELS, input_size=SIZE, min_score=MIN_SCORE,
                                 max_overlap=MAX_OVERLAP, top_k=TOP_K)
                m.load_state_dict(self.sd, strict=True)
                self.model = m.eval()
                self.kind = "reference"
            except Exception as exc:      # noqa: BLE001  (fall back to the port, say why)
                self.why_port = repr(exc)
        if self.model is None:
            self.priors = O.prior_boxes_fast(SIZE, in_channels=CHANNELS)

    def run(self, volumes: np.ndarray, threads: int) -> float:
        """Seconds per volume."""
        torch.set_num_threads(threads)
        x = torch.from_numpy(volumes)
        with torch.no_grad():
            t0 = time.perf_counter()
            for i in range(x.shape[0]):
                if self.model is not None:
                    self.model.predict_step({"img": x[i:i + 1]}, 0)
                else:
                    locs, scores = self.O.forward(self.sd, x[i:i + 1])
                    self.O.detect_objects(locs, scores, self.priors, MIN_SCORE, MAX_OVERLAP, TOP_K)
            return (time.perf_counter() - t0) / x.shape[0]

    def best_threads(self, volume: np.ndarray, budget_s: float = 40.0):
        """Sweep thread counts (oversubscription can be far slower than 1 thread) and keep the best."""
        ncpu = os.cpu_count() or 1
        cands = sorted({t for t in (1, 2, 4, 8, 16, 32, 64, ncpu) if t <= ncpu})
        self.run(volume, cands[-1] if len(cands) < 3 else cands[2])      # warm-up: thread pool, mkldnn primitives
        best, t_start = None, time.perf_counter()
        for t in cands:
            if time.perf_counter() - t_start > budget_s:
                break
            spv = self.run(volume, t)
            if best is None or spv < best[0]:
                best = (spv, t)
        return best


def reference_line(steps: int, warmup: int, n_gpus: int, volumes_per_step: int = 2):
    """ONE definition of the CPU number (used by --impl reference and, through a subprocess, by the repo arm's
    cpu_baseline): best thread count of a sweep, then `steps` timed steps of `volumes_per_step` volumes."""
    from mslesions3d_b200 import synthetic
    ref = CpuReference()
    sample = synthetic.make_batch(volumes_per_step, CHANNELS, SIZE)
    _, threads = ref.best_threads(sample[:1])
    for _ in range(warmup):
        ref.run(sample[:1], threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        ref.run(sample, threads)
    dt = time.perf_counter() - t0
    vps = steps * sample.shape[0] / dt
    what = ("the unmodified reference (oracle/_ref: lesions3d/ssd3d.py LSSD3D.predict_step = forward + detect_objects)"
            if ref.kind == "reference" else "oracle port of the reference's torch-CPU path (forward + detect_objects)")
    return {
        "impl": "reference", "metric": METRIC, "value": vps, "unit": UNIT, "n_gpus": n_gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": 1000.0 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "step": "%d volumes (bounded sample of the batch-8 workload), batch 1 each, "
                   "fp32 torch-CPU" % volumes_per_step},
        "cpu_baseline": {"value": vps, "unit": UNIT, "cores": threads, "kind": ref.kind,
                         "sample": "%d volumes per step x %d steps, %s, best thread count of a sweep (host has %d cpus)"
                                   % (volumes_per_step, steps, what, os.cpu_count() or 1)},
        "e2e": {"value": vps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def cpu_baseline_subprocess():
    """The repo arm's cpu_baseline = the reference arm on a bounded sample, in a process that sees no GPU (the
    reference picks its device at import).  Never fatal."""
    try:
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
            env.pop(k, None)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3",
                            "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)["cpu_baseline"]
        return {"error": (r.stderr or r.stdout)[-400:]}
    except Exception as exc:      # noqa: BLE001
        return {"error": repr(exc)}


# ------------------------------------------------------------------------------------------------------
# BASELINE.json configs[2]: the training step, on every N
# ------------------------------------------------------------------------------------------------------
def train_leg(dev, rank, world, steps, warmup, barrier, max_over_ranks):
    """LSSD3D.fit_step on 1ch 96^3, batch 16 per GPU, threshold [0.1, 0.2] (train.py:38), Adam + cosine
    schedule, flat-gradient NCCL all-reduce when world > 1.  Inputs resident on the device (3 rotating batches =
    170 MB of activations per step >> L2 anyway).  -> dict for extras.train."""
    import torch.distributed as dist
    from mslesions3d_b200 import ops, synthetic
    from mslesions3d_b200.ssd3d import LSSD3D
    sd = synthetic.random_state_dict(TRAIN_CHANNELS, seed=0)
    model = LSSD3D(n_classes=2, input_channels=TRAIN_CHANNELS, input_size=TRAIN_SIZE, threshold=[0.1, 0.2], lr=1e-4)
    model.load_state_dict(sd)
    model = model.to(dev).train()
    n_rot = 3
    batches = []
    for r in range(n_rot):
        x, b, l = synthetic.make_batch(TRAIN_BATCH, TRAIN_CHANNELS, TRAIN_SIZE,
                                       first_idx=(rank * n_rot + r) * TRAIN_BATCH, with_boxes=True)
        batches.append({"img": torch.from_numpy(x).to(dev), "boxes": [torch.from_numpy(v).to(dev) for v in b],
                        "labels": [torch.from_numpy(v).to(dev) for v in l]})
    for i in range(max(warmup, 3)):
        model.fit_step(batches[i % n_rot])
    torch.cuda.synchronize()

    def region(n, **kw):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        last = None
        for i in range(n):
            last = model.fit_step(batches[i % n_rot], **kw)
        e1.record()
        host_ms = 1000.0 * (time.perf_counter() - t0)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), dev), host_ms, last

    ops.LAUNCHES[0] = 0
    ms, host_ms, last = region(steps)
    launches = ops.LAUNCHES[0] / float(steps)
    out = {"metric": "SSD3D training volumes/sec (fwd + IoU matching + MultiBox loss + bwd + all-reduce + Adam)",
           "volumes_per_s": world * TRAIN_BATCH * steps / (ms / 1000.0), "ms_per_step": ms / steps,
           "host_ms_per_step": host_ms / steps, "steps": steps, "timed_region_ms": ms,
           "launches_per_step": launches, "n_gpus": world, "scaling": "weak", "dtype": "bf16 activations, fp32 "
           "gradients / optimizer", "loss": [float(v) for v in last.cpu()],
           "skipped_steps": model.fit_skipped_steps(),
           "config": {"workload": "SSD3D training step, %dch %d^3, batch %d per GPU, threshold [0.1,0.2], Adam + cosine "
                      "schedule, flat-gradient NCCL all-reduce" % (TRAIN_CHANNELS, TRAIN_SIZE[0], TRAIN_BATCH),
                      "global_batch": TRAIN_BATCH * world, "parallelism": "dp%d" % world,
                      "collective": getattr(model.train_engine(), "collective_mode", "none") if world > 1 else "none"}}
    if world > 1:
        # the collective alone (same buffer, same communicator), and the step without it
        flat = model.train_engine().flat
        g = flat.grad.clone()
        for _ in range(5):
            dist.all_reduce(g)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            dist.all_reduce(g)
        e1.record()
        barrier()
        out["allreduce_ms"] = max_over_ranks(e0.elapsed_time(e1), dev) / 20.0
        out["allreduce_bytes"] = int(g.numel() * 4)
    else:
        out["allreduce_ms"] = 0.0
    del model, batches
    torch.cuda.empty_cache()
    return out


def train_roofline(dev):
    """Roofline object of the training step's largest kernel: the BatchNorm + ReLU backward of the stem-sized map
    (16 x 48^3 x 32 bf16 = 113 MB per tensor; csrc/bn_unit.cu bn_tile_kernel<1>).  Algorithmic bytes per launch: the
    saved raw conv output z and the incoming gradient read once, dz written once (the kernel reads z and g a second
    time for the apply phase -- that shows as the distance from the peak).  20 back-to-back launches over three
    rotating (z, g) pairs (680 MB > L2) between one CUDA event pair.  Never fatal."""
    from mslesions3d_b200 import ops
    n, c = TRAIN_BATCH, 32
    d, h, w = (TRAIN_SIZE[0] + 1) // 2, (TRAIN_SIZE[1] + 1) // 2, (TRAIN_SIZE[2] + 1) // 2
    peak, peak_src = load_peaks()
    bn = torch.nn.BatchNorm3d(c).to(dev).train()
    sets = []
    gen = torch.Generator(device=dev).manual_seed(3)
    for _ in range(3):
        z = torch.randn((n, c, d, h, w), device=dev, generator=gen).to(torch.bfloat16).contiguous(
            memory_format=torch.channels_last_3d)
        g = torch.randn((n, c, d, h, w), device=dev, generator=gen).to(torch.bfloat16).contiguous(
            memory_format=torch.channels_last_3d)
        _, st = ops.bn_train_relu(z, bn, None)
        sets.append((z, g, st))
    dgamma, dbeta = torch.empty(c, device=dev), torch.empty(c, device=dev)
    for z, g, st in sets:
        ops.bn_relu_backward(z, g, st, dgamma, dbeta)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 21
    e0.record()
    for i in range(launches):
        z, g, st = sets[i % 3]
        ops.bn_relu_backward(z, g, st, dgamma, dbeta)
    e1.record()
    torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1) / launches
    algo = 3 * n * c * d * h * w * 2
    achieved = algo / (k_ms * 1e-3) / 1e9
    return {"kernel": "bn_tile_kernel<1> (train-mode BatchNorm + ReLU backward of the stem map, 16 x 48^3 x 32: column "
                      "statistics, one barrier per channel group, dz in place)",
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
            "algorithmic_bytes_per_launch": algo, "kernel_ms": k_ms, "peak_source": peak_src,
            "timing": "%d back-to-back launches between one CUDA event pair, three rotating (z, g) pairs = 680 MB" % launches}


def dump_outputs(out_dir, boxes, labels, scores):
    """Per-volume detections of one step (lists of device tensors) -> out_dir/{boxes,labels,scores,counts}.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"boxes": torch.cat(boxes).reshape(-1, 6), "labels": torch.cat(labels), "scores": torch.cat(scores),
              "counts": torch.tensor([b.shape[0] for b in boxes])}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the extras.train leg (configs[2])")
    ap.add_argument("--no-extras", action="store_true", help="skip every secondary measurement")
    ap.add_argument("--eager", action="store_true",
                    help="launch every kernel individually (no CUDA graph): for ncu launch lists, not for numbers")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the detections of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from mslesions3d_b200.parallel import rank_world, max_over_ranks
    rank, local_rank, world = rank_world()

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(reference_line(args.steps, args.warmup, args.gpus)), flush=True)
        return

    import torch.distributed as dist
    from mslesions3d_b200 import _lib, ops
    from mslesions3d_b200.ssd3d import LSSD3D

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    _lib.load()
    if world > 1:
        from mslesions3d_b200.parallel import bind_to_gpu_cpus
        bind_to_gpu_cpus(local_rank)      # pinned staging buffers next to the GPU they feed
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- model + inputs -------------------------------------------------------------------------
    from mslesions3d_b200 import synthetic
    sd = synthetic.random_state_dict(CHANNELS, seed=0)
    model = LSSD3D(n_classes=2, input_channels=CHANNELS, input_size=SIZE, min_score=MIN_SCORE,
                   max_overlap=MAX_OVERLAP, top_k=TOP_K)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    host_f32_np = make_inputs(N_ROTATE, rank)
    host_f32 = [torch.from_numpy(h).pin_memory() for h in host_f32_np]
    host_bf16 = [h.to(torch.bfloat16).pin_memory() for h in host_f32]
    dev_bf16 = [h.to(dev) for h in host_bf16]
    in_bytes = host_bf16[0].numel() * 2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        """fn() inside ONE event pair, barrier + synchronize on both sides; max over ranks, in ms."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        fn()
        e1.record()
        barrier()
        sampler.window(t0, time.time())
        return max_over_ranks(e0.elapsed_time(e1), dev)    # the job is as slow as its slowest rank

    depth = int(model.pipeline_depth)

    def run_stream(src, warmup, steps, to_host=False):
        """Batches rotating over src through ONE pass of LSSD3D.predict_batches (one predict_step per batch on the
        device-resident path with --eager).  The CUDA event pair opens when the result of the warmup-th batch is
        handed back and closes at the result of the `steps`-th batch after it, with depth - 1 more batches still
        queued behind it: both ends see the same batches in flight, so the region holds exactly `steps` steps of a
        full pipeline; its fill and drain are outside.  -> (ms max over ranks, results of the last timed step)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        batches = ({"img": src[i % N_ROTATE]} for i in range(warmup + steps + depth - 1))
        if args.eager and not to_host:
            model.use_cuda_graph = False
            results = (model.predict_step(b, 0) for b in batches)
        else:
            results = model.predict_batches(batches, to_host=to_host)
        with torch.no_grad():
            for i, out in enumerate(results):
                assert out[0][0].is_cuda != to_host
                if i == warmup - 1:
                    t0 = time.time()
                    e0.record()
                elif i == warmup + steps - 1:
                    e1.record()
                    t1, last = time.time(), out
        barrier()
        sampler.window(t0, t1)
        return max_over_ranks(e0.elapsed_time(e1), dev), last    # the job is as slow as its slowest rank

    def capture(src, to_host=False):
        """Build (capture) the inference plan of every pipeline slot: one-off setup, not a step."""
        with torch.no_grad():
            for _ in model.predict_batches(({"img": src[i % N_ROTATE]} for i in range(depth)), to_host=to_host):
                pass

    # ---- resident-input throughput (value) --------------------------------------------------------
    if not args.eager:
        capture(dev_bf16)
    ops.LAUNCHES[0] = 0
    ms, last = run_stream(dev_bf16, args.warmup, args.steps)
    launches = round(ops.LAUNCHES[0] * args.steps / (args.warmup + args.steps + depth - 1))   # same every step
    n_timed = args.steps
    value = world * BATCH * n_timed / (ms / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last

    # ---- end to end from pinned host memory --------------------------------------------------------
    # every batch is copied from pinned host memory inside the timed region and its detections are read back
    # to the host; per step: padded boxes/labels/scores (top_k rows per volume) + the count/status/flag words
    d2h_bytes = BATCH * TOP_K * (24 + 4 + 8 + 8) + 4 * (BATCH + 2)
    e2e = {}
    for name, host in (("bf16", host_bf16), ("fp32", host_f32)):
        capture(host, to_host=True)
        ms_e, _ = run_stream(host, args.warmup, args.steps, to_host=True)
        e2e[name] = {"value": world * BATCH * args.steps / (ms_e / 1000.0), "ms_per_step": ms_e / args.steps,
                     "h2d_bytes_per_step": host[0].numel() * host[0].element_size(), "timed_region_ms": ms_e}
    # bare copy loop: what the host fabric gives `world` ranks copying at once, no compute
    stage = torch.empty_like(dev_bf16[0])
    copy_stream = torch.cuda.Stream(device=dev)

    def copy_loop(n):
        with torch.cuda.stream(copy_stream):
            for i in range(n):
                stage.copy_(host_bf16[i % N_ROTATE], non_blocking=True)
        torch.cuda.current_stream().wait_stream(copy_stream)

    copy_loop(3)
    n_copy = max(20, int(math.ceil(MIN_REGION_MS / 1.3)))
    ms_copy = timed(lambda: copy_loop(n_copy))
    ceiling_gbs = world * in_bytes * n_copy / (ms_copy / 1000.0) / 1e9
    ceiling_vps = world * BATCH * n_copy / (ms_copy / 1000.0)
    del stage

    # ---- dominant kernel alone: roofline ------------------------------------------------------------
    peak, peak_src = load_peaks()
    stem = model.base.features[0]
    w, scale, shift = stem._pack()
    sd_stride = 2

    def kernel_ms(fn, n_launch):
        """Average duration of n_launch back-to-back launches (one event pair around all of them, so the
        per-launch event/launch overhead is not attributed to the kernel); inputs rotate over > L2 bytes."""
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n_launch):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n_launch

    # HBM WRITE ceiling of this box, measured live: a memset of a buffer >> L2.  The copy peak in MEASURED_PEAKS.json
    # is 3.2 TB/s of reads + 3.2 TB/s of writes at once; pure writes top out well below the sum (3.9 TB/s on the
    # round-2 boxes, scripts/probe_hbm.py), which is what bounds the stem: two thirds of its bytes are writes.
    wbuf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
    write_gbs = wbuf.numel() / (kernel_ms(lambda i: wbuf.zero_(), 10) / 1000.0) / 1e9
    del wbuf
    stem_out = ops.stem_conv_bn_relu(dev_bf16[0], w, scale, shift, sd_stride)
    n_launch = max(20, args.steps)
    k_ms = kernel_ms(lambda i: ops.stem_conv_bn_relu(dev_bf16[i % N_ROTATE], w, scale, shift, sd_stride, out=stem_out),
                     n_launch)
    vox_out = BATCH * (SIZE[0] // 2) * (SIZE[1] // 2) * (SIZE[2] // 2)
    algo_bytes = in_bytes + vox_out * 32 * 2 + 27 * CHANNELS * 32 * 4
    achieved = algo_bytes / (k_ms / 1000.0) / 1e9
    stem_tz = os.environ.get("SSD3D_STEM_TZ", "") != "0"      # the library's own choice for rows of 128 voxels
    stem_name = ("stem_tz_kernel<2> (dense 3x3x3 conv 2->32 + BN + ReLU, banded-B tcgen05 GEMM on raw TMA rows)" if stem_tz
                 else "stem_tc_kernel<bf16,2> (dense 3x3x3 conv 2->32 + BN + ReLU, tcgen05 implicit GEMM)")
    traffic, traffic_src = (ncu_traffic("r02_ncu_stem_tz.json") if stem_tz else
                            ncu_traffic("r02_ncu_full_stem.json", "r01_ncu_full_stem_final.json"))
    roofline = {"kernel": stem_name, "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_source": "%s (ncu --set full, dram read+write per launch; part of the 134 MB output is still "
                                  "in the 126 MB L2 when the kernel ends)" % traffic_src,
                "timing": "%d back-to-back launches between one CUDA event pair, inputs rotating over 268 MB" % n_launch,
                "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": k_ms, "peak_source": peak_src,
                "write_ceiling": {"measured_write_gbs": write_gbs, "how": "torch zero_ of 512 MiB, 10 back-to-back launches",
                                  "write_bytes_per_launch": vox_out * 32 * 2,
                                  "write_floor_ms": vox_out * 32 * 2 / write_gbs / 1e6,
                                  "frac_of_write_floor": (vox_out * 32 * 2 / write_gbs / 1e6) / k_ms,
                                  "note": "the kernel cannot finish before its 134 MB of output has been written at the "
                                          "HBM write rate; reads overlap (a copy sustains read + write at once)"}}

    # second HBM-bound kernel the north star names: the first depthwise conv (32 ch, stride 2, 64^3 -> 32^3)
    blk = model.base.features[1]
    wd, s1, b1 = blk._pack()[:3]
    f0 = stem_out
    f0s = [f0, f0.clone()]      # 2 x 134 MB > L2
    dw_ms = kernel_ms(lambda i: ops.dwconv3d_bn_relu(f0s[i % 2], wd, s1, b1, 2), n_launch)
    dw_bytes = f0.numel() * 2 + (f0.numel() // 8) * 2 + 54 * 32
    dw_traffic, _ = ncu_traffic("r02_ncu_full_dw.json", "r01_ncu_full_dw_final.json")
    roofline_dw = {"kernel": "dw_tma_kernel<2,2,4,4,8> (depthwise 3x3x3, 32 ch, stride 2 + BN + ReLU, TMA halo tiles)",
                   "bound": "hbm", "achieved": dw_bytes / (dw_ms / 1000.0) / 1e9, "peak": peak, "unit": "GB/s",
                   "frac": dw_bytes / (dw_ms / 1000.0) / 1e9 / peak, "traffic": dw_traffic,
                   "algorithmic_bytes_per_launch": dw_bytes, "kernel_ms": dw_ms}
    del f0s, f0, stem_out

    # ---- secondary measurements; never allowed to break the bench line: any failure is recorded instead -----
    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            n_nms = 2500000
            gen = torch.Generator(device=dev).manual_seed(n_nms)
            ctr = torch.rand((n_nms, 3), device=dev, generator=gen)
            side = 0.02 + 0.08 * torch.rand((n_nms, 1), device=dev, generator=gen)
            nms_boxes = torch.cat([ctr - side / 2, ctr + side / 2], 1).contiguous()
            keep, kept = ops.nms3d_sorted_chunked(nms_boxes, MAX_OVERLAP, return_count=True)
            torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ops.nms3d_sorted_chunked(nms_boxes, MAX_OVERLAP)
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            extras["nms_any_length"] = {"candidates": n_nms, "kept": int(kept.item()), "ms": sorted(ts)[1],
                                        "workload": "greedy 3-D NMS over ALL score-sorted candidates (no 10*top_k "
                                                    "truncation), cubic boxes of side 0.02-0.1 at uniform centres, "
                                                    "threshold 0.5 (SURVEY 8d C5); the reference's n x n IoU matrix "
                                                    "would be 25 TB"}
            del nms_boxes, keep
        except Exception as exc:      # noqa: BLE001
            extras["nms_any_length_error"] = repr(exc)
    if not (args.no_train or args.no_extras or args.eager):
        # every rank takes part (the all-reduce is a collective); a failure on any rank is a failure on all
        try:
            model._plans.clear()
            del dev_bf16
            torch.cuda.empty_cache()
            extras["train"] = train_leg(dev, rank, world, args.steps, args.warmup, barrier, max_over_ranks)
        except Exception as exc:      # noqa: BLE001
            if world > 1:
                raise
            extras["train_error"] = repr(exc)
        if rank == 0 and "train" in extras:
            try:
                extras["train"]["roofline"] = train_roofline(dev)
            except Exception as exc:      # noqa: BLE001
                extras["train"]["roofline_error"] = repr(exc)
            torch.cuda.empty_cache()

    clocks = sampler.stop() if rank == 0 else None

    # ---- CPU baseline (rank 0, N = 1 only) -----------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / n_timed, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "timed_steps": n_timed, "timed_region_ms": ms,
            "config": {"workload": WORKLOAD, "global_batch": BATCH * world, "parallelism": "dp%d" % world,
                       "l2": "inputs rotate over %d resident batches (%d MB) > 126 MB L2" %
                             (N_ROTATE, N_ROTATE * in_bytes // 2 ** 20),
                       "min_score": MIN_SCORE, "max_overlap": MAX_OVERLAP, "top_k": TOP_K, "priors": 9344,
                       "timed_region": "%d steps inside one CUDA event pair, in the middle of one pipelined pass (after "
                                       "%d warm-up batches, before the drain)" % (args.steps, args.warmup),
                       "pipeline": "%d batches in flight (LSSD3D.predict_batches: one captured plan per slot, own "
                                   "stream each; a step = one batch through stem + graph replay + result read-back)" % depth},
            "e2e": {"value": e2e["bf16"]["value"], "unit": UNIT, "h2d_bytes_per_step": in_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e["bf16"]["ms_per_step"],
                    "host_format": "bf16 pinned batches (bit-identical detections: the stem rounds fp32 inputs to bf16 "
                                   "on load)",
                    "timed_region_ms": e2e["bf16"]["timed_region_ms"],
                    "fp32_host": {"value": e2e["fp32"]["value"], "ms_per_step": e2e["fp32"]["ms_per_step"],
                                  "h2d_bytes_per_step": e2e["fp32"]["h2d_bytes_per_step"],
                                  "note": "the fp32 batches the reference's loader yields (datasets.py:403)"},
                    "h2d_ceiling_gbs": ceiling_gbs, "h2d_ceiling_volumes_per_s": ceiling_vps,
                    "frac_of_h2d_ceiling": e2e["bf16"]["value"] / ceiling_vps,
                    "h2d_ceiling_how": "%d ranks x %d pinned->device copies of the same 67 MB bf16 batches on a copy "
                                       "stream, no compute, one event pair, max over ranks" % (world, n_copy)},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_depthwise": roofline_dw,
            "cpu_baseline": cpu,
            "extras": extras or None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # The training step's CUDA graph holds captured NCCL work; tearing the communicator down under it
        # (destroy_process_group) was seen to block forever after the line had been printed.  Everything that had
        # to be measured and reported is done: leave together, without the teardown.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
