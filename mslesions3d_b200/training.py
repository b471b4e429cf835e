"""Training step of the SSD3D network on the sm_100a kernels (``LSSD3D.training_step`` /
``configure_optimizers``, ssd3d.py:467-531,704-722).

The reference gets the backward pass from torch autograd over ``nn.Conv3d`` / ``nn.BatchNorm3d`` /
``nn.ReLU`` and steps ``torch.optim.Adam``.  Here the whole network is ONE autograd node: ``TrainEngine``
runs the train-mode forward (raw conv -> batch-statistic BN -> ReLU per unit, fused SSD heads) while
recording a tape of saved activations, and walks it backwards with hand-written kernels (BN/ReLU backward,
pointwise / depthwise / stem / head weight and data gradients).  Two ways in:

* ``LSSD3D.training_step(batch)`` returns a loss tensor whose ``backward()`` fills ``p.grad`` of every
  parameter -- the reference's contract, any torch optimizer can follow;
* ``LSSD3D.fit_step(batch)`` is the fused loop body: forward, MultiBox loss with its analytic gradient,
  backward straight into one flat fp32 gradient buffer, one NCCL all-reduce of that buffer when
  ``torch.distributed`` is initialised (data parallel over volumes, SURVEY.md section 8e), one fused Adam
  launch over the flat parameter buffer (weight decay 5e-4, biases at 2x lr, cosine schedule).

PyTorch is plumbing (memory, streams, autograd hand-off, NCCL); every arithmetic step is a library kernel.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib, ops
from .mobilenet import Block, ConvBN, _stride3


SIDE_STREAMS = 3                 # side streams of a training step (TrainEngine._side_streams)
HEAVY_LEAF_BYTES = 32 * 2 ** 20  # weight-gradient leaves that read this much or more stay on the main stream


class _Grads:
    """Destination tensors of the parameter gradients, keyed by parameter name."""

    def __init__(self, named_params, flat: Optional["FlatParams"] = None):
        self.t: Dict[str, torch.Tensor] = {}
        for name, p in named_params:
            if not p.requires_grad:
                continue
            if flat is not None and name in flat.views_grad:
                self.t[name] = flat.views_grad[name]
            else:
                self.t[name] = torch.empty_like(p, dtype=torch.float32, memory_format=torch.contiguous_format)

    def __getitem__(self, name):
        return self.t[name]


class FlatParams:
    """All trainable parameters re-homed as views of ONE fp32 buffer, gradients and Adam moments likewise.
    Layout: [weights ...][biases ...] (``name.endswith('.bias')``, the reference's 2x-lr group,
    ssd3d.py:706-715), every tensor padded to a multiple of 8 elements so that kernels may use 16/32-byte
    accesses on any view.  Parameters that never receive a gradient (``rescale_factors``, SURVEY.md B2) stay
    outside, exactly as torch.optim.Adam skips ``grad is None``."""

    def __init__(self, model: nn.Module, skip=("rescale_factors",)):
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad and n not in skip]
        weights = [(n, p) for n, p in named if not n.endswith(".bias")]
        biases = [(n, p) for n, p in named if n.endswith(".bias")]
        dev = named[0][1].device
        off = 0
        self.offsets: Dict[str, int] = {}
        for n, p in weights:
            self.offsets[n] = off
            off += (p.numel() + 7) // 8 * 8
        self.bias_start = off
        for n, p in biases:
            self.offsets[n] = off
            off += (p.numel() + 7) // 8 * 8
        self.numel = off
        self.param = torch.zeros((off,), dtype=torch.float32, device=dev)
        self.grad = torch.zeros((off,), dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros((off,), dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros((off,), dtype=torch.float32, device=dev)
        self.views_grad: Dict[str, torch.Tensor] = {}
        # optimizer state on the device (the whole step is one captured graph: no host scalars):
        # [non-finite gradient this step, skipped steps, APPLIED steps, -] and the per-step scalars derived from it
        self.status = torch.zeros((4,), dtype=torch.int32, device=dev)
        self.scalars = torch.zeros((8,), dtype=torch.float32, device=dev)
        with torch.no_grad():
            for n, p in weights + biases:
                o = self.offsets[n]
                view = self.param[o:o + p.numel()].view(p.shape)
                view.copy_(p.detach().float())
                p.data = view
                self.views_grad[n] = self.grad[o:o + p.numel()].view(p.shape)

    @property
    def step(self) -> int:
        """Optimizer steps APPLIED so far (reads the device counter: synchronises)."""
        return int(self.status[2].item())


class PackedWeights:
    """bf16 copies of every conv weight in the layouts the kernels read (stem (32,KPAD), depthwise (27,C),
    pointwise (Cout,Cin) and its transpose for the data gradient, head (16,27*C)) plus the fp32 head biases, all
    views of two buffers that ONE gather launch each refreshes from the flat fp32 parameter buffer after an
    optimizer step (instead of ~45 small torch launches per step inside the captured graph).  The index maps are
    built once on the host by pushing flat indices through the same reshapes / permutes the packing does."""

    def __init__(self, model, flat: "FlatParams"):
        dev = flat.param.device
        segs, fsegs = [], []           # (name, index tensor (int64, CPU), shape)
        self.views: Dict[str, torch.Tensor] = {}

        def idx(name):
            p = dict(model.named_parameters())[name]
            o = flat.offsets[name]
            return (o + torch.arange(p.numel(), dtype=torch.int64)).view(p.shape)

        for i, feat in enumerate(model.base.features):
            p = "base.features.%d" % i
            if isinstance(feat, ConvBN):
                w = idx(p + ".0.weight")
                co, ci = w.shape[0], w.shape[1]
                kpad = 64 if 27 * ci <= 64 else 128
                m = torch.full((co, kpad), -1, dtype=torch.int64)
                m[:, :27 * ci] = w.reshape(co, 27 * ci)
                segs.append((p + ".stem", m))
            else:
                w1 = idx(p + ".conv1.weight")
                segs.append((p + ".dw", w1.reshape(w1.shape[0], 27).t().contiguous()))
                w2 = idx(p + ".conv2.weight")
                w2 = w2.reshape(w2.shape[0], w2.shape[1])
                segs.append((p + ".pw", w2.contiguous()))
                segs.append((p + ".pwT", w2.t().contiguous()))
        for j in range(len(model.pred_convs.loc_convs)):
            lw = idx("pred_convs.loc_convs.%d.weight" % j)
            cw = idx("pred_convs.cl_convs.%d.weight" % j)
            c = lw.shape[1]
            rows = lw.shape[0] + cw.shape[0]
            npad = (rows + 15) // 16 * 16
            m = torch.full((npad, 27 * c), -1, dtype=torch.int64)
            m[:lw.shape[0]] = lw.permute(0, 2, 3, 4, 1).reshape(lw.shape[0], 27 * c)
            m[lw.shape[0]:rows] = cw.permute(0, 2, 3, 4, 1).reshape(cw.shape[0], 27 * c)
            segs.append(("head%d.w" % j, m))
            b = torch.full((npad,), -1, dtype=torch.int64)
            b[:lw.shape[0]] = idx("pred_convs.loc_convs.%d.bias" % j)
            b[lw.shape[0]:rows] = idx("pred_convs.cl_convs.%d.bias" % j)
            fsegs.append(("head%d.b" % j, b))

        def build(seg_list, dtype):
            offs, total = [], 0
            for _, m in seg_list:
                offs.append(total)
                total += (m.numel() + 127) // 128 * 128          # 256-byte aligned segments (TMA bases)
            index = torch.full((total,), -1, dtype=torch.int32)
            for (name, m), o in zip(seg_list, offs):
                index[o:o + m.numel()] = m.reshape(-1).to(torch.int32)
            buf = torch.zeros((total,), dtype=dtype, device=dev)
            for (name, m), o in zip(seg_list, offs):
                self.views[name] = buf[o:o + m.numel()].view(m.shape)
            return index.to(dev), buf

        self.index_bf16, self.buf_bf16 = build(segs, torch.bfloat16)
        self.index_f32, self.buf_f32 = build(fsegs, torch.float32)
        self.flat = flat

    def refresh(self):
        ops.gather_cast(self.flat.param, self.index_bf16, self.buf_bf16)
        ops.gather_cast(self.flat.param, self.index_f32, self.buf_f32)


def broadcast_replica_state(model, flat: "FlatParams", src: int = 0) -> None:
    """Make every rank a replica of rank ``src`` before the first data-parallel step -- what DistributedDataParallel
    does at construction (parameter broadcast) and with ``broadcast_buffers``: the flat parameter buffer, the Adam
    moments and step counter, and every BatchNorm buffer (running_mean / running_var / num_batches_tracked) and
    ``rescale_factors``.  Without it, ranks built from different RNG states or checkpoints would silently train
    divergent replicas on averaged gradients.  During training the BatchNorm statistics stay rank-local (each rank
    sees its own volumes; the reference has no SyncBN, SURVEY.md 8e); ``sync_batchnorm_buffers`` averages them on
    demand (e.g. before validation / checkpointing)."""
    with torch.no_grad():
        for t in (flat.param, flat.exp_avg, flat.exp_avg_sq, flat.status):
            dist.broadcast(t, src)
        for _, b in model.named_buffers():
            dist.broadcast(b, src)
        for n, p in model.named_parameters():
            if n not in flat.offsets:          # parameters outside the flat buffer (rescale_factors)
                dist.broadcast(p.data, src)


def sync_batchnorm_buffers(model) -> None:
    """Average the BatchNorm running statistics over the ranks (num_batches_tracked: maximum)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    world = float(dist.get_world_size())
    with torch.no_grad():
        for n, b in model.named_buffers():
            if b.is_floating_point():
                dist.all_reduce(b)
                b.div_(world)
            else:
                dist.all_reduce(b, op=dist.ReduceOp.MAX)
    model.invalidate_packed()


def replica_checksum_matches(flat: "FlatParams") -> bool:
    """True when every rank holds bit-identical parameters (a cheap health check for long runs)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return True
    v = flat.param.view(torch.int32).to(torch.int64)
    mine = torch.stack([v.sum(), (v * torch.arange(1, v.numel() + 1, device=v.device)).sum()])
    lo, hi = mine.clone(), mine.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return bool(torch.equal(lo, hi))


def dims_of(x, count, bpl):
    """Spatial shape of ``x`` if it holds ``count`` priors at ``bpl`` boxes per location, else ()."""
    sp = tuple(x.shape[2:])
    return sp if sp[0] * sp[1] * sp[2] * bpl == count else ()


class TrainEngine:
    """Train-mode forward with a tape + hand-written backward for ``LSSD3D`` (MobileNet base + SSD heads)."""

    def __init__(self, model):
        self.model = model
        self.flat: Optional[FlatParams] = None
        self.packed: Optional[PackedWeights] = None
        self.tape = None
        self.plans = {}
        self._side = None
        # tests set this to a dict: backward() then stores the tape and clones of every gradient that flows through
        # a unit (the in-situ stage-wise parity test replays each stage through torch-CPU autograd)
        self.record = None
        self.collective_mode = "none"

    def _side_streams(self, main):
        """The side streams of the step, on ``main``'s device: the weight-gradient leaves are dealt round-robin over
        them (each is a few small launches -- tens of CTAs -- so independent leaves run next to each other instead
        of queueing behind one another); every stream has its own scratch slot.  The forward pass issues the heads
        on the first one."""
        if self._side is None or self._side[0].device != main.device:
            self._side = [torch.cuda.Stream(device=main.device) for _ in range(SIDE_STREAMS)]
        return self._side

    # ------------------------------------------------------------------------------------------
    def flatten(self) -> FlatParams:
        if self.flat is None or self.flat.param.device != self.model.device:
            self.flat = FlatParams(self.model)
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                broadcast_replica_state(self.model, self.flat)
            self.packed = PackedWeights(self.model, self.flat)
            self.packed.refresh()
            self.plans.clear()
            self.model.invalidate_packed()
        return self.flat

    # ------------------------------------------------------------------------------------------
    def forward(self, image: torch.Tensor, packed: Optional[PackedWeights] = None):
        """image (N, Cin, D, H, W) -> locs (N,P,6), scores (N,P,n_classes); records the tape.  ``packed``: the
        fused step's pre-packed weights (kept current by the optimizer step); otherwise the weights are packed
        from the parameters here."""
        m = self.model
        dev = m.device
        if dev.type != "cuda":
            raise RuntimeError("training needs the model on a CUDA device; there is no CPU path")
        if image.device != dev:
            image = image.to(dev, non_blocking=True)
        if image.dtype not in (torch.float32, torch.bfloat16):
            image = image.float()
        image = image.contiguous()
        flag = m.base.nan_flag(dev)
        tape = {"image": image, "units": [], "heads": []}
        x = image
        feats = {}
        keys = list(m.aspect_ratios.keys())
        pc = m.pred_convs
        n = image.shape[0]
        # head outputs are allocated up front (feature-map sizes follow from the strides) so that each head can be
        # issued on the side stream as soon as its feature map exists, overlapping the rest of the backbone
        dims, counts_at = tuple(image.shape[2:]), {}
        for i, feat in enumerate(m.base.features):
            st3 = _stride3(feat[0].stride if isinstance(feat, ConvBN) else feat.conv1.stride)
            dims = tuple(ops.conv_out(v, s_) for v, s_ in zip(dims, st3))
            if i in keys:
                counts_at[i] = dims[0] * dims[1] * dims[2] * pc.n_boxes[i]
        counts = [counts_at[k] for k in keys]
        offs = [int(sum(counts[:j])) for j in range(len(keys))]
        total = int(sum(counts))
        locs = torch.empty((n, total, 6), dtype=torch.float32, device=dev)
        scores = torch.empty((n, total, pc.n_classes), dtype=torch.float32, device=dev)
        head_w = ([(packed.views["head%d.w" % j], packed.views["head%d.b" % j]) for j in range(len(keys))]
                  if packed else pc._pack())
        main = torch.cuda.current_stream()
        side = self._side_streams(main)[0]
        for i, feat in enumerate(m.base.features):
            if isinstance(feat, ConvBN):
                conv, bn = feat[0], feat[1]
                sd = _stride3(conv.stride)[0]
                w = packed.views["base.features.%d.stem" % i] if packed else ops.pack_stem_weight(conv.weight)
                z = ops.stem_conv_raw(x, w, sd)
                a, st = ops.bn_train_relu(z, bn, flag)
                tape["units"].append(dict(kind="stem", idx=i, x=x, z=z, st=st, stride=sd))
                x = a
            elif isinstance(feat, Block):
                s = _stride3(feat.conv1.stride)[0]
                pre = "base.features.%d" % i
                wd = packed.views[pre + ".dw"] if packed else ops.pack_dw_weight(feat.conv1.weight)
                z1 = ops.dwconv3d_raw(x, wd, s)
                a1, st1 = ops.bn_train_relu(z1, feat.bn1, None)
                wp = packed.views[pre + ".pw"] if packed else ops.pack_pw_weight(feat.conv2.weight)
                z2 = ops.pwconv_raw(a1, wp)
                a2, st2 = ops.bn_train_relu(z2, feat.bn2, flag)
                wpt = packed.views[pre + ".pwT"] if packed else None
                tape["units"].append(dict(kind="block", idx=i, x=x, z1=z1, st1=st1, a1=a1, z2=z2, st2=st2, wd=wd, wp=wp,
                                          wpt=wpt, stride=s))
                x = a2
            else:
                raise NotImplementedError("unexpected backbone layer %r" % type(feat))
            if i in keys:
                feats[i] = x
                j = keys.index(i)
                if tuple(x.shape[2:]) != dims_of(x, counts_at[i], pc.n_boxes[i]):
                    raise RuntimeError("feature map %d has an unexpected shape %r" % (i, tuple(x.shape)))
                side.wait_stream(main)
                ops._WS_SLOT[0] = "ws_side"
                try:
                    with torch.cuda.stream(side):
                        ops.head_conv(x, head_w[j][0], head_w[j][1], locs, scores, pc.n_boxes[i], pc.n_classes,
                                      offs[j], flag)
                finally:
                    ops._WS_SLOT[0] = "ws"
                tape["heads"].append(dict(j=j, layer=i, feat=x, w=head_w[j][0], off=offs[j], bpl=pc.n_boxes[i]))
        main.wait_stream(side)
        self.tape = tape
        return locs, scores

    # ------------------------------------------------------------------------------------------
    def take_tape(self):
        """Hand the tape of the latest forward to its owner (the autograd node): later train-mode forwards then
        record their own tape without disturbing a backward that has not run yet."""
        tape, self.tape = self.tape, None
        return tape

    def backward(self, dlocs: torch.Tensor, dscores: torch.Tensor, grads: _Grads, tape=None) -> None:
        """d(loss)/d(locs), d(loss)/d(scores) -> every parameter gradient (written into ``grads``).
        ``tape``: the forward's tape (``take_tape``); default: the latest forward of this engine."""
        if tape is None:
            tape = self.tape
            self.tape = None
        if tape is None:
            raise RuntimeError("TrainEngine.backward without a recorded forward")
        m = self.model
        pc = m.pred_convs
        dlocs = dlocs.float().contiguous()
        dscores = dscores.float().contiguous()
        rec = self.record
        if rec is not None:
            rec.clear()
            rec.update(tape=tape, dlocs=dlocs.clone(), dscores=dscores.clone(), units={}, heads={})

        def snap(t):
            return None if t is None else t.clone(memory_format=torch.preserve_format)
        n = tape["image"].shape[0]
        head_at = {h["layer"]: h for h in tape["heads"]}
        # Weight gradients are leaves of the backward graph: they go to a second (lower-priority) stream and
        # overlap the critical chain BN-backward -> data gradient -> BN-backward ..., whose small-map kernels
        # fill a fraction of the SMs.  Inside a CUDA-graph capture the fork/join become graph edges.  The
        # gradient tensors the side stream reads are kept alive until the join (the allocator would hand their
        # memory to a later main-stream tensor otherwise); the side stream has its own scratch slot.
        main = torch.cuda.current_stream()
        sides = self._side_streams(main)
        keep = []
        n_leaf = [0]

        # ... except the heavy ones (the first blocks' maps, tens of MB): they are HBM-bound like the main-chain kernels
        # around them, so overlapping buys nothing, and their persistent CTAs (180 registers, ~200 KB of shared
        # memory) would keep the all-resident BatchNorm grids of the main chain (csrc/bn_unit.cu) waiting for SMs.
        # They run in order on the main stream.
        def leaf(fn, *tensors, nbytes=0):
            if nbytes >= HEAVY_LEAF_BYTES:
                fn()
                return
            k = n_leaf[0] % len(sides)
            n_leaf[0] += 1
            sides[k].wait_stream(main)
            ops._WS_SLOT[0] = "ws_side" if k == 0 else "ws_side%d" % k
            try:
                with torch.cuda.stream(sides[k]):
                    fn()
            finally:
                ops._WS_SLOT[0] = "ws"
            keep.extend(tensors)

        dO = {}
        for h in tape["heads"]:
            j = h["j"]
            _, c, d, hh, w = h["feat"].shape
            bpl = h["bpl"]
            dO[h["layer"]] = ops.head_grad_pack(dlocs, dscores, n, d, hh, w, bpl, pc.n_classes, h["off"],
                                                grads["pred_convs.loc_convs.%d.bias" % j],
                                                grads["pred_convs.cl_convs.%d.bias" % j])
            leaf(lambda h=h, j=j, bpl=bpl: ops.head_wgrad(
                dO[h["layer"]], h["feat"], bpl * 6, bpl * pc.n_classes,
                grads["pred_convs.loc_convs.%d.weight" % j], grads["pred_convs.cl_convs.%d.weight" % j]))
        g = None    # gradient w.r.t. the output of the unit being processed (channels-last bf16)
        for u in reversed(tape["units"]):
            i = u["idx"]
            p = "base.features.%d" % i
            r = None
            if rec is not None:
                r = rec["units"][i] = {}
            if i in head_at:
                h = head_at[i]
                if rec is not None:
                    rec["heads"][i] = dict(dO=snap(dO[i]), addend=snap(g))
                g = ops.head_dgrad(dO[i], h["w"], h["feat"], addend=g, n_cols=h["bpl"] * (6 + pc.n_classes))
                if rec is not None:
                    rec["heads"][i]["out"] = snap(g)
            if g is None:
                raise RuntimeError("no gradient reaches backbone layer %d" % i)
            if u["kind"] == "block":
                if r is not None:
                    r["g2"] = snap(g)
                dz2 = ops.bn_relu_backward(u["z2"], g, u["st2"], grads[p + ".bn2.weight"], grads[p + ".bn2.bias"])
                if r is not None:
                    r["dz2"] = snap(dz2)
                leaf(lambda dz2=dz2, u=u, p=p: ops.pwconv_wgrad(dz2, u["a1"], grads[p + ".conv2.weight"]), dz2,
                     nbytes=2 * (dz2.numel() + u["a1"].numel()))
                g1 = torch.empty_like(u["a1"])
                nn_, c1, d1, h1, w1 = u["a1"].shape
                wt = u["wpt"] if u["wpt"] is not None else u["wp"].t().contiguous()   # (Cin, Cout): dx = dz . W
                ops.pw_gemm_raw(nn_ * d1 * h1 * w1, dz2, wt, g1)
                if r is not None:
                    r["g1"] = snap(g1)
                dz1 = ops.bn_relu_backward(u["z1"], g1, u["st1"], grads[p + ".bn1.weight"], grads[p + ".bn1.bias"])
                if r is not None:
                    r["dz1"] = snap(dz1)
                leaf(lambda dz1=dz1, u=u, p=p: ops.dwconv3d_wgrad(dz1, u["x"], u["stride"],
                                                                  grads[p + ".conv1.weight"]), dz1,
                     nbytes=2 * (dz1.numel() + u["x"].numel()))
                g = ops.dwconv3d_dgrad(dz1, u["wd"], u["x"], u["stride"])
                if r is not None:
                    r["dx"] = snap(g)
            else:
                if r is not None:
                    r["g"] = snap(g)
                # first layer: nothing upstream needs dz, so (outside the tests' recording mode) it is never written --
                # the weight-gradient kernel applies the BatchNorm + ReLU backward to the rows it loads
                fused = (r is None and
                         ops.stem_unit_backward(u["z"], g, u["st"], grads[p + ".1.weight"], grads[p + ".1.bias"],
                                                u["x"], u["stride"], grads[p + ".0.weight"]))
                if not fused:
                    dz = ops.bn_relu_backward(u["z"], g, u["st"], grads[p + ".1.weight"], grads[p + ".1.bias"])
                    if r is not None:
                        r["dz"] = snap(dz)
                    ops.stem_wgrad(dz, u["x"], u["stride"], grads[p + ".0.weight"])
                g = None
        for st in sides:
            main.wait_stream(st)
        del keep


class _NetFn(torch.autograd.Function):
    """The whole network as one autograd node: forward = TrainEngine.forward, backward = TrainEngine.backward
    returning one gradient per parameter (autograd accumulates them into ``p.grad``)."""

    @staticmethod
    def forward(ctx, engine, image, names, *params):
        ctx.engine, ctx.names, ctx.params = engine, names, params
        locs, scores = engine.forward(image)
        ctx.tape = engine.take_tape()
        return locs, scores

    @staticmethod
    def backward(ctx, dlocs, dscores):
        eng = ctx.engine
        grads = _Grads(zip(ctx.names, ctx.params))
        tape, ctx.tape = ctx.tape, None
        if tape is None:
            raise RuntimeError("backward through the same LSSD3D forward twice (the saved activations were released)")
        eng.backward(dlocs, dscores, grads, tape=tape)
        out = []
        for name, p in zip(ctx.names, ctx.params):
            out.append(grads.t.get(name) if name != "rescale_factors" else None)
        return (None, None, None, *out)


def forward_train(model, image):
    """Autograd-visible train-mode forward of ``model`` (an ``LSSD3D``)."""
    eng = model.train_engine()
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    names = tuple(n for n, _ in named)
    return _NetFn.apply(eng, image, names, *[p for _, p in named])


def cosine_lr(base_lr: float, step: int, t_max: int = 40, eta_min: float = 0.0) -> float:
    """CosineAnnealingLR(T_max) in closed form (ssd3d.py:718-720; stepped once per batch, ssd3d.py:525-527)."""
    return eta_min + (base_lr - eta_min) * (1.0 + math.cos(math.pi * step / t_max)) / 2.0


class _TrainPlan:
    """One whole optimisation step for one input signature, captured into ONE CUDA graph (the eager step is
    host-bound: ~190 launches): forward, matching, loss, backward, the gradient all-reduce (NCCL, captured like any
    other node), Adam and the re-packing of the bf16 weights.  Nothing in it depends on a host scalar: the step
    counter, the cosine learning-rate schedule and the skip-on-NaN decision live on the device
    (``ssd3d_adam_step_dev``).  Inputs are staged into static buffers: the image batch, the concatenated
    ground-truth boxes / labels (capacity ``tmax`` rows) and the per-image offsets.  Without ``use_cuda_graph`` the
    plan is not captured and ``_step`` runs the same step body on the staged buffers eagerly."""

    def __init__(self, model, shape, dtype, tmax: int, world_size: int, allreduce):
        eng = model.train_engine()
        self.flat = eng.flatten()
        dev = model.device
        n = shape[0]
        self.n, self.tmax = n, tmax
        self.world_size, self.allreduce = world_size, allreduce
        self.image = torch.empty(tuple(shape), dtype=dtype, device=dev)
        self.gt_boxes = torch.zeros((tmax, 6), dtype=torch.float32, device=dev)
        self.gt_labels = torch.zeros((tmax,), dtype=torch.int64, device=dev)
        self.offsets = torch.zeros((n + 1,), dtype=torch.int32, device=dev)
        self.loss = None
        self.n_kernels = 0
        self.graph = None
        self.optimizer_in_graph = False
        self.extra_state = []       # device state besides the model's that the warm-up steps change (restored)

    def load(self, images, gt_boxes, gt_labels):
        self.image.copy_(images, non_blocking=True)
        counts = [int(b.shape[0]) for b in gt_boxes]
        total = sum(counts)
        if total > self.tmax:
            raise RuntimeError("more ground-truth boxes (%d) than the captured plan holds (%d)" % (total, self.tmax))
        offs = [0]
        for c in counts:
            offs.append(offs[-1] + c)
        # a fresh pageable tensor per step: the copy is staged before copy_ returns, so the host may run
        # steps ahead of the device without rewriting memory an earlier copy still has to read
        self.offsets.copy_(torch.tensor(offs, dtype=torch.int32))
        if total:
            dev = self.gt_boxes.device
            boxes = [b.reshape(-1, 6) for b in gt_boxes]
            labels = [l.reshape(-1) for l in gt_labels]
            if all(b.device == dev and b.dtype == torch.float32 for b in boxes) and \
                    all(l.device == dev and l.dtype == torch.int64 for l in labels):
                # device-resident ground truth: concatenate straight into the staging buffers (one launch each)
                torch.cat(boxes, out=self.gt_boxes[:total])
                torch.cat(labels, out=self.gt_labels[:total])
            else:
                self.gt_boxes[:total].copy_(torch.cat(boxes).float(), non_blocking=True)
                self.gt_labels[:total].copy_(torch.cat(labels).long(), non_blocking=True)

    def _run(self, model, with_optimizer: bool):
        self._prepare(model)
        eng = model.train_engine()
        lf = model.loss_fn
        t0, t1 = (lf.threshold, lf.threshold) if lf.thresholding_mode == "hard" else lf.threshold
        locs, scores = eng.forward(self.image, eng.packed)
        m = ops.match_priors_packed(self.gt_boxes, self.gt_labels, self.offsets, self.n, self.tmax,
                                    model._prior_source(model.device), t0, t1)
        out, n_pos, g_locs, g_scores = ops.multibox_loss(locs, scores, m["true_classes"], m["true_locs"],
                                                         alpha=float(lf.alpha),
                                                         hard_negative_mining=lf.hard_negative_mining,
                                                         neg_pos_ratio=lf.neg_pos_ratio, want_grads=True)
        grads = _Grads(((n, p) for n, p in model.named_parameters() if p.requires_grad and n != "rescale_factors"),
                       self.flat)
        eng.backward(g_locs, g_scores, grads)
        if with_optimizer:
            _optimizer_step(model, self.flat, self.world_size, self.allreduce)
        self.loss = out

    def _prepare(self, model):
        """Work of the step before the forward pass (nothing: the host stages the batch, ``load``)."""

    def capture(self, model):
        """Warm up (lazy module loading, workspaces, the NCCL communicator) and record.  The warm-up steps run
        for real, so everything they touch -- BatchNorm buffers, parameters, Adam moments and counters -- is
        restored afterwards."""
        flat = self.flat
        buffers = {k: v.clone() for k, v in model.named_buffers()}
        state = (flat.param, flat.exp_avg, flat.exp_avg_sq, flat.status, *self.extra_state)
        saved = [t.clone() for t in state]
        side = torch.cuda.Stream(device=model.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(2):
                self._run(model, True)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()

        def restore():
            with torch.no_grad():
                for k, v in model.named_buffers():
                    v.copy_(buffers[k])
                for t, v in zip(state, saved):
                    t.copy_(v)
                model.train_engine().packed.refresh()
            torch.cuda.synchronize()

        restore()
        # the capture stream is high priority: the critical chain then wins free SM slots over the weight-gradient
        # side stream (kernel nodes inherit the priority of the stream they were captured on)
        cap = torch.cuda.Stream(device=model.device, priority=-1)
        before = ops.LAUNCHES[0]
        graph = torch.cuda.CUDAGraph()
        try:
            # thread_local: the NCCL watchdog thread may query events of earlier collectives while we capture
            with torch.no_grad(), torch.cuda.graph(graph, stream=cap, capture_error_mode="thread_local"):
                self._run(model, True)
            self.optimizer_in_graph = True
        except Exception:
            if self.allreduce is None:
                raise
            # a collective that cannot be captured (a custom ``allreduce`` callable): optimizer outside the graph
            torch.cuda.synchronize()
            restore()
            ops.LAUNCHES[0] = before
            graph = torch.cuda.CUDAGraph()
            with torch.no_grad(), torch.cuda.graph(graph, stream=cap, capture_error_mode="thread_local"):
                self._run(model, False)
            self.optimizer_in_graph = False
        self.n_kernels = ops.LAUNCHES[0] - before
        ops.LAUNCHES[0] = before
        self.graph = graph
        ops.pin_workspaces()     # the graph bakes the scratch addresses in: they must outlive it


T_MAX = 40      # CosineAnnealingLR(optimizer, T_max=40), ssd3d.py:719


def _optimizer_step(model, flat, world_size, allreduce):
    """(all-reduce) + Adam + re-pack; everything on the device, capturable."""
    if allreduce is not None:
        allreduce(flat.grad)
    ops.adam_step_dev(flat.param, flat.grad, flat.exp_avg, flat.exp_avg_sq, flat.bias_start, float(model.lr),
                      flat.status, flat.scalars, t_max=(T_MAX if model.scheduler != "none" else 0), bias_lr_mult=2.0,
                      weight_decay=0.0005, grad_scale=1.0 / float(world_size))
    model.train_engine().packed.refresh()      # every packed weight layout for the next step: two launches


def _install(model, key, plan: _TrainPlan) -> None:
    """Capture ``plan`` (its inputs staged: the warm-up steps run on them) unless the model runs its steps eagerly,
    and cache it under ``key``; at most 4 plans are kept."""
    if model.use_cuda_graph:
        model.invalidate_packed()
        plan.capture(model)
    plans = model.train_engine().plans
    plans.pop(key, None)
    if len(plans) >= 4:
        plans.clear()
    plans[key] = plan


def _step(model, plan: _TrainPlan) -> None:
    """One optimisation step on ``plan``'s staged inputs: its graph replayed, then the optimizer if the collective
    could not be captured; without a graph (``use_cuda_graph`` False) the same step body runs eagerly."""
    eng = model.train_engine()
    if plan.allreduce is None:
        eng.collective_mode = "none"
    elif plan.optimizer_in_graph:
        eng.collective_mode = "nccl all_reduce of the flat gradient, captured in the step's CUDA graph"
    else:
        eng.collective_mode = "all_reduce after the graph replay"
    with torch.no_grad():
        if plan.graph is None:
            plan._run(model, True)
        else:
            plan.graph.replay()
            ops.LAUNCHES[0] += plan.n_kernels
            if not plan.optimizer_in_graph:
                _optimizer_step(model, plan.flat, plan.world_size, plan.allreduce)


def fit_step(model, batch, world_size: int = 1, allreduce=None):
    """One fused optimisation step: forward, MultiBox loss + its gradient, backward into the flat gradient
    buffer, (all-reduce), fused Adam.  Returns a (2,) device tensor [conf_loss, loc_loss] -- no host sync.
    With ``model.use_cuda_graph`` the whole step is one CUDA-graph replay."""
    images, gt_boxes, gt_labels = batch["img"], batch["boxes"], batch["labels"]
    if images.dtype not in (torch.float32, torch.bfloat16):
        images = images.float()
    model.train_engine().flatten()
    total = sum(int(b.shape[0]) for b in gt_boxes)
    key = (tuple(images.shape), images.dtype, int(world_size), allreduce, bool(model.use_cuda_graph))
    plan = model.train_engine().plans.get(key)
    if plan is None or plan.tmax < total:
        tmax = 64
        while tmax < total:
            tmax *= 2
        plan = _TrainPlan(model, images.shape, images.dtype, tmax, world_size, allreduce)
        plan.load(images, gt_boxes, gt_labels)
        _install(model, key, plan)
    else:
        plan.load(images, gt_boxes, gt_labels)
    _step(model, plan)
    model.invalidate_packed()
    return plan.loss.clone()


class _EpochPlan(_TrainPlan):
    """The fused step fed from a ``DeviceDataset``: the captured graph also samples and augments the batch straight
    into the static image buffer (``ssd3d_augment_batch``; ``ssd3d_augment_affine_batch`` when the augmentation
    draws a rotation and zoom; ``ssd3d_augment_elastic_batch`` when it draws an elastic deformation), then, when the
    augmentation draws MR intensity changes, applies them in place (``ssd3d_augment_intensity_batch``), extracts the
    ground truth of the augmented masks (``ssd3d_gt_boxes_from_segmentation``) and packs it into the static GT
    buffers (``ssd3d_gt_pack``).  The draw state advances inside the graph, so every replay is the next step of the epoch with no host copy or sync."""

    def __init__(self, model, dataset, augment, n: int, per_volume: int, world_size: int, allreduce):
        dev = model.device
        d, h, w = (int(v) for v in model.input_size)
        c = dataset.channels
        super().__init__(model, (n, c, d, h, w), torch.bfloat16, n * per_volume, world_size, allreduce)
        self.dataset, self.augment, self.per_volume = dataset, augment, per_volume
        self.mask = torch.empty((n, d, h, w), dtype=torch.uint8, device=dev)
        words = 33 if augment.elastic_prob > 0 else (32 if augment.affine_prob > 0 else 16)
        self.record = torch.empty((n, words), dtype=torch.int32, device=dev)
        self.order = torch.zeros((len(dataset),), dtype=torch.int32, device=dev)
        # {seed, draw counter, step in epoch, rank, world size, kernel scratch, -, -}
        self.state = torch.zeros((8,), dtype=torch.int64, device=dev)
        self.pack_status = torch.zeros((2,), dtype=torch.int32, device=dev)
        self.gt_out = (torch.empty((n, per_volume, 6), dtype=torch.float32, device=dev),
                       torch.empty((n, per_volume), dtype=torch.int64, device=dev),
                       torch.empty((2, n), dtype=torch.int32, device=dev))
        lib = _lib.load()
        self.gt_ws = torch.empty((lib.ssd3d_gt_boxes_workspace_bytes(n, d, h, w, per_volume),), dtype=torch.uint8,
                                 device=dev)
        if augment.intensity:
            self.intensity_record = torch.empty((n, 27), dtype=torch.int32, device=dev)
            self.intensity_ws = torch.empty((max(1, ops.augment_intensity_workspace_bytes(n, c, d, h, w)),),
                                            dtype=torch.uint8, device=dev)
        self.extra_state = [self.state, self.pack_status]

    def _prepare(self, model):
        a, ds = self.augment, self.dataset
        args = (ds.images, ds.masks, self.order, self.state, ds.boxes, ds.box_offsets, self.n, model.input_size,
                a.pos_ratio, a.flip_prob, a.rot90_prob, a.rot90_axes, a.scale, a.shift)
        if a.elastic_prob > 0:
            ops.augment_elastic_batch(*args, a.affine_prob, a.rotate_range, a.zoom_range, a.elastic_prob,
                                      a.elastic_points, a.elastic_magnitude, out=(self.image, self.mask, self.record))
        elif a.affine_prob > 0:
            ops.augment_affine_batch(*args, a.affine_prob, a.rotate_range, a.zoom_range,
                                     out=(self.image, self.mask, self.record))
        else:
            ops.augment_batch(*args, out=(self.image, self.mask, self.record))
        if a.intensity:
            ops.augment_intensity_batch(self.image, self.state, self.n, a.bias_prob, a.bias_coefficient, a.gamma_prob,
                                        a.gamma_log_range, a.noise_prob, a.noise_std,
                                        out_record=self.intensity_record, workspace=self.intensity_ws)
        boxes, labels, meta = ops.gt_boxes_padded(self.mask, ds.n_classes, self.per_volume, out=self.gt_out,
                                                  workspace=self.gt_ws)
        ops.gt_pack(boxes, labels, meta, self.per_volume, out=(self.gt_boxes, self.gt_labels, self.offsets),
                    status=self.pack_status)

    def start_epoch(self, epoch: int, steps: int, rank: int):
        """Host writes of one epoch, before its first step: the order, the draw state, the overflow count."""
        from .data import epoch_order
        seed = int(self.augment.seed)
        self.order.copy_(epoch_order(len(self.dataset), epoch, seed))
        seed = seed - (1 << 64) if seed >= (1 << 63) else seed
        # draws are a pure function of (seed, epoch, step, slot): the counter of step t of epoch e is e * steps + t
        self.state.copy_(torch.tensor([seed, int(epoch) * steps, 0, rank, self.world_size, 0, 0, 0],
                                      dtype=torch.int64))
        self.pack_status.zero_()


def fit_epoch(model, dataset, batch_size: int, augment=None, epoch: int = 0, world_size: int = 1, allreduce=None,
              rank: int = 0, max_boxes_per_volume: int = 64):
    """One epoch of fused steps over a ``DeviceDataset``; see ``LSSD3D.fit_epoch``."""
    from .data import Augment
    if augment is None:
        augment = Augment()
    if not model.use_cuda_graph:
        raise RuntimeError("fit_epoch runs every step as a CUDA-graph replay; it needs model.use_cuda_graph")
    if dataset.images.device != model.device:
        raise RuntimeError("the data set lives on %s, the model on %s" % (dataset.images.device, model.device))
    if dataset.channels != model.input_channels:
        raise ValueError("the data set has %d channels, the model expects %d" % (dataset.channels,
                                                                                 model.input_channels))
    augment.validate(model.input_size, dataset.shape)
    n, per_volume = int(batch_size), int(max_boxes_per_volume)
    if n < 1 or per_volume < 1:
        raise ValueError("batch_size and max_boxes_per_volume must be >= 1")
    model.train_engine().flatten()
    steps = -(-len(dataset) // (n * world_size))
    key = ("epoch", id(dataset), augment, n, per_volume, tuple(model.input_size), int(world_size), int(rank),
           allreduce)
    plan = model.train_engine().plans.get(key)
    if plan is None or plan.dataset is not dataset:
        plan = _EpochPlan(model, dataset, augment, n, per_volume, world_size, allreduce)
        plan.start_epoch(epoch, steps, rank)
        _install(model, key, plan)
    plan.start_epoch(epoch, steps, rank)
    dev = model.device
    losses = torch.empty((steps, 2), dtype=torch.float32, device=dev)
    subjects = torch.empty((steps, n), dtype=torch.int32, device=dev)
    for i in range(steps):
        _step(model, plan)
        losses[i].copy_(plan.loss)
        subjects[i].copy_(plan.record[:, 0])
    model.invalidate_packed()
    overflows = int(plan.pack_status[1].item())         # the one host read of the epoch
    if overflows:
        raise RuntimeError("%d of %d steps had more ground-truth boxes in a volume than max_boxes_per_volume=%d (or "
                           "more connected components than that); their updates were skipped -- raise "
                           "max_boxes_per_volume" % (overflows, steps, per_volume))
    return losses, subjects
