"""SSD3D detector with the reference's class / method surface (``lesions3d/ssd3d.py``), running on
hand-written sm_100a kernels (``libssd3d_b200.so``).

Drop-in points kept verbatim: ``LSSD3D`` constructor kwargs (ssd3d.py:177-200), ``forward`` ->
``(locs (N,P,6), classes_scores (N,P,n_classes))``, ``detect_objects`` -> three lists of per-image
tensors, ``create_prior_boxes``, ``predict_step``, ``init``, ``configure_optimizers``,
``load_from_checkpoint``; ``MobileNetBase``, ``PredictionConvolutions``, ``MultiBoxLoss`` with their
signatures; parameter names / ``state_dict`` keys (103 tensors incl. the unused ``rescale_factors``).
``SSD3D`` is an alias of ``LSSD3D`` (the name BASELINE.json uses).

What differs from the reference by design (SURVEY.md section 8b):
  * all arithmetic is in CUDA kernels; activations are channels-last-3d bf16 with fp32 accumulation;
  * the reference's per-layer ``isnan().sum() > 0`` host syncs are one device flag, read once;
  * ``detect_objects`` runs fully on the device and reads back only the per-image counts;
  * equal scores are ordered by ascending prior index (the reference's sort leaves ties unspecified);
  * no CPU path: CPU tensors handed to the kernels raise.
"""
from __future__ import annotations

import inspect
import operator
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .mobilenet import MOBILENET_CONFIGS, Block, conv_bn
from .utils import *  # noqa: F401,F403  (the reference does `from utils import *`)
from .utils import cxcycz_to_xyz

try:  # the reference derives from pytorch_lightning.LightningModule; it is optional here
    import pytorch_lightning as pl  # type: ignore
    _LightningBase = pl.LightningModule
    _HAVE_PL = True
except Exception:  # pragma: no cover - PL is absent in the build image
    _HAVE_PL = False

    class _LightningBase(nn.Module):
        """The small part of ``LightningModule`` the SSD3D path touches."""

        def __init__(self):
            super().__init__()
            self.hparams = {}
            self.current_epoch = 0
            self.global_step = 0

        def save_hyperparameters(self, *args, **kwargs):
            frame = inspect.currentframe().f_back
            names = inspect.signature(type(self).__init__).parameters
            self.hparams = {k: frame.f_locals[k] for k in names if k != "self" and k in frame.f_locals}

        def log(self, *args, **kwargs):
            pass

        def lr_schedulers(self):
            return None

        @property
        def device(self):
            for p in self.parameters():
                return p.device
            return torch.device("cpu")

        @classmethod
        def load_from_checkpoint(cls, checkpoint_path, map_location=None, strict=True, **kwargs):
            """Read a PyTorch-Lightning checkpoint dict (``state_dict`` + ``hyper_parameters``), predict.py:257."""
            ckpt = torch.load(checkpoint_path, map_location=map_location or "cpu", weights_only=False)
            hp = dict(ckpt.get("hyper_parameters", {}))
            hp.update(kwargs)
            allowed = inspect.signature(cls.__init__).parameters
            model = cls(**{k: v for k, v in hp.items() if k in allowed})
            model.load_state_dict(ckpt["state_dict"], strict=strict)
            return model


device = torch.device("cuda" if torch.cuda.is_available() else "cpu")   # ssd3d.py:23
_VERSION_OF = operator.attrgetter("_version")

ASPECT_RATIOS = {3: [1.], 5: [1.], 7: [1]}   # ssd3d.py:25


class MobileNetBase(nn.Module):
    """Truncated 3-D MobileNet-v1 feature extractor (ssd3d.py:47-110)."""

    def __init__(self, config="mobilenet", in_channels=1, width_mult=1., cube=False, aspect_ratios=None):
        super(MobileNetBase, self).__init__()
        if aspect_ratios is None:
            aspect_ratios = ASPECT_RATIOS
        self.aspect_ratios = aspect_ratios
        self.in_channels = in_channels
        self.config = MOBILENET_CONFIGS[config]
        input_channel = int(self.config[0] * width_mult)
        cfg = self.config[1:]
        first_stride = (1, 2, 2) if not cube else (2, 2, 2)
        features = [conv_bn(in_channels, input_channel, first_stride)]
        last = max(self.aspect_ratios.keys())
        for c, n, s in cfg:
            if len(features) - 1 == last:   # truncate the network after the last prediction layer
                break
            output_channel = int(c * width_mult)
            for i in range(n):
                if len(features) - 1 == last:
                    break
                stride = s if i == 0 else 1
                features.append(Block(input_channel, output_channel, stride))
                input_channel = output_channel
        self.features = nn.Sequential(*features)
        self._nan_flag: Optional[torch.Tensor] = None

    def init(self):
        for c in self.children():
            if isinstance(c, nn.Conv3d):
                nn.init.kaiming_uniform_(c.weight)
                nn.init.constant_(c.bias, 0.)

    def nan_flag(self, dev) -> torch.Tensor:
        """Device int32 the kernels OR NaN bits into (replaces the syncs at mobilenet.py:46, ssd3d.py:95)."""
        if self._nan_flag is None or self._nan_flag.device != dev:
            self._nan_flag = torch.zeros((1,), dtype=torch.int32, device=dev)
            for f in self.features:
                if isinstance(f, Block):
                    f.nan_flag = self._nan_flag
        return self._nan_flag

    def use_nan_flag(self, flag: torch.Tensor) -> torch.Tensor:
        """Route the blocks' NaN bits into ``flag`` (a captured inference plan owns its word); returns the
        previous one."""
        prev = self._nan_flag
        self._nan_flag = flag
        for f in self.features:
            if isinstance(f, Block):
                f.nan_flag = flag
        return prev

    def forward(self, image, check_nan: bool = True, stem_out=None, fuse: bool = True):
        """``stem_out``: the already-computed output of features[0] (the captured inference plan runs the
        stem eagerly on the caller's tensor and replays the rest from a static buffer).  ``fuse``: see
        ``Block.forward``."""
        flag = self.nan_flag(image.device if stem_out is None else stem_out.device)
        out = image
        wanted = list(self.aspect_ratios.keys())
        out_features = {}
        for i, feat in enumerate(self.features):
            if i == 0:
                out = feat(out) if stem_out is None else stem_out
            else:
                out = feat(out, fuse=fuse)
            if i in wanted:
                out_features[i] = out
        if check_nan and int(flag.item()) & _lib.NAN_BACKBONE:
            flag.zero_()
            print("Yesssss this NaN error again in the base network")
            raise Exception("Yesssss this NaN error again in the base network")   # ssd3d.py:95-98
        return out_features

    def get_feature_map_infos(self, input_size, device=None):
        """Spatial size and channel count after every layer (ssd3d.py:102-110), computed from the layer
        parameters instead of a dummy forward."""
        cur = tuple(int(v) for v in input_size)
        dims, chans = {}, []
        for i, l in enumerate(self.features):
            conv = l[0] if isinstance(l, nn.Sequential) else l.conv1
            st = conv.stride if isinstance(conv.stride, tuple) else (conv.stride,) * 3
            cur = tuple(ops.conv_out(cur[a], st[a]) for a in range(3))
            dims[i] = cur
            chans.append(l[0].out_channels if isinstance(l, nn.Sequential) else l.conv2.out_channels)
        return dims, chans


class PredictionConvolutions(nn.Module):
    """Localisation and class prediction convolutions over the selected feature maps (ssd3d.py:113-169).
    Both 3x3x3 convs of a feature map run as one tcgen05 implicit GEMM."""

    def __init__(self, n_classes, width_mult, aspect_ratios, features_n_channels, boxes_per_location=2):
        super(PredictionConvolutions, self).__init__()
        self.n_classes = n_classes
        self.aspect_ratios = aspect_ratios
        n_boxes = {feat: len(aspect_ratios[feat]) + boxes_per_location - 1 for feat in aspect_ratios}
        self.n_boxes = n_boxes
        loc_convs, cl_convs = [], []
        for f in aspect_ratios:
            f_n_channels = int(features_n_channels[f] * width_mult)   # width_mult applied twice, as ssd3d.py:130
            loc_convs.append(nn.Conv3d(f_n_channels, n_boxes[f] * 6, kernel_size=3, padding=1))
            cl_convs.append(nn.Conv3d(f_n_channels, n_boxes[f] * n_classes, kernel_size=3, padding=1))
        self.loc_convs = nn.ModuleList(loc_convs)
        self.cl_convs = nn.ModuleList(cl_convs)
        self._packed = None
        self._packed_kw = None
        self._packed_key = None

    def init(self):
        for c in self.children():
            if isinstance(c, nn.Conv3d):
                nn.init.kaiming_uniform_(c.weight)
                nn.init.constant_(c.bias, 0.)

    def _pack(self):
        tensors = []
        for lc, cc in zip(self.loc_convs, self.cl_convs):
            tensors += [lc.weight, lc.bias, cc.weight, cc.bias]
        key = tuple((t.data_ptr(), t._version) for t in tensors)
        if self._packed is None or key != self._packed_key:
            self._packed = [ops.pack_head_weight(lc.weight, lc.bias, cc.weight, cc.bias)
                            for lc, cc in zip(self.loc_convs, self.cl_convs)]
            # the kw-GEMM head kernel's own tiling, once per weight version (C % 64 == 0, 16 output columns)
            self._packed_kw = [ops.pack_head_weight_kw(w) if (w.is_cuda and w.shape[0] == 16 and (w.shape[1] // 27) % 64 == 0)
                               else None for w, _ in self._packed]
            self._packed_key = key
        return self._packed

    def forward(self, feats, nan_flag: Optional[torch.Tensor] = None, out=None):
        if self.training and torch.is_grad_enabled() and out is None:
            # stand-alone use with gradients (ssd3d.py:134-169 under autograd): one autograd node over the head kernels
            from .train_modules import heads_train
            return heads_train(self, feats, nan_flag)
        feat_keys = list(feats.keys())
        first = feats[min(feat_keys)]
        batch_size = first.size(0)
        packed = self._pack()
        counts = []
        for i, key in enumerate(feat_keys):
            _, _, d, h, w = feats[key].shape
            counts.append(d * h * w * self.n_boxes[list(self.aspect_ratios.keys())[i]])
        total = int(sum(counts))
        if out is None:
            locs = torch.empty((batch_size, total, 6), dtype=torch.float32, device=first.device)
            classes_scores = torch.empty((batch_size, total, self.n_classes), dtype=torch.float32, device=first.device)
        else:
            locs, classes_scores = out
        off = 0
        for i, key in enumerate(feat_keys):
            self.run_head(i, feats[key], locs, classes_scores, off, nan_flag)
            off += counts[i]
        return locs, classes_scores

    def run_head(self, i, feat, locs, classes_scores, prior_offset, nan_flag=None):
        """Head ``i`` (i-th prediction layer) on its feature map, written at ``prior_offset``."""
        w, b = self._pack()[i]
        bpl = self.n_boxes[list(self.aspect_ratios.keys())[i]]
        w_kw = self._packed_kw[i]
        if w_kw is not None and ops.head_kw_supported(feat, w.shape[0]):
            ops.head_conv(feat, w_kw, b, locs, classes_scores, bpl, self.n_classes, prior_offset, nan_flag, algo=4)
        else:
            ops.head_conv(feat, w, b, locs, classes_scores, bpl, self.n_classes, prior_offset, nan_flag)


TAIL_FROM = 3   # first backbone layer of a captured inference plan on the high-priority stream


def _checked_counts(meta: List[int], n_out: int) -> List[int]:
    """Decode a read-back vector ``[per-output counts | detect status words | NaN bits]``: raise on its NaN bits
    and status words, return the counts."""
    status = 0
    for word in meta[n_out:-1]:
        status |= word
    ops.raise_on_status(meta[-1], status)
    return meta[:n_out]


class _InferencePlan:
    """forward + detect_objects for one input signature, captured once into a CUDA graph.

    The network is 19 small kernels (~20 us each at the benchmark size) plus 4 detection kernels: launched
    one by one from Python the step is host-bound, so the whole sequence is recorded on first use and
    replayed with a single launch.  Outputs live in static buffers; the per-output counts, the detect status
    words and the plan's NaN word are one int32 vector that is read back with a single device->host copy.

    A batch plan (``overlap`` None) takes an image batch of ``shape``.  The stem runs outside the graph, so that
    a device-resident batch is consumed in place (no staging copy of the largest tensor of the step); a host batch
    goes through the static input buffer.

    A window plan (``overlap`` given) takes ``shape[0]`` whole scans of ``shape``: the graph also gathers their
    ``input_size`` windows into the network's input batch (csrc/windows.cu) in front -- so the stem is inside, its
    input being the plan's own buffer -- and merges the per-window detections into per-scan ones behind.  The scans
    are copied into the static input buffer before each replay."""

    def __init__(self, model: "LSSD3D", shape, dtype, fuse_blocks: bool, overlap: Optional[float] = None):
        dev = model.device
        self.fuse_blocks = fuse_blocks      # Blocks run as the fused depthwise->pointwise kernel where it applies
        self.args = (model.min_score, model.max_overlap, int(model.top_k))
        self.inp = torch.zeros(shape, dtype=dtype, device=dev)
        self.windowed = overlap is not None
        if self.windowed:
            from .data import window_origins
            s, c = int(shape[0]), int(shape[1])
            self.window = tuple(int(v) for v in model.input_size)
            self.overlap = float(overlap)
            self.scan_spatial = tuple(int(v) for v in shape[2:])
            nd, nh, nw, origins = window_origins(self.scan_spatial, self.window, self.overlap)
            self.offset = ops.window_map(self.scan_spatial, self.window, origins)[1].to(dev)
            self.merge_ws = torch.empty((_lib.load().ssd3d_merge_windows_workspace_bytes(
                s, nd * nh * nw, self.args[2], model.n_classes, self.args[2]),), dtype=torch.uint8, device=dev)
            self.windows = torch.zeros((s * nd * nh * nw, c) + self.window, dtype=torch.bfloat16, device=dev)
            net_in = self.windows
        else:
            net_in = self.inp
        self.n, self.n_out = int(net_in.shape[0]), int(shape[0])
        # [per-output counts | detect status (| merge status) | NaN bits]; the NaN word is the plan's own (plans may
        # overlap), the last element of this vector
        n_status = 2 if self.windowed else 1
        self.meta = torch.zeros((self.n_out + n_status + 1,), dtype=torch.int32, device=dev)
        self.host_meta = torch.zeros_like(self.meta, device="cpu").pin_memory()
        self.flag = self.meta[-1:]
        self.out = None
        self.done = torch.cuda.Event()       # graph + metadata read-back of the latest launch finished
        self.cloned = torch.cuda.Event()     # results of the latest launch were copied out of the static buffers
        self.copied = torch.cuda.Event()     # the latest host input has arrived in the static input buffer
        self.stem = model.base.features[0]
        self.stream = torch.cuda.Stream(device=dev)                     # compute stream of the streaming API
        # Later stages run at higher stream priority (recorded into the graph's kernel nodes): when two batches
        # are in flight, the latency-bound tail of the older one (small maps, heads, sort/NMS: a few CTAs each)
        # takes SM slots as soon as CTAs of the younger batch's big layers retire, instead of queueing behind them.
        self.head_streams = [torch.cuda.Stream(device=dev, priority=-1) for _ in model.aspect_ratios]
        self.tail_stream = torch.cuda.Stream(device=dev, priority=-1)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            self.stem_out = self.stem(net_in)   # static buffer the captured graph reads
            for _ in range(2):                # warm-up: lazy module loading, function attributes, packing
                self._run(model)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        before = ops.LAUNCHES[0]
        with torch.no_grad(), torch.cuda.graph(graph):
            self._run(model)
        self.n_kernels = ops.LAUNCHES[0] - before     # library kernels in the graph
        self.graph = graph

    def _run(self, model: "LSSD3D"):
        model.base.nan_flag(self.inp.device)
        prev_flag = model.base.use_nan_flag(self.flag)
        try:
            self._run_with_flag(model, self.flag)
        finally:
            model.base.use_nan_flag(prev_flag)

    def _run_with_flag(self, model: "LSSD3D", flag: torch.Tensor):
        dev = self.inp.device
        flag.zero_()
        net_in = self.inp
        if self.windowed:
            net_in = ops.window_gather(self.inp, self.window, self.overlap, out=self.windows)
            self.stem(net_in, out=self.stem_out)
        # Backbone on the main stream; every head forks onto its own stream as soon as its feature map
        # exists, so the head GEMMs overlap the small tail layers (which leave most SMs idle) and join
        # before detection.  Captured, these become parallel branches of the graph.
        main = torch.cuda.current_stream()
        base, pc = model.base, model.pred_convs
        keys = list(model.aspect_ratios.keys())
        dims, _ = base.get_feature_map_infos(tuple(net_in.shape[2:]))
        counts = [dims[k][0] * dims[k][1] * dims[k][2] * pc.n_boxes[k] for k in keys]
        offs = [int(sum(counts[:j])) for j in range(len(keys))]
        locs = torch.empty((self.n, int(sum(counts)), 6), dtype=torch.float32, device=dev)
        scores = torch.empty((self.n, int(sum(counts)), pc.n_classes), dtype=torch.float32, device=dev)
        out, keep_alive = self.stem_out, []
        cur = main
        tail = self.tail_stream
        for i, feat in enumerate(base.features):
            if i == TAIL_FROM and cur is main:
                tail.wait_stream(main)
                cur = tail
            with torch.cuda.stream(cur):
                if i > 0:
                    out = feat(out, fuse=self.fuse_blocks)
                if i in keys:
                    j = keys.index(i)
                    keep_alive.append(out)
                    hs = self.head_streams[j]
                    hs.wait_stream(cur)
                    with torch.cuda.stream(hs):
                        pc.run_head(j, out, locs, scores, offs[j], flag)
        if cur is main:
            tail.wait_stream(main)
        ms, mo, k = self.args
        n_out = self.n_out
        # one packed result buffer (labels | prior | boxes | scores) so that handing results out is ONE copy
        detected = torch.empty((self.n * k * 44,), dtype=torch.uint8, device=dev)
        with torch.cuda.stream(tail):
            for hs in self.head_streams:
                tail.wait_stream(hs)
            self.out = ops.detect_objects_padded(locs, scores, model._prior_source(dev), ms, mo, k,
                                                 out_count=None if self.windowed else self.meta[:n_out],
                                                 status=self.meta[n_out:n_out + 1], out=self._views(detected, k))
        main.wait_stream(tail)
        self.locs, self.scores = locs, scores
        if self.windowed:
            self.result = torch.empty((n_out * k * 44,), dtype=torch.uint8, device=dev)
            win = self.out
            ops.merge_windows(win.boxes, win.scores, win.labels, win.count, n_out, self.scan_spatial, self.window,
                              self.overlap, model.n_classes, ms, mo, k, offset=self.offset, workspace=self.merge_ws,
                              out=self._views(self.result, k), out_count=self.meta[:n_out],
                              status=self.meta[n_out + 1:n_out + 2])
        else:
            self.result = detected

    @staticmethod
    def _views(buf: torch.Tensor, k: int):
        """(boxes (N,K,6) f32, scores (N,K) f32, labels (N,K) i64, prior (N,K) i64) views of a packed buffer."""
        n = buf.numel() // (44 * k)
        nk = n * k
        labels = buf[:nk * 8].view(torch.int64).view(n, k)
        prior = buf[nk * 8:nk * 16].view(torch.int64).view(n, k)
        boxes = buf[nk * 16:nk * 40].view(torch.float32).view(n, k, 6)
        scores = buf[nk * 40:nk * 44].view(torch.float32).view(n, k)
        return boxes, scores, labels, prior

    def launch(self, x: torch.Tensor, copy_stream=None, own_stream: bool = False, caller_stream=None):
        """Queue one step: a host input is first copied into the static input buffer (on ``copy_stream`` if given,
        so that the copy overlaps the previous step), then a batch plan runs the stem, then the captured graph is
        replayed and the read-back vector copied to the host asynchronously.  With ``own_stream`` the step runs on
        this plan's stream (after everything already queued on the caller's stream), so that consecutive steps on
        different plan slots overlap: the small tail layers of one step leave most SMs idle for the big first
        layers of the next."""
        if own_stream:
            caller = caller_stream if caller_stream is not None else torch.cuda.current_stream()
            self.stream.wait_stream(caller)
            torch.cuda.set_stream(self.stream)       # (the context manager costs several current_stream() calls)
            try:
                self._launch(x, copy_stream, self.stream)
            finally:
                torch.cuda.set_stream(caller)
        else:
            self._launch(x, copy_stream, caller_stream if caller_stream is not None else torch.cuda.current_stream())

    def _launch(self, x: torch.Tensor, copy_stream, compute):
        compute.wait_event(self.cloned)          # static outputs of the previous use of this plan were consumed
        if x.is_cuda and not self.windowed:
            # the batch (or its dtype-converted temporary) was allocated on the caller's stream but is read by the
            # stem on `compute`: tell the caching allocator, or the block could be handed out again while the
            # kernel still reads it (up to pipeline_depth batches are in flight)
            x.record_stream(compute)
            self.stem(x, out=self.stem_out)
        else:
            if x.is_cuda or copy_stream is None:
                self.inp.copy_(x, non_blocking=True)
            else:
                torch.cuda.set_stream(copy_stream)
                try:
                    copy_stream.wait_event(self.done)    # the previous step that read this buffer has run
                    self.inp.copy_(x, non_blocking=True)
                    self.copied.record(copy_stream)
                finally:
                    torch.cuda.set_stream(compute)
                compute.wait_event(self.copied)
            if not self.windowed:
                self.stem(self.inp, out=self.stem_out)
        self.graph.replay()
        ops.LAUNCHES[0] += self.n_kernels
        self.host_meta.copy_(self.meta, non_blocking=True)
        self.done.record(compute)

    def results(self, post_stream=None, to_host: bool = False, caller_stream=None):
        """Wait for this plan's latest launch (not for later work on the stream), check the flags, and hand
        out fresh per-output tensors: the static buffers are copied on ``post_stream`` (device clones, or
        pinned-host copies when ``to_host``) so that the next steps already queued are not delayed."""
        self.done.synchronize()
        counts = _checked_counts(self.host_meta.tolist(), self.n_out)
        current = caller_stream if caller_stream is not None else torch.cuda.current_stream()
        stream = post_stream if post_stream is not None else current
        if stream is not current:
            torch.cuda.set_stream(stream)
        try:
            buf = self.result.to("cpu", non_blocking=False) if to_host else self.result.clone()
            self.cloned.record(stream)
        finally:
            if stream is not current:
                torch.cuda.set_stream(current)
        if not to_host and stream is not current:
            current.wait_event(self.cloned)      # later work on the caller's stream sees complete tensors
            buf.record_stream(current)           # allocated on `stream`, used (and eventually freed) by the caller's
        boxes, scores, labels, _ = self._views(buf, self.args[2])
        return ([boxes[i, :k] for i, k in enumerate(counts)], [labels[i, :k] for i, k in enumerate(counts)],
                [scores[i, :k] for i, k in enumerate(counts)])


class LSSD3D(_LightningBase):
    """The SSD 3D network - the base MobileNet network and the prediction convolutions (ssd3d.py:172-738)."""

    def __init__(self,
                 n_classes,
                 input_channels=3,
                 input_size=(64, 64, 64),
                 threshold=0.5,  # threshold for box matching in MultiBoxLoss
                 alpha=1.,
                 lr=1.3e-5,
                 base_network_config="mobilenet",
                 width_mult=1.,
                 min_score=0.5,
                 max_overlap=0.5,  # for box matching
                 min_overlap=0.5,  # for evaluation metrics
                 top_k=100,
                 scheduler="CosineAnnealingLR",
                 use_wandb=False,
                 batch_size=8,
                 compute_metric_every_n_epochs=1,
                 comments="",
                 aspect_ratios={},
                 min_object_size=6,
                 max_object_size=14,
                 scales={},
                 boxes_per_location=2
                 ):
        super(LSSD3D, self).__init__()
        if aspect_ratios == {}:
            aspect_ratios = ASPECT_RATIOS
        self.save_hyperparameters()
        self.base_network_config = base_network_config
        self.cube = input_size[0] == input_size[1] == input_size[2]
        self.input_size = input_size
        self.input_channels = input_channels
        self.width_mult = width_mult
        self.aspect_ratios = aspect_ratios
        self.boxes_per_location = 2   # the kwarg is ignored, as in ssd3d.py:213

        self.n_classes = n_classes
        self._make_base_and_prediction_layers()
        self.lr = lr
        self.min_score = min_score
        self.max_overlap = max_overlap
        self.min_overlap = min_overlap
        self.top_k = top_k
        self.scheduler = scheduler
        self.use_wandb = use_wandb
        self.batch_size = batch_size
        self.compute_metric_every_n_epochs = compute_metric_every_n_epochs
        self.comments = comments

        if scales == {}:
            self.scales = {layer: scale for layer, scale in zip(self.aspect_ratios.keys(),
                                                                np.linspace(min_object_size / input_size[0],
                                                                            max_object_size / input_size[0],
                                                                            len(self.aspect_ratios)))}
        else:
            self.scales = scales

        features_n_channels = self.base.get_feature_map_infos(self.input_size)[1]
        n_channel_rescale = int(features_n_channels[min(self.aspect_ratios.keys())] * self.width_mult)
        # kept for checkpoint compatibility; unused in forward exactly as in the reference (ssd3d.py:240-254)
        self.rescale_factors = nn.Parameter(torch.FloatTensor(1, n_channel_rescale, 1, 1, 1))
        nn.init.constant_(self.rescale_factors, 20)

        self.priors_cxcycz = self.create_prior_boxes()
        self.__dict__["_priors_origin"] = self.priors_cxcycz
        self.__dict__["_priors_version"] = self.priors_cxcycz._version
        self.loss_fn = MultiBoxLoss(self.priors_cxcycz, threshold=threshold, alpha=alpha)
        self.defer_nan_check = False
        self.use_cuda_graph = True     # predict_step replays a captured forward+detect graph
        self.pipeline_depth = 6        # batches in flight in predict_batches
        self._plans = {}

    # ------------------------------------------------------------------------------------------
    def _make_base_and_prediction_layers(self):
        if 'mobilenet' in self.base_network_config:
            self.base = MobileNetBase(config=self.base_network_config, in_channels=self.input_channels,
                                      width_mult=self.width_mult, cube=self.cube, aspect_ratios=self.aspect_ratios)
            features_n_channels = self.base.get_feature_map_infos(self.input_size)[1]
            # The reference measures the shapes with a dummy forward of torch.randn(...) here
            # (ssd3d.py:102-103,270); drawing the same numbers keeps the global RNG stream -- and hence the
            # default initialisation of the head convs that follow -- identical for a given manual_seed.
            torch.randn((1, self.input_channels, *self.input_size))
            self.pred_convs = PredictionConvolutions(self.n_classes, width_mult=self.width_mult,
                                                     aspect_ratios=self.aspect_ratios,
                                                     features_n_channels=features_n_channels,
                                                     boxes_per_location=self.boxes_per_location)
        elif 'convnet' in self.base_network_config:
            # the reference's branch is itself broken (self.boxes.per_location, ssd3d.py:281) and needs MONAI
            raise NotImplementedError("the 'convnet' base network is outside the accelerated SSD3D-MobileNet path")
        else:
            raise Exception(
                f"Unknown base network name. Expected 'mobilenet' or 'convnet' but got {self.base_network_config}")

    def create_prior_boxes(self, per_feature_map=False):
        """Prior (default) boxes in centre-size coordinates, (P, 6) fp32 (ssd3d.py:286-342).

        Same float64 arithmetic per box as the reference's Python triple loop, vectorised; note the axis
        quirk kept from ssd3d.py:304-309 (cx follows array axis 1, cy axis 0)."""
        features = list(self.aspect_ratios.keys())
        fmd = self.base.get_feature_map_infos(self.input_size)[0]
        chunks, per_map = [], {}
        for fmap in features:
            d0, d1, d2 = fmd[fmap]
            s = float(self.scales[fmap])
            cy = (np.arange(d0, dtype=np.float64) + 0.5) / d0
            cx = (np.arange(d1, dtype=np.float64) + 0.5) / d1
            cz = (np.arange(d2, dtype=np.float64) + 0.5) / d2
            CY, CX, CZ = np.meshgrid(cy, cx, cz, indexing="ij")
            sizes = self._prior_sizes(fmap)
            per = np.empty((d0, d1, d2, len(sizes), 6), dtype=np.float64)
            per[..., 0] = CX[..., None]
            per[..., 1] = CY[..., None]
            per[..., 2] = CZ[..., None]
            per[..., 3:] = np.asarray(sizes, dtype=np.float64)[None, None, None, :, None]
            chunks.append(per.reshape(-1, 6))
            per_map[fmap] = per.reshape(-1, 6).tolist() if per_feature_map else None
        if per_feature_map:
            return per_map
        prior_boxes = torch.tensor(np.concatenate(chunks, 0), dtype=torch.float32).to(device)
        prior_boxes.clamp_(0, 1)
        return prior_boxes

    def _prior_sizes(self, fmap):
        """Box edges at one location of prediction layer ``fmap`` as Python floats (ssd3d.py:311-330)."""
        s = float(self.scales[fmap])
        sizes = []
        for ratio in self.aspect_ratios[fmap]:
            sizes.append(s)
            if ratio == 1.:
                for div in list(range(1, self.boxes_per_location)):
                    sizes.append(s + s / div)
        return sizes

    # ------------------------------------------------------------------------------------------
    def _priors_on(self, dev) -> torch.Tensor:
        if self.priors_cxcycz.device != dev:
            mine = (self.priors_cxcycz is self.__dict__.get("_priors_origin")
                    and self.priors_cxcycz._version == self.__dict__.get("_priors_version"))
            self.priors_cxcycz = self.priors_cxcycz.to(dev)
            if mine:
                self.__dict__["_priors_origin"] = self.priors_cxcycz
                self.__dict__["_priors_version"] = self.priors_cxcycz._version
            self.loss_fn.set_priors(self.priors_cxcycz)
        return self.priors_cxcycz

    def _prior_source(self, dev):
        """What the decode / matching kernels take their priors from: the closed-form table (SURVEY.md 8f rank 3:
        every prior is recomputed from its index in float64 -> fp32, bit-identical to ``create_prior_boxes`` -- no
        24-byte read per prior) while ``priors_cxcycz`` is still the constructor's tensor; the tensor itself once a
        caller has replaced or edited it (it is a public attribute of the reference's class)."""
        pri = self._priors_on(dev)
        if pri is not self.__dict__.get("_priors_origin") or pri._version != self.__dict__.get("_priors_version"):
            return pri
        tbl = self.__dict__.get("_prior_table")
        if tbl is None or tbl.dev.device != dev:
            fmd = self.base.get_feature_map_infos(self.input_size)[0]
            keys = list(self.aspect_ratios.keys())
            if len(keys) > _lib.MAX_PRIOR_LAYERS or any(len(self._prior_sizes(k)) > _lib.MAX_PRIOR_SIZES for k in keys):
                return pri
            tbl = ops.PriorTable([fmd[k] for k in keys], [self._prior_sizes(k) for k in keys], dev)
            if tbl.count != pri.shape[0]:
                return pri
            self.__dict__["_prior_table"] = tbl
        return tbl

    def _raise_on_nan(self, flag: torch.Tensor):
        bits = int(flag.item())
        if bits:
            flag.zero_()
        ops.raise_on_status(bits)

    def forward(self, image):
        """image (N, Cin, D, H, W) -> locs (N,P,6), classes_scores (N,P,n_classes) fp32 (ssd3d.py:248-263).
        In training mode BatchNorm uses batch statistics (and updates its running ones) and the outputs carry
        an autograd node whose backward runs the hand-written gradient kernels (training.py)."""
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("LSSD3D.forward needs the model on a CUDA device; there is no CPU path")
        if self.training:
            from . import training
            if torch.is_grad_enabled():
                locs, classes_scores = training.forward_train(self, image)
            else:
                locs, classes_scores = self.train_engine().forward(image)
            if not self.defer_nan_check:
                self._raise_on_nan(self.base.nan_flag(dev))
            return locs, classes_scores
        if image.device != dev:
            image = image.to(dev, non_blocking=True)
        flag = self.base.nan_flag(dev)
        feats = self.base(image, check_nan=False)
        locs, classes_scores = self.pred_convs(feats, flag)
        if not self.defer_nan_check:
            self._raise_on_nan(flag)
        return locs, classes_scores

    def detect_objects(self, predicted_locs, predicted_scores, min_score, max_overlap, top_k, return_prior=False):
        """Decode + per-class NMS + top-k (ssd3d.py:344-460) -> lists of per-image boxes, labels, scores."""
        priors = self._prior_source(predicted_locs.device)
        if ops.detect_needs_long_lists(self.priors_cxcycz.shape[0], top_k):
            # NMS-stress settings (model_insight.py:146: min_score=0, top_k=50000): lists of any length
            return ops.detect_objects_long(predicted_locs, predicted_scores, priors, min_score, max_overlap, top_k,
                                           return_prior=return_prior)
        out = ops.detect_objects_padded(predicted_locs, predicted_scores, priors, min_score, max_overlap, top_k)
        return ops.detect_lists(out, return_prior=return_prior)

    def init(self):
        print("[INFO] Initializing model weights")
        self.base.init()
        self.pred_convs.init()

    # ------------------------------------------------------------------------------------------
    def _state_version(self):
        """Cheap fingerprint of everything a captured plan depends on besides the input signature: in-place
        updates of any parameter / buffer bump its version counter; moves and dtype changes go through
        ``_apply`` which drops the plans."""
        ts = self.__dict__.get("_state_tensors")
        if ts is None:
            ts = list(self.parameters()) + list(self.buffers())
            self.__dict__["_state_tensors"] = ts
        return sum(map(_VERSION_OF, ts))

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.get("_plans", {}).clear()
        self.__dict__["_state_tensors"] = None
        eng = self.__dict__.get("_train_engine")
        if eng is not None:      # parameters are about to be replaced: the flat buffers / packed views die with them
            eng.flat, eng.packed = None, None
            eng.plans.clear()
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self.__dict__.get("_plans", {}).clear()
        self.__dict__["_state_tensors"] = None
        out = super().load_state_dict(*args, **kwargs)
        eng = self.__dict__.get("_train_engine")
        if eng is not None and eng.packed is not None:
            eng.packed.refresh()     # values were copied into the flat buffer in place
        return out

    def _plan_for(self, image: torch.Tensor, slot: int = 0, fuse_blocks: bool = True,
                  overlap: Optional[float] = None) -> _InferencePlan:
        """The captured plan of pipeline slot ``slot`` for ``image``: a batch, or with ``overlap`` scans to tile into
        windows.  Plans are recaptured when the model's state changed since, and all are dropped past 24."""
        if self.training:
            raise RuntimeError("predict_step needs eval() mode (BatchNorm running statistics)")
        dtype = image.dtype if image.dtype in (torch.float32, torch.bfloat16) else torch.float32
        key = (tuple(image.shape), dtype, None if overlap is None else float(overlap), str(self.device),
               float(self.min_score), float(self.max_overlap), int(self.top_k), slot, fuse_blocks)
        ver = self._state_version()
        plan = self._plans.get(key)
        if plan is None or plan.key != ver:
            if len(self._plans) > 24:
                self._plans.clear()
            plan = _InferencePlan(self, tuple(image.shape), dtype, fuse_blocks, overlap)
            plan.key = ver
            self._plans[key] = plan
        return plan

    def _pipelined(self, inputs, depth: int, fuse_blocks: bool, overlap: Optional[float], to_host: bool):
        """Generator of per-step (boxes, labels, scores) over the tensors ``inputs``, software-pipelined over ``depth``
        plan slots: input i+1 is copied (copy stream) and launched before the host waits for step i, and step i's
        results leave the static buffers on a third stream."""
        if self.__dict__.get("_copy_stream") is None:
            self.__dict__["_copy_stream"] = torch.cuda.Stream(device=self.device)
            self.__dict__["_post_stream"] = torch.cuda.Stream(device=self.device)
        copy_stream, post_stream = self.__dict__["_copy_stream"], self.__dict__["_post_stream"]
        caller = torch.cuda.current_stream()
        inflight = []
        slot = 0
        for x in inputs:
            if len(inflight) == depth:
                yield inflight.pop(0).results(post_stream, to_host, caller)
            plan = self._plan_for(x, slot, fuse_blocks, overlap)
            if x.dtype != plan.inp.dtype:
                x = x.to(plan.inp.dtype)
            plan.launch(x, copy_stream, own_stream=True, caller_stream=caller)
            inflight.append(plan)
            slot = (slot + 1) % depth
        while inflight:
            yield inflight.pop(0).results(post_stream, to_host, caller)

    def predict_step(self, batch, batch_idx: int = 0, dataloader_idx: int = None):
        """forward + detect_objects (ssd3d.py:692-702): eager stem + one CUDA-graph replay and a single host
        sync for the whole batch.  ``batch["img"]`` may live on the host (pinned memory makes the copy
        asynchronous)."""
        image = batch["img"]
        if not self.use_cuda_graph or ops.detect_needs_long_lists(self.priors_cxcycz.shape[0], self.top_k):
            return self._predict_step_eager(image)
        if self.device.type != "cuda":
            raise RuntimeError("LSSD3D.predict_step needs the model on a CUDA device; there is no CPU path")
        plan = self._plan_for(image)
        plan.launch(image if image.dtype == plan.inp.dtype else image.to(plan.inp.dtype))
        return plan.results()

    def predict_batches(self, batches, to_host: bool = False):
        """Generator over an iterable of batches (dicts with "img", as a DataLoader yields them) -> per-batch
        (boxes, labels, scores).  What ``Trainer.predict(model, loader)`` does in the reference
        (predict.py:262-263), software-pipelined over ``pipeline_depth`` plan slots: batch i+1 is copied (copy
        stream) and launched before the host waits for batch i, and batch i's results leave the static buffers on a
        third stream.  ``to_host=True`` returns CPU tensors (one device->host copy per output)."""
        if self.device.type != "cuda":
            raise RuntimeError("LSSD3D.predict_batches needs the model on a CUDA device; there is no CPU path")
        if ops.detect_needs_long_lists(self.priors_cxcycz.shape[0], self.top_k):
            for batch in batches:          # candidate lists of any length: no captured plan, one batch at a time
                b, l, s = self._predict_step_eager(batch["img"])
                yield ([t.cpu() for t in b], [t.cpu() for t in l], [t.cpu() for t in s]) if to_host else (b, l, s)
            return
        yield from self._pipelined((batch["img"] for batch in batches), max(1, int(self.pipeline_depth)), False,
                                   None, to_host)

    def predict_scans(self, scans, overlap: float = 0.5, scans_per_step: int = 1, to_host: bool = False):
        """Sliding-window detection over whole scans larger than ``input_size`` -> per-scan lists (boxes, labels,
        scores), boxes as fractions of the scan's shape (the coordinates ``gt_boxes_from_segmentation`` gives for the
        scan's mask).  ``scans``: normalised volumes (S, C, D, H, W) on the host or the device, or a
        ``data.DeviceDataset``.  Every scan is tiled into ``input_size`` windows (``data.window_origins``); each
        step -- one CUDA-graph replay over ``scans_per_step`` scans -- gathers the windows, runs the network and
        ``detect_objects`` on them as one batch, maps the detections into the scan and merges them per scan and
        class with the same sort -> truncation -> greedy NMS -> top-k (``min_score``, ``max_overlap``, ``top_k``
        apply per window and in the merge).  One device->host read per step; steps are pipelined over plan slots
        like ``predict_batches``.  One window over a scan of exactly ``input_size`` gives ``predict_step``'s result."""
        from .data import DeviceDataset, window_origins
        if self.device.type != "cuda":
            raise RuntimeError("LSSD3D.predict_scans needs the model on a CUDA device; there is no CPU path")
        if self.training:
            raise RuntimeError("predict_scans needs eval() mode (BatchNorm running statistics)")
        vols = scans.images if isinstance(scans, DeviceDataset) else scans
        if not isinstance(vols, torch.Tensor):
            vols = torch.as_tensor(np.ascontiguousarray(vols))
        if vols.dim() != 5:
            raise ValueError("scans must be (S, C, D, H, W), got %r" % (tuple(vols.shape),))
        if int(vols.shape[1]) != int(self.input_channels):
            raise ValueError("scans have %d channels, the model takes %d" % (int(vols.shape[1]), self.input_channels))
        nd, nh, nw, _ = window_origins(vols.shape[2:], self.input_size, overlap)
        if ops.detect_needs_long_lists(nd * nh * nw * int(self.top_k), self.top_k):
            raise ValueError("top_k = %d over %d windows needs the any-length merge, which is not supported; lower "
                             "top_k or the window count" % (int(self.top_k), nd * nh * nw))
        if vols.dtype not in (torch.float32, torch.bfloat16):
            vols = vols.float()
        per = max(1, int(scans_per_step))
        chunks = (vols[first:first + per] for first in range(0, int(vols.shape[0]), per))
        # a step is a whole window batch: two in flight overlap one step's tail with the next one's big layers
        steps = self._pipelined((c if c.is_cuda else c.contiguous().pin_memory() for c in chunks),
                                max(1, min(2, int(self.pipeline_depth))), True, overlap, to_host)
        boxes, labels, scores = [], [], []
        for b, l, s in steps:
            boxes.extend(b)
            labels.extend(l)
            scores.extend(s)
        return boxes, labels, scores

    def _predict_step_eager(self, image):
        prev = self.defer_nan_check
        self.defer_nan_check = True
        try:
            predicted_locs, predicted_scores = self(image)
        finally:
            self.defer_nan_check = prev
        priors = self._prior_source(predicted_locs.device)
        if ops.detect_needs_long_lists(self.priors_cxcycz.shape[0], self.top_k):
            flag = self.base.nan_flag(predicted_locs.device)
            if int(flag.cpu()[0]):
                self._raise_on_nan(flag)
            return ops.detect_objects_long(predicted_locs, predicted_scores, priors, self.min_score,
                                           self.max_overlap, self.top_k)
        out = ops.detect_objects_padded(predicted_locs, predicted_scores, priors, self.min_score, self.max_overlap,
                                        self.top_k)
        flag = self.base.nan_flag(predicted_locs.device)
        meta = torch.cat([out.count, out.status, flag]).tolist()   # the one device->host read of the step
        if meta[-1]:
            flag.zero_()
        counts = _checked_counts(meta, out.count.shape[0])
        det_boxes = [out.boxes[i, :k] for i, k in enumerate(counts)]
        det_label = [out.labels[i, :k] for i, k in enumerate(counts)]
        det_scores = [out.scores[i, :k] for i, k in enumerate(counts)]
        return det_boxes, det_label, det_scores

    def train_engine(self):
        eng = self.__dict__.get("_train_engine")
        if eng is None:
            from .training import TrainEngine
            eng = TrainEngine(self)
            self.__dict__["_train_engine"] = eng
        return eng

    def invalidate_packed(self):
        """Drop every packed-weight cache and captured plan (the fused optimizer updates parameters through
        raw pointers, which does not bump their version counters)."""
        for mod in self.modules():
            if getattr(mod, "_packed", None) is not None:
                mod._packed = None
        self.__dict__.get("_plans", {}).clear()

    @staticmethod
    def _distributed(world_size, allreduce):
        """(world size, gradient all-reduce, rank) of a training call; what the caller leaves None comes from
        torch.distributed when it is initialised."""
        import torch.distributed as dist
        dist_on = dist.is_available() and dist.is_initialized()
        if world_size is None:
            world_size = dist.get_world_size() if dist_on else 1
        if allreduce is None and world_size > 1:
            allreduce = dist.all_reduce
        rank = dist.get_rank() if dist_on and world_size > 1 else 0
        return world_size, allreduce, rank

    def fit_step(self, batch, world_size: int = None, allreduce=None):
        """forward + MultiBox loss + backward + (gradient all-reduce) + Adam in one call, everything on the
        device (training.py).  With torch.distributed initialised the flat gradient buffer is summed over
        ranks with one NCCL all-reduce and averaged inside the Adam kernel (DDP semantics, SURVEY.md 8e).
        Returns the (2,) device tensor [conf_loss, loc_loss]."""
        from . import training
        world_size, allreduce, _ = self._distributed(world_size, allreduce)
        if not self.training:
            raise RuntimeError("fit_step needs train() mode")
        return training.fit_step(self, batch, world_size, allreduce)

    def fit_epoch(self, dataset, batch_size: int, augment=None, epoch: int = 0, world_size: int = None,
                  allreduce=None, max_boxes_per_volume: int = 64):
        """One epoch over a ``data.DeviceDataset``, every step ONE CUDA-graph replay: sample the batch (this rank's
        share of ``data.epoch_order``), augment it (``data.Augment``; default: none, which needs a data set of
        ``input_size`` volumes) into bf16 images, extract and pack the ground truth of the augmented masks, then
        forward, loss, backward, (all-reduce) and Adam as ``fit_step``.  ceil(S / (batch_size * world_size)) steps;
        the last batch wraps around to the start of the order.  No host copy or sync inside the epoch.
        Returns (losses (steps, 2) [conf, loc], subjects (steps, batch_size) int32) as device tensors.
        A step in which a volume has more than ``max_boxes_per_volume`` boxes (a crop can split a lesion) is
        skipped like a non-finite one; the epoch then raises at its end."""
        from . import training
        world_size, allreduce, rank = self._distributed(world_size, allreduce)
        if not self.training:
            raise RuntimeError("fit_epoch needs train() mode")
        return training.fit_epoch(self, dataset, batch_size, augment, epoch, world_size, allreduce, rank,
                                  max_boxes_per_volume)

    def fit_skipped_steps(self) -> int:
        """Number of fit_step calls whose gradient was NaN / Inf (e.g. a batch without one positive prior: the
        reference raises "Loss is NaN", ssd3d.py:938-940) and whose update was therefore skipped on the device.
        Reading it synchronises with the device."""
        eng = self.__dict__.get("_train_engine")
        if eng is None or eng.flat is None:
            return 0
        return int(eng.flat.status[1].item())

    def training_step(self, batch):
        """forward + MultiBox loss (ssd3d.py:467-531): matching, hard/soft labelling, CE + L1 and their
        gradients w.r.t. the head outputs run in the loss kernels; ``loss.backward()`` continues through the
        network's hand-written backward (training.py) and fills ``p.grad`` for every parameter."""
        images, gt_boxes, gt_labels = batch["img"], batch['boxes'], batch["labels"]
        dev = self.device
        gt_boxes = [b.to(dev) for b in gt_boxes]
        gt_labels = [l.to(dev) for l in gt_labels]
        predicted_locs, predicted_scores = self(images)
        conf_loss, loc_loss = self.loss_fn(predicted_locs, predicted_scores, gt_boxes, gt_labels)
        loss = conf_loss + self.loss_fn.alpha * loc_loss
        logs = {"train_total_loss": loss, "train_conf_loss": conf_loss, "train_loc_loss": loc_loss}
        # mAP every 2n epochs (ssd3d.py:497-518)
        if self.current_epoch % (self.compute_metric_every_n_epochs * 2) == 0:
            logs.update(self._detection_metrics(predicted_locs, predicted_scores, gt_boxes, gt_labels))
        sch = self.lr_schedulers()
        if sch is not None:
            sch.step()
        return {'loss': loss, "log": logs}

    def _detection_metrics(self, predicted_locs, predicted_scores, gt_boxes, gt_labels, wrap_map50: bool = False):
        """detect_objects + calculate_mAP at IoU 0.1 and 0.5 (ssd3d.py:499-518,563-584), all on the device."""
        from .utils import calculate_mAP
        with torch.no_grad():
            det_boxes, det_labels, det_scores = self.detect_objects(predicted_locs.detach(), predicted_scores.detach(),
                                                                    self.min_score, self.max_overlap, self.top_k)
            if predicted_locs.size(1) <= 500:          # the reference only computes mAP with more than 500 priors
                raise NotImplementedError
            gt_difficulties = [torch.zeros((lbls.size(0),), dtype=torch.bool, device=lbls.device) for lbls in gt_labels]
            metrics_10 = calculate_mAP(det_boxes, det_labels, det_scores, gt_boxes, gt_labels, gt_difficulties,
                                       min_overlap=0.1, return_detail=True)
            metrics_50 = calculate_mAP(det_boxes, det_labels, det_scores, gt_boxes, gt_labels, gt_difficulties,
                                       min_overlap=0.5, return_detail=True)
            if wrap_map50:
                metrics_50["mAP"] = torch.FloatTensor([metrics_50["mAP"]])   # ssd3d.py:580
        return {"metrics_10": metrics_10, "metrics_50": metrics_50}

    def validation_step(self, batch, batch_idx=0):
        """forward + MultiBox loss (+ mAP every n epochs) on a validation batch (ssd3d.py:533-586);
        ``batch["seg"]`` = [gt_boxes, gt_labels]."""
        import warnings
        images, (gt_boxes, gt_labels) = batch["img"], batch['seg']
        dev = self.device
        gt_boxes = [b.to(dev) for b in gt_boxes]
        gt_labels = [l.to(dev) for l in gt_labels]
        predicted_locs, predicted_scores = self(images)
        subjects = batch.get("subject", list(range(len(gt_boxes))))
        for i, subj_boxes in enumerate(gt_boxes):
            sb = subj_boxes.detach().cpu()
            for axis in (0, 1, 2):
                negatives = int((sb[:, axis + 3] < sb[:, axis]).sum())
                zeros = int((sb[:, axis + 3] == sb[:, axis]).sum())
                if negatives > 0:
                    warnings.warn(f"Given boxes has invalid values (subject {subjects[i]}). The box size must "
                                  f"be non-negative but got {negatives} boxes with negative sizes.")
                if zeros > 0:
                    warnings.warn(f"Given boxes has invalid values (subject {subjects[i]}). The box size must "
                                  f"be non-zero but got {zeros} boxes with size of zero.")
        conf_loss, loc_loss = self.loss_fn(predicted_locs, predicted_scores, gt_boxes, gt_labels)
        loss = conf_loss + self.loss_fn.alpha * loc_loss
        logs = {"val_total_loss": loss, "val_conf_loss": conf_loss, "val_loc_loss": loc_loss}
        if self.current_epoch % self.compute_metric_every_n_epochs == 0:
            logs.update(self._detection_metrics(predicted_locs, predicted_scores, gt_boxes, gt_labels, wrap_map50=True))
        return {'val_loss': loss, "log": logs}

    def configure_optimizers(self):
        """Adam, weight decay 5e-4, biases at twice the learning rate, cosine schedule (ssd3d.py:704-722)."""
        biases, not_biases = list(), list()
        for param_name, param in self.named_parameters():
            if param.requires_grad:
                if param_name.endswith('.bias'):
                    biases.append(param)
                else:
                    not_biases.append(param)
        params = [{'params': biases, 'lr': 2 * self.lr}, {'params': not_biases}]
        optimizer = torch.optim.Adam(params=params, lr=self.lr, weight_decay=0.0005)
        if self.scheduler != "none":
            scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, T_max=40)
            return [optimizer], [scheduler]
        return optimizer


SSD3D = LSSD3D


class _MultiBoxLossFn(torch.autograd.Function):
    """conf / loc losses with the analytic gradient computed by the loss kernel in the same pass."""

    @staticmethod
    def forward(ctx, locs, scores, true_classes, true_locs, hnm, ratio):
        out, n_pos, g_locs, g_scores = ops.multibox_loss(locs, scores, true_classes, true_locs, alpha=1.0,
                                                         hard_negative_mining=hnm, neg_pos_ratio=ratio,
                                                         want_grads=True)
        ctx.save_for_backward(g_locs, g_scores)
        return out[0], out[1]

    @staticmethod
    def backward(ctx, g_conf, g_loc):
        g_locs, g_scores = ctx.saved_tensors
        return g_locs * g_loc, g_scores * g_conf, None, None, None, None


class MultiBoxLoss(nn.Module):
    """The MultiBox loss: L1 localisation loss over positive priors + cross-entropy confidence loss over
    all non-ignored priors, normalised by the number of positives (ssd3d.py:741-941).

    ``hard_negative_mining=True`` (not in the reference's signature) switches to the variant the
    reference ships commented out (ssd3d.py:926-932): per image only the ``neg_pos_ratio * n_positives``
    hardest negatives count."""

    def __init__(self, priors_cxcycz, threshold=0.5, neg_pos_ratio=3, alpha=1., hard_negative_mining=False):
        super(MultiBoxLoss, self).__init__()
        self.threshold = threshold
        self.neg_pos_ratio = neg_pos_ratio
        self.alpha = alpha
        self.hard_negative_mining = hard_negative_mining
        if type(self.threshold) == list:
            if len(self.threshold) == 1:
                self.thresholding_mode = "hard"
                self.threshold = self.threshold[0]
            else:
                self.thresholding_mode = "soft"
                assert (len(self.threshold) == 2)
        elif type(self.threshold) == float:
            self.thresholding_mode = "hard"
        else:
            raise Exception(
                "Type error. Expected float or list of floats for threshold but got {type(self.threshold))}")
        self.set_priors(priors_cxcycz)

    def set_priors(self, priors_cxcycz):
        self.priors_cxcycz = priors_cxcycz
        # centre-size -> boundary is +-(w/2): exact in fp32 on any device, so the CPU build container can
        # construct the module; the kernels recompute it from priors_cxcycz anyway
        half = priors_cxcycz[:, 3:] / 2
        self.priors_xyz = torch.cat([priors_cxcycz[:, :3] - half, priors_cxcycz[:, :3] + half], 1)

    def match(self, boxes, labels):
        """Prior <-> object matching, labelling and target encoding for a batch (ssd3d.py:786-888)."""
        if self.thresholding_mode == "hard":
            t0 = t1 = self.threshold
        else:
            t0, t1 = self.threshold
        dev = boxes[0].device if len(boxes) else self.priors_cxcycz.device
        if self.priors_cxcycz.device != dev:
            self.set_priors(self.priors_cxcycz.to(dev))
        return ops.match_priors(boxes, labels, self.priors_cxcycz, t0, t1)

    def forward(self, predicted_locs, predicted_scores, boxes, labels):
        n_priors = self.priors_cxcycz.size(0)
        assert n_priors == predicted_locs.size(1) == predicted_scores.size(1)
        m = self.match(boxes, labels)
        conf_loss, loc_loss = _MultiBoxLossFn.apply(predicted_locs, predicted_scores, m["true_classes"],
                                                    m["true_locs"], self.hard_negative_mining, self.neg_pos_ratio)
        if torch.isnan(loc_loss):   # no positive prior at all (ssd3d.py:938-940, without the breakpoint)
            raise Exception("Loss is NaN")
        return conf_loss, loc_loss
