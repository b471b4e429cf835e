"""Tensor-level wrappers over the C ABI: argument checking, output allocation (torch's caching
allocator), launch on torch's current stream.  PyTorch is plumbing here -- device memory and streams;
all arithmetic happens in ``libssd3d_b200.so``.  CPU tensors are an error, never a fallback.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib

BF16 = torch.bfloat16

# kernels launched by this process through the library (bench.py reports it as ``gpu_launches``)
LAUNCHES = [0]


def _stream() -> int:
    # raw handle of torch's current stream on the current device (torch.cuda.current_stream() costs ~14 us of
    # host time per call, which matters when a pipelined inference step is ~250 us)
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def _need_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("ssd3d_b200 ops need CUDA tensors (got a %s tensor); there is no CPU path" % t.device)


def _ptr(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


def f32(v: float) -> float:
    """Round a Python float to fp32 the way torch does when comparing it with a float32 tensor."""
    return float(np.float32(v))


def conv_out(d: int, s: int) -> int:
    return (d - 1) // s + 1


# ----------------------------------------------------------------------------------------------
# activations: logical (N, C, D, H, W) tensors stored channels-last-3d in bf16
# ----------------------------------------------------------------------------------------------
def to_channels_last_bf16(x: torch.Tensor) -> torch.Tensor:
    """Bring a 5-D activation to the kernels' storage format (a no-op for tensors produced by the ops)."""
    if x.dim() != 5:
        raise RuntimeError("expected a 5-D (N, C, D, H, W) tensor, got %s" % (tuple(x.shape),))
    if x.dtype != BF16:
        x = x.to(BF16)
    if not x.is_contiguous(memory_format=torch.channels_last_3d):
        x = x.contiguous(memory_format=torch.channels_last_3d)
    return x


def _alloc_ndhwc(n, c, d, h, w, device) -> torch.Tensor:
    # physical (N, D, H, W, C), returned as its logical NCDHW view
    return torch.empty((n, d, h, w, c), dtype=BF16, device=device).permute(0, 4, 1, 2, 3)


def stem_conv_bn_relu(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor,
                      stride_d: int, force_simt: bool = False, out: Optional[torch.Tensor] = None,
                      kernel: Optional[str] = None) -> torch.Tensor:
    """x (N,Cin,D,H,W) contiguous fp32|bf16 -> (N,32,Do,Ho,Wo) channels-last bf16.  mobilenet.py:28-30.
    The library picks the kernel: banded-B tcgen05 GEMM on raw TMA rows (bf16 volumes, Cin <= 2), gather-based
    tcgen05 implicit GEMM when TMA can address the rows, CUDA-core kernel otherwise.  ``kernel`` = "tz" | "tc" |
    "simt" forces one (tests; "tz" raises when it does not apply)."""
    _need_cuda(x, w_packed, scale, shift)
    if x.dim() != 5:
        raise RuntimeError("expected (N, C, D, H, W) input")
    if x.dtype not in (torch.float32, BF16):
        x = x.float()
    x = x.contiguous()
    n, cin, d, h, w = x.shape
    y = out if out is not None else _alloc_ndhwc(n, 32, conv_out(d, stride_d), conv_out(h, 2), conv_out(w, 2),
                                                 x.device)
    lib = _lib.load()
    if kernel in ("tz", "tc"):
        fn = lib.ssd3d_stem_conv_affine_tz if kernel == "tz" else lib.ssd3d_stem_conv_affine_tc
        rc = fn(x.data_ptr(), int(x.dtype == BF16), w_packed.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                y.data_ptr(), n, cin, d, h, w, stride_d, 1, _stream())
        _lib.check(rc, "ssd3d_stem_conv_affine_" + kernel)
        LAUNCHES[0] += 1
        return y
    fn = lib.ssd3d_stem_conv_bn_relu_simt if (force_simt or kernel == "simt") else lib.ssd3d_stem_conv_bn_relu
    rc = fn(x.data_ptr(), int(x.dtype == BF16), w_packed.data_ptr(), scale.data_ptr(), shift.data_ptr(), y.data_ptr(),
            n, cin, d, h, w, stride_d, _stream())
    _lib.check(rc, "ssd3d_stem_conv_bn_relu")
    LAUNCHES[0] += 1
    return y


def dwconv3d_bn_relu(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor,
                     stride: int, force_direct: bool = False) -> torch.Tensor:
    """Depthwise 3x3x3 + BN + ReLU on a channels-last bf16 activation.  mobilenet.py:38,44.
    TMA halo-tile kernel on large maps, direct kernel otherwise (or when forced)."""
    _need_cuda(x, w_packed, scale, shift)
    x = to_channels_last_bf16(x)
    n, c, d, h, w = x.shape
    y = _alloc_ndhwc(n, c, conv_out(d, stride), conv_out(h, stride), conv_out(w, stride), x.device)
    lib = _lib.load()
    if force_direct:
        rc = lib.ssd3d_dwconv3d_affine_direct(x.data_ptr(), w_packed.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                              y.data_ptr(), n, c, d, h, w, stride, 1, _stream())
    else:
        rc = lib.ssd3d_dwconv3d_bn_relu(x.data_ptr(), w_packed.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                        y.data_ptr(), n, c, d, h, w, stride, _stream())
    _lib.check(rc, "ssd3d_dwconv3d_bn_relu")
    LAUNCHES[0] += 1
    return y


def pwconv_bn_relu(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor,
                   nan_flag: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Pointwise conv + BN + ReLU (tcgen05 GEMM).  w_packed (Cout, Cin) bf16.  mobilenet.py:40,45."""
    _need_cuda(x, w_packed, scale, shift, nan_flag)
    x = to_channels_last_bf16(x)
    n, c, d, h, w = x.shape
    cout = w_packed.shape[0]
    y = _alloc_ndhwc(n, cout, d, h, w, x.device)
    rc = _lib.load().ssd3d_pwconv_bn_relu(x.data_ptr(), w_packed.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                          y.data_ptr(), n * d * h * w, c, cout, _ptr(nan_flag), _stream())
    _lib.check(rc, "ssd3d_pwconv_bn_relu")
    LAUNCHES[0] += 1
    return y


def block_fused_supported(x: torch.Tensor, cout: int, stride: int) -> bool:
    n, c, d, h, w = x.shape
    return bool(_lib.load().ssd3d_block_fused_supported(c, cout, d, h, w, stride))


def block_dwpw_bn_relu(x: torch.Tensor, w_dw: torch.Tensor, scale1: torch.Tensor, shift1: torch.Tensor,
                       w_pw: torch.Tensor, scale2: torch.Tensor, shift2: torch.Tensor, stride: int,
                       nan_flag: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A whole Block (depthwise + BN + ReLU -> pointwise + BN + ReLU, mobilenet.py:34-49) in one kernel: the
    depthwise tile stays in shared memory as the tcgen05 A operand.  Check ``block_fused_supported`` first."""
    _need_cuda(x, w_dw, scale1, shift1, w_pw, scale2, shift2, nan_flag)
    x = to_channels_last_bf16(x)
    n, c, d, h, w = x.shape
    cout = w_pw.shape[0]
    y = _alloc_ndhwc(n, cout, conv_out(d, stride), conv_out(h, stride), conv_out(w, stride), x.device)
    rc = _lib.load().ssd3d_block_dwpw_bn_relu(x.data_ptr(), w_dw.data_ptr(), scale1.data_ptr(), shift1.data_ptr(),
                                              w_pw.data_ptr(), scale2.data_ptr(), shift2.data_ptr(), y.data_ptr(), n, c,
                                              cout, d, h, w, stride, _ptr(nan_flag), _stream())
    _lib.check(rc, "ssd3d_block_dwpw_bn_relu")
    LAUNCHES[0] += 1
    return y


def head_conv(x: torch.Tensor, w_packed: torch.Tensor, bias: torch.Tensor, locs: torch.Tensor, scores: torch.Tensor,
              bpl: int, n_classes: int, prior_offset: int, nan_flag: Optional[torch.Tensor] = None,
              algo: int = 0) -> None:
    """Fused loc+class 3x3x3 head of one feature map, written into locs (N,P,6) / scores (N,P,n_classes).
    algo: 0 auto, 1 per-tap TMA kernel, 2 halo-tile kernel, 3 kw-GEMM + stencil (large maps)."""
    _need_cuda(x, w_packed, bias, locs, scores, nan_flag)
    x = to_channels_last_bf16(x)
    n, c, d, h, w = x.shape
    lib = _lib.load()
    npad = w_packed.shape[0] if algo != 4 else 16
    need = lib.ssd3d_head_workspace_bytes(n, c, d, h, w, npad) if algo != 1 else 0
    ws = torch.empty((need,), dtype=torch.uint8, device=x.device) if need else None
    rc = lib.ssd3d_head_conv(x.data_ptr(), w_packed.data_ptr(), bias.data_ptr(), locs.data_ptr(), scores.data_ptr(),
                             n, c, d, h, w, bpl, n_classes, npad, locs.shape[1], prior_offset, _ptr(nan_flag),
                             _ptr(ws), need, algo, _stream())
    _lib.check(rc, "ssd3d_head_conv")
    LAUNCHES[0] += 2 if need else 1


def head_kw_supported(x: torch.Tensor, npad: int) -> bool:
    n, c, d, h, w = x.shape
    return bool(_lib.load().ssd3d_head_kw_supported(n, c, d, h, w, npad))


def pack_head_weight_kw(w_packed: torch.Tensor) -> torch.Tensor:
    """(16, 27*C) packed head weight -> (144, 3*C) tiling of the kw-GEMM head kernel (once per weight version)."""
    _need_cuda(w_packed)
    c = w_packed.shape[1] // 27
    out = torch.empty((144, 3 * c), dtype=BF16, device=w_packed.device)
    rc = _lib.load().ssd3d_head_weight_kw(w_packed.data_ptr(), c, out.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_head_weight_kw")
    return out


# ----------------------------------------------------------------------------------------------
# weight packing (host-side layout work, done once per state_dict)
# ----------------------------------------------------------------------------------------------
def fold_bn(bn: torch.nn.BatchNorm3d) -> Tuple[torch.Tensor, torch.Tensor]:
    """Eval-mode BatchNorm as y = x*scale + shift (fp32)."""
    w = bn.weight.detach().float() if bn.weight is not None else torch.ones_like(bn.running_mean)
    b = bn.bias.detach().float() if bn.bias is not None else torch.zeros_like(bn.running_mean)
    scale = w / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    shift = b - bn.running_mean.detach().float() * scale
    return scale.contiguous(), shift.contiguous()


def pack_stem_weight(w: torch.Tensor) -> torch.Tensor:
    """(32, Cin, 3,3,3) -> (32, KPAD) bf16: the weight flattened in its own (Cin,3,3,3) order, K zero-padded
    to 64 (Cin <= 2) or 128."""
    co, ci = w.shape[0], w.shape[1]
    kpad = 64 if 27 * ci <= 64 else 128
    p = torch.zeros((co, kpad), dtype=BF16, device=w.device)
    p[:, :27 * ci] = w.detach().reshape(co, 27 * ci).to(BF16)
    return p.contiguous()


def pack_dw_weight(w: torch.Tensor) -> torch.Tensor:
    """(C, 1, 3,3,3) -> (27, C) bf16."""
    c = w.shape[0]
    return w.detach().reshape(c, 27).t().contiguous().to(BF16)


def pack_pw_weight(w: torch.Tensor) -> torch.Tensor:
    """(Cout, Cin, 1,1,1) -> (Cout, Cin) bf16."""
    return w.detach().reshape(w.shape[0], w.shape[1]).contiguous().to(BF16)


def pack_head_weight(loc_w, loc_b, cl_w, cl_b) -> Tuple[torch.Tensor, torch.Tensor]:
    """loc (bpl*6, C,3,3,3) and class (bpl*n_classes, C,3,3,3) convs -> (NPAD, 27*C) bf16 + (NPAD) fp32 bias."""
    c = loc_w.shape[1]
    rows = loc_w.shape[0] + cl_w.shape[0]
    npad = ((rows + 15) // 16) * 16
    w = torch.zeros((npad, 27 * c), dtype=torch.float32, device=loc_w.device)
    w[:loc_w.shape[0]] = loc_w.detach().float().permute(0, 2, 3, 4, 1).reshape(loc_w.shape[0], 27 * c)
    w[loc_w.shape[0]:rows] = cl_w.detach().float().permute(0, 2, 3, 4, 1).reshape(cl_w.shape[0], 27 * c)
    b = torch.zeros((npad,), dtype=torch.float32, device=loc_w.device)
    b[:loc_w.shape[0]] = loc_b.detach().float()
    b[loc_w.shape[0]:rows] = cl_b.detach().float()
    return w.to(BF16).contiguous(), b.contiguous()


# ----------------------------------------------------------------------------------------------
# box geometry (utils.py:42-149)
# ----------------------------------------------------------------------------------------------
def _boxes(t: torch.Tensor, what: str) -> torch.Tensor:
    _need_cuda(t)
    if t.dim() != 2 or t.shape[1] != 6:
        raise RuntimeError("%s must be (n, 6), got %s" % (what, tuple(t.shape)))
    return t.float().contiguous()


def box_transform(mode: int, boxes: torch.Tensor, priors: Optional[torch.Tensor] = None) -> torch.Tensor:
    boxes = _boxes(boxes, "boxes")
    if priors is not None:
        priors = _boxes(priors, "priors")
        if priors.shape[0] != boxes.shape[0]:
            raise RuntimeError("boxes and priors must have the same length")
    out = torch.empty_like(boxes)
    rc = _lib.load().ssd3d_box_transform(mode, boxes.data_ptr(), _ptr(priors), out.data_ptr(), boxes.shape[0], _stream())
    _lib.check(rc, "ssd3d_box_transform")
    LAUNCHES[0] += 1
    return out


def iou3d_pairwise(a: torch.Tensor, b: torch.Tensor, want_iou: bool = True) -> torch.Tensor:
    a, b = _boxes(a, "set_1"), _boxes(b, "set_2")
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device=a.device)
    rc = _lib.load().ssd3d_iou3d_pairwise(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.shape[0], b.shape[0],
                                          int(want_iou), _stream())
    _lib.check(rc, "ssd3d_iou3d_pairwise")
    LAUNCHES[0] += 1
    return out


# ----------------------------------------------------------------------------------------------
# prior boxes as a function of the prior index (ssd3d.py:286-342)
# ----------------------------------------------------------------------------------------------
class PriorTable:
    """Device copy of ``ssd3d_prior_table`` + the prior count.  ``fmap_dims``: (d0, d1, d2) per prediction layer in
    prior order; ``sizes``: per layer the box edges as Python floats (float64), e.g. [s, s + s/1] -- rounded to
    fp32 and clamped to [0, 1] here exactly like ``torch.FloatTensor(...).clamp_(0, 1)`` does."""

    def __init__(self, fmap_dims, sizes, device):
        if len(fmap_dims) != len(sizes) or not 0 < len(fmap_dims) <= _lib.MAX_PRIOR_LAYERS:
            raise ValueError("1..%d prediction layers expected" % _lib.MAX_PRIOR_LAYERS)
        t = _lib.PriorTable()
        t.n_layers = len(fmap_dims)
        start = 0
        for l, ((d0, d1, d2), sz) in enumerate(zip(fmap_dims, sizes)):
            if not 0 < len(sz) <= _lib.MAX_PRIOR_SIZES:
                raise ValueError("1..%d boxes per location expected" % _lib.MAX_PRIOR_SIZES)
            t.d0[l], t.d1[l], t.d2[l], t.n_boxes[l] = int(d0), int(d1), int(d2), len(sz)
            t.start[l] = start
            for b, v in enumerate(sz):
                t.size[l][b] = float(min(max(np.float32(v), np.float32(0.0)), np.float32(1.0)))
            start += int(d0) * int(d1) * int(d2) * len(sz)
        t.start[len(fmap_dims)] = start
        self.count = start
        self.host = t
        raw = np.frombuffer(bytes(t), dtype=np.uint8).copy()
        self.dev = torch.from_numpy(raw).to(device)

    def data_ptr(self) -> int:
        return self.dev.data_ptr()

    def materialize(self) -> torch.Tensor:
        """(P, 6) fp32 priors computed on the device: bit-identical to ``LSSD3D.create_prior_boxes()``."""
        out = torch.empty((self.count, 6), dtype=torch.float32, device=self.dev.device)
        rc = _lib.load().ssd3d_prior_boxes(self.dev.data_ptr(), self.count, out.data_ptr(), _stream())
        _lib.check(rc, "ssd3d_prior_boxes")
        LAUNCHES[0] += 1
        return out


def _prior_arg(priors):
    """-> (pointer, analytic?) for a (P, 6) tensor or a PriorTable."""
    if isinstance(priors, PriorTable):
        return priors.data_ptr(), True
    return priors.data_ptr(), False


def _prior_count(priors) -> int:
    return priors.count if isinstance(priors, PriorTable) else int(priors.shape[0])


# ----------------------------------------------------------------------------------------------
# detection
# ----------------------------------------------------------------------------------------------
def decode_softmax(locs: torch.Tensor, scores: torch.Tensor, priors: torch.Tensor):
    """-> (probs (N,P,C), boxes_xyz (N,P,6)); ssd3d.py:363,373-374."""
    _need_cuda(locs, scores)
    locs, scores = locs.float().contiguous(), scores.float().contiguous()
    if not isinstance(priors, PriorTable):
        _need_cuda(priors)
        priors = priors.float().contiguous()
    n, p, c = scores.shape
    probs = torch.empty_like(scores)
    boxes = torch.empty_like(locs)
    pp, analytic = _prior_arg(priors)
    lib = _lib.load()
    fn = lib.ssd3d_decode_softmax_analytic if analytic else lib.ssd3d_decode_softmax
    rc = fn(locs.data_ptr(), scores.data_ptr(), pp, n, p, c, probs.data_ptr(), boxes.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_decode_softmax")
    LAUNCHES[0] += 1
    return probs, boxes


def nms3d_sorted(boxes_xyz: torch.Tensor, max_overlap: float) -> torch.Tensor:
    """Greedy NMS over score-sorted boxes -> bool keep mask (ssd3d.py:407-426)."""
    boxes_xyz = _boxes(boxes_xyz, "boxes")
    n = boxes_xyz.shape[0]
    keep = torch.empty((n,), dtype=torch.uint8, device=boxes_xyz.device)
    if n == 0:
        return keep.bool()
    words = (n + 63) // 64
    ws = torch.empty((n * words,), dtype=torch.int64, device=boxes_xyz.device)
    rc = _lib.load().ssd3d_nms3d_sorted(boxes_xyz.data_ptr(), n, f32(max_overlap), keep.data_ptr(), ws.data_ptr(),
                                        _stream())
    _lib.check(rc, "ssd3d_nms3d_sorted")
    LAUNCHES[0] += 2
    return keep.bool()


def nms3d_sorted_chunked(boxes_xyz: torch.Tensor, max_overlap: float, chunk: int = 0,
                         return_count: bool = False, use_grid: bool = True):
    """Greedy NMS over a score-sorted list of any length (ssd3d.py:407-426): chunks of ``chunk`` boxes
    (0 = the library default), each tested against the boxes kept so far (found through a uniform grid when
    ``max_overlap >= 0`` and ``use_grid``, else the whole kept list), then resolved with the bit matrix.
    -> bool keep mask (and the device int64 kept count)."""
    boxes_xyz = _boxes(boxes_xyz, "boxes")
    n = boxes_xyz.shape[0]
    dev = boxes_xyz.device
    keep = torch.empty((n,), dtype=torch.uint8, device=dev)
    count = torch.zeros((1,), dtype=torch.int64, device=dev)
    if n == 0:
        return (keep.bool(), count) if return_count else keep.bool()
    lib = _lib.load()
    need = lib.ssd3d_nms3d_chunked_workspace_bytes(n, int(chunk))
    if need <= 0:
        raise ValueError("nms3d_sorted_chunked: chunk must be 0 or a multiple of 64 in [64, %d]" % _lib.SORT_MAX)
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    rc = lib.ssd3d_nms3d_sorted_chunked(boxes_xyz.data_ptr(), n, f32(max_overlap), keep.data_ptr(), count.data_ptr(),
                                        ws.data_ptr(), need, int(chunk), 0 if use_grid else _lib.NMS_NO_GRID,
                                        _stream())
    _lib.check(rc, "ssd3d_nms3d_sorted_chunked")
    per = int(chunk) if chunk else 4096
    LAUNCHES[0] += 2 * ((n + per - 1) // per) + (4 if use_grid and n > per else 0)   # delta + fused launch per chunk
    return (keep.bool(), count) if return_count else keep.bool()


def sort_keys_u64(keys: torch.Tensor) -> torch.Tensor:
    """Ascending stable in-place sort of packed 64-bit keys held in an int64 tensor (compared as unsigned)."""
    _need_cuda(keys)
    if keys.dtype != torch.int64 or not keys.is_contiguous() or keys.dim() != 1:
        raise ValueError("sort_keys_u64 needs a contiguous 1-D int64 tensor")
    n = keys.numel()
    if n <= 1:
        return keys
    tmp = torch.empty_like(keys) if n > _lib.SORT_MAX else None
    rc = _lib.load().ssd3d_sort_keys_u64(keys.data_ptr(), n, tmp.data_ptr() if tmp is not None else None, _stream())
    _lib.check(rc, "ssd3d_sort_keys_u64")
    runs = (n + _lib.SORT_MAX - 1) // _lib.SORT_MAX
    LAUNCHES[0] += 1 + max(0, (runs - 1).bit_length())
    return keys


def decode_filter(locs: torch.Tensor, scores: torch.Tensor, priors: torch.Tensor, min_score: float):
    """Stage 1 of detect_objects -> (boxes_xyz (N,P,6), cand (S,P) int64 keys, count (S,) int32), S = N*(C-1)."""
    _need_cuda(locs, scores)
    locs, scores = locs.float().contiguous(), scores.float().contiguous()
    if not isinstance(priors, PriorTable):
        _need_cuda(priors)
        priors = priors.float().contiguous()
    n, p, c = scores.shape
    if locs.shape[0] != n or locs.shape[1] != p or _prior_count(priors) != p:
        raise AssertionError("prior / prediction count mismatch")  # ssd3d.py:370
    dev = locs.device
    boxes = torch.empty((n, p, 6), dtype=torch.float32, device=dev)
    cand = torch.empty((n * (c - 1), p), dtype=torch.int64, device=dev)
    count = torch.empty((n * (c - 1),), dtype=torch.int32, device=dev)
    pp, analytic = _prior_arg(priors)
    lib = _lib.load()
    fn = lib.ssd3d_decode_filter_analytic if analytic else lib.ssd3d_decode_filter
    rc = fn(locs.data_ptr(), scores.data_ptr(), pp, n, p, c, f32(min_score), boxes.data_ptr(), cand.data_ptr(),
            count.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_decode_filter")
    LAUNCHES[0] += 1
    return boxes, cand, count


def _key_scores(keys: torch.Tensor) -> torch.Tensor:
    """fp32 score packed in the high word of a candidate key ({~orderable(score) << 32 | index})."""
    u = (~(keys >> 32)) & 0xFFFFFFFF                       # orderable(score)
    bits = torch.where((u & 0x80000000) != 0, u & 0x7FFFFFFF, (~u) & 0xFFFFFFFF)
    return bits.to(torch.int32).view(torch.float32) if bits.numel() else bits.to(torch.float32)


def detect_needs_long_lists(n_priors: int, top_k: int) -> bool:
    """True where the fused ssd3d_detect_objects stops (P > SORT_MAX and 10*top_k > SORT_MAX/2): the
    NMS-stress settings (model_insight.py:146) go through ``detect_objects_long`` instead."""
    return n_priors > _lib.SORT_MAX and 10 * int(top_k) > _lib.SORT_MAX // 2


def detect_objects_long(locs: torch.Tensor, scores: torch.Tensor, priors: torch.Tensor, min_score: float,
                        max_overlap: float, top_k: int, return_prior: bool = False, chunk: int = 0):
    """``detect_objects`` (ssd3d.py:344-460) for candidate lists of any length: filter/decode, key sort and
    greedy NMS are this library's kernels (decode_filter, sort_keys_u64, nms3d_sorted_chunked); the host
    reads the per-(image, class) candidate counts once and strings the stages together with tensor slicing.
    Same outputs as the fused path (ties: ascending prior index)."""
    top_k = int(top_k)
    n, p, c = scores.shape
    boxes, cand, count = decode_filter(locs, scores, priors, min_score)
    dev = boxes.device
    counts = count.cpu().tolist()                          # the one read-back before the per-segment stages
    out_b, out_l, out_s, out_p = [], [], [], []
    for i in range(n):
        ib, ik, il = [], [], []
        for cls in range(1, c):
            seg = i * (c - 1) + (cls - 1)
            m = counts[seg]
            if m == 0:                                     # ssd3d.py:390-391
                continue
            keys = sort_keys_u64(cand[seg, :m])
            keys = keys[:min(m, 10 * top_k)]               # ssd3d.py:401
            prior = keys & 0xFFFFFFFF
            sboxes = boxes[i].index_select(0, prior)
            keep = nms3d_sorted_chunked(sboxes, max_overlap, chunk)
            ib.append(sboxes[keep])
            ik.append(keys[keep])
            il.append(torch.full((ib[-1].shape[0],), cls, dtype=torch.int64, device=dev))
        if not ib:                                         # ssd3d.py:437-440
            out_b.append(torch.tensor([[0., 0., 0., 1., 1., 1.]], device=dev))
            out_l.append(torch.zeros((1,), dtype=torch.int64, device=dev))
            out_s.append(torch.zeros((1,), dtype=torch.float32, device=dev))
            out_p.append(torch.full((1,), -1, dtype=torch.int64, device=dev))
            continue
        b, k, l = torch.cat(ib), torch.cat(ik), torch.cat(il)
        if b.shape[0] > top_k:                             # ssd3d.py:449-453, stable: class order on ties
            order_keys = ((k >> 32) << 32) | torch.arange(k.shape[0], dtype=torch.int64, device=dev)
            order = (sort_keys_u64(order_keys.contiguous()) & 0xFFFFFFFF)[:top_k]
            b, k, l = b[order], k[order], l[order]
        out_b.append(b)
        out_l.append(l)
        out_s.append(_key_scores(k))
        out_p.append(k & 0xFFFFFFFF)
    if return_prior:
        return out_b, out_l, out_s, out_p
    return out_b, out_l, out_s


class DetectOutput:
    """Padded device-side result of one detect call (rows >= count[i] are undefined)."""
    __slots__ = ("boxes", "scores", "labels", "prior", "count", "status")

    def __init__(self, boxes, scores, labels, prior, count, status):
        self.boxes, self.scores, self.labels, self.prior, self.count, self.status = (boxes, scores, labels, prior,
                                                                                   count, status)


def detect_objects_padded(locs: torch.Tensor, scores: torch.Tensor, priors: torch.Tensor, min_score: float,
                          max_overlap: float, top_k: int, workspace: Optional[torch.Tensor] = None,
                          out_count: Optional[torch.Tensor] = None,
                          status: Optional[torch.Tensor] = None, out=None) -> DetectOutput:
    """The whole of ``detect_objects`` on the device, no host sync; see include/ssd3d_b200.h.
    ``out_count`` (N,) / ``status`` (1,) int32 may be supplied (e.g. slices of one buffer that is read back
    with a single copy)."""
    _need_cuda(locs, scores)
    locs, scores = locs.float().contiguous(), scores.float().contiguous()
    if not isinstance(priors, PriorTable):
        _need_cuda(priors)
        priors = priors.float().contiguous()
    n, p, c = scores.shape
    if locs.shape[0] != n or locs.shape[1] != p or _prior_count(priors) != p:
        raise AssertionError("prior / prediction count mismatch")  # ssd3d.py:370
    dev = locs.device
    top_k = int(top_k)
    lib = _lib.load()
    need = lib.ssd3d_detect_workspace_bytes(n, p, c, top_k)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((need,), dtype=torch.uint8, device=dev)
    if out is not None:          # caller-provided (boxes, scores, labels, prior), e.g. views of one packed buffer
        out_boxes, out_scores, out_labels, out_prior = out
    else:
        out_boxes = torch.empty((n, top_k, 6), dtype=torch.float32, device=dev)
        out_scores = torch.empty((n, top_k), dtype=torch.float32, device=dev)
        out_labels = torch.empty((n, top_k), dtype=torch.int64, device=dev)
        out_prior = torch.empty((n, top_k), dtype=torch.int64, device=dev)
    if out_count is None:
        out_count = torch.empty((n,), dtype=torch.int32, device=dev)
    if status is None:
        status = torch.empty((1,), dtype=torch.int32, device=dev)
    pp, analytic = _prior_arg(priors)
    fn = lib.ssd3d_detect_objects_analytic if analytic else lib.ssd3d_detect_objects
    rc = fn(locs.data_ptr(), scores.data_ptr(), pp, n, p, c, f32(min_score), f32(max_overlap), top_k,
            out_boxes.data_ptr(), out_scores.data_ptr(), out_labels.data_ptr(), out_prior.data_ptr(),
            out_count.data_ptr(), workspace.data_ptr(), workspace.numel(), status.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_detect_objects")
    LAUNCHES[0] += 4
    return DetectOutput(out_boxes, out_scores, out_labels, out_prior, out_count, status)


def raise_on_status(nan_bits: int, detect_status: int = 0) -> None:
    """Raise on the NaN bits a forward ORed into its flag (the reference's exceptions, ssd3d.py:95-98,255-262) and
    on the status word of ``detect_objects`` (bit 0: an (image, class) list outgrew one sort block)."""
    if nan_bits & _lib.NAN_BACKBONE:
        print("Yesssss this NaN error again in the base network")
        raise Exception("Yesssss this NaN error again in the base network")
    if nan_bits & _lib.NAN_SCORES:
        raise Exception("Oh no not this NaN error again... (forward SSD), CLASSES_SCORES is nan!")
    if nan_bits & _lib.NAN_LOCS:
        raise Exception("Oh no not this NaN error again... (forward SSD), LOCS is nan!")
    if detect_status & 1:
        raise RuntimeError("detect_objects: more than %d candidates above min_score for one (image, class); "
                           "raise min_score (limit of this version)" % _lib.SORT_MAX)


def detect_lists(out: DetectOutput, return_prior: bool = False):
    """Turn the padded result into the reference's three Python lists (one D2H read of the counts)."""
    host = torch.cat([out.count, out.status]).tolist()
    raise_on_status(0, host[-1])
    counts = host[:-1]
    b = [out.boxes[i, :k] for i, k in enumerate(counts)]
    l = [out.labels[i, :k] for i, k in enumerate(counts)]
    s = [out.scores[i, :k] for i, k in enumerate(counts)]
    if return_prior:
        return b, l, s, [out.prior[i, :k] for i, k in enumerate(counts)]
    return b, l, s


# ----------------------------------------------------------------------------------------------
# matching + loss
# ----------------------------------------------------------------------------------------------
def match_priors(boxes: Sequence[torch.Tensor], labels: Sequence[torch.Tensor], priors_cxcycz: torch.Tensor,
                 t0: float, t1: float):
    """-> dict(true_classes (N,P) int64, true_locs (N,P,6), overlap, object_for_prior, prior_for_object)."""
    _need_cuda(*boxes, *labels)
    dev = priors_cxcycz.dev.device if isinstance(priors_cxcycz, PriorTable) else priors_cxcycz.device
    n = len(boxes)
    counts = [int(b.shape[0]) for b in boxes]
    offsets = torch.tensor(np.concatenate([[0], np.cumsum(counts)]).astype(np.int32), device=dev)
    total = int(sum(counts))
    if total:
        gt_boxes = torch.cat([b.reshape(-1, 6).float() for b in boxes]).contiguous()
        gt_labels = torch.cat([l.reshape(-1).long() for l in labels]).contiguous()
    else:
        gt_boxes = gt_labels = None
    return match_priors_packed(gt_boxes, gt_labels, offsets, n, total, priors_cxcycz, t0, t1)


def match_priors_packed(gt_boxes: Optional[torch.Tensor], gt_labels: Optional[torch.Tensor], offsets: torch.Tensor,
                        n: int, total: int, priors_cxcycz: torch.Tensor, t0: float, t1: float):
    """Same, on already concatenated ground truth: gt_boxes (>= total, 6) fp32, gt_labels (>= total) int64,
    offsets (n+1) int32 on the device.  ``total`` may be a CAPACITY larger than offsets[-1] (static buffers of a
    captured training step): rows past offsets[-1] are never read."""
    analytic = isinstance(priors_cxcycz, PriorTable)
    dev = priors_cxcycz.dev.device if analytic else priors_cxcycz.device
    p = _prior_count(priors_cxcycz)
    tc = torch.empty((n, p), dtype=torch.int64, device=dev)
    tl = torch.empty((n, p, 6), dtype=torch.float32, device=dev)
    ov = torch.empty((n, p), dtype=torch.float32, device=dev)
    ofp = torch.empty((n, p), dtype=torch.int32, device=dev)
    pfo = torch.empty((max(total, 1),), dtype=torch.int32, device=dev)
    ws = torch.empty((max(total, 1),), dtype=torch.int64, device=dev)
    pri = priors_cxcycz if analytic else priors_cxcycz.float().contiguous()
    lib = _lib.load()
    fn = lib.ssd3d_match_priors_analytic if analytic else lib.ssd3d_match_priors
    rc = fn(_ptr(gt_boxes), _ptr(gt_labels), offsets.data_ptr(), n, total, pri.data_ptr(), p, f32(t0), f32(t1),
            tc.data_ptr(), tl.data_ptr(), ov.data_ptr(), ofp.data_ptr(), pfo.data_ptr(), ws.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_match_priors")
    LAUNCHES[0] += 2
    return dict(true_classes=tc, true_locs=tl, overlap=ov, object_for_prior=ofp, prior_for_object=pfo[:total])


def multibox_loss(locs: torch.Tensor, scores: torch.Tensor, true_classes: torch.Tensor, true_locs: torch.Tensor,
                  alpha: float = 1.0, hard_negative_mining: bool = False, neg_pos_ratio: int = 3,
                  want_grads: bool = True):
    """-> (loss (2,) = [conf, loc], n_pos (1,) int32, grad_locs | None, grad_scores | None)."""
    _need_cuda(locs, scores, true_classes, true_locs)
    locs, scores = locs.float().contiguous(), scores.float().contiguous()
    n, p, c = scores.shape
    dev = locs.device
    lib = _lib.load()
    ws = torch.empty((lib.ssd3d_multibox_workspace_bytes(n, p),), dtype=torch.uint8, device=dev)
    out = torch.empty((2,), dtype=torch.float32, device=dev)
    n_pos = torch.empty((1,), dtype=torch.int32, device=dev)
    gl = torch.empty_like(locs) if want_grads else None
    gs = torch.empty_like(scores) if want_grads else None
    rc = lib.ssd3d_multibox_loss(locs.data_ptr(), scores.data_ptr(), true_classes.contiguous().data_ptr(),
                                 true_locs.contiguous().data_ptr(), n, p, c, float(alpha), int(hard_negative_mining),
                                 int(neg_pos_ratio), out.data_ptr(), n_pos.data_ptr(), _ptr(gl), _ptr(gs),
                                 ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_multibox_loss")
    LAUNCHES[0] += 3
    return out, n_pos, gl, gs


# ----------------------------------------------------------------------------------------------
# training step: raw convolutions, train-mode BatchNorm, backward kernels, Adam
# ----------------------------------------------------------------------------------------------
_CONST = {}


def _ones_zeros(n: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """Identity epilogue vectors (scale = 1, shift = 0) for the raw-conv launches."""
    key = (str(device), "oz")
    cur = _CONST.get(key)
    if cur is None or cur[0].numel() < n:
        m = max(n, 1024)
        cur = (torch.ones((m,), dtype=torch.float32, device=device), torch.zeros((m,), dtype=torch.float32, device=device))
        _CONST[key] = cur
    return cur


_WS_SLOT = ["ws"]      # scratch slot of the stream being issued to (training.py switches it for its side stream)
_WS_PINNED = set()     # data_ptr of scratch buffers whose address a captured CUDA graph has baked in
_WS_RETIRED = []       # pinned buffers that were outgrown: kept alive for the graphs that still replay into them


def _workspace(nbytes: int, device, slot: Optional[str] = None) -> torch.Tensor:
    """Grow-only scratch buffer per (device, slot); kernels of one stream use it strictly in order.  A buffer a
    captured graph refers to (``pin_workspaces``) is never freed: when a later call needs more, a new buffer takes
    over for eager launches and the old one stays alive for the graph's replays."""
    key = (str(device), slot or _WS_SLOT[0])
    cur = _CONST.get(key)
    if cur is None or cur.numel() < nbytes:
        if cur is not None and cur.data_ptr() in _WS_PINNED:
            _WS_RETIRED.append(cur)
        cur = torch.empty((max(int(nbytes), 1 << 20),), dtype=torch.uint8, device=device)
        _CONST[key] = cur
    return cur


def pin_workspaces() -> None:
    """Called after a CUDA-graph capture that used the scratch slots: their current buffers must outlive the graph."""
    for key, cur in _CONST.items():
        if isinstance(cur, torch.Tensor) and cur.dtype == torch.uint8:
            _WS_PINNED.add(cur.data_ptr())


def _sync_words(device) -> torch.Tensor:
    """Barrier words of the single-launch BatchNorm kernels (csrc/bn_unit.cu): zero-initialised once per (device,
    scratch slot) -- the kernels leave them zero -- and never freed (captured graphs bake the address in)."""
    key = (str(device), "bn_sync", _WS_SLOT[0])
    cur = _CONST.get(key)
    if cur is None:
        cur = torch.zeros((512,), dtype=torch.int32, device=device)
        _CONST[key] = cur
    return cur


def stem_conv_raw(x: torch.Tensor, w_packed: torch.Tensor, stride_d: int) -> torch.Tensor:
    """Raw stem conv output (no BN, no ReLU), channels-last bf16."""
    _need_cuda(x, w_packed)
    if x.dtype not in (torch.float32, BF16):
        x = x.float()
    x = x.contiguous()
    n, cin, d, h, w = x.shape
    y = _alloc_ndhwc(n, 32, conv_out(d, stride_d), conv_out(h, 2), conv_out(w, 2), x.device)
    one, zero = _ones_zeros(32, x.device)
    rc = _lib.load().ssd3d_stem_conv_affine(x.data_ptr(), int(x.dtype == BF16), w_packed.data_ptr(), one.data_ptr(),
                                            zero.data_ptr(), y.data_ptr(), n, cin, d, h, w, stride_d, 0, _stream())
    _lib.check(rc, "ssd3d_stem_conv_affine")
    LAUNCHES[0] += 1
    return y


def dwconv3d_raw(x: torch.Tensor, w_packed: torch.Tensor, stride: int) -> torch.Tensor:
    _need_cuda(x, w_packed)
    x = to_channels_last_bf16(x)
    n, c, d, h, w = x.shape
    y = _alloc_ndhwc(n, c, conv_out(d, stride), conv_out(h, stride), conv_out(w, stride), x.device)
    one, zero = _ones_zeros(c, x.device)
    rc = _lib.load().ssd3d_dwconv3d_affine(x.data_ptr(), w_packed.data_ptr(), one.data_ptr(), zero.data_ptr(),
                                           y.data_ptr(), n, c, d, h, w, stride, 0, _stream())
    _lib.check(rc, "ssd3d_dwconv3d_affine")
    LAUNCHES[0] += 1
    return y


def pw_gemm_raw(x2d_rows: int, x: torch.Tensor, w_packed: torch.Tensor, out: torch.Tensor) -> None:
    """out (M, Cout) bf16 = x (M, Cin) bf16 . w (Cout, Cin)^T -- the pointwise GEMM with an identity epilogue
    (raw pointwise conv, and the pointwise data gradient with the transposed weight)."""
    cout, cin = w_packed.shape
    one, zero = _ones_zeros(cout, x.device)
    rc = _lib.load().ssd3d_pwconv_affine(x.data_ptr(), w_packed.data_ptr(), one.data_ptr(), zero.data_ptr(),
                                         out.data_ptr(), x2d_rows, cin, cout, 0, 0, _stream())
    _lib.check(rc, "ssd3d_pwconv_affine")
    LAUNCHES[0] += 1


def pwconv_raw(x: torch.Tensor, w_packed: torch.Tensor) -> torch.Tensor:
    _need_cuda(x, w_packed)
    x = to_channels_last_bf16(x)
    n, c, d, h, w = x.shape
    y = _alloc_ndhwc(n, w_packed.shape[0], d, h, w, x.device)
    pw_gemm_raw(n * d * h * w, x, w_packed, y)
    return y


class BNState:
    """What the backward of one conv -> BN -> ReLU unit needs from the forward."""
    __slots__ = ("scale", "shift", "mean", "invstd")

    def __init__(self, c, device):
        buf = torch.empty((4, c), dtype=torch.float32, device=device)
        self.scale, self.shift, self.mean, self.invstd = buf[0], buf[1], buf[2], buf[3]


def bn_train_relu(z: torch.Tensor, bn: torch.nn.BatchNorm3d, nan_flag: Optional[torch.Tensor] = None):
    """Training-mode BatchNorm3d + ReLU on a raw conv output (channels-last bf16) -> (a, BNState); updates the
    module's running statistics and num_batches_tracked like nn.BatchNorm3d does."""
    return _bn_train_relu(z, bn, nan_flag, single_launch=True)


def _bn_train_relu_passes(z: torch.Tensor, bn: torch.nn.BatchNorm3d, nan_flag: Optional[torch.Tensor] = None):
    """``bn_train_relu`` on the three-launch passes of train.cu: what it falls back to when ``bn_unit`` does not take
    the shape or the driver refuses its launch, and the reference the single launch is tested against."""
    return _bn_train_relu(z, bn, nan_flag, single_launch=False)


def _bn_train_relu(z, bn, nan_flag, single_launch: bool):
    _need_cuda(z, nan_flag)
    n, c, d, h, w = z.shape
    m = n * d * h * w
    st = BNState(c, z.device)
    a = _alloc_ndhwc(n, c, d, h, w, z.device)
    lib = _lib.load()
    need = lib.ssd3d_bn_workspace_bytes(c)
    ws = _workspace(need, z.device)
    track = bn.track_running_stats and bn.running_mean is not None
    momentum = 0.1 if bn.momentum is None else float(bn.momentum)
    if track and bn.momentum is None:
        raise NotImplementedError("cumulative-average BatchNorm (momentum=None) is not used by the reference")
    nbt = bn.num_batches_tracked if (track and bn.num_batches_tracked is not None) else None
    args = (z.data_ptr(), m, c, _ptr(bn.weight.detach() if bn.weight is not None else None),
            _ptr(bn.bias.detach() if bn.bias is not None else None), float(bn.eps), momentum,
            _ptr(bn.running_mean if track else None), _ptr(bn.running_var if track else None), _ptr(nbt),
            st.scale.data_ptr(), st.shift.data_ptr(), st.mean.data_ptr(), st.invstd.data_ptr(),
            a.data_ptr(), _ptr(nan_flag), ws.data_ptr(), ws.numel())
    rc = _lib.SSD3D_ERR_UNSUPPORTED
    if single_launch and lib.ssd3d_bn_unit_supported(m, c):
        rc = lib.ssd3d_bn_unit_fwd(*args, _sync_words(z.device).data_ptr(), _stream())
        if rc != _lib.SSD3D_ERR_UNSUPPORTED:     # unsupported = the driver refused the launch: three-launch path
            _lib.check(rc, "ssd3d_bn_unit_fwd")
            LAUNCHES[0] += 1
    if rc == _lib.SSD3D_ERR_UNSUPPORTED:
        rc = lib.ssd3d_bn_train_fwd(*args, _stream())
        _lib.check(rc, "ssd3d_bn_train_fwd")
        LAUNCHES[0] += 3
    if track:
        # the kernel updated the running statistics through raw pointers: bump their version counters (host-side
        # only, no launch) so that caches keyed on (data_ptr, _version) -- folded eval-mode BN, captured inference
        # plans -- see the change
        bufs = [t for t in (bn.running_mean, bn.running_var, nbt) if t is not None]
        torch._C._autograd._unsafe_set_version_counter(bufs, [t._version + 1 for t in bufs])
    return a, st


def bn_relu_backward(z: torch.Tensor, grad_a: torch.Tensor, st: BNState, dgamma: torch.Tensor, dbeta: torch.Tensor):
    """-> dz, written over grad_a (both channels-last bf16); dgamma / dbeta (C) fp32 are filled."""
    return _bn_relu_backward(z, grad_a, st, dgamma, dbeta, single_launch=True)


def _bn_relu_backward_passes(z: torch.Tensor, grad_a: torch.Tensor, st: BNState, dgamma: torch.Tensor,
                             dbeta: torch.Tensor):
    """``bn_relu_backward`` on the three-launch passes of train.cu (see ``_bn_train_relu_passes``)."""
    return _bn_relu_backward(z, grad_a, st, dgamma, dbeta, single_launch=False)


def _bn_relu_backward(z, grad_a, st, dgamma, dbeta, single_launch: bool):
    n, c, d, h, w = z.shape
    lib = _lib.load()
    ws = _workspace(lib.ssd3d_bn_workspace_bytes(c), z.device)
    m = n * d * h * w
    args = (z.data_ptr(), grad_a.data_ptr(), m, c, st.scale.data_ptr(), st.shift.data_ptr(), st.mean.data_ptr(),
            st.invstd.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), grad_a.data_ptr(), ws.data_ptr(), ws.numel())
    rc = _lib.SSD3D_ERR_UNSUPPORTED
    if single_launch and lib.ssd3d_bn_unit_supported(m, c):
        rc = lib.ssd3d_bn_unit_bwd(*args, _sync_words(z.device).data_ptr(), _stream())
        if rc != _lib.SSD3D_ERR_UNSUPPORTED:
            _lib.check(rc, "ssd3d_bn_unit_bwd")
            LAUNCHES[0] += 1
    if rc == _lib.SSD3D_ERR_UNSUPPORTED:
        rc = lib.ssd3d_bn_relu_bwd(*args, _stream())
        _lib.check(rc, "ssd3d_bn_relu_bwd")
        LAUNCHES[0] += 3
    return grad_a


def pwconv_wgrad(dz: torch.Tensor, x: torch.Tensor, dw: torch.Tensor) -> None:
    """dw (Cout, Cin, 1,1,1) fp32 <- dz (M, Cout)^T . x (M, Cin)."""
    n, cin, d, h, w = x.shape
    cout = dz.shape[1]
    m = n * d * h * w
    lib = _lib.load()
    ws = _workspace(lib.ssd3d_wgrad_workspace_bytes(m, cout, cin), x.device)
    rc = lib.ssd3d_pwconv_wgrad(dz.data_ptr(), x.data_ptr(), m, cin, cout, dw.data_ptr(), ws.data_ptr(), ws.numel(),
                                _stream())
    _lib.check(rc, "ssd3d_pwconv_wgrad")
    LAUNCHES[0] += 2


def stem_wgrad(dz: torch.Tensor, x: torch.Tensor, stride_d: int, dw: torch.Tensor) -> None:
    n, cin, d, h, w = x.shape
    do, ho, wo = conv_out(d, stride_d), conv_out(h, 2), conv_out(w, 2)
    lib = _lib.load()
    ws = _workspace(lib.ssd3d_wgrad_workspace_bytes(n * do * ho * wo, 32, 27 * cin), x.device)
    rc = lib.ssd3d_stem_wgrad(dz.data_ptr(), x.data_ptr(), int(x.dtype == BF16), n, cin, d, h, w, stride_d,
                              dw.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_stem_wgrad")
    LAUNCHES[0] += 2


def stem_unit_backward(z: torch.Tensor, grad_a: torch.Tensor, st: BNState, dgamma: torch.Tensor, dbeta: torch.Tensor,
                       x: torch.Tensor, stride_d: int, dw: torch.Tensor) -> bool:
    """Backward of the stem unit (conv -> BN -> ReLU) in two launches: BatchNorm statistics only (dgamma, dbeta), then the
    weight-gradient kernel applies the BatchNorm + ReLU backward to the gradient rows as it loads them -- dz is never
    written.  False (nothing launched) where that path does not take the shape: the caller then runs
    ``bn_relu_backward`` + ``stem_wgrad``."""
    n, c, do, ho, wo = z.shape
    m = n * do * ho * wo
    _, cin, d, h, w = x.shape
    lib = _lib.load()
    if not lib.ssd3d_bn_unit_supported(m, c) or m < 128 * 148 or cin > 4:
        return False
    if not lib.ssd3d_stem_tc_supported(int(x.dtype == BF16), cin, w):
        return False
    ws = _workspace(max(lib.ssd3d_bn_workspace_bytes(c), lib.ssd3d_wgrad_workspace_bytes(m, 32, 27 * cin)), x.device)
    rc = lib.ssd3d_bn_unit_bwd(z.data_ptr(), grad_a.data_ptr(), m, c, st.scale.data_ptr(), st.shift.data_ptr(),
                               st.mean.data_ptr(), st.invstd.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), 0,
                               ws.data_ptr(), ws.numel(), _sync_words(z.device).data_ptr(), _stream())
    if rc == _lib.SSD3D_ERR_UNSUPPORTED:         # the driver refused the launch: nothing ran, take the two-step path
        return False
    _lib.check(rc, "ssd3d_bn_unit_bwd (statistics only)")
    rc = lib.ssd3d_stem_wgrad_bn(z.data_ptr(), grad_a.data_ptr(), x.data_ptr(), int(x.dtype == BF16), n, cin, d, h, w,
                                 stride_d, st.scale.data_ptr(), st.shift.data_ptr(), st.mean.data_ptr(),
                                 st.invstd.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), dw.data_ptr(), ws.data_ptr(),
                                 ws.numel(), _stream())
    _lib.check(rc, "ssd3d_stem_wgrad_bn")
    LAUNCHES[0] += 3
    return True


def head_grad_pack(dlocs, dscores, n, d, h, w, bpl, n_classes, prior_offset, dbias_loc, dbias_cls) -> torch.Tensor:
    """-> dO (G, N*D*H*W, 16) bf16 gradient rows of one head in G = ceil(bpl*(6+n_classes)/16) column groups;
    fills the two bias gradients."""
    lib = _lib.load()
    n_cols = bpl * (6 + n_classes)
    dO = torch.empty(((n_cols + 15) // 16, n * d * h * w, 16), dtype=BF16, device=dlocs.device)
    ws = _workspace(lib.ssd3d_head_grad_workspace_bytes(n, d, h, w, n_cols), dlocs.device)
    rc = lib.ssd3d_head_grad_pack(dlocs.data_ptr(), dscores.data_ptr(), n, d, h, w, bpl, n_classes, dlocs.shape[1],
                                  prior_offset, dO.data_ptr(), dbias_loc.data_ptr(), dbias_cls.data_ptr(),
                                  ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_head_grad_pack")
    LAUNCHES[0] += 3
    return dO


def head_wgrad(dO: torch.Tensor, x: torch.Tensor, n_loc: int, n_cls: int, dw_loc: torch.Tensor, dw_cls: torch.Tensor):
    n, c, d, h, w = x.shape
    lib = _lib.load()
    ws = _workspace(lib.ssd3d_wgrad_workspace_bytes(n * d * h * w, 16, 27 * c), x.device)
    rc = lib.ssd3d_head_wgrad(dO.data_ptr(), x.data_ptr(), n, c, d, h, w, n_loc, n_cls, dw_loc.data_ptr(),
                              dw_cls.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_head_wgrad")
    LAUNCHES[0] += 3 * ((n_loc + n_cls + 15) // 16)


def head_dgrad(dO: torch.Tensor, w_packed: torch.Tensor, like: torch.Tensor, addend: Optional[torch.Tensor] = None,
               n_cols: Optional[int] = None):
    """-> d(loss)/d(feature map) (channels-last bf16, shape of ``like``) [+ addend, written in place].
    ``n_cols`` = bpl*(6+n_classes) real gradient columns (default: all 16*G of dO)."""
    n, c, d, h, w = like.shape
    out = addend if addend is not None else _alloc_ndhwc(n, c, d, h, w, like.device)
    groups = dO.shape[0] if dO.dim() == 3 else 1
    n_cols = 16 * groups if n_cols is None else int(n_cols)
    rc = _lib.load().ssd3d_head_dgrad(dO.data_ptr(), w_packed.data_ptr(), _ptr(addend), out.data_ptr(), n, c, d, h, w,
                                      n_cols, _stream())
    _lib.check(rc, "ssd3d_head_dgrad")
    LAUNCHES[0] += 1
    return out


def dwconv3d_dgrad(dz: torch.Tensor, w_packed: torch.Tensor, like: torch.Tensor, stride: int) -> torch.Tensor:
    n, c, d, h, w = like.shape
    dx = _alloc_ndhwc(n, c, d, h, w, like.device)
    rc = _lib.load().ssd3d_dwconv3d_dgrad(dz.data_ptr(), w_packed.data_ptr(), dx.data_ptr(), n, c, d, h, w, stride,
                                          _stream())
    _lib.check(rc, "ssd3d_dwconv3d_dgrad")
    LAUNCHES[0] += 1
    return dx


def dwconv3d_wgrad(dz: torch.Tensor, x: torch.Tensor, stride: int, dw: torch.Tensor) -> None:
    n, c, d, h, w = x.shape
    lib = _lib.load()
    ws = _workspace(lib.ssd3d_dw_wgrad_workspace_bytes(c), x.device)
    rc = lib.ssd3d_dwconv3d_wgrad(dz.data_ptr(), x.data_ptr(), n, c, d, h, w, stride, dw.data_ptr(), ws.data_ptr(),
                                  ws.numel(), _stream())
    _lib.check(rc, "ssd3d_dwconv3d_wgrad")
    LAUNCHES[0] += 2


def adam_step(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
              bias_start: int, lr: float, lr_bias: float, step: int, betas=(0.9, 0.999), eps: float = 1e-8,
              weight_decay: float = 0.0, grad_scale: float = 1.0, status: Optional[torch.Tensor] = None) -> None:
    """``status`` (2,) int32: steps with a non-finite gradient are skipped and counted (see the header)."""
    _need_cuda(param, grad, exp_avg, exp_avg_sq, status)
    rc = _lib.load().ssd3d_adam_step(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                     param.numel(), bias_start, lr, lr_bias, betas[0], betas[1], eps, weight_decay,
                                     int(step), grad_scale, _ptr(status), _stream())
    _lib.check(rc, "ssd3d_adam_step")
    LAUNCHES[0] += 2 if status is not None else 1


def adam_step_dev(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
                  bias_start: int, base_lr: float, state: torch.Tensor, scalars: torch.Tensor, t_max: int = 0,
                  bias_lr_mult: float = 2.0, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                  grad_scale: float = 1.0) -> None:
    """Adam with the step counter, the cosine schedule and the skip-on-non-finite logic on the device (see the
    header): ``state`` (4,) int32 = [non-finite, skipped, applied, -], ``scalars`` (8,) fp32 scratch."""
    _need_cuda(param, grad, exp_avg, exp_avg_sq, state, scalars)
    rc = _lib.load().ssd3d_adam_step_dev(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                         param.numel(), bias_start, float(base_lr), float(bias_lr_mult), int(t_max),
                                         betas[0], betas[1], eps, weight_decay, grad_scale, state.data_ptr(),
                                         scalars.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_adam_step_dev")
    LAUNCHES[0] += 3


# ----------------------------------------------------------------------------------------------
# detection metrics (utils.py:155-396)
# ----------------------------------------------------------------------------------------------
def map_class(det_boxes: torch.Tensor, det_scores: torch.Tensor, det_images: torch.Tensor, true_boxes: torch.Tensor,
              true_difficulties: torch.Tensor, true_images: torch.Tensor, min_overlap: float,
              recall_thresholds: torch.Tensor):
    """Metrics of one class on the device (no host sync) -> dict of tensors; see include/ssd3d_b200.h."""
    _need_cuda(det_boxes, det_scores, det_images)
    dev = det_boxes.device
    nd, nt = int(det_boxes.shape[0]), int(true_boxes.shape[0])
    if nd == 0:
        raise RuntimeError("map_class needs at least one detection")
    db = det_boxes.float().contiguous()
    ds = det_scores.float().contiguous()
    di = det_images.to(torch.int32).contiguous()
    tb = true_boxes.to(dev).float().contiguous()
    td = true_difficulties.to(dev).to(torch.uint8).contiguous()
    ti = true_images.to(dev).to(torch.int32).contiguous()
    thr = recall_thresholds.to(dev).float().contiguous()
    k = int(thr.numel())
    out = dict(sorted_scores=torch.empty((nd,), dtype=torch.float32, device=dev),
               sort_index=torch.empty((nd,), dtype=torch.int32, device=dev),
               tp=torch.empty((nd,), dtype=torch.float32, device=dev),
               fp=torch.empty((nd,), dtype=torch.float32, device=dev),
               detected=torch.empty((nt,), dtype=torch.uint8, device=dev),
               volumes=torch.empty((nt,), dtype=torch.float32, device=dev),
               cum_precision=torch.empty((nd,), dtype=torch.float32, device=dev),
               cum_recall=torch.empty((nd,), dtype=torch.float32, device=dev),
               stats=torch.empty((4 + k,), dtype=torch.float32, device=dev))
    lib = _lib.load()
    ws = torch.empty((lib.ssd3d_map_workspace_bytes(nd, nt),), dtype=torch.uint8, device=dev)
    rc = lib.ssd3d_map_class(db.data_ptr(), ds.data_ptr(), di.data_ptr(), nd, _ptr(tb if nt else None),
                             _ptr(td if nt else None), _ptr(ti if nt else None), nt, f32(min_overlap), thr.data_ptr(), k,
                             out["sorted_scores"].data_ptr(), out["sort_index"].data_ptr(), out["tp"].data_ptr(),
                             out["fp"].data_ptr(), _ptr(out["detected"] if nt else None),
                             _ptr(out["volumes"] if nt else None), out["cum_precision"].data_ptr(),
                             out["cum_recall"].data_ptr(), out["stats"].data_ptr(), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_map_class")
    LAUNCHES[0] += 5 if nt else 4
    return out


def gather_cast(src: torch.Tensor, index: torch.Tensor, dst: torch.Tensor) -> None:
    """dst[i] = src[index[i]] (0 where index < 0), cast to dst's dtype (bf16 or fp32): one-launch weight packing."""
    _need_cuda(src, index, dst)
    rc = _lib.load().ssd3d_gather_cast(src.data_ptr(), index.data_ptr(), dst.numel(), dst.data_ptr(),
                                       int(dst.dtype == BF16), _stream())
    _lib.check(rc, "ssd3d_gather_cast")
    LAUNCHES[0] += 1


def normalize_intensity_nonzero(x: torch.Tensor, out_dtype: torch.dtype = BF16) -> torch.Tensor:
    """MONAI ``NormalizeIntensity(nonzero=True)`` (datasets.py:403) per (volume, channel) on the device:
    x (N, C, D, H, W) fp32 -> z-scored over its non-zero voxels, fp32 or bf16 (the stem's input format)."""
    _need_cuda(x)
    if x.dim() != 5:
        raise RuntimeError("expected a 5-D (N, C, D, H, W) tensor")
    if out_dtype not in (torch.float32, BF16):
        raise RuntimeError("out_dtype must be float32 or bfloat16")
    x = x.float().contiguous()
    n, c = x.shape[0], x.shape[1]
    vox = x.numel() // (n * c)
    y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    lib = _lib.load()
    ws = torch.empty((lib.ssd3d_normalize_workspace_bytes(n * c),), dtype=torch.uint8, device=x.device)
    rc = lib.ssd3d_normalize_intensity_nonzero(x.data_ptr(), n * c, vox, y.data_ptr(), int(out_dtype == BF16),
                                               ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_normalize_intensity_nonzero")
    LAUNCHES[0] += 3
    return y


def gt_boxes_from_segmentation(seg: torch.Tensor, n_classes: int = 0, max_boxes: int = 1024):
    """Ground-truth boxes of segmentation volumes on the device (utils.py:438-513 ``BoundingBoxesGeneratord``,
    "binary" mode for ``n_classes == 0``, "classes" mode with ``classes = [1..n_classes]`` otherwise).
    seg (N, D, H, W) or (N, 1, D, H, W), uint8 or floating -> (boxes list[(n_i, 6) fp32], labels list[(n_i,) int64]),
    fractional [min, max] index boxes in array-axis order, the reference's order and zero-volume filter."""
    _need_cuda(seg)
    if seg.dim() == 5 and seg.shape[1] == 1:
        seg = seg[:, 0]
    if seg.dim() != 4:
        raise RuntimeError("expected (N, D, H, W) or (N, 1, D, H, W) segmentations")
    boxes, labels, meta = gt_boxes_padded(seg, n_classes, max_boxes)
    n = boxes.shape[0]
    counts, comps = meta.cpu().tolist()
    if max(comps) > max_boxes:
        raise RuntimeError("segmentation has %d connected components, max_boxes=%d" % (max(comps), max_boxes))
    return [boxes[i, :counts[i]] for i in range(n)], [labels[i, :counts[i]] for i in range(n)]


def gt_boxes_padded(seg: torch.Tensor, n_classes: int = 0, max_boxes: int = 1024, out=None, workspace=None):
    """``gt_boxes_from_segmentation`` without the host read: -> (boxes (N, max_boxes, 6), labels (N, max_boxes),
    meta (2, N) int32 = [counts, n_components]); rows [0, counts[i]) are valid, and only if n_components[i] <=
    max_boxes.  ``out`` / ``workspace`` (from an earlier call) make it capturable in a CUDA graph."""
    if seg.dtype == torch.uint8:
        dt = 0
    else:
        seg, dt = seg.float(), 1
    seg = seg.contiguous()
    n, d, h, w = seg.shape
    dev = seg.device
    lib = _lib.load()
    if out is None:
        out = (torch.empty((n, max_boxes, 6), dtype=torch.float32, device=dev),
               torch.empty((n, max_boxes), dtype=torch.int64, device=dev),
               torch.empty((2, n), dtype=torch.int32, device=dev))
    boxes, labels, meta = out
    if workspace is None:
        workspace = torch.empty((lib.ssd3d_gt_boxes_workspace_bytes(n, d, h, w, max_boxes),), dtype=torch.uint8,
                                device=dev)
    rc = lib.ssd3d_gt_boxes_from_segmentation(seg.data_ptr(), dt, n, d, h, w, int(n_classes), int(max_boxes),
                                              boxes.data_ptr(), labels.data_ptr(), meta[0].data_ptr(),
                                              meta[1].data_ptr(), workspace.data_ptr(), workspace.numel(), _stream())
    _lib.check(rc, "ssd3d_gt_boxes_from_segmentation")
    LAUNCHES[0] += 6
    return boxes, labels, meta


def gt_boxes_from_instances(seg: torch.Tensor, thresholds, max_boxes: int = 1024):
    """``BoundingBoxesGeneratord`` in "instances" mode on the device (utils.py:439-441,483-513): ``seg`` holds one
    integer id per object, ``thresholds`` = [(min_c, max_c), ...] maps the id range [min_c, max_c) to class c+1
    (``max_c`` may be ``inf``).  One box per id over all its voxels, ordered by class then ascending id; same output
    format, box convention and zero-volume filter as ``gt_boxes_from_segmentation``."""
    _need_cuda(seg)
    if seg.dim() == 5 and seg.shape[1] == 1:
        seg = seg[:, 0]
    if seg.dim() != 4:
        raise RuntimeError("expected (N, D, H, W) or (N, 1, D, H, W) segmentations")
    if seg.dtype == torch.uint8:
        dt = 0
    else:
        seg, dt = seg.float(), 1
    seg = seg.contiguous()
    n, d, h, w = seg.shape
    dev = seg.device
    thr = [(float(a), float(b)) for a, b in thresholds]
    if not thr:
        raise ValueError("instances mode needs thresholds")          # utils.py:417
    srt = sorted(thr)
    if any(srt[i][1] > srt[i + 1][0] for i in range(len(srt) - 1)):
        raise NotImplementedError("overlapping id ranges are not supported")
    top = max(b for _, b in thr)
    if top == float("inf"):                       # open range: the largest id present decides the table size
        top = float(seg.max().item()) + 1.0
    id_limit = int(min(max(2.0, top), 2.0 ** 30))
    import math
    thr_dev = torch.tensor([[int(math.ceil(max(a, 0.0))), int(min(math.ceil(b), id_limit)) if b != float("inf")
                             else id_limit] for a, b in thr], dtype=torch.int32, device=dev)
    boxes = torch.empty((n, max_boxes, 6), dtype=torch.float32, device=dev)
    labels = torch.empty((n, max_boxes), dtype=torch.int64, device=dev)
    meta = torch.empty((2, n), dtype=torch.int32, device=dev)
    lib = _lib.load()
    need = lib.ssd3d_gt_boxes_instances_workspace_bytes(n, id_limit, max_boxes)
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    rc = lib.ssd3d_gt_boxes_from_instances(seg.data_ptr(), dt, n, d, h, w, thr_dev.data_ptr(), len(thr), id_limit,
                                           int(max_boxes), boxes.data_ptr(), labels.data_ptr(), meta[0].data_ptr(),
                                           meta[1].data_ptr(), ws.data_ptr(), ws.numel(), _stream())
    _lib.check(rc, "ssd3d_gt_boxes_from_instances")
    LAUNCHES[0] += 4
    counts, comps = meta.cpu().tolist()
    if max(comps) > max_boxes:
        raise RuntimeError("segmentation has %d instances, max_boxes=%d" % (max(comps), max_boxes))
    return [boxes[i, :counts[i]] for i in range(n)], [labels[i, :counts[i]] for i in range(n)]


def generate_volumes(n: int, channels: int, image_size, first_idx: int = 0, seed: int = 0, num_objects=(1, 5),
                     object_size=(6, 14), device=None, max_cubes: int = 64):
    """Raw synthetic volumes on the device (generate_artificial_dataset.py:63-105 with a counter-based RNG, see
    the header): -> (raw (N, C, D, H, W) fp32, mask (N, D, H, W) uint8, cubes (N, max_cubes, 4) int32, n_cubes (N,))."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("generate_volumes runs on a CUDA device; the host generator is synthetic.make_batch")
    d, h, w = (int(v) for v in image_size)
    raw = torch.empty((n, channels, d, h, w), dtype=torch.float32, device=dev)
    mask = torch.empty((n, d, h, w), dtype=torch.uint8, device=dev)
    cubes = torch.zeros((n, max_cubes, 4), dtype=torch.int32, device=dev)
    n_cubes = torch.zeros((n,), dtype=torch.int32, device=dev)
    smin, smax = sorted(int(v) for v in object_size)
    with torch.cuda.device(dev):
        rc = _lib.load().ssd3d_generate_volumes(int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_idx), n, channels, d, h, w,
                                                int(num_objects[0]), int(num_objects[1]), smin, smax, max_cubes,
                                                raw.data_ptr(), mask.data_ptr(), cubes.data_ptr(), n_cubes.data_ptr(),
                                                _stream())
    _lib.check(rc, "ssd3d_generate_volumes")
    LAUNCHES[0] += 2
    return raw, mask, cubes, n_cubes


# ----------------------------------------------------------------------------------------------
# training batches from a device-resident data set (data.py, training.fit_epoch)
# ----------------------------------------------------------------------------------------------
def augment_batch(src: torch.Tensor, masks: torch.Tensor, order: torch.Tensor, state: torch.Tensor,
                  boxes: torch.Tensor, box_offsets: torch.Tensor, batch_size: int, out_size, pos_ratio: float = 0.0,
                  flip_prob: float = 0.0, rot90_prob: float = 0.0, rot90_axes=(0, 1), scale: float = 0.0,
                  shift: float = 0.0, out=None):
    """One augmented training batch (see ``ssd3d_augment_batch`` in the header): src (S, C, Ds, Hs, Ws) fp32 / bf16,
    masks (S, Ds, Hs, Ws) uint8, order (S) int32, state (8) int64 (advanced by the call), boxes (B, 6) int32 voxel
    boxes, box_offsets (S + 1) int32 -> (images (N, C, d, h, w) bf16, masks (N, d, h, w) uint8, record (N, 16)
    int32).  ``out``: the three output tensors to write (static buffers of a captured step)."""
    args, out = _augment_args(src, masks, order, state, boxes, box_offsets, batch_size, out_size, pos_ratio,
                              flip_prob, rot90_prob, rot90_axes, scale, shift, 16, out)
    rc = _lib.load().ssd3d_augment_batch(*args, *(t.data_ptr() for t in out), _stream())
    _lib.check(rc, "ssd3d_augment_batch")
    LAUNCHES[0] += 1
    return out


def augment_affine_batch(src: torch.Tensor, masks: torch.Tensor, order: torch.Tensor, state: torch.Tensor,
                         boxes: torch.Tensor, box_offsets: torch.Tensor, batch_size: int, out_size,
                         pos_ratio: float = 0.0, flip_prob: float = 0.0, rot90_prob: float = 0.0, rot90_axes=(0, 1),
                         scale: float = 0.0, shift: float = 0.0, affine_prob: float = 0.0, rotate_range=(0, 0, 0),
                         zoom_range=(0, 0, 0), out=None):
    """``augment_batch`` with a random rotation (``rotate_range`` radians per plane) and zoom (``zoom_range`` per
    axis) of the crop, applied with probability ``affine_prob`` (see ``ssd3d_augment_affine_batch`` in the header)
    -> (images, masks, record (N, 32) int32: words 0-15 those of ``augment_batch``, 16 affine drawn, 17-19 theta,
    20-22 z, 23-31 the 3x3 matrix M, fp32 bits)."""
    args, out = _augment_args(src, masks, order, state, boxes, box_offsets, batch_size, out_size, pos_ratio,
                              flip_prob, rot90_prob, rot90_axes, scale, shift, 32, out)
    rot, zoom = (ctypes.c_float * 3)(*(float(v) for v in rotate_range)), (ctypes.c_float * 3)(*(float(v) for v in
                                                                                                 zoom_range))
    rc = _lib.load().ssd3d_augment_affine_batch(*args, float(affine_prob), rot, zoom, *(t.data_ptr() for t in out),
                                                _stream())
    _lib.check(rc, "ssd3d_augment_affine_batch")
    LAUNCHES[0] += 1
    return out


def augment_elastic_batch(src: torch.Tensor, masks: torch.Tensor, order: torch.Tensor, state: torch.Tensor,
                          boxes: torch.Tensor, box_offsets: torch.Tensor, batch_size: int, out_size,
                          pos_ratio: float = 0.0, flip_prob: float = 0.0, rot90_prob: float = 0.0, rot90_axes=(0, 1),
                          scale: float = 0.0, shift: float = 0.0, affine_prob: float = 0.0, rotate_range=(0, 0, 0),
                          zoom_range=(0, 0, 0), elastic_prob: float = 0.0, elastic_points=(7, 7, 7),
                          elastic_magnitude=(0, 0, 0), out=None):
    """``augment_affine_batch`` with a random cubic B-spline deformation of the crop (``elastic_points`` control
    points and at most ``elastic_magnitude`` source voxels of displacement per axis), applied with probability
    ``elastic_prob`` (see ``ssd3d_augment_elastic_batch`` in the header) -> (images, masks, record (N, 33) int32:
    words 0-31 those of ``augment_affine_batch``, 32 field drawn)."""
    args, out = _augment_args(src, masks, order, state, boxes, box_offsets, batch_size, out_size, pos_ratio,
                              flip_prob, rot90_prob, rot90_axes, scale, shift, 33, out)
    rot, zoom = (ctypes.c_float * 3)(*(float(v) for v in rotate_range)), (ctypes.c_float * 3)(*(float(v) for v in
                                                                                                 zoom_range))
    pts = (ctypes.c_int32 * 3)(*(int(v) for v in elastic_points))
    mag = (ctypes.c_float * 3)(*(float(v) for v in elastic_magnitude))
    rc = _lib.load().ssd3d_augment_elastic_batch(*args, float(affine_prob), rot, zoom, float(elastic_prob), pts, mag,
                                                 *(t.data_ptr() for t in out), _stream())
    _lib.check(rc, "ssd3d_augment_elastic_batch")
    LAUNCHES[0] += 1
    return out


def augment_intensity_batch(images: torch.Tensor, state: torch.Tensor, batch_size: int, bias_prob: float = 0.0,
                            bias_coefficient: float = 0.0, gamma_prob: float = 0.0, gamma_log_range: float = 0.0,
                            noise_prob: float = 0.0, noise_std: float = 0.0, out_record=None, workspace=None):
    """MR intensity augmentation in place on a batch an augment launch has just written (see
    ``ssd3d_augment_intensity_batch`` in the header): per slot, with their probabilities, gamma = exp(U(-r, r)) on the
    slot's [min, max], an order-3 polynomial bias field exp(sum c u_d^i u_h^j u_w^k) with c ~ U(-bias_coefficient,
    bias_coefficient), and Gaussian noise of sigma ~ U(0, noise_std); ``state`` is read, not advanced.  images
    (N, C, d, h, w) bf16 -> record (N, 27) int32: gamma / bias / noise drawn, gamma, lo, hi, sigma, the 20
    coefficients (fp32 bits).  ``workspace``: ``augment_intensity_workspace_bytes`` bytes (allocated if None)."""
    _need_cuda(images, state)
    if images.dim() != 5 or images.dtype != BF16 or not images.is_contiguous():
        raise RuntimeError("expected contiguous bf16 images (N, C, d, h, w)")
    if state.dtype != torch.int64 or not state.is_contiguous():
        raise RuntimeError("state must be contiguous int64")
    n, c, d, h, w = images.shape
    if n != int(batch_size):
        raise RuntimeError("images hold %d volumes, batch_size is %d" % (n, int(batch_size)))
    lib = _lib.load()
    if out_record is None:
        out_record = torch.empty((n, 27), dtype=torch.int32, device=images.device)
    if workspace is None:
        workspace = torch.empty((max(1, augment_intensity_workspace_bytes(n, c, d, h, w)),), dtype=torch.uint8,
                                device=images.device)
    rc = lib.ssd3d_augment_intensity_batch(images.data_ptr(), n, c, d, h, w, state.data_ptr(), float(bias_prob),
                                           float(bias_coefficient), float(gamma_prob), float(gamma_log_range),
                                           float(noise_prob), float(noise_std), out_record.data_ptr(),
                                           workspace.data_ptr(), workspace.numel(), _stream())
    _lib.check(rc, "ssd3d_augment_intensity_batch")
    LAUNCHES[0] += 2
    return out_record


def augment_intensity_workspace_bytes(n: int, c: int, d: int, h: int, w: int) -> int:
    return int(_lib.load().ssd3d_augment_intensity_workspace_bytes(int(n), int(c), int(d), int(h), int(w)))


def _augment_args(src, masks, order, state, boxes, box_offsets, batch_size, out_size, pos_ratio, flip_prob,
                  rot90_prob, rot90_axes, scale, shift, record_words, out):
    """The checked leading arguments shared by ssd3d_augment_batch, ssd3d_augment_affine_batch and
    ssd3d_augment_elastic_batch, and the three output tensors (allocated unless ``out`` is given)."""
    _need_cuda(src, masks, order, state, boxes, box_offsets)
    if src.dim() != 5 or masks.dim() != 4 or src.dtype not in (torch.float32, BF16) or masks.dtype != torch.uint8:
        raise RuntimeError("expected src (S, C, D, H, W) fp32/bf16 and masks (S, D, H, W) uint8")
    for t, dt in ((order, torch.int32), (state, torch.int64), (boxes, torch.int32), (box_offsets, torch.int32)):
        if t.dtype != dt or not t.is_contiguous():
            raise RuntimeError("order / boxes / box_offsets must be contiguous int32 and state int64")
    s, c, ds, hs, ws = src.shape
    d, h, w = (int(v) for v in out_size)
    n = int(batch_size)
    if out is None:
        out = (torch.empty((n, c, d, h, w), dtype=BF16, device=src.device),
               torch.empty((n, d, h, w), dtype=torch.uint8, device=src.device),
               torch.empty((n, record_words), dtype=torch.int32, device=src.device))
    args = (src.data_ptr(), int(src.dtype == BF16), masks.data_ptr(), s, c, ds, hs, ws, order.data_ptr(),
            state.data_ptr(), boxes.data_ptr(), box_offsets.data_ptr(), n, d, h, w, float(pos_ratio), float(flip_prob),
            float(rot90_prob), int(rot90_axes[0]), int(rot90_axes[1]), float(scale), float(shift))
    return args, tuple(out)


def gt_pack(boxes: torch.Tensor, labels: torch.Tensor, meta: torch.Tensor, per_volume: int, out=None,
            status: Optional[torch.Tensor] = None):
    """The output of ``gt_boxes_padded`` -> the packed ground truth of a training step, no host sync:
    (gt_boxes (N * per_volume, 6), gt_labels (N * per_volume) int64, offsets (N + 1) int32, status (2) int32 =
    [overflow of this batch, overflowing batches so far]).  An overflowing batch is packed without ground truth."""
    _need_cuda(boxes, labels, meta)
    n, max_boxes = int(boxes.shape[0]), int(boxes.shape[1])
    dev = boxes.device
    if out is None:
        out = (torch.zeros((n * per_volume, 6), dtype=torch.float32, device=dev),
               torch.zeros((n * per_volume,), dtype=torch.int64, device=dev),
               torch.zeros((n + 1,), dtype=torch.int32, device=dev))
    if status is None:
        status = torch.zeros((2,), dtype=torch.int32, device=dev)
    gb, gl, offs = out
    if gb.shape[0] < n * per_volume or gl.shape[0] < n * per_volume or offs.shape[0] != n + 1:
        raise RuntimeError("gt_pack: output buffers smaller than N * per_volume rows")
    rc = _lib.load().ssd3d_gt_pack(boxes.data_ptr(), labels.data_ptr(), meta[0].data_ptr(), meta[1].data_ptr(), n,
                                   max_boxes, int(per_volume), gb.data_ptr(), gl.data_ptr(), offs.data_ptr(),
                                   status.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_gt_pack")
    LAUNCHES[0] += 1
    return gb, gl, offs, status


# ----------------------------------------------------------------------------------------------
# sliding-window inference over scans larger than the network input (csrc/windows.cu, LSSD3D.predict_scans)
# ----------------------------------------------------------------------------------------------
def window_map(scan_shape, window, origins) -> Tuple[Tuple[float, float, float], torch.Tensor]:
    """Factors of the window -> scan coordinate map x' = x * scale_k + offset[t, k] (spatial axis k), each rounded
    to fp32 once: scale_k = fp32(w_k / S_k), offset[t, k] = fp32(o_k / S_k).  -> (scale (3 floats), offset (T, 3)
    fp32 CPU tensor)."""
    scale = tuple(f32(int(w) / int(s)) for w, s in zip(window, scan_shape))
    o = np.asarray(origins, dtype=np.float64).reshape(-1, 3)
    offset = (o / np.asarray([float(s) for s in scan_shape])).astype(np.float32)
    return scale, torch.from_numpy(offset)


def window_gather(src: torch.Tensor, window, overlap: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The sliding windows of scans src (S, C, D, H, W) fp32 / bf16 (grid of ``data.window_origins``) -> (S*T, C, d, h, w)
    bf16 NCDHW, scan-major; ``out`` may be a static buffer of that shape (a captured step)."""
    from .data import window_origins, window_strides
    _need_cuda(src)
    if src.dim() != 5 or src.dtype not in (torch.float32, BF16) or not src.is_contiguous():
        raise RuntimeError("expected contiguous scans (S, C, D, H, W) fp32/bf16")
    s, c, dd, hh, ww = src.shape
    d, h, w = (int(v) for v in window)
    nd, nh, nw, _ = window_origins((dd, hh, ww), (d, h, w), overlap)
    sd, sh, sw = window_strides((d, h, w), overlap)
    n = s * nd * nh * nw
    if out is None:
        out = torch.empty((n, c, d, h, w), dtype=BF16, device=src.device)
    if tuple(out.shape) != (n, c, d, h, w) or out.dtype != BF16 or not out.is_contiguous():
        raise RuntimeError("window_gather: out must be a contiguous (%d, %d, %d, %d, %d) bf16 tensor" % (n, c, d, h, w))
    rc = _lib.load().ssd3d_window_gather(src.data_ptr(), int(src.dtype == BF16), s, c, dd, hh, ww, d, h, w, sd, sh, sw,
                                         out.data_ptr(), _stream())
    _lib.check(rc, "ssd3d_window_gather")
    LAUNCHES[0] += 1
    return out


def merge_windows(boxes: torch.Tensor, scores: torch.Tensor, labels: torch.Tensor, count: torch.Tensor, n_scans: int,
                  scan_shape, window, overlap: float, n_classes: int, min_score: float, max_overlap: float,
                  top_k: int, offset: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None,
                  out=None, out_count: Optional[torch.Tensor] = None,
                  status: Optional[torch.Tensor] = None) -> DetectOutput:
    """Per-window detections -- the padded ``detect_objects_padded`` outputs over n_scans * T windows: boxes
    (S*T, K, 6), scores (S*T, K), labels (S*T, K) int64, count (S*T) int32 -- merged into per-scan detections in the
    scan's fractional coordinates (see ``ssd3d_merge_windows`` in the header), no host sync.  ``offset``: the
    (T, 3) fp32 device tensor of ``window_map`` (made here when None); ``out`` / ``out_count`` / ``status``: static
    buffers like ``detect_objects_padded``'s.  ``prior`` of the result holds the candidate index t * K + r."""
    from .data import window_origins
    _need_cuda(boxes, scores, labels, count)
    nd, nh, nw, origins = window_origins(scan_shape, window, overlap)
    t = nd * nh * nw
    n, k = int(scores.shape[0]), int(scores.shape[1])
    if n != int(n_scans) * t or tuple(boxes.shape) != (n, k, 6) or tuple(labels.shape) != (n, k) or \
            tuple(count.shape) != (n,):
        raise RuntimeError("merge_windows: expected boxes (S*T, K, 6), scores / labels (S*T, K), count (S*T) with "
                           "S*T = %d * %d" % (n_scans, t))
    if boxes.dtype != torch.float32 or scores.dtype != torch.float32 or labels.dtype != torch.int64 or \
            count.dtype != torch.int32 or not all(x.is_contiguous() for x in (boxes, scores, labels, count)):
        raise RuntimeError("merge_windows: boxes / scores fp32, labels int64 and count int32, all contiguous")
    top_k = int(top_k)
    if detect_needs_long_lists(t * k, top_k):
        raise ValueError("merge_windows: top_k = %d over %d windows (%d candidates per scan) needs the any-length "
                         "merge, which is not supported; lower top_k or the window count" % (top_k, t, t * k))
    dev = boxes.device
    scale, off_host = window_map(scan_shape, window, origins)
    if offset is None:
        offset = off_host.to(dev)
    lib = _lib.load()
    s = int(n_scans)
    need = lib.ssd3d_merge_windows_workspace_bytes(s, t, k, int(n_classes), top_k)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((need,), dtype=torch.uint8, device=dev)
    if out is None:
        out = (torch.empty((s, top_k, 6), dtype=torch.float32, device=dev),
               torch.empty((s, top_k), dtype=torch.float32, device=dev),
               torch.empty((s, top_k), dtype=torch.int64, device=dev),
               torch.empty((s, top_k), dtype=torch.int64, device=dev))
    ob, osc, ol, op = out
    if out_count is None:
        out_count = torch.empty((s,), dtype=torch.int32, device=dev)
    if status is None:
        status = torch.empty((1,), dtype=torch.int32, device=dev)
    rc = lib.ssd3d_merge_windows(boxes.data_ptr(), scores.data_ptr(), labels.data_ptr(), count.data_ptr(), s, t, k,
                                 offset.data_ptr(), scale[0], scale[1], scale[2], int(n_classes), f32(min_score),
                                 f32(max_overlap), top_k, ob.data_ptr(), osc.data_ptr(), ol.data_ptr(), op.data_ptr(),
                                 out_count.data_ptr(), workspace.data_ptr(), workspace.numel(), status.data_ptr(),
                                 _stream())
    _lib.check(rc, "ssd3d_merge_windows")
    LAUNCHES[0] += 4
    return DetectOutput(ob, osc, ol, op, out_count, status)
