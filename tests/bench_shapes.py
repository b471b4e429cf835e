"""The shapes each kernel sees in the two workloads ``bench.py`` times, read off the model itself, and the
shape-selected kernel switches restated where the library has no query for them.

The per-kernel parity tests take their benchmark cases from here, so the paths a user runs most are the paths the
suite checks; ``tests/test_host_bench_shapes.py`` pins the table against a hand-written list, so a change to the
model or to the benchmark's configuration shows up as a failing test rather than as coverage that drifts away.
Nothing here needs a GPU.
"""
from __future__ import annotations

import functools
from collections import namedtuple

import torch

# bench.py:65 (CHANNELS, SIZE, BATCH) and bench.py:69 (TRAIN_CHANNELS, TRAIN_SIZE, TRAIN_BATCH), restated: importing
# bench.py puts the repository root on sys.path and, for some command lines, hides the GPU (bench.py:54-57).
Config = namedtuple("Config", "name channels size batch")
INFER = Config("infer", 2, (128, 128, 128), 8)       # predict_step on bf16 batches
TRAIN = Config("train", 1, (96, 96, 96), 16)         # fit_step on fp32 batches
CONFIGS = (INFER, TRAIN)

SMS = 148                      # B200 multiprocessors: the BatchNorm tile plan and the kw head size their grids by it

# one record per kernel input; `unit` names the layer (stem, f1..f7 = base.features[1..7])
Stem = namedtuple("Stem", "unit cin n size stride_d dtype")          # input (n, cin, *size), output stride (sd, 2, 2)
BN = namedtuple("BN", "unit n c size")                               # train-mode BatchNorm over n * prod(size) rows
Depthwise = namedtuple("Depthwise", "unit c n size stride")          # input (n, c, *size)
Pointwise = namedtuple("Pointwise", "unit cin cout n size")          # M = n * prod(size) rows
Head = namedtuple("Head", "unit c n size bpl")                       # feature map (n, c, *size), bpl boxes per location
Block = namedtuple("Block", "unit cin cout stride n size")           # fused depthwise -> pointwise, input (n, cin, *size)


def rows(n, size):
    return n * size[0] * size[1] * size[2]


def _conv_out(size, conv):
    return tuple((size[a] + 2 * conv.padding[a] - conv.kernel_size[a]) // conv.stride[a] + 1 for a in range(3))


@functools.lru_cache(maxsize=None)
def table(cfg: Config) -> dict:
    """Per kernel family, the inputs one step of ``cfg`` hands each kernel, in network order: LSSD3D built on the
    CPU, its ``base.features`` walked (stem, then depthwise -> BN -> pointwise -> BN per Block) and its prediction
    layers read off ``pred_convs``.  Every family is listed for both configurations; the training kernels (BatchNorm,
    the gradients) run at TRAIN's shapes, the eval-mode forward kernels (stem + BN + ReLU, fused Block) at INFER's."""
    from mslesions3d_b200.mobilenet import ConvBN
    from mslesions3d_b200.ssd3d import LSSD3D
    model = LSSD3D(n_classes=2, input_channels=cfg.channels, input_size=cfg.size)
    n = cfg.batch
    out = {k: [] for k in ("stem", "bn", "dw", "pw", "head", "block")}
    size, maps = tuple(cfg.size), {}
    dtype = torch.bfloat16 if cfg.name == "infer" else torch.float32
    for i, f in enumerate(model.base.features):
        unit = "stem" if i == 0 else "f%d" % i
        if isinstance(f, ConvBN):
            conv = f[0]
            out["stem"].append(Stem(unit, conv.in_channels, n, size, conv.stride[0], dtype))
            size = _conv_out(size, conv)
            out["bn"].append(BN(unit, n, conv.out_channels, size))
            maps[i] = (size, conv.out_channels)
        else:
            dw, pw = f.conv1, f.conv2
            assert len(set(dw.stride)) == 1
            out["dw"].append(Depthwise(unit, dw.in_channels, n, size, dw.stride[0]))
            out["block"].append(Block(unit, dw.in_channels, pw.out_channels, dw.stride[0], n, size))
            size = _conv_out(size, dw)
            out["bn"].append(BN(unit + ".bn1", n, dw.out_channels, size))
            out["pw"].append(Pointwise(unit, pw.in_channels, pw.out_channels, n, size))
            out["bn"].append(BN(unit + ".bn2", n, pw.out_channels, size))
            maps[i] = (size, pw.out_channels)
    pc = model.pred_convs
    for j, layer in enumerate(model.aspect_ratios):
        fsize, c = maps[layer]
        assert pc.loc_convs[j].in_channels == c
        out["head"].append(Head("f%d" % layer, c, n, fsize, pc.n_boxes[layer]))
    return out


def distinct(records, key):
    """First record of each distinct ``key(record)``, in order."""
    seen, keep = set(), []
    for r in records:
        if key(r) not in seen:
            seen.add(key(r))
            keep.append(r)
    return keep


def bn_shapes(cfg: Config = TRAIN):
    """Every distinct (rows, channels) BatchNorm input of a training step, as (n, c, size)."""
    return [(b.n, b.c, b.size) for b in distinct(table(cfg)["bn"], lambda b: (rows(b.n, b.size), b.c))]


# ---------------------------------------------------------------------------------------------------------------
# Kernel switches the library chooses from the shape and does not report.  Each restates the C it mirrors; the
# boundary cases below sit on both sides of every one of them.
# ---------------------------------------------------------------------------------------------------------------
def bn_kernel(m: int, c: int, sms: int = SMS) -> str:
    """The train-mode BatchNorm kernel ``ops.bn_train_relu`` / ``ops.bn_relu_backward`` launch for m rows of c
    channels: "cluster" (bn_cluster_plan, csrc/bn_unit.cu:634-636: at most BC_MAX_K * BC_MAX_R * BC_THREADS = 8192
    rows), "tile<CG>-keep" / "tile<CG>-stream" (bn_tile_plan, bn_unit.cu:961-980: CG = 64, or 32 when C is an odd
    multiple of 32; the forward keeps its rows in registers when rows_per_cta <= 8 * RL, bn_unit.cu:984), "unit"
    (bn_unit_plan), or "passes" (the three launches of train.cu) where ssd3d_bn_unit_supported (bn_unit.cu:1034-1040)
    refuses the shape."""
    if c <= 0 or c % 8 or m <= 0:
        return "passes"
    if m <= 8 * 4 * 256:
        return "cluster"
    cv = c // 8
    if cv < 4 or cv > 512 or cv & (cv - 1):
        return "passes"
    if c % 32 == 0:
        cg = 64 if c % 64 == 0 else 32
        ng = c // cg
        if ng <= sms and ng <= 256:
            rl = 512 // (cg // 8)
            rc = max(1, min(sms // ng, -(-m // (rl * 4))))
            rpc = -(-m // rc)
            return "tile%d-%s" % (cg, "keep" if rpc <= 8 * rl else "stream")
    return "unit"


def dw_wgrad_kernel(c: int, n: int, size, stride: int):
    """The depthwise weight-gradient kernel ``ops.dwconv3d_wgrad`` runs: ("tma",) for the halo-tile kernel
    (csrc/conv_dw_tma.cu:572: C % 32 == 0, Wo >= 8, Ho >= 4, Do >= 4), else ("simt", voxels per lane, blocks,
    capped) for the CUDA-core kernel (dw_wgrad_plan, csrc/train.cu:1638-1652: Mo / (G * 222) voxels per lane
    clamped to [2, 8], at most 592 blocks)."""
    do, ho, wo = ((s - 1) // stride + 1 for s in size)
    if c % 32 == 0 and wo >= 8 and ho >= 4 and do >= 4:
        return ("tma",)
    mo = n * do * ho * wo
    g = 256 // (c // 8 * 3)
    vpl = min(8, max(2, mo // (g * 222)))
    blocks = -(-mo // (g * vpl))
    return ("simt", vpl, min(blocks, 592), blocks > 592)


def stem_kernel(dtype, cin: int, w: int) -> str:
    """The stem forward ``ops.stem_conv_bn_relu(kernel=None)`` runs (stem_tz_wanted and ssd3d_stem_conv_affine,
    csrc/conv_stem_tc.cu:740-770): the banded-B "tz" kernel for bf16 volumes with Cin <= 2 and W % 64 == 0, the
    gather "tc" kernel when TMA can address the rows, the CUDA-core "simt" kernel otherwise."""
    bf16 = dtype == torch.bfloat16
    if bf16 and 1 <= cin <= 2 and w % 64 == 0:
        return "tz"
    if 1 <= cin <= 4 and (w * (2 if bf16 else 4)) % 16 == 0:
        return "tc"
    return "simt"


STEM_WGRAD_TILE_ROWS = 128 * 148     # csrc/train.cu:1507,1530 and ops.stem_unit_backward: the TMA tile kernel from here


def head_kw_columns(c: int, n: int, size) -> int:
    """Output columns per CTA of the kw-GEMM head kernel (ssd3d_head_conv_kw, csrc/conv_head_kw.cu:260-274): 144
    when the map has at least 148 tiles of 128 voxels, 48 (three column tiles) below."""
    def p2ceil(v):
        r = 1
        while r < v:
            r <<= 1
        return r
    d, h, w = size
    tw, th = min(p2ceil(w), 8), min(p2ceil(h), 4)
    td = min(p2ceil(d), 128 // (tw * th))
    tn = 128 // (tw * th * td)
    m_tiles = -(-w // tw) * -(-h // th) * -(-d // td) * -(-n // tn)
    return 144 if m_tiles >= 148 else 48


# ---------------------------------------------------------------------------------------------------------------
# Boundary cases, one on each side of every switch
# ---------------------------------------------------------------------------------------------------------------
BN_BOUNDARY = [
    # (n, c, size): cluster up to 8192 rows, tile kernel from 8193 (8193 = 3 * 2731)
    (2, 32, (16, 16, 16)), (1, 32, (3, 1, 2731)), (2, 128, (16, 16, 16)), (1, 128, (3, 1, 2731)),
    # tile kernel, forward rows kept in registers up to rows_per_cta = 8 * RL, streamed above:
    # C = 32 (CG = 32, RL = 128): 148 * 1024 rows and one more (151553 is prime)
    (1, 32, (37, 64, 64)), (1, 32, (1, 1, 151553)),
    # C = 64 (CG = 64, RL = 64): 148 * 512 rows and one more
    (1, 64, (37, 32, 64)), (1, 64, (39, 29, 67)),
]
# C = 96 is an odd multiple of 32 with three 32-channel groups, but ssd3d_bn_unit_supported takes channel counts whose
# C / 8 is a power of two only: above 8192 rows it runs the three-launch passes (checked against torch, not against them)
BN_BOUNDARY_PASSES = [(1, 96, (20, 20, 24))]

DW_BOUNDARY = [
    # (c, n, size, stride): halo-tile vs CUDA-core weight gradient at Wo = 8 / 7 and at Do = 4 / 3
    (32, 2, (16, 16, 16), 2), (32, 2, (16, 16, 14), 2), (64, 1, (4, 8, 16), 1), (64, 1, (3, 8, 16), 1),
    # CUDA-core kernel: 2 voxels per lane (clamped up), 8 (clamped down), 8 with the 592-block cap
    (128, 1, (5, 6, 7), 1), (128, 4, (24, 24, 7), 1), (128, 2, (40, 48, 7), 1),
]

# (cin, n, size, sd, dtype): stem weight gradient below / at M = 128 * 148 output voxels.  18943 = 19 * 997 has no
# factorisation with rows the TMA tile kernel can address (W * element size a multiple of 16 bytes), so the fp32 case
# below sits at 18942 and the bf16 one at 18940, the largest such counts.
STEM_WGRAD_BOUNDARY = [
    (1, 1, (21, 82, 44), 1, torch.float32), (1, 1, (37, 32, 64), 1, torch.float32),
    (1, 1, (1, 1894, 40), 1, torch.bfloat16), (1, 1, (37, 32, 64), 1, torch.bfloat16),
]

# (cin, size, sd, dtype, batch): bf16, Cin <= 2, W = 64k runs the banded-B kernel, W = 64k +- 16 the gather kernel
STEM_FWD_BOUNDARY = [
    (2, (16, 24, 128), 2, torch.bfloat16, 2), (2, (16, 24, 112), 2, torch.bfloat16, 2),
    (2, (16, 24, 144), 2, torch.bfloat16, 2), (1, (12, 20, 64), 1, torch.bfloat16, 3),
    (1, (12, 20, 48), 1, torch.bfloat16, 3), (1, (12, 20, 80), 1, torch.bfloat16, 3),
]

# (c, size, batch, n_classes): kw head at 147 and 148 tiles of 128 voxels (3 x 7 x 7 and 1 x 37 x 4)
HEAD_KW_BOUNDARY = [(128, (28, 28, 8), 3, 2), (128, (16, 145, 8), 1, 2)]


def extend(cases, *more):
    """``cases`` followed by every case of ``more`` not already in it: existing parametrisations keep their ids."""
    out = list(cases)
    for group in more:
        out += [c for c in group if c not in out]
    return out
