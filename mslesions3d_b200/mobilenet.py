"""3-D MobileNet building blocks with the reference's names and constructor signatures
(``lesions3d/mobilenet.py:13-49``), executing on the sm_100a kernels.

``conv_bn`` and ``Block`` hold ordinary ``nn.Conv3d`` / ``nn.BatchNorm3d`` children, so parameter names,
shapes, default initialisation and ``state_dict`` keys are the reference's (``0.weight``, ``1.running_mean``,
``conv1.weight``, ``bn2.bias`` ...) and its checkpoints load unchanged.  Those children are containers
only: ``forward`` packs their tensors once (bf16, channels-last, BN folded to scale/shift) and launches
the CUDA kernels; activations travel between modules as logical (N,C,D,H,W) tensors stored
channels-last-3d in bf16.

In ``eval()`` mode BatchNorm is folded into the conv epilogues.  In training mode (the reference's modules work
stand-alone there too, mobilenet.py:34-49) each module is one autograd node over the train-mode kernels
(``train_modules.py``: batch-statistic BatchNorm, running-statistic update, hand-written backward); inside
``LSSD3D`` the fused ``training.TrainEngine`` drives the same kernels for the whole network at once.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops

# mobilenet.py:13-24
config_mobilenet = [32,
                    # channel, n, stride
                    [64, 1, (2, 2, 2)],
                    [128, 2, (2, 2, 2)],
                    [256, 2, (2, 2, 2)],
                    [512, 6, (2, 2, 2)],
                    [1024, 2, (1, 1, 1)],
                    ]

MOBILENET_CONFIGS = {
    "mobilenet": config_mobilenet
}


def _versions(*tensors):
    return tuple((t.data_ptr(), t._version) for t in tensors if t is not None)


def _bn_tensors(bn):
    return (bn.weight, bn.bias, bn.running_mean, bn.running_var)


def _stride3(stride):
    if isinstance(stride, int):
        return (stride, stride, stride)
    return tuple(int(s) for s in stride)


class ConvBN(nn.Sequential):
    """``conv_bn``: dense 3x3x3 conv (no bias) + BN + ReLU -- the network stem (mobilenet.py:26-31)."""

    def __init__(self, inp, oup, stride):
        super().__init__(
            nn.Conv3d(inp, oup, kernel_size=3, stride=stride, padding=(1, 1, 1), bias=False),
            nn.BatchNorm3d(oup),
            nn.ReLU(inplace=True),
        )
        self._packed = None
        self._packed_key = None

    def _pack(self):
        conv, bn = self[0], self[1]
        key = _versions(conv.weight, *_bn_tensors(bn))
        if self._packed is None or key != self._packed_key:
            scale, shift = ops.fold_bn(bn)
            self._packed = (ops.pack_stem_weight(conv.weight), scale, shift)
            self._packed_key = key
        return self._packed

    def forward(self, x, out=None):
        conv = self[0]
        sd, sh, sw = _stride3(conv.stride)
        if conv.out_channels != 32 or (sh, sw) != (2, 2) or sd not in (1, 2):
            raise NotImplementedError("stem kernel is built for Cout=32 and stride (1|2, 2, 2), as ssd3d.py:60-61 uses it")
        if self.training:
            from .train_modules import conv_bn_train
            return conv_bn_train(self, x)
        w, scale, shift = self._pack()
        return ops.stem_conv_bn_relu(x, w, scale, shift, sd, out=out)


def conv_bn(inp, oup, stride):
    return ConvBN(inp, oup, stride)


class Block(nn.Module):
    '''Depthwise conv + Pointwise conv (mobilenet.py:34-49)'''

    def __init__(self, in_planes, out_planes, stride=1):
        super(Block, self).__init__()
        self.conv1 = nn.Conv3d(in_planes, in_planes, kernel_size=3, stride=stride, padding=1, groups=in_planes,
                               bias=False)
        self.bn1 = nn.BatchNorm3d(in_planes)
        self.conv2 = nn.Conv3d(in_planes, out_planes, kernel_size=1, stride=1, padding=0, bias=False)
        self.bn2 = nn.BatchNorm3d(out_planes)
        self._packed = None
        self._packed_key = None
        self.nan_flag = None   # device int32 shared by the owning network (set by MobileNetBase)

    def _pack(self):
        key = _versions(self.conv1.weight, self.conv2.weight, *_bn_tensors(self.bn1), *_bn_tensors(self.bn2))
        if self._packed is None or key != self._packed_key:
            s1, b1 = ops.fold_bn(self.bn1)
            s2, b2 = ops.fold_bn(self.bn2)
            self._packed = (ops.pack_dw_weight(self.conv1.weight), s1, b1, ops.pack_pw_weight(self.conv2.weight), s2, b2)
            self._packed_key = key
        return self._packed

    def forward(self, x, fuse: bool = True):
        """``fuse``: run the shapes the fused depthwise -> pointwise kernel (csrc/conv_dwpw.cu) is built for as that one
        kernel.  Measured on B200 at the benchmark size (profiles/r02_block_fused.md): alone, every fused block beats
        its two kernels (f1 41 vs 47, f2 16.5 vs 20.6, f3 18.8 vs 22.8 us) and f1 keeps 33.6 MB per step out of HBM,
        so eager calls and the lone ``predict_step`` (latency) fuse.  In the 6-deep ``predict_batches`` pipeline
        (throughput) the fused CTAs own their SM (200 KB of shared memory) while the stand-alone pointwise GEMMs they
        replace run underneath other batches' kernels: there the plans pass False."""
        s = _stride3(self.conv1.stride)
        if s[0] != s[1] or s[1] != s[2] or s[0] not in (1, 2):
            raise NotImplementedError("depthwise kernel is built for isotropic stride 1 or 2 (mobilenet.py:13-20)")
        if self.training:
            from .train_modules import block_train
            return block_train(self, x)
        wd, s1, b1, wp, s2, b2 = self._pack()
        own_flag = self.nan_flag is None
        flag = torch.zeros((1,), dtype=torch.int32, device=x.device) if own_flag else self.nan_flag
        if fuse and x.is_cuda and x.dim() == 5 and ops.block_fused_supported(x, wp.shape[0], s[0]):
            # the three large blocks: depthwise tile -> shared memory -> tcgen05 pointwise GEMM, one kernel
            out = ops.block_dwpw_bn_relu(x, wd, s1, b1, wp, s2, b2, s[0], flag)
        else:
            out = ops.dwconv3d_bn_relu(x, wd, s1, b1, s[0])
            out = ops.pwconv_bn_relu(out, wp, s2, b2, flag)
        if own_flag and int(flag.item()) != 0:   # stand-alone use keeps the reference's check (mobilenet.py:46-48)
            raise Exception("NaN Loss in MobileNet Block")
        return out
