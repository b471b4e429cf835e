"""Training data that lives in HBM: ``DeviceDataset`` (normalised volumes, label masks and every subject's lesion
boxes, prepared once at load), ``Augment`` (the augmentation drawn per slot inside the captured training step,
csrc/augment.cu) and ``epoch_order`` (the per-epoch permutation).  ``LSSD3D.fit_epoch`` trains on them with one
CUDA-graph replay per step: sampling, augmentation, ground-truth extraction and packing, then the fused step.

The reference prepares its batches with MONAI transform pipelines on CPU workers (datasets.py): a host pipeline
cannot augment at the rate the fused step consumes volumes.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops


@dataclasses.dataclass(frozen=True)
class Augment:
    """Per-volume augmentation, applied in this order (exact semantics: ``ssd3d_augment_batch`` in the header):

    * crop to the model's ``input_size``: with probability ``pos_ratio`` (and only if the subject has a lesion)
      around one of its lesions, otherwise anywhere;
    * ``np.rot90(x, k, axes=rot90_axes)``, k uniform in {1, 2, 3}, with probability ``rot90_prob``;
    * ``np.flip`` of each spatial axis with probability ``flip_prob``;
    * ``x * (1 + f) + o`` with ``f ~ U(-scale, scale)``, ``o ~ U(-shift, shift)`` per volume (shared by its channels).

    ``Augment()`` on a data set of ``input_size`` volumes is the identity (up to the bf16 rounding of the input)."""
    pos_ratio: float = 0.0
    flip_prob: float = 0.0
    rot90_prob: float = 0.0
    rot90_axes: Tuple[int, int] = (0, 1)
    scale: float = 0.0
    shift: float = 0.0
    seed: int = 0

    def validate(self, input_size: Sequence[int], source_size: Sequence[int]) -> None:
        """Raise ValueError unless this augmentation can turn ``source_size`` volumes into ``input_size`` ones."""
        out, src = tuple(int(v) for v in input_size), tuple(int(v) for v in source_size)
        for name in ("pos_ratio", "flip_prob", "rot90_prob"):
            p = getattr(self, name)
            if not 0.0 <= p <= 1.0:
                raise ValueError("%s=%r is not a probability in [0, 1]" % (name, p))
        if self.scale < 0 or self.shift < 0:
            raise ValueError("scale and shift are half-widths and must be >= 0")
        if len(out) != 3 or len(src) != 3 or any(s < o for s, o in zip(src, out)):
            raise ValueError("source volumes %r are smaller than the model's input_size %r" % (src, out))
        a0, a1 = (int(v) for v in self.rot90_axes)
        if len(self.rot90_axes) != 2 or a0 == a1 or not (0 <= a0 <= 2 and 0 <= a1 <= 2):
            raise ValueError("rot90_axes must be two different spatial axes in 0..2, got %r" % (self.rot90_axes,))
        if self.rot90_prob > 0 and out[a0] != out[a1]:
            raise ValueError("rot90 over axes %r needs equal input_size extents, got %d and %d"
                             % (self.rot90_axes, out[a0], out[a1]))
        if out[2] % 16:
            raise ValueError("the last input_size extent must be a multiple of 16, got %d" % out[2])


def epoch_order(n_subjects: int, epoch: int, seed: int = 0) -> torch.Tensor:
    """The subject permutation of one epoch (int32, host): ``torch.randperm`` with a generator seeded from
    (seed, epoch), as DistributedSampler shuffles.  Every rank computes the same one and takes its slots of it."""
    g = torch.Generator()
    g.manual_seed((int(seed) * 1000003 + int(epoch)) & 0x7FFFFFFFFFFFFFFF)
    return torch.randperm(int(n_subjects), generator=g).to(torch.int32)


class DeviceDataset:
    """Normalised volumes (S, C, D, H, W) fp32 or bf16 and label masks (S, D, H, W) uint8 on one CUDA device, with
    the lesion boxes of every subject in voxel indices: ``boxes`` (B, 6) int32 [lo d, lo h, lo w, hi d, hi h, hi w]
    (inclusive), subject s owning rows ``box_offsets[s]:box_offsets[s + 1]``.  ``n_classes`` = 0: binary masks
    (every non-zero voxel is lesion, label 1); otherwise masks hold classes 1..n_classes."""

    def __init__(self, images: torch.Tensor, masks: torch.Tensor, boxes: torch.Tensor, box_offsets: torch.Tensor,
                 n_classes: int = 0):
        self.images, self.masks, self.boxes, self.box_offsets = images, masks, boxes, box_offsets
        self.n_classes = int(n_classes)

    def __len__(self) -> int:
        return int(self.images.shape[0])

    @property
    def shape(self) -> Tuple[int, int, int]:
        """Spatial shape (D, H, W) of every volume."""
        return tuple(int(v) for v in self.images.shape[2:])

    @property
    def channels(self) -> int:
        return int(self.images.shape[1])

    @classmethod
    def from_arrays(cls, images, masks, n_classes: int = 0, dtype: torch.dtype = torch.float32, device=None,
                    chunk: int = 64) -> "DeviceDataset":
        """images: raw intensities, a (S, C, D, H, W) array or a sequence of (C, D, H, W) arrays; masks: (S, D, H, W)
        (or (S, 1, D, H, W)) or a sequence of (D, H, W).  All volumes must have one shape.  Normalises on the
        device (MONAI NormalizeIntensity(nonzero=True), datasets.py:403) into ``dtype`` and extracts every
        subject's lesion boxes once (BoundingBoxesGeneratord, utils.py:438-513)."""
        if dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("dtype must be torch.float32 or torch.bfloat16")
        imgs, msks = _stack(images, 4, "images"), _stack(masks, 3, "masks")
        if msks.dim() == 5 and msks.shape[1] == 1:
            msks = msks[:, 0]
        if imgs.dim() != 5 or msks.dim() != 4:
            raise ValueError("expected images (S, C, D, H, W) and masks (S, D, H, W)")
        if imgs.shape[0] != msks.shape[0] or tuple(imgs.shape[2:]) != tuple(msks.shape[1:]):
            raise ValueError("images %r and masks %r do not match" % (tuple(imgs.shape), tuple(msks.shape)))
        if imgs.shape[0] == 0:
            raise ValueError("empty data set")
        if msks.is_floating_point() and not bool((msks == msks.round()).all()):
            raise ValueError("masks must hold integer labels")
        if int(msks.min()) < 0 or int(msks.max()) > 255:
            raise ValueError("mask labels must fit uint8")
        s = int(imgs.shape[0])
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        out = torch.empty(tuple(imgs.shape), dtype=dtype, device=dev)
        mask_dev = torch.empty(tuple(msks.shape), dtype=torch.uint8, device=dev)
        boxes, offsets = [], [0]
        dims = torch.tensor(list(imgs.shape[2:]) * 2, dtype=torch.float64)
        for i in range(0, s, chunk):
            out[i:i + chunk] = ops.normalize_intensity_nonzero(imgs[i:i + chunk].to(dev, torch.float32), dtype)
            mask_dev[i:i + chunk] = msks[i:i + chunk].to(dev).to(torch.uint8)
            bl, _ = ops.gt_boxes_from_segmentation(mask_dev[i:i + chunk], n_classes)
            for b in bl:          # fractional [index / dim] -> voxel index (exact: far below half a voxel off)
                boxes.append(torch.round(b.cpu().double() * dims).to(torch.int32))
                offsets.append(offsets[-1] + int(b.shape[0]))
        table = torch.cat(boxes) if offsets[-1] else torch.zeros((0, 6), dtype=torch.int32)
        if table.shape[0] == 0:
            table = torch.zeros((1, 6), dtype=torch.int32)        # keeps a valid device pointer; no subject owns it
        return cls(out, mask_dev, table.to(dev), torch.tensor(offsets, dtype=torch.int32, device=dev), n_classes)

    @classmethod
    def from_directory(cls, path: str, n_classes: int = 0, dtype: torch.dtype = torch.float32,
                       device=None) -> "DeviceDataset":
        """The generator's layout (``images/sub-XXXX_image.nii.gz`` + ``labels/sub-XXXX_seg.nii.gz``, as
        ``synthetic.write_dataset`` writes and ``synthetic.load_dataset_dir`` reads)."""
        from .nifti import load_nifti
        image_dir, seg_dir = os.path.join(path, "images"), os.path.join(path, "labels")
        names = sorted(f for f in os.listdir(image_dir) if f.endswith("_image.nii.gz") or f.endswith("_image.nii"))
        if not names:
            raise ValueError("no *_image.nii[.gz] volumes under %s" % image_dir)
        images, masks = [], []
        for f in names:
            data, _ = load_nifti(os.path.join(image_dir, f))
            seg, _ = load_nifti(os.path.join(seg_dir, f.replace("_image", "_seg")))
            images.append(np.asarray(data, dtype=np.float32)[None] if data.ndim == 3 else np.asarray(data, np.float32))
            masks.append(np.asarray(seg))
        return cls.from_arrays(images, masks, n_classes, dtype, device)


def _stack(x, item_dim: int, what: str) -> torch.Tensor:
    """An array / tensor, or a sequence of equally shaped per-volume arrays, as one CPU-or-device tensor."""
    if isinstance(x, torch.Tensor):
        return x
    if isinstance(x, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(x))
    items = [torch.as_tensor(np.ascontiguousarray(v)) if not isinstance(v, torch.Tensor) else v for v in x]
    if not items:
        raise ValueError("empty data set")
    shapes = {tuple(v.shape) for v in items}
    if len(shapes) != 1:
        raise ValueError("all %s must have one shape (mixed shapes are not supported), got %s"
                         % (what, sorted(shapes)))
    if len(next(iter(shapes))) != item_dim:
        raise ValueError("each of the %s must be %d-D" % (what, item_dim))
    return torch.stack(items)
