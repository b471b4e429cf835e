"""numpy restatement of the training-batch sampling and augmentation (mslesions3d_b200/csrc/augment.cu) --
TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``draws`` restates the Philox draws of every slot (through ``philox_oracle.philox4x32_10`` / ``randint_ms``) and
``apply`` the crop -> ``np.rot90`` -> ``np.flip`` -> intensity steps with numpy's own array functions, in fp32
with a final bf16 round to nearest.  ``signed_permutation`` / ``gather`` state the same geometry as the kernel
evaluates it (one signed axis permutation plus an offset); the CPU tests check the two statements agree.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.philox_oracle import philox4x32_10, randint_ms

F32 = np.float32


def u01(u) -> np.float32:
    return F32(int(u) >> 8) * F32(2.0 ** -24)


def _signed_unit(u, scale) -> np.float32:
    return F32(scale) * (F32(2.0) * u01(u) - F32(1.0))


def draws(seed, counter, step, rank, world, n, order, boxes, box_offsets, src_shape, out_shape, pos_ratio=0.0,
          flip_prob=0.0, rot90_prob=0.0, scale=0.0, shift=0.0):
    """-> (n, 16) int32 record of slot draws (layout of ssd3d_augment_batch).  ``boxes`` (B, 6) int voxel boxes
    [lo d, lo h, lo w, hi d, hi h, hi w] inclusive, ``box_offsets`` (S + 1)."""
    order = np.asarray(order)
    s = len(order)
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    c_lo, c_hi = int(counter) & 0xFFFFFFFF, (int(counter) >> 32) & 0xFFFFFFFF
    rec = np.zeros((n, 16), dtype=np.int32)
    for b in range(n):
        g = rank * n + b
        subj = int(order[(step * n * world + g) % s])
        r = [[int(v) for v in philox4x32_10(g, c_lo, c_hi, i, k0, k1)] for i in range(4)]
        b0, nb = int(box_offsets[subj]), int(box_offsets[subj + 1]) - int(box_offsets[subj])
        pos = nb > 0 and u01(r[0][0]) < F32(pos_ratio)
        box = randint_ms(r[0][1], 0, nb) if pos else -1
        rec[b, 0] = subj
        for ax in range(3):
            lo, hi = 0, src_shape[ax] - out_shape[ax]
            if pos:
                bl, bh = int(boxes[b0 + box][ax]), int(boxes[b0 + box][3 + ax])
                if bh - bl + 1 <= out_shape[ax]:
                    lo, hi = max(0, bh - out_shape[ax] + 1), min(bl, src_shape[ax] - out_shape[ax])
                else:
                    c = (bl + bh) // 2
                    lo, hi = max(0, c - out_shape[ax] + 1), min(c, src_shape[ax] - out_shape[ax])
            rec[b, 1 + ax] = randint_ms(r[1][ax], lo, hi + 1)
            rec[b, 5 + ax] = int(u01(r[2][ax]) < F32(flip_prob))
        rec[b, 4] = randint_ms(r[0][3], 1, 4) if u01(r[0][2]) < F32(rot90_prob) else 0
        rec[b, 8], rec[b, 9] = int(pos), box
        rec[b, 10] = np.array([_signed_unit(r[3][0], scale)], dtype=np.float32).view(np.int32)[0]
        rec[b, 11] = np.array([_signed_unit(r[3][1], shift)], dtype=np.float32).view(np.int32)[0]
        rec[b, 12], rec[b, 13], rec[b, 14], rec[b, 15] = step, np.uint32(c_lo).view(np.int32), g, nb
    return rec


def scale_shift(rec_row):
    return rec_row[10:12].astype(np.int32).view(np.float32)


def crop_rot_flip(vol, rec_row, out_shape, rot_axes=(0, 1)):
    """Geometry of one slot on the spatial axes of ``vol`` (..., Ds, Hs, Ws) with numpy's own functions."""
    lead = vol.ndim - 3
    o = [int(v) for v in rec_row[1:4]]
    x = vol[(Ellipsis, slice(o[0], o[0] + out_shape[0]), slice(o[1], o[1] + out_shape[1]),
             slice(o[2], o[2] + out_shape[2]))]
    if rec_row[4]:
        x = np.rot90(x, int(rec_row[4]), axes=(lead + rot_axes[0], lead + rot_axes[1]))
    for ax in range(3):
        if rec_row[5 + ax]:
            x = np.flip(x, lead + ax)
    return np.ascontiguousarray(x)


def intensity_bf16(x, rec_row):
    """y = bf16_rn((x * (1 + f)) + o) with two fp32 roundings -> torch bf16 tensor."""
    f, o = scale_shift(rec_row)
    y = (np.asarray(x, dtype=np.float32) * (F32(1.0) + F32(f))).astype(np.float32) + F32(o)
    return torch.from_numpy(y.astype(np.float32)).to(torch.bfloat16)


def apply(image, mask, rec_row, out_shape, rot_axes=(0, 1)):
    """image (C, Ds, Hs, Ws) fp32 values (a bf16 source as its fp32 values), mask (Ds, Hs, Ws) -> (bf16 image
    tensor, uint8 mask tensor)."""
    img = crop_rot_flip(np.asarray(image, dtype=np.float32), rec_row, out_shape, rot_axes)
    m = crop_rot_flip(np.asarray(mask), rec_row, out_shape, rot_axes)
    return intensity_bf16(img, rec_row), torch.from_numpy(m)


def signed_permutation(rec_row, rot_axes=(0, 1)):
    """(q, rev): crop axis c reads output axis q[c], reversed when rev[c] -- the kernel's statement of the geometry."""
    q, rev = [0, 1, 2], [0, 0, 0]
    k, (a0, a1) = int(rec_row[4]), rot_axes
    if k == 1:
        q[a0], q[a1], rev[a1] = a1, a0, 1
    elif k == 2:
        rev[a0] = rev[a1] = 1
    elif k == 3:
        q[a0], q[a1], rev[a0] = a1, a0, 1
    return q, [rev[c] ^ int(rec_row[5 + q[c]]) for c in range(3)]


def gather(vol, rec_row, out_shape, rot_axes=(0, 1)):
    """The geometry as an index gather: out[o] = vol[off + (rev ? n - 1 - o[q] : o[q])] per source axis."""
    q, rev = signed_permutation(rec_row, rot_axes)
    grids = np.meshgrid(*[np.arange(n) for n in out_shape], indexing="ij")
    idx = []
    for c in range(3):
        oq = grids[q[c]]
        idx.append(int(rec_row[1 + c]) + (out_shape[q[c]] - 1 - oq if rev[c] else oq))
    return vol[(Ellipsis, idx[0], idx[1], idx[2])]


def epoch_subjects(order, n, world, steps):
    """(world, steps, n) subjects every rank's slots take over one epoch."""
    order = np.asarray(order)
    s = len(order)
    return np.array([[[order[(t * n * world + r * n + b) % s] for b in range(n)] for t in range(steps)]
                     for r in range(world)])
