"""numpy restatement of the rotation / zoom augmentation (ssd3d_augment_affine_batch, mslesions3d_b200/csrc/augment.cu)
-- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``affine_draws`` restates record words 16-22 (Philox calls 4 and 5), ``affine_matrix`` the float64 matrix
R0 R1 R2 diag(1 / z) from the recorded theta and z, and ``affine_apply`` the per-voxel geometry, trilinear and
nearest resampling in numpy float32 (every operation rounded separately, in the header's order) from the recorded
fp32 matrix, followed by ``augment_oracle.intensity_bf16``.  The draws, the signed permutation and the intensity
step of ssd3d_augment_batch come from ``oracle/augment_oracle.py`` unchanged.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.augment_oracle import F32, _signed_unit, intensity_bf16, signed_permutation, u01
from oracle.philox_oracle import philox4x32_10


def affine_draws(seed, counter, rank, n, affine_prob=0.0, rotate_range=(0, 0, 0), zoom_range=(0, 0, 0)):
    """-> (n, 7) int32: record words 16-22 of ssd3d_augment_affine_batch (affine drawn, theta (fp32 bits),
    z (fp32 bits)) from Philox calls 4 and 5 of every slot."""
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    c_lo, c_hi = int(counter) & 0xFFFFFFFF, (int(counter) >> 32) & 0xFFFFFFFF
    rec = np.zeros((n, 7), dtype=np.int32)
    for b in range(n):
        g = rank * n + b
        r4 = [int(v) for v in philox4x32_10(g, c_lo, c_hi, 4, k0, k1)]
        r5 = [int(v) for v in philox4x32_10(g, c_lo, c_hi, 5, k0, k1)]
        on = bool(u01(r4[0]) < F32(affine_prob))
        th = [_signed_unit(r4[1 + i], rotate_range[i]) if on else F32(0.0) for i in range(3)]
        z = [F32(1.0) + _signed_unit(r5[i], zoom_range[i]) if on else F32(1.0) for i in range(3)]
        rec[b, 0] = int(on)
        rec[b, 1:7] = np.array(th + z, dtype=np.float32).view(np.int32)
    return rec


def affine_matrix(rec_row):
    """float64 M = R0 R1 R2 diag(1 / z) from the recorded theta and z (words 17-22), axes (d, h, w): R0 rotates in
    the (h, w) plane, R1 in (d, w), R2 in (d, h), each [[c, -s], [s, c]] on its (lower, higher) axis pair."""
    w = np.asarray(rec_row, dtype=np.int32)
    th = w[17:20].view(np.float32).astype(np.float64)
    z = w[20:23].view(np.float32).astype(np.float64)
    rots = []
    for (lo, hi), t in zip(((1, 2), (0, 2), (0, 1)), th):
        r = np.eye(3)
        r[lo, lo] = r[hi, hi] = np.cos(t)
        r[lo, hi], r[hi, lo] = -np.sin(t), np.sin(t)
        rots.append(r)
    return rots[0] @ rots[1] @ rots[2] @ np.diag(1.0 / z)


def recorded_matrix(rec_row):
    """The fp32 M of record words 23-31 (row = source axis, column = crop axis)."""
    return np.asarray(rec_row, dtype=np.int32)[23:32].view(np.float32).reshape(3, 3)


def affine_coords(rec_row, out_shape, M, rot_axes=(0, 1), dtype=np.float32):
    """Source coordinates (3, d, h, w) of every output voxel: the signed permutation to the crop index p, then
    x_a = ((M[a][0] u_0 + M[a][1] u_1) + M[a][2] u_2) + (o_a + (n_a - 1) / 2), u_c = p_c - (n_c - 1) / 2, in
    ``dtype`` with every operation rounded separately (numpy does not contract)."""
    q, rev = signed_permutation(rec_row, rot_axes)
    grids = np.meshgrid(*[np.arange(n) for n in out_shape], indexing="ij")
    M = np.asarray(M, dtype=dtype)
    half = [dtype((n - 1) / 2) for n in out_shape]
    u = []
    for c in range(3):
        oq = grids[q[c]]
        p = out_shape[c] - 1 - oq if rev[c] else oq
        u.append(p.astype(dtype) - half[c])
    x = []
    for a in range(3):
        cen = dtype(int(rec_row[1 + a])) + half[a]
        x.append(((M[a, 0] * u[0] + M[a, 1] * u[1]) + M[a, 2] * u[2]) + cen)
    return np.stack(x)


def _taps(vol, idx):
    """vol[..., i_d, i_h, i_w] with 0 wherever an index lies outside the volume."""
    shape = vol.shape[-3:]
    ok = np.ones(idx[0].shape, dtype=bool)
    clamped = []
    for a in range(3):
        ok &= (idx[a] >= 0) & (idx[a] < shape[a])
        clamped.append(np.clip(idx[a], 0, shape[a] - 1))
    return np.where(ok, vol[(Ellipsis, *clamped)], np.zeros((), dtype=vol.dtype))


def affine_apply(image, mask, rec_row, out_shape, rot_axes=(0, 1)):
    """ssd3d_augment_affine_batch for one slot from its record row (the recorded M): image (C, Ds, Hs, Ws) fp32
    values, mask (Ds, Hs, Ws) -> (bf16 image tensor, uint8 mask tensor).  Trilinear in fp32 (lerp along W, then H,
    then D; v0 * (1 - t) + v1 * t with every operation rounded), nearest floor(x + 0.5) for the mask, zeros outside
    the source, then ``intensity_bf16``."""
    image = np.asarray(image, dtype=np.float32)
    x = affine_coords(rec_row, out_shape, recorded_matrix(rec_row), rot_axes)
    fl = np.floor(x)
    i0, t = fl.astype(np.int64), (x - fl).astype(np.float32)
    omt = F32(1.0) - t

    def lerp(v0, v1, a):
        return v0 * omt[a] + v1 * t[a]

    c = {}
    for dd in (0, 1):
        for dh in (0, 1):
            v0 = _taps(image, (i0[0] + dd, i0[1] + dh, i0[2]))
            v1 = _taps(image, (i0[0] + dd, i0[1] + dh, i0[2] + 1))
            c[dd, dh] = lerp(v0, v1, 2)
    val = lerp(lerp(c[0, 0], c[0, 1], 1), lerp(c[1, 0], c[1, 1], 1), 0)
    nn = np.floor(x + F32(0.5)).astype(np.int64)
    m = _taps(np.asarray(mask), (nn[0], nn[1], nn[2]))
    return intensity_bf16(val, rec_row), torch.from_numpy(np.ascontiguousarray(m))


