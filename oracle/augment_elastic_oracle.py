"""numpy restatement of the elastic deformation (ssd3d_augment_elastic_batch, mslesions3d_b200/csrc/augment.cu) --
TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``elastic_draws`` restates record word 32 (Philox call 6), ``control_points`` the displacements of every control
point (Philox call 7 + k), ``bspline`` the per-axis interval and weights, ``elastic_field`` the 64-term sum in the
header's fp32 order (R innermost, then K, then L: the crop axes output h, d and w read), and ``elastic_apply`` the
deformed coordinates followed by the trilinear / nearest resampling and intensity step of
``augment_affine_oracle.affine_apply``, in numpy float32 with every operation rounded separately.  The draws, the
signed permutation, the recorded matrix, the taps and the intensity step come from ``oracle/augment_oracle.py``,
``oracle/augment_affine_oracle.py`` and ``oracle/philox_oracle.py`` unchanged.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle.augment_affine_oracle import _taps, recorded_matrix
from oracle.augment_oracle import F32, intensity_bf16, signed_permutation, u01
from oracle.philox_oracle import philox4x32_10

SIXTH, TWO_THIRDS = F32(1) / F32(6), F32(2) / F32(3)


def elastic_draws(seed, counter, rank, n, elastic_prob=0.0):
    """-> (n,) int32: record word 32 of ssd3d_augment_elastic_batch (field drawn) from Philox call 6 of every slot."""
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    c_lo, c_hi = int(counter) & 0xFFFFFFFF, (int(counter) >> 32) & 0xFFFFFFFF
    return np.array([int(u01(int(philox4x32_10(rank * n + b, c_lo, c_hi, 6, k0, k1)[0])) < F32(elastic_prob))
                     for b in range(n)], dtype=np.int32)


def control_points(seed, counter, slot, points, magnitude):
    """(G_d, G_h, G_w, 3) float32 displacements of global slot ``slot``: point k = (k_d G_h + k_h) G_w + k_w takes
    Philox call 7 + k, component c = fp32(m_c * fp32(fp32(2 u01(word c)) - 1))."""
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    c_lo, c_hi = int(counter) & 0xFFFFFFFF, (int(counter) >> 32) & 0xFFFFFFFF
    n = int(np.prod(points))
    words = philox4x32_10(slot, c_lo, c_hi, 7 + np.arange(n, dtype=np.uint64), k0, k1)
    out = np.empty((n, 3), dtype=np.float32)
    for c in range(3):
        u = (np.asarray(words[c]) >> np.uint64(8)).astype(np.float32) * F32(2.0 ** -24)
        out[:, c] = F32(magnitude[c]) * (F32(2) * u - F32(1))
    return out.reshape(*points, 3)


def inverse_spacing(n, g):
    """r = fp32((G - 3) / (n - 1)), 0 for a single-voxel axis."""
    return F32(g - 3) / F32(n - 1) if n > 1 else F32(0)


def _h(x):
    return ((x * x) * x) * SIXTH


def _c(x):
    x2 = x * x
    return (F32(0.5) * (x2 * x) - x2) + TWO_THIRDS


def bspline(p, r, g):
    """Crop indices p (int array) -> (j int64 array, [B0, B1, B2, B3] float32 arrays): t = fp32(p r),
    j = min(floor(t), G - 4), f = t - j, weights {h(1 - f), c(f), c(1 - f), h(f)}."""
    t = np.asarray(p).astype(np.float32) * F32(r)
    j = np.minimum(np.floor(t).astype(np.int64), g - 4)
    f = (t - j.astype(np.float32)).astype(np.float32)
    gm = F32(1) - f
    return j, [_h(gm), _c(f), _c(gm), _h(f)]


def crop_indices(rec_row, out_shape, rot_axes=(0, 1)):
    """(p (3, d, h, w) int64 crop index of every output voxel, q): the signed permutation of the record."""
    q, rev = signed_permutation(rec_row, rot_axes)
    grids = np.meshgrid(*[np.arange(n) for n in out_shape], indexing="ij")
    p = [out_shape[c] - 1 - grids[q[c]] if rev[c] else grids[q[c]] for c in range(3)]
    return np.stack(p), q


def elastic_field(P, p, q, out_shape):
    """delta (3, ...) float32 at crop indices p (3, ...) for control points P (G_d, G_h, G_w, 3), in the header's
    order: crop axes K, R, L = those output d, h, w read (q[c] = 0, 1, 2); V = sum_b B_b(R) P, T = sum_a B_a(K) V,
    delta = sum_e B_e(L) T, each sum from +0 in index order, every product rounded."""
    g = P.shape[:3]
    cK, cR, cL = (q.index(o) for o in range(3))
    j, w = {}, {}
    for c in range(3):
        j[c], w[c] = bspline(p[c], inverse_spacing(out_shape[c], g[c]), g[c])
    delta = np.zeros((3,) + p.shape[1:], dtype=np.float32)
    for e in range(4):
        T = np.zeros_like(delta)
        for a in range(4):
            V = np.zeros_like(delta)
            for b in range(4):
                k = [None] * 3
                k[cK], k[cR], k[cL] = j[cK] + a, j[cR] + b, j[cL] + e
                V = V + w[cR][b] * np.moveaxis(P[k[0], k[1], k[2]], -1, 0)
            T = T + w[cK][a] * V
        delta = delta + w[cL][e] * T
    return delta


def elastic_coords(rec_row, out_shape, M, P, rot_axes=(0, 1)):
    """Source coordinates (3, d, h, w): u_c = p_c - (n_c - 1) / 2, u' = fp32(u + delta) (delta = 0 without P),
    x_a = ((M[a][0] u'_0 + M[a][1] u'_1) + M[a][2] u'_2) + (o_a + (n_a - 1) / 2), in float32."""
    p, q = crop_indices(rec_row, out_shape, rot_axes)
    half = [F32((n - 1) / 2) for n in out_shape]
    u = np.stack([p[c].astype(np.float32) - half[c] for c in range(3)])
    if P is not None:
        u = u + elastic_field(P, p, q, out_shape)
    M = np.asarray(M, dtype=np.float32)
    return np.stack([((M[a, 0] * u[0] + M[a, 1] * u[1]) + M[a, 2] * u[2]) + (F32(int(rec_row[1 + a])) + half[a])
                     for a in range(3)])


def resample(image, mask, x, rec_row):
    """The resampling of ``augment_affine_oracle.affine_apply`` at coordinates x: trilinear (lerp along W, then H,
    then D) and nearest floor(x + 0.5), zeros outside the source, then ``intensity_bf16``."""
    image = np.asarray(image, dtype=np.float32)
    fl = np.floor(x)
    i0, t = fl.astype(np.int64), (x - fl).astype(np.float32)
    omt = F32(1.0) - t

    def lerp(v0, v1, a):
        return v0 * omt[a] + v1 * t[a]

    c = {}
    for dd in (0, 1):
        for dh in (0, 1):
            c[dd, dh] = lerp(_taps(image, (i0[0] + dd, i0[1] + dh, i0[2])),
                             _taps(image, (i0[0] + dd, i0[1] + dh, i0[2] + 1)), 2)
    val = lerp(lerp(c[0, 0], c[0, 1], 1), lerp(c[1, 0], c[1, 1], 1), 0)
    nn = np.floor(x + F32(0.5)).astype(np.int64)
    m = _taps(np.asarray(mask), (nn[0], nn[1], nn[2]))
    return intensity_bf16(val, rec_row), torch.from_numpy(np.ascontiguousarray(m))


def elastic_apply(image, mask, rec_row, out_shape, P, rot_axes=(0, 1)):
    """ssd3d_augment_elastic_batch for one slot from its record row (the recorded M) and its control points P
    (``control_points``; used only when record word 32 is set): image (C, Ds, Hs, Ws) fp32 values, mask
    (Ds, Hs, Ws) -> (bf16 image tensor, uint8 mask tensor)."""
    x = elastic_coords(rec_row, out_shape, recorded_matrix(rec_row), P if int(rec_row[32]) else None, rot_axes)
    return resample(image, mask, x, rec_row)
