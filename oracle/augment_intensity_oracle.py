"""numpy restatement of the MR intensity augmentation (ssd3d_augment_intensity_batch, mslesions3d_b200/csrc/augment.cu)
-- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``slot_draws`` restates the per-slot Philox draws (calls 2^16 + j) with the u01 and fp32 arithmetic of the header,
``record`` the (N, 27) record they and the batch's min / max give, ``normals`` the per-voxel Box-Muller normals
(calls 2^24 + quad) in float64, and ``apply`` the gamma -> bias field -> noise steps in float64 from the input bf16
values and a record row.  The device's expf / exp2f / __log2f / __expf / logf / sincospif are not numpy's, so the
image is compared within a bf16 ulp; the recorded gamma is the only record word computed through a transcendental.
"""
from __future__ import annotations

import numpy as np

from oracle.augment_oracle import F32, u01
from oracle.philox_oracle import MASK32, philox4x32_10

WORDS = 27
CALL_SLOT, CALL_NOISE = 1 << 16, 1 << 24
# the 20 monomials (i, j, k) of u_d^i u_h^j u_w^k, i + j + k <= 3, in the header's order
MONOMIALS = [(i, j, k) for i in range(4) for j in range(4 - i) for k in range(4 - i - j)]


def _key(seed, counter):
    """(k0, k1, c_lo, c_hi) of the draws: the counter the preceding augment launch consumed."""
    return (int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF, int(counter) & 0xFFFFFFFF,
            (int(counter) >> 32) & 0xFFFFFFFF)


def slot_draws(seed, counter, slot, bias_prob=0.0, bias_coefficient=0.0, gamma_prob=0.0, gamma_log_range=0.0,
               noise_prob=0.0, noise_std=0.0):
    """The draws of global slot ``slot`` at draw counter ``counter`` -> dict: flags (gamma, bias, noise), g (the fp32
    log-gamma; 0 without gamma), gamma64 = exp(g) in float64 (1 without gamma), sigma (fp32), coef (20 fp32)."""
    k0, k1, c_lo, c_hi = _key(seed, counter)
    r = [[int(v) for v in philox4x32_10(slot, c_lo, c_hi, CALL_SLOT + j, k0, k1)] for j in range(7)]
    gon = bool(u01(r[0][0]) < F32(gamma_prob))
    bon = bool(u01(r[0][1]) < F32(bias_prob))
    non = bool(u01(r[0][2]) < F32(noise_prob))
    g = F32(gamma_log_range) * (F32(2) * u01(r[0][3]) - F32(1)) if gon else F32(0)
    sigma = F32(noise_std) * u01(r[1][0]) if non else F32(0)
    coef = np.array([F32(bias_coefficient) * (F32(2) * u01(r[2 + m // 4][m % 4]) - F32(1)) if bon else F32(0)
                     for m in range(20)], dtype=np.float32)
    return {"flags": (gon, bon, non), "g": F32(g), "gamma64": float(np.exp(np.float64(g))) if gon else 1.0,
            "sigma": F32(sigma), "coef": coef}


def _bits(v):
    return int(np.array([v], dtype=np.float32).view(np.int32)[0])


def record(images, seed, counter, rank, **kw):
    """(N, 27) int32 record of a batch ``images`` (N, C, d, h, w) (the bf16 input, as float32 / float64 values):
    gamma is fp32(exp(g)) of float64 exp (the device's expf is within 2 fp32 ulps of it), lo / hi the slot's min /
    max when gamma is drawn."""
    images = np.asarray(images)
    n = images.shape[0]
    rec = np.zeros((n, WORDS), dtype=np.int32)
    for b in range(n):
        s = slot_draws(seed, counter, rank * n + b, **kw)
        gon, bon, non = s["flags"]
        rec[b, :3] = (int(gon), int(bon), int(non))
        rec[b, 3] = _bits(np.float32(s["gamma64"]))
        if gon:
            rec[b, 4], rec[b, 5] = _bits(images[b].min()), _bits(images[b].max())
        rec[b, 6] = _bits(s["sigma"])
        rec[b, 7:] = s["coef"].view(np.int32)
    return rec


def unpack(rec_row):
    """A record row -> (flags, gamma, lo, hi, sigma, coef) with the fp32 words as float64."""
    rec_row = np.asarray(rec_row, dtype=np.int32)
    f = rec_row.view(np.float32).astype(np.float64)
    return (bool(rec_row[0]), bool(rec_row[1]), bool(rec_row[2])), f[3], f[4], f[5], f[6], f[7:]


def normals(seed, counter, slot, shape):
    """The standard normals (C, d, h, w) float64 of global slot ``slot``: voxel i (C-order index in the slot) of quad
    q = i // 4 takes Philox call 2^24 + q; Box-Muller on words (0, 1) gives voxels 4q, 4q + 1 and on words (2, 3)
    4q + 2, 4q + 3, with u1 = ((word >> 8) + 1) 2^-24 and u2 = (word >> 8) 2^-24."""
    k0, k1, c_lo, c_hi = _key(seed, counter)
    n = int(np.prod(shape))
    q = np.arange(n // 4, dtype=np.uint64)
    w = philox4x32_10(slot, c_lo, c_hi, (np.uint64(CALL_NOISE) + q) & MASK32, k0, k1)
    out = np.empty((n // 4, 4), dtype=np.float64)
    for p in range(2):
        u1 = ((np.asarray(w[2 * p]) >> np.uint64(8)) + np.uint64(1)).astype(np.float64) * 2.0 ** -24
        u2 = (np.asarray(w[2 * p + 1]) >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
        rad = np.sqrt(-2.0 * np.log(u1))
        out[:, 2 * p] = rad * np.cos(2 * np.pi * u2)
        out[:, 2 * p + 1] = rad * np.sin(2 * np.pi * u2)
    return out.reshape(shape)


def coords(n):
    """u = 2 p / (n - 1) - 1 of the indices of an axis of extent n (0 when n = 1), float64."""
    return 2.0 * np.arange(n) / (n - 1) - 1.0 if n > 1 else np.zeros(1)


def bias_field(coef, shape):
    """exp(sum_m c_m u_d^i u_h^j u_w^k) over a (d, h, w) grid, float64."""
    ud, uh, uw = (coords(n) for n in shape)
    p = np.zeros(shape)
    for c, (i, j, k) in zip(np.asarray(coef, dtype=np.float64), MONOMIALS):
        p += c * (ud[:, None, None] ** i) * (uh[None, :, None] ** j) * (uw[None, None, :] ** k)
    return np.exp(p)


def apply(x, rec_row, seed=0, counter=0, slot=0, n=None):
    """One slot in float64: x (C, d, h, w) the input bf16 values, rec_row its record (the recorded gamma, lo, hi,
    sigma and coefficients are used as recorded); ``n`` the slot's ``normals`` (computed if None) -> (y, noise):
    y before the bf16 round, noise = sigma * n where the noise step applies (else 0)."""
    (gon, bon, non), gamma, lo, hi, sigma, coef = unpack(rec_row)
    y = np.asarray(x, dtype=np.float64).copy()
    if gon and gamma != 1.0 and hi != lo:
        y = lo + (hi - lo) * ((y - lo) / (hi - lo)) ** gamma
    if bon:
        y = y * bias_field(coef, y.shape[1:])[None]
    noise = np.zeros_like(y)
    if non and sigma != 0.0:
        noise = sigma * (normals(seed, counter, slot, y.shape) if n is None else n)
        y = y + noise
    return y, noise
