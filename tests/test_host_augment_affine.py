"""CPU-only checks of the rotation / zoom augmentation (ssd3d_augment_affine_batch): ``Augment`` validation of the
new fields, the C entry point's argument errors, and the numpy oracle (oracle/augment_affine_oracle.py) -- its
identity path against numpy's crop / rot90 / flip, its draws against Philox calls 4 and 5 written out here, and its
resampling against scipy.ndimage.map_coordinates at coordinates built independently from the header's matrices."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import augment_affine_oracle as AAO
from oracle import augment_oracle as AO
from oracle.philox_oracle import philox4x32_10

F32 = np.float32


def header_matrix(theta, z):
    """float64 M = R0 R1 R2 diag(1 / z), written out from the header: R0 in the (h, w) plane, R1 in (d, w), R2 in
    (d, h), axes (d, h, w)."""
    c, s = np.cos(theta), np.sin(theta)
    r0 = np.array([[1, 0, 0], [0, c[0], -s[0]], [0, s[0], c[0]]])
    r1 = np.array([[c[1], 0, -s[1]], [0, 1, 0], [s[1], 0, c[1]]])
    r2 = np.array([[c[2], -s[2], 0], [s[2], c[2], 0], [0, 0, 1]])
    return r0 @ r1 @ r2 @ np.diag(1.0 / np.asarray(z, dtype=np.float64))


def scipy_affine_reference(image, mask, rec_row, out_shape, rot_axes):
    """(image (C, d, h, w) float64, mask, clean): the crop resampled in float64 by scipy (order 1 / order 0, zeros
    outside the source) at x = M (p - c) + o + c over the crop index p, then np.rot90 and np.flip; ``clean`` marks
    the voxels whose coordinates lie more than 1e-3 from a half-integer on every axis (where order 0 is unambiguous)."""
    rec = np.asarray(rec_row, dtype=np.int32)
    m = header_matrix(rec[17:20].view(np.float32).astype(np.float64), rec[20:23].view(np.float32).astype(np.float64))
    p = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64) for n in out_shape], indexing="ij"))
    half = (np.asarray(out_shape, dtype=np.float64) - 1) / 2
    x = np.einsum("ac,c...->a...", m, p - half[:, None, None, None])
    x += (rec[1:4].astype(np.float64) + half)[:, None, None, None]
    img = np.stack([ndimage.map_coordinates(np.asarray(ch, dtype=np.float64), x, order=1, mode="grid-constant",
                                            cval=0.0) for ch in image])
    msk = ndimage.map_coordinates(np.asarray(mask), x, order=0, mode="grid-constant", cval=0)
    clean = (np.abs(x - np.floor(x) - 0.5) > 1e-3).all(0)
    out = []
    for v, lead in ((img, 1), (msk, 0), (clean, 0)):
        if rec[4]:
            v = np.rot90(v, int(rec[4]), axes=(lead + rot_axes[0], lead + rot_axes[1]))
        for ax in range(3):
            if rec[5 + ax]:
                v = np.flip(v, lead + ax)
        out.append(np.ascontiguousarray(v))
    return tuple(out)


def assert_close_to_scipy(got_img, got_msk, ref_img, ref_msk, clean):
    """Images within 1 bf16 ulp of the float64 value (plus 1e-4 absolute: near zero, the fp32 rounding of the
    coordinates exceeds a bf16 ulp), masks equal wherever order 0 is unambiguous."""
    got = got_img.float().numpy().astype(np.float64)
    ulp = np.exp2(np.floor(np.log2(np.maximum(np.abs(ref_img), 2.0 ** -126))) - 7)
    err = np.abs(got - ref_img)
    assert (err <= ulp + 1e-4).all(), "max error %g (ulp there %g)" % (err.max(), ulp.flat[err.argmax()])
    assert clean.mean() > 0.9
    assert np.array_equal(got_msk.numpy()[clean], ref_msk[clean])


def _record(rs, src, out, k, flips, theta, z, rot_axes, affine=True):
    rec = np.zeros(32, dtype=np.int32)
    rec[1:4] = [rs.randint(0, s - o + 1) for s, o in zip(src, out)]
    rec[4], rec[5:8] = k, flips
    rec[16] = int(affine)
    rec[17:23] = np.array(list(theta) + list(z), dtype=np.float32).view(np.int32)
    m = header_matrix(np.asarray(theta, dtype=np.float64), np.asarray(z, dtype=np.float64))
    rec[23:32] = m.astype(np.float32).reshape(-1).view(np.int32)
    return rec


def test_augment_affine_validation_errors():
    from mslesions3d_b200.data import Augment
    ok = dict(affine_prob=0.5, rotate_range=(0.3, 0.0, math.pi), zoom_range=(0.2, 0.0, 0.99))
    Augment(**ok).validate((64, 64, 64), (64, 64, 64))
    for bad in (dict(affine_prob=1.5), dict(affine_prob=-0.1)):
        with pytest.raises(ValueError, match="probability"):
            Augment(**bad).validate((64, 64, 64), (64, 64, 64))
    for bad in (dict(rotate_range=(-0.1, 0, 0)), dict(rotate_range=(0, 0, 3.2))):
        with pytest.raises(ValueError, match="rotate_range"):
            Augment(**bad).validate((64, 64, 64), (64, 64, 64))
    for bad in (dict(zoom_range=(0, -0.1, 0)), dict(zoom_range=(0, 0, 1.0))):
        with pytest.raises(ValueError, match="zoom_range"):
            Augment(**bad).validate((64, 64, 64), (64, 64, 64))
    for bad in (dict(rotate_range=(0.1, 0.1)), dict(zoom_range=(0.1, 0.1, 0.1, 0.1)), dict(zoom_range=0.1),
                dict(rotate_range=(0.1, "a", 0.1)), dict(rotate_range=[0.1, 0.1, 0.1]),
                dict(zoom_range=(0.1, None, 0.1))):
        with pytest.raises(ValueError, match="three numbers"):
            Augment(**bad).validate((64, 64, 64), (64, 64, 64))


def test_affine_symbol_reports_argument_errors_without_a_gpu():
    from mslesions3d_b200 import _lib, build
    build.build(verbose=False)
    lib = _lib.load()
    e = _lib.SSD3D_ERR_ARG

    def f3(*v):
        return (ctypes.c_float * 3)(*v)
    args = [1, 0, 1, 4, 1, 64, 64, 64, 1, 1, 1, 1, 2, 32, 32, 32, 0.0, 0.0, 0.0, 0, 1, 0.0, 0.0,
            0.5, f3(0.1, 0.1, 0.1), f3(0.1, 0.1, 0.1), 1, 1, 1, None]

    def call(**changes):
        a = list(args)
        for i, v in changes.items():
            a[int(i[1:])] = v
        return lib.ssd3d_augment_affine_batch(*a)
    assert call(a0=None) == e                                                      # no source
    assert call(a13=65) == e                                                       # output larger than the source
    assert call(a16=1.5) == e                                                      # pos_ratio outside [0, 1]
    assert call(a19=1, a20=1) == e                                                 # one axis twice
    assert call(a13=16, a18=1.0) == e                                              # rot90 over unequal extents
    assert call(a15=24) == _lib.SSD3D_ERR_UNSUPPORTED                              # W not a multiple of 16
    assert call(a23=1.5) == e and call(a23=-0.5) == e and call(a23=float("nan")) == e     # affine_prob
    assert call(a24=None) == e and call(a25=None) == e                             # no ranges
    assert call(a24=f3(0.1, -0.1, 0.1)) == e and call(a24=f3(0.1, 0.1, 3.2)) == e  # rotate_range outside [0, pi]
    assert call(a24=f3(float("nan"), 0, 0)) == e
    assert call(a25=f3(0.1, 1.0, 0.1)) == e and call(a25=f3(-0.1, 0, 0)) == e      # zoom_range outside [0, 1)
    assert call(a25=f3(0, 0, float("inf"))) == e


@pytest.mark.parametrize("k,axes", [(0, (0, 1)), (1, (0, 1)), (2, (1, 2)), (3, (0, 2)), (1, (2, 1))])
def test_oracle_identity_matrix_equals_crop_rot_flip(k, axes):
    rs = np.random.RandomState(k + 7 * axes[0])
    out = [12, 12, 12]
    out[3 - axes[0] - axes[1]] = 8
    out, src = tuple(out), (15, 17, 19)
    img = rs.randn(2, *src).astype(np.float32)
    msk = rs.randint(0, 3, size=src).astype(np.uint8)
    for trial in range(3):
        rec = _record(rs, src, out, k, rs.randint(0, 2, size=3), (0, 0, 0), (1, 1, 1), axes, affine=trial > 0)
        rec[10:12] = np.array([0.1, -0.2], dtype=np.float32).view(np.int32)
        got_img, got_msk = AAO.affine_apply(img, msk, rec, out, axes)
        want_img, want_msk = AO.apply(img, msk, rec, out, axes)
        assert torch.equal(got_img, want_img) and torch.equal(got_msk, want_msk)


def test_oracle_affine_draws_follow_philox_calls_4_and_5():
    seed, counter, rank, n = 0x1234_5678_9ABC, (3 << 32) + 17, 1, 6
    rot, zoom = (0.5, 0.25, 0.125), (0.2, 0.1, 0.3)
    got = AAO.affine_draws(seed, counter, rank, n, 0.5, rot, zoom)
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    kinds = set()
    for b in range(n):
        r4 = philox4x32_10(rank * n + b, 17, 3, 4, k0, k1)
        r5 = philox4x32_10(rank * n + b, 17, 3, 5, k0, k1)
        on = (int(r4[0]) >> 8) / 2.0 ** 24 < 0.5
        kinds.add(on)
        th, z = got[b, 1:4].view(np.float32), got[b, 4:7].view(np.float32)
        assert got[b, 0] == int(on)
        if not on:
            assert (th == 0).all() and (z == 1).all()
            continue
        for i in range(3):
            want_t = F32(rot[i]) * (F32(2) * F32((int(r4[1 + i]) >> 8) * 2.0 ** -24) - F32(1))
            want_z = F32(1) + F32(zoom[i]) * (F32(2) * F32((int(r5[i]) >> 8) * 2.0 ** -24) - F32(1))
            assert th[i] == want_t and z[i] == want_z
            assert abs(th[i]) <= F32(rot[i]) and abs(z[i] - 1) <= F32(zoom[i]) * 1.0000001
    assert kinds == {True, False}
    assert (AAO.affine_draws(seed, counter, rank, n, 0.0, rot, zoom)[:, 0] == 0).all()
    assert (AAO.affine_draws(seed, counter, rank, n, 1.0, rot, zoom)[:, 0] == 1).all()
    # the oracle's float64 matrix is the header's
    rec = np.zeros(32, dtype=np.int32)
    rec[17:23] = np.array([0.3, -0.2, 0.1, 1.1, 0.9, 1.05], dtype=np.float32).view(np.int32)
    th, z = rec[17:20].view(np.float32).astype(np.float64), rec[20:23].view(np.float32).astype(np.float64)
    assert np.allclose(AAO.affine_matrix(rec), header_matrix(th, z), rtol=0, atol=1e-15)


@pytest.mark.parametrize("k,axes,src", [(0, (0, 1), (30, 33, 35)), (1, (1, 2), (28, 26, 27)),
                                        (3, (0, 2), (40, 31, 29))])
def test_oracle_affine_apply_matches_scipy(k, axes, src):
    rs = np.random.RandomState(k + 11)
    out = (24, 24, 24)
    img = ndimage.gaussian_filter(rs.randn(2, *src), (0, 1.5, 1.5, 1.5)).astype(np.float32) * 4
    msk = (ndimage.gaussian_filter(rs.rand(*src), 2) > 0.5).astype(np.uint8) * rs.randint(1, 3, size=src).astype(np.uint8)
    for trial in range(2):
        theta = rs.uniform(-0.5, 0.5, size=3)
        z = rs.uniform(0.8, 1.2, size=3)
        rec = _record(rs, src, out, k, rs.randint(0, 2, size=3), theta, z, axes)
        got_img, got_msk = AAO.affine_apply(img, msk, rec, out, axes)
        ref_img, ref_msk, clean = scipy_affine_reference(img, msk, rec, out, axes)
        assert_close_to_scipy(got_img, got_msk, ref_img, ref_msk, clean)
        assert (ref_img == 0).any()                     # the rotated crop reaches outside these small sources
