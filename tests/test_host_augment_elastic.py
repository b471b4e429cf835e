"""CPU-only checks of the elastic deformation (ssd3d_augment_elastic_batch): ``Augment`` validation of the new fields
(the folding limit included), the C entry point's argument errors, and the numpy oracle
(oracle/augment_elastic_oracle.py) -- its field against a constant control grid, an independent float64 evaluation of
the tensor-product sum and the bound |delta| <= m, its draws against Philox calls 6 and 7 + k written out here, and
its zero field against the affine oracle."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import augment_affine_oracle as AAO
from oracle import augment_elastic_oracle as AEO
from oracle.philox_oracle import philox4x32_10
from tests.test_host_augment_affine import _record

F32 = np.float32


def test_augment_elastic_validation():
    from mslesions3d_b200.data import Augment
    out = (64, 64, 64)                                    # G = 7: spacing 63 / 4 = 15.75, limit 6.3 voxels
    Augment(elastic_prob=0.5, elastic_points=(7, 4, 16), elastic_magnitude=(6.2, 0.0, 1.0)).validate(out, out)
    Augment(elastic_prob=1.0, elastic_points=(7, 7, 7), elastic_magnitude=(0, 0, 0)).validate(out, out)
    Augment().validate((1, 16, 16), (1, 16, 16))          # a single-voxel axis with the field off
    for bad in (dict(elastic_prob=1.5), dict(elastic_prob=-0.1)):
        with pytest.raises(ValueError, match="probability"):
            Augment(**bad).validate(out, out)
    for bad in ((3, 7, 7), (7, 17, 7), (7, 7), (7, 7, 7, 7), [7, 7, 7], (7.0, 7, 7), (7, True, 7), 7):
        with pytest.raises(ValueError, match="elastic_points"):
            Augment(elastic_points=bad).validate(out, out)
    for bad in ((-0.1, 0, 0), (0, float("nan"), 0), (0, 0, float("inf")), (1, 1), [1, 1, 1], (1, "a", 1),
                (1, None, 1), 1.0):
        with pytest.raises(ValueError, match="elastic_magnitude"):
            Augment(elastic_magnitude=bad).validate(out, out)
    for m, g in (((0.4 * 63 / 4, 0, 0), (7, 7, 7)), ((0, 7.0, 0), (7, 7, 7)), ((0, 0, 2.0), (7, 7, 16))):
        with pytest.raises(ValueError, match="fold"):          # 0.4 * 63 / 13 = 1.94 for G = 16
            Augment(elastic_magnitude=m, elastic_points=g).validate(out, out)
    with pytest.raises(ValueError, match="6.3"):
        Augment(elastic_magnitude=(7, 0, 0)).validate(out, out)


def test_elastic_symbol_reports_argument_errors_without_a_gpu():
    from mslesions3d_b200 import _lib, build
    build.build(verbose=False)
    lib = _lib.load()
    e = _lib.SSD3D_ERR_ARG

    def f3(*v):
        return (ctypes.c_float * 3)(*v)

    def i3(*v):
        return (ctypes.c_int32 * 3)(*v)
    args = [1, 0, 1, 4, 1, 64, 64, 64, 1, 1, 1, 1, 2, 32, 32, 32, 0.0, 0.0, 0.0, 0, 1, 0.0, 0.0,
            0.5, f3(0.1, 0.1, 0.1), f3(0.1, 0.1, 0.1), 0.5, i3(7, 7, 7), f3(1.0, 1.0, 1.0), 1, 1, 1, None]

    def call(**changes):
        a = list(args)
        for i, v in changes.items():
            a[int(i[1:])] = v
        return lib.ssd3d_augment_elastic_batch(*a)
    assert call(a31=None) == e                                                     # no record
    assert call(a0=None) == e and call(a13=65) == e                                # the shared checks
    assert call(a15=24) == _lib.SSD3D_ERR_UNSUPPORTED                              # W not a multiple of 16
    assert call(a23=1.5) == e and call(a24=None) == e                              # the affine checks
    assert call(a26=1.5) == e and call(a26=-0.1) == e and call(a26=float("nan")) == e     # elastic_prob
    assert call(a27=None) == e and call(a28=None) == e                             # no points / magnitudes
    assert call(a27=i3(3, 7, 7)) == e and call(a27=i3(7, 17, 7)) == e and call(a27=i3(7, 7, -1)) == e
    assert call(a28=f3(-0.5, 0, 0)) == e and call(a28=f3(0, float("nan"), 0)) == e
    assert call(a28=f3(0, 0, float("inf"))) == e
    # the folding limit: 0.4 * (32 - 1) / (7 - 3) = 3.1 voxels; with G = 16, 0.4 * 31 / 13 = 0.954
    assert call(a28=f3(3.11, 0, 0)) == e and call(a27=i3(7, 7, 16), a28=f3(0, 0, 0.96)) == e


def _float64_field(P, p, g, n):
    """sum_{a,b,e} B_a B_b B_e P[j + (a, b, e)] in float64 with the textbook weights at p / s, s = (n - 1) / (G - 3)."""
    j, w = [], []
    for c in range(3):
        t = p[c] / ((n[c] - 1) / (g[c] - 3))
        jc = np.minimum(np.floor(t).astype(np.int64), g[c] - 4)
        f = t - jc
        j.append(jc)
        w.append([(1 - f) ** 3 / 6, (3 * f ** 3 - 6 * f ** 2 + 4) / 6, (-3 * f ** 3 + 3 * f ** 2 + 3 * f + 1) / 6,
                  f ** 3 / 6])
    P = P.astype(np.float64)
    out = np.zeros((3,) + p.shape[1:])
    for a in range(4):
        for b in range(4):
            for e in range(4):
                out += w[0][a] * w[1][b] * w[2][e] * np.moveaxis(P[j[0] + a, j[1] + b, j[2] + e], -1, 0)
    return out


CASES = [((24, 20, 32), (7, 7, 7), (0, 0, 0), (0, 1)), ((16, 16, 16), (4, 16, 9), (1, 0, 0), (0, 1)),
         ((32, 12, 32), (16, 4, 5), (1, 0, 1), (0, 2)), ((20, 32, 32), (5, 6, 7), (2, 1, 1), (1, 2)),
         ((20, 32, 32), (5, 6, 7), (3, 0, 1), (2, 1))]


@pytest.mark.parametrize("out,g,flips_k,axes", CASES)
def test_oracle_field_matches_float64_and_is_bounded(out, g, flips_k, axes):
    rs = np.random.RandomState(sum(out) + sum(g))
    k = flips_k[0]
    rec = np.zeros(33, dtype=np.int32)
    rec[4], rec[5:8] = k, rs.randint(0, 2, size=3)
    p, q = AEO.crop_indices(rec, out, axes)
    m = np.array([0.4 * (n - 1) / (gc - 3) * 0.99 for n, gc in zip(out, g)], dtype=np.float32)
    P = AEO.control_points(0xABCDEF12345, 5, 3, g, m)
    delta = AEO.elastic_field(P, p, q, out)
    want = _float64_field(P, p.astype(np.float64), g, out)
    err = np.abs(delta - want)
    assert err.max() <= 4e-6 * float(m.max()), err.max()
    for c in range(3):                                    # |delta_c| <= m_c up to fp32 rounding
        assert np.abs(delta[c]).max() <= m[c] * (1 + 1e-6)
        assert np.abs(delta[c]).max() > 0.2 * m[c]
    # every control point equal to one vector v: the field is v up to the rounding of the weights' sum
    v = np.array([1.75, -0.5, 3.25], dtype=np.float32)
    const = AEO.elastic_field(np.broadcast_to(v, P.shape).copy(), p, q, out)
    for c in range(3):
        assert np.abs(const[c] - v[c]).max() <= 8 * np.spacing(np.float32(abs(v[c])))


def test_oracle_weights_are_the_cubic_b_spline():
    f = np.linspace(0, 1, 1001)
    j, w = AEO.bspline(np.arange(1001), F32(1) / F32(1000), 4)
    assert (j[:-1] == 0).all() and j[-1] == 0                                     # clamped to G - 4 at the end
    want = [(1 - f) ** 3 / 6, (3 * f ** 3 - 6 * f ** 2 + 4) / 6, (-3 * f ** 3 + 3 * f ** 2 + 3 * f + 1) / 6, f ** 3 / 6]
    for a in range(4):
        assert w[a].dtype == np.float32 and np.abs(w[a] - want[a]).max() < 1e-6
    assert np.abs(sum(x.astype(np.float64) for x in w) - 1).max() < 3e-7
    assert AEO.SIXTH == F32(1 / 6) and AEO.TWO_THIRDS == F32(2 / 3)


def test_oracle_draws_follow_philox_calls_6_and_7_plus_k():
    seed, counter, rank, n = 0x1234_5678_9ABC, (3 << 32) + 17, 1, 8
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    on = AEO.elastic_draws(seed, counter, rank, n, 0.5)
    for b in range(n):
        r6 = philox4x32_10(rank * n + b, 17, 3, 6, k0, k1)
        assert on[b] == int((int(r6[0]) >> 8) / 2.0 ** 24 < 0.5)
    assert set(on.tolist()) == {0, 1}
    assert (AEO.elastic_draws(seed, counter, rank, n, 0.0) == 0).all()
    assert (AEO.elastic_draws(seed, counter, rank, n, 1.0) == 1).all()
    g, m = (4, 5, 6), (1.5, 0.25, 2.0)
    P = AEO.control_points(seed, counter, 9, g, m)
    assert P.shape == (4, 5, 6, 3) and P.dtype == np.float32
    for kd, kh, kw in ((0, 0, 0), (1, 2, 3), (3, 4, 5)):
        r = philox4x32_10(9, 17, 3, 7 + (kd * 5 + kh) * 6 + kw, k0, k1)
        for c in range(3):
            want = F32(m[c]) * (F32(2) * F32((int(r[c]) >> 8) * 2.0 ** -24) - F32(1))
            assert P[kd, kh, kw, c] == want
    assert (np.abs(P) <= np.array(m, dtype=np.float32)).all()


@pytest.mark.parametrize("k,axes", [(0, (0, 1)), (1, (1, 2)), (3, (0, 2))])
def test_oracle_without_the_field_equals_the_affine_oracle(k, axes):
    rs = np.random.RandomState(k + 3)
    out, src = (16, 16, 16), (21, 19, 23)
    img = rs.randn(2, *src).astype(np.float32)
    msk = rs.randint(0, 3, size=src).astype(np.uint8)
    rec = np.zeros(33, dtype=np.int32)
    rec[:32] = _record(rs, src, out, k, rs.randint(0, 2, size=3), rs.uniform(-0.4, 0.4, 3), rs.uniform(0.9, 1.1, 3),
                       axes)
    want = AAO.affine_apply(img, msk, rec, out, axes)
    P = AEO.control_points(1, 2, 3, (7, 7, 7), (0.0, 0.0, 0.0))
    for word, pts in ((0, P), (1, P)):               # not drawn, or drawn with m = 0: delta = 0 exactly
        rec[32] = word
        got = AEO.elastic_apply(img, msk, rec, out, pts, axes)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    rec[32] = 1
    moved = AEO.elastic_apply(img, msk, rec, out, AEO.control_points(1, 2, 3, (7, 7, 7), (1.0, 1.0, 1.0)), axes)
    assert not torch.equal(moved[0], want[0])
