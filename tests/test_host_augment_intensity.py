"""CPU-only checks of the MR intensity augmentation (ssd3d_augment_intensity_batch): ``Augment`` validation of the six
new fields, the C entry point's argument errors before any CUDA call, and the numpy oracle
(oracle/augment_intensity_oracle.py) -- its draws against the Philox calls written out here and as a pure function of
(seed, counter, slot), its normals, and its float64 image against closed-form values of a hand-built case."""
import ctypes
import math

import numpy as np
import pytest

from oracle import augment_intensity_oracle as AIO
from oracle.philox_oracle import philox4x32_10

F32 = np.float32
FIELDS = ("bias_prob", "bias_coefficient", "gamma_prob", "gamma_log_range", "noise_prob", "noise_std")


def test_augment_intensity_validation():
    from mslesions3d_b200.data import Augment
    out = (32, 32, 32)
    a = Augment()
    assert all(getattr(a, f) == 0 for f in FIELDS) and not a.intensity
    good = [Augment(bias_prob=1.0, bias_coefficient=1.0, gamma_prob=0.5, gamma_log_range=0.999, noise_prob=0,
                    noise_std=2.5),
            Augment(gamma_prob=1, gamma_log_range=0.3), Augment(noise_prob=0.25, noise_std=1e30),
            Augment(bias_prob=np.float64(0.5), bias_coefficient=0)]
    for g in good:
        g.validate(out, out)
        hash(g)
        assert g.intensity
    assert len({*good, Augment(gamma_prob=1, gamma_log_range=0.3)}) == len(good)
    for name in ("bias_prob", "gamma_prob", "noise_prob", "bias_coefficient"):
        for v in (-0.1, 1.0 + 1e-6, 2):
            with pytest.raises(ValueError, match=name):
                Augment(**{name: v}).validate(out, out)
    for v in (-0.1, 1.0, 1.5, 1 - 1e-9):                # 1 - 1e-9 rounds to fp32 1.0: the kernel would refuse it
        with pytest.raises(ValueError, match="gamma_log_range"):
            Augment(gamma_log_range=v).validate(out, out)
    for v in (-1e-3, 1e39):
        with pytest.raises(ValueError, match="noise_std"):
            Augment(noise_std=v).validate(out, out)
    for name in FIELDS:
        for v in (float("nan"), float("inf"), "0.5", None, [0.5], (0.5,), True, np.float32(0.5)):
            with pytest.raises(ValueError, match=name):
                Augment(**{name: v}).validate(out, out)


def test_intensity_symbol_reports_argument_errors_without_a_gpu():
    from mslesions3d_b200 import _lib, build
    build.build(verbose=False)
    lib = _lib.load()
    e = _lib.SSD3D_ERR_ARG
    ws = lib.ssd3d_augment_intensity_workspace_bytes(4, 2, 32, 32, 32)
    assert ws == 4 * 4 * 8                                        # 2 * 32^3 / 16384 = 4 chunks of (lo, hi) fp32
    assert lib.ssd3d_augment_intensity_workspace_bytes(4, 1, 33, 32, 32) == 4 * 3 * 8
    assert lib.ssd3d_augment_intensity_workspace_bytes(0, 1, 32, 32, 32) == 0
    # image, N, C, d, h, w, state, bias p, bias c, gamma p, gamma r, noise p, noise std, record, ws, ws bytes, stream
    args = [1, 4, 2, 32, 32, 32, 1, 0.5, 0.5, 0.5, 0.5, 0.5, 0.5, 1, 1, ws, None]

    def call(**changes):
        a = list(args)
        for i, v in changes.items():
            a[int(i[1:])] = v
        return lib.ssd3d_augment_intensity_batch(*a)
    nan = float("nan")
    assert call(a0=None) == e and call(a6=None) == e and call(a13=None) == e
    for i in range(1, 6):
        assert call(**{"a%d" % i: 0}) == e and call(**{"a%d" % i: -1}) == e
    assert call(a5=24) == e and call(a5=8) == e                                  # w % 16
    for i in (7, 9, 11):                                                         # probabilities
        assert call(**{"a%d" % i: 1.5}) == e and call(**{"a%d" % i: -0.1}) == e and call(**{"a%d" % i: nan}) == e
    assert call(a8=1.01) == e and call(a8=-0.1) == e and call(a8=nan) == e       # bias_coefficient
    assert call(a10=1.0) == e and call(a10=-0.1) == e and call(a10=nan) == e     # gamma_log_range
    assert call(a12=-0.1) == e and call(a12=nan) == e and call(a12=float("inf")) == e      # noise_std
    assert call(a14=None) == e and call(a15=ws - 1) == e                        # gamma needs the workspace
    assert call(a1=65536, a14=None, a9=0.0) == _lib.SSD3D_ERR_UNSUPPORTED
    assert call(a2=16, a3=1024, a4=1024, a5=1024, a14=None, a9=0.0) == _lib.SSD3D_ERR_UNSUPPORTED  # noise calls


def test_oracle_draws_follow_philox_and_depend_only_on_the_slot():
    seed, counter = 0x1234_5678_9ABC, (3 << 32) + 17
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    kw = dict(bias_prob=0.5, bias_coefficient=0.75, gamma_prob=0.5, gamma_log_range=0.4, noise_prob=0.5,
              noise_std=0.3)
    seen = set()
    for slot in range(16):
        s = AIO.slot_draws(seed, counter, slot, **kw)
        r0 = [int(v) for v in philox4x32_10(slot, 17, 3, 1 << 16, k0, k1)]
        u = [F32((v >> 8) * 2.0 ** -24) for v in r0]
        assert s["flags"] == (u[0] < F32(0.5), u[1] < F32(0.5), u[2] < F32(0.5))
        gon, bon, non = s["flags"]
        seen.add(s["flags"])
        assert s["g"] == (F32(0.4) * (F32(2) * u[3] - F32(1)) if gon else 0)
        assert s["gamma64"] == (math.exp(float(s["g"])) if gon else 1.0)
        r1 = int(philox4x32_10(slot, 17, 3, (1 << 16) + 1, k0, k1)[0])
        assert s["sigma"] == (F32(0.3) * F32((r1 >> 8) * 2.0 ** -24) if non else 0)
        for m in (0, 7, 19):
            rm = int(philox4x32_10(slot, 17, 3, (1 << 16) + 2 + m // 4, k0, k1)[m % 4])
            assert s["coef"][m] == (F32(0.75) * (F32(2) * F32((rm >> 8) * 2.0 ** -24) - F32(1)) if bon else 0)
        assert np.abs(s["coef"]).max() <= 0.75 and 0 <= s["sigma"] < 0.3 and abs(s["g"]) <= 0.4
    assert len(seen) > 3
    # the record of slot b of an N-batch at rank r is that of global slot r * N + b, whatever N
    imgs = np.random.RandomState(0).randn(8, 2, 4, 4, 16).astype(np.float32)
    big = AIO.record(imgs, seed, counter, 0, **kw)
    for rank, n in ((0, 1), (1, 4), (3, 2)):
        part = AIO.record(imgs[rank * n:(rank + 1) * n], seed, counter, rank, **kw)
        assert np.array_equal(part, big[rank * n:(rank + 1) * n])
    for b in range(8):
        gon = big[b, 0]
        assert (big[b, 4:6].view(np.float32) == ([imgs[b].min(), imgs[b].max()] if gon else [0, 0])).all()
    assert not np.array_equal(AIO.record(imgs, seed, counter + 1, 0, **kw), big)
    none = AIO.record(imgs, seed, counter, 0)
    assert (none[:, :3] == 0).all() and (none[:, 3] == np.float32(1).view(np.int32)).all() and (none[:, 4:] == 0).all()


def test_oracle_normals_are_standard_and_follow_philox_quads():
    seed, counter, slot = 99, 5, 3
    n = AIO.normals(seed, counter, slot, (2, 32, 32, 64))
    assert abs(n.mean()) < 4 / math.sqrt(n.size) and abs(n.std() - 1) < 4 / math.sqrt(2 * n.size)
    w = [int(v) for v in philox4x32_10(slot, 5, 0, (1 << 24) + 7, 99, 0)]
    rad = math.sqrt(-2 * math.log(((w[0] >> 8) + 1) * 2.0 ** -24))
    flat = n.reshape(-1)
    assert flat[28] == pytest.approx(rad * math.cos(2 * math.pi * (w[1] >> 8) * 2.0 ** -24), abs=1e-15)
    assert flat[29] == pytest.approx(rad * math.sin(2 * math.pi * (w[1] >> 8) * 2.0 ** -24), abs=1e-15)
    assert np.array_equal(AIO.normals(seed, counter, slot, (1, 32, 32, 64)), n[:1])      # channel 0 is a prefix
    assert np.isfinite(n).all() and np.abs(n).max() <= math.sqrt(-2 * math.log(2.0 ** -24))


def _row(flags, gamma, lo, hi, sigma, coef):
    rec = np.zeros(27, dtype=np.int32)
    rec[:3] = flags
    rec[3:7] = np.array([gamma, lo, hi, sigma], dtype=np.float32).view(np.int32)
    rec[7:] = np.asarray(coef, dtype=np.float32).view(np.int32)
    return rec


def test_oracle_image_matches_closed_form():
    shape = (1, 3, 5, 16)
    x = np.linspace(-1.0, 3.0, int(np.prod(shape))).reshape(shape)
    coef = np.zeros(20)
    coef[AIO.MONOMIALS.index((0, 0, 1))] = 0.5          # u_w
    coef[AIO.MONOMIALS.index((1, 1, 0))] = -0.25        # u_d u_h
    coef[AIO.MONOMIALS.index((0, 0, 3))] = 0.125        # u_w^3
    lo, hi, gamma, sigma = -1.0, 3.0, 1.5, 0.25
    n = AIO.normals(1, 2, 3, shape)
    y, noise = AIO.apply(x, _row((1, 1, 1), gamma, lo, hi, sigma, coef), n=n)
    for (c, z, h, w) in ((0, 0, 0, 0), (0, 1, 2, 7), (0, 2, 4, 15), (0, 2, 1, 3)):
        ud, uh, uw = z - 1.0, h / 2 - 1.0, 2 * w / 15 - 1.0
        t = (x[c, z, h, w] + 1) / 4
        want = (-1 + 4 * t ** 1.5) * math.exp(0.5 * uw - 0.25 * ud * uh + 0.125 * uw ** 3) + 0.25 * n[c, z, h, w]
        assert y[c, z, h, w] == pytest.approx(want, rel=1e-12, abs=1e-12)
        assert noise[c, z, h, w] == 0.25 * n[c, z, h, w]
    # each step alone, and none
    assert np.array_equal(AIO.apply(x, _row((0, 0, 0), 1, 0, 0, 0, np.zeros(20)))[0], x)
    g = AIO.apply(x, _row((1, 0, 0), 0.5, lo, hi, 0, np.zeros(20)))[0]
    assert np.allclose(g, -1 + 4 * np.sqrt((x + 1) / 4), rtol=0, atol=1e-12)
    assert g.min() == lo and g.max() == pytest.approx(hi)
    assert np.array_equal(AIO.apply(x, _row((1, 0, 0), 1.0, lo, hi, 0, np.zeros(20)))[0], x)   # gamma 1: identity
    assert np.array_equal(AIO.apply(x, _row((0, 1, 0), 1, 0, 0, 0, np.zeros(20)))[0], x)       # zero field
    assert np.array_equal(AIO.apply(x, _row((0, 0, 1), 1, 0, 0, 0, np.zeros(20)), n=n)[0], x)  # sigma 0
    b = AIO.apply(x, _row((0, 1, 0), 1, 0, 0, 0, np.full(20, 0.1)))[0]
    assert b[0, 0, 0, 0] / x[0, 0, 0, 0] == pytest.approx(math.exp(0.1 * sum((-1) ** (i + j + k)
                                                                         for i, j, k in AIO.MONOMIALS)))
    # a single-voxel axis has u = 0
    one = AIO.bias_field(coef, (1, 1, 16))
    assert np.allclose(one[0, 0], np.exp(0.5 * AIO.coords(16) + 0.125 * AIO.coords(16) ** 3))
