"""MR intensity augmentation (ssd3d_augment_intensity_batch, Augment.bias_prob / gamma_prob / noise_prob,
LSSD3D.fit_epoch): zero strengths and slots that draw nothing leave the batch bit for bit; records equal the numpy
oracle (oracle/augment_intensity_oracle.py) -- gamma within 2 fp32 ulps of float64 exp -- after each geometric kernel;
every voxel is within one bf16 ulp of the oracle's float64 image; a slot's result does not depend on N; the noise is
N(0, sigma^2) and uncorrelated; an MR epoch equals host-fed fit_step calls, is deterministic and leaves the masks and
ground truth of the epoch without the pass."""
import dataclasses
import math

import numpy as np
import pytest
import torch

from oracle import augment_intensity_oracle as AIO
from tests.test_gpu_augment_affine import _affine, _dataset, _model, _state, _train_state
from tests.test_gpu_augment_elastic import _elastic, _epoch_plan

pytestmark = pytest.mark.gpu

GEOM = dict(pos_ratio=0.5, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1)
AFFINE = dict(affine_prob=0.75, rotate_range=(0.26, 0.26, 0.26), zoom_range=(0.1, 0.1, 0.1))
ELASTIC = dict(elastic_prob=0.75, elastic_magnitude=(3.0, 3.0, 3.0))
STRENGTH = dict(bias_coefficient=0.5, gamma_log_range=0.4, noise_std=0.3)
ONLY = {"all": dict(bias_prob=0.8, gamma_prob=0.8, noise_prob=0.8), "gamma": dict(gamma_prob=0.8),
        "bias": dict(bias_prob=0.8), "noise": dict(noise_prob=0.8)}


FIELDS = ("bias_prob", "bias_coefficient", "gamma_prob", "gamma_log_range", "noise_prob", "noise_std")


def _kw(a):
    return {f: getattr(a, f) for f in FIELDS}


def _intensity(img, state, a, **kw):
    from mslesions3d_b200 import ops
    return ops.augment_intensity_batch(img, state, img.shape[0], a.bias_prob, a.bias_coefficient, a.gamma_prob,
                                       a.gamma_log_range, a.noise_prob, a.noise_std, **kw)


def _geometric(kind, ds, a, n, out, order, state):
    from mslesions3d_b200 import ops
    if kind == "elastic":
        return _elastic(ds, a, n, out, order, state)
    if kind == "affine":
        return _affine(ds, a, n, out, order, state)
    return ops.augment_batch(ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, n, out, a.pos_ratio,
                             a.flip_prob, a.rot90_prob, a.rot90_axes, a.scale, a.shift)


def _augment(kind, seed, **kw):
    from mslesions3d_b200.data import Augment
    geo = dict(GEOM, **(AFFINE if kind != "batch" else {}), **(ELASTIC if kind == "elastic" else {}))
    return Augment(seed=seed, **geo, **kw)


def bf16_ulp(m):
    """The spacing of bf16 values at magnitude m (8 significant bits)."""
    m = np.maximum(np.abs(m), 2.0 ** -126)
    return 2.0 ** (np.floor(np.log2(m)) - 7)


def assert_within_one_ulp(got, x, rec_row, seed, counter, slot, what):
    y, noise = AIO.apply(x, rec_row, seed, counter, slot)
    _, _, lo, hi, _, _ = AIO.unpack(rec_row)
    tol = bf16_ulp(np.maximum.reduce([np.abs(y), np.full_like(y, abs(lo)), np.full_like(y, abs(hi)), np.abs(noise)]))
    err = np.abs(got - y)
    i = np.unravel_index(np.argmax(err / tol), err.shape)
    assert (err <= tol).all(), "%s: voxel %s got %r, float64 %r (tolerance %g)" % (what, i, got[i], y[i], tol[i])


def test_zero_strengths_and_undrawn_slots_leave_the_batch():
    from mslesions3d_b200.data import Augment, epoch_order
    out, n = (48, 32, 32), 8
    ds = _dataset(6, 2, (52, 40, 40), object_size=(4, 12))
    base = _augment("affine", 3)
    order = epoch_order(len(ds), 0, base.seed).cuda()
    state = _state(base.seed, 4)
    img, _, _ = _geometric("affine", ds, base, n, out, order, state)
    before, s0 = img.clone(), state.clone()
    zero = dataclasses.replace(base, bias_prob=1.0, gamma_prob=1.0, noise_prob=1.0)       # strengths 0
    rec = _intensity(img, state, zero)
    assert torch.equal(img, before) and torch.equal(state, s0)
    assert (rec[:, :3] == 1).all()
    r = rec.cpu().numpy()
    assert (r[:, 3].view(np.float32) == 1).all() and (r[:, 6:].view(np.float32) == 0).all()   # gamma 1, sigma 0, c = +-0
    assert (r[:, 4:6].view(np.float32)[:, 0] < r[:, 4:6].view(np.float32)[:, 1]).all()    # lo < hi recorded
    # probabilities 0.3 with strengths: the slots that draw none of the three keep their input bit for bit
    mixed = dataclasses.replace(base, bias_prob=0.3, gamma_prob=0.3, noise_prob=0.3, **STRENGTH)
    rec = _intensity(img, state, mixed).cpu().numpy()
    idle = [b for b in range(n) if not rec[b, :3].any()]
    busy = [b for b in range(n) if rec[b, :3].any()]
    assert idle and busy
    for b in idle:
        assert torch.equal(img[b], before[b])
    for b in busy:
        assert not torch.equal(img[b], before[b])
    assert not Augment().intensity


CASES = [
    (torch.float32, 1, 16, "batch", "all"), (torch.bfloat16, 2, 5, "affine", "all"),
    (torch.float32, 2, 1, "elastic", "all"), (torch.bfloat16, 1, 16, "elastic", "all"),
    (torch.float32, 1, 5, "batch", "gamma"), (torch.bfloat16, 2, 5, "affine", "bias"),
    (torch.float32, 2, 5, "elastic", "noise"), (torch.float32, 1, 16, "affine", "noise"),
]


@pytest.mark.parametrize("dtype,channels,n,kind,only", CASES)
def test_record_and_image_match_oracle(dtype, channels, n, kind, only):
    from mslesions3d_b200.data import epoch_order
    out, src = (32, 32, 32), (36, 40, 36)
    probs = dict(ONLY[only])
    if n == 1:
        probs = {k: 1.0 for k in probs}
    a = _augment(kind, 987654321 + n, **probs, **STRENGTH)
    a.validate(out, src)
    ds = _dataset(6, channels, src, dtype, object_size=(4, 12))
    order = epoch_order(len(ds), 1, a.seed).cuda()
    state = _state(a.seed, 7)
    drawn = np.zeros(3, dtype=np.int64)
    for step in range(2):
        img, msk, _ = _geometric(kind, ds, a, n, out, order, state)
        x, m0, s0 = img.clone(), msk.clone(), state.clone()
        rec = _intensity(img, state, a).cpu().numpy()
        assert torch.equal(state, s0) and torch.equal(msk, m0)
        xs = x.float().cpu().numpy()
        want = AIO.record(xs, a.seed, 7 + step, 0, **_kw(a))
        assert np.array_equal(np.delete(rec, 3, 1), np.delete(want, 3, 1)), "record of step %d" % step
        for b in range(n):
            g64 = AIO.slot_draws(a.seed, 7 + step, b, **_kw(a))["gamma64"]
            gamma = float(rec[b, 3:4].view(np.float32)[0])
            assert abs(gamma - g64) <= 2 * np.spacing(np.float32(g64)), "gamma of slot %d: %r vs %r" % (b, gamma, g64)
            assert_within_one_ulp(img[b].float().cpu().numpy(), xs[b].astype(np.float64), rec[b], a.seed, 7 + step,
                                  b, "slot %d step %d %s" % (b, step, rec[b, :3].tolist()))
        drawn += rec[:, :3].sum(0)
    assert drawn.sum() > 0
    for i, name in enumerate(("gamma", "bias", "noise")):
        assert (drawn[i] > 0) == (only in ("all", name))


def test_slot_alone_equals_slot_of_the_batch():
    """The pass on slot 0 alone (N = 1, the same volume and state) gives slot 0 of the N = 16 run, bit for bit."""
    from mslesions3d_b200.data import epoch_order
    out = (32, 32, 32)
    a = _augment("elastic", 11, bias_prob=1.0, gamma_prob=1.0, noise_prob=1.0, **STRENGTH)
    ds = _dataset(6, 2, (36, 40, 36), object_size=(4, 12))
    order = epoch_order(len(ds), 0, a.seed).cuda()
    state = _state(a.seed, 2)
    img, _, _ = _geometric("elastic", ds, a, 16, out, order, state)
    one = img[:1].clone()
    rec16 = _intensity(img, state, a)
    rec1 = _intensity(one, state, a)
    assert torch.equal(one[0], img[0]) and torch.equal(rec1[0], rec16[0])
    assert not torch.equal(rec16[0], rec16[1])


def test_noise_statistics():
    """96^3, 2 channels, noise alone with recorded sigma >= 0.25: the residual against the noise-free input has mean
    0 (within 4 sigma / sqrt(n)), standard deviation sigma (within 1 %), and no correlation between neighbouring
    voxels or between the channels."""
    from mslesions3d_b200.data import Augment, epoch_order
    size = (96, 96, 96)
    kw = dict(noise_prob=1.0, noise_std=0.5)
    seed = next(s for s in range(100) if AIO.slot_draws(s, 0, 0, **kw)["sigma"] >= 0.25)
    a = Augment(seed=seed, **kw)
    ds = _dataset(2, 2, size, object_size=(4, 12))
    order = epoch_order(len(ds), 0, a.seed).cuda()
    state = _state(a.seed, 0)
    img, _, _ = _geometric("batch", ds, a, 1, size, order, state)
    x = img.float().cpu().numpy()[0].astype(np.float64)
    rec = _intensity(img, state, a).cpu().numpy()
    sigma = float(rec[0, 6:7].view(np.float32)[0])
    assert sigma >= 0.25 and rec[0, 2] == 1
    res = img.float().cpu().numpy()[0].astype(np.float64) - x
    n = res.size
    assert abs(res.mean()) <= 4 * sigma / math.sqrt(n)
    assert abs(res.std() / sigma - 1) <= 0.01
    lim = 5 / math.sqrt(n / 2)
    for ax in (1, 2, 3):
        lo, hi = [slice(None)] * 4, [slice(None)] * 4
        lo[ax], hi[ax] = slice(None, -1), slice(1, None)
        r = np.corrcoef(res[tuple(lo)].ravel(), res[tuple(hi)].ravel())[0, 1]
        assert abs(r) <= lim, "correlation along axis %d: %g" % (ax, r)
    assert abs(np.corrcoef(res[0].ravel(), res[1].ravel())[0, 1]) <= lim


MR = dict(bias_prob=0.5, bias_coefficient=0.5, gamma_prob=0.5, gamma_log_range=0.3, noise_prob=0.5, noise_std=0.1)


def test_mr_epoch_equals_host_fed_steps_and_is_deterministic():
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment, epoch_order
    size, epoch, n = (64, 64, 64), 2, 4
    ds = _dataset(12, 1, (72, 80, 72), seed=5)
    plain = _augment("elastic", 17)
    aug = dataclasses.replace(plain, **MR)
    m1, m2, m3, m4 = _model(size), _model(size), _model(size), _model(size)
    losses, subjects = m1.fit_epoch(ds, n, aug, epoch=epoch)
    assert losses.shape == (3, 2) and bool(torch.isfinite(losses).all())
    p1 = _epoch_plan(m1, aug)
    # host-fed: the same batches from the elastic kernel and the intensity pass at the epoch's draw state
    steps = 3
    order = epoch_order(len(ds), epoch, aug.seed).cuda()
    state = _state(aug.seed, epoch * steps)
    drawn = 0
    for i in range(steps):
        img, msk, rec = _elastic(ds, aug, n, size, order, state)
        irec = _intensity(img, state, aug)
        assert torch.equal(rec[:, 0], subjects[i])
        drawn += int(irec[:, :3].sum())
        boxes, labels = ops.gt_boxes_from_segmentation(msk)
        loss = m2.fit_step({"img": img.clone(), "boxes": boxes, "labels": labels})
        assert torch.equal(loss, losses[i]), "loss of step %d" % i
    assert drawn > 0
    assert torch.equal(p1.image, img) and torch.equal(p1.intensity_record, irec)      # the last step's batch
    for x, y in zip(_train_state(m1), _train_state(m2)):
        assert torch.equal(x, y)
    again, subjects3 = m3.fit_epoch(ds, n, aug, epoch=epoch)
    assert torch.equal(again, losses) and torch.equal(subjects3, subjects)
    for x, y in zip(_train_state(m1), _train_state(m3)):
        assert torch.equal(x, y)
    # without the pass: the same masks, ground truth and draw state, two kernels fewer per step
    m4.fit_epoch(ds, n, plain, epoch=epoch)
    p4 = _epoch_plan(m4, plain)
    assert torch.equal(p1.mask, p4.mask) and torch.equal(p1.record, p4.record)
    k = int(p1.offsets[-1])
    assert k > 0 and torch.equal(p1.offsets, p4.offsets) and torch.equal(p1.gt_boxes[:k], p4.gt_boxes[:k])
    assert torch.equal(p1.gt_labels[:k], p4.gt_labels[:k]) and torch.equal(p1.state, p4.state)
    assert not torch.equal(p1.image, p4.image)
    assert p1.n_kernels == p4.n_kernels + 2 and not hasattr(p4, "intensity_record")
    m5 = _model(size)
    m5.fit_epoch(ds, n, Augment(seed=17), epoch=epoch)
    assert not hasattr(_epoch_plan(m5, Augment(seed=17)), "intensity_record")
