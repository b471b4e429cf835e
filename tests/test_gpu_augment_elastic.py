"""Elastic deformation (ssd3d_augment_elastic_batch, Augment.elastic_prob, LSSD3D.fit_epoch): without the field, and
with a zero one, the batches and records equal ssd3d_augment_affine_batch's; with it, images, masks and records equal
the numpy oracle (oracle/augment_elastic_oracle.py) bit for bit under every rot90 plane, with and without the affine,
and are within a bf16 ulp of scipy's float64 resampling at independently built coordinates; the in-graph ground truth
follows the deformed masks; an elastic epoch equals host-fed fit_step calls, is deterministic and advances the draw
state as an epoch without the field does."""
import dataclasses

import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import augment_affine_oracle as AAO
from oracle import augment_elastic_oracle as AEO
from oracle import augment_oracle as AO
from tests.test_gpu_augment_affine import AFFINE, EXISTING, _affine, _dataset, _model, _state, _train_state
from tests.test_host_augment_affine import assert_close_to_scipy, header_matrix
from tests.test_host_augment_elastic import _float64_field

pytestmark = pytest.mark.gpu


def _elastic(ds, aug, n, out_size, order, state):
    from mslesions3d_b200 import ops
    return ops.augment_elastic_batch(ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, n, out_size,
                                     aug.pos_ratio, aug.flip_prob, aug.rot90_prob, aug.rot90_axes, aug.scale,
                                     aug.shift, aug.affine_prob, aug.rotate_range, aug.zoom_range, aug.elastic_prob,
                                     aug.elastic_points, aug.elastic_magnitude)


ROT_ZOOM = dict(rotate_range=(0.5, 0.5, 0.5), zoom_range=(0.2, 0.2, 0.2))


@pytest.mark.parametrize("field", ["prob0", "magnitude0"])
@pytest.mark.parametrize("affine_prob", [0.0, 1.0, 0.5])
@pytest.mark.parametrize("dtype,channels,src,out,aug", EXISTING + AFFINE)
def test_without_a_field_equals_augment_affine_batch(dtype, channels, src, out, aug, affine_prob, field):
    """elastic_prob = 0, and elastic_prob = 1 with zero magnitudes (delta = 0 exactly): the batch and record words
    0-31 of ssd3d_augment_affine_batch, the same state advance."""
    from mslesions3d_b200.data import Augment, epoch_order
    ranges = ROT_ZOOM if affine_prob == 0.5 else {}
    el = dict(elastic_prob=0.0, elastic_magnitude=(2.0, 1.0, 2.0)) if field == "prob0" else dict(elastic_prob=1.0)
    a = Augment(seed=12345678901, affine_prob=affine_prob, **ranges, **el, **aug)
    a.validate(out, src)
    ds = _dataset(6, channels, src, dtype, object_size=(4, 12))
    n = 4
    order = epoch_order(len(ds), 1, a.seed).cuda()
    s_old, s_new = _state(a.seed, 7), _state(a.seed, 7)
    for step in range(3):
        img0, msk0, rec0 = _affine(ds, a, n, out, order, s_old)
        img1, msk1, rec1 = _elastic(ds, a, n, out, order, s_new)
        assert rec1.shape == (n, 33) and torch.equal(rec1[:, :32], rec0), "draws of step %d" % step
        assert (rec1[:, 32] == int(field == "magnitude0")).all()
        assert torch.equal(img1, img0) and torch.equal(msk1, msk0), "batch of step %d" % step
        assert torch.equal(s_new, s_old)
    assert s_new.cpu().tolist()[1:3] == [10, 3]


# fp32 / bf16, 1 / 2 channels, odd sources, every rot90 plane (both orders) with flips, with and without the affine,
# G in {4, 7, 16} and anisotropic G and m (each m below 0.4 control-point spacings)
ELASTIC = [
    (torch.float32, 1, (97, 120, 101), (64, 64, 64), dict(pos_ratio=0.5, flip_prob=0.5, rot90_prob=1.0,
     rot90_axes=(0, 1), scale=0.1, shift=0.2), 0.5, (7, 7, 7), (4.0, 4.0, 4.0)),
    (torch.bfloat16, 2, (71, 80, 77), (64, 64, 64), dict(pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.75,
     rot90_axes=(1, 2), scale=0.3, shift=0.05), 0.0, (4, 7, 16), (12.0, 5.0, 1.5)),
    (torch.float32, 2, (50, 40, 61), (48, 32, 48), dict(pos_ratio=0.0, flip_prob=0.5, rot90_prob=1.0,
     rot90_axes=(0, 2)), 0.5, (16, 5, 16), (1.4, 3.0, 1.4)),
    (torch.bfloat16, 1, (35, 37, 35), (32, 32, 32), dict(pos_ratio=0.5, flip_prob=1.0, rot90_prob=1.0,
     rot90_axes=(2, 0), scale=0.5), 0.5, (16, 16, 16), (0.9, 0.9, 0.9)),
    (torch.float32, 1, (33, 50, 49), (32, 48, 48), dict(pos_ratio=1.0, flip_prob=0.25, rot90_prob=1.0,
     rot90_axes=(2, 1), shift=1.0), 0.0, (4, 4, 4), (8.0, 12.0, 12.0)),
    (torch.float32, 1, (40, 100, 70), (20, 80, 64), dict(pos_ratio=0.5, flip_prob=0.5), 1.0, (5, 11, 7),
     (3.0, 2.5, 4.0)),
]


@pytest.mark.parametrize("dtype,channels,src,out,aug,affine_prob,points,magnitude", ELASTIC)
def test_elastic_kernel_matches_oracle(dtype, channels, src, out, aug, affine_prob, points, magnitude):
    from mslesions3d_b200.data import Augment, epoch_order
    a = Augment(seed=987654321, affine_prob=affine_prob, **ROT_ZOOM, elastic_prob=0.75, elastic_points=points,
                elastic_magnitude=magnitude, **aug)
    a.validate(out, src)
    ds = _dataset(6, channels, src, dtype, object_size=(4, 12))
    n = 4
    order = epoch_order(len(ds), 1, a.seed).cuda()
    state = _state(a.seed, 7)
    images, masks = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy()
    boxes, offs = ds.boxes.cpu().numpy(), ds.box_offsets.cpu().numpy()
    kinds, ks = set(), set()
    for step in range(2):
        img, msk, rec = _elastic(ds, a, n, out, order, state)
        rec = rec.cpu().numpy()
        want = AO.draws(a.seed, 7 + step, step, 0, 1, n, order.cpu().numpy(), boxes, offs, src, out, a.pos_ratio,
                        a.flip_prob, a.rot90_prob, a.scale, a.shift)
        want_aff = AAO.affine_draws(a.seed, 7 + step, 0, n, a.affine_prob, a.rotate_range, a.zoom_range)
        want_el = AEO.elastic_draws(a.seed, 7 + step, 0, n, a.elastic_prob)
        assert np.array_equal(rec[:, :16], want) and np.array_equal(rec[:, 16:23], want_aff), "draws of step %d" % step
        assert np.array_equal(rec[:, 32], want_el)
        for b in range(n):
            P = AEO.control_points(a.seed, 7 + step, b, points, magnitude)
            wi, wm = AEO.elastic_apply(images[rec[b, 0]], masks[rec[b, 0]], rec[b], out, P, a.rot90_axes)
            assert torch.equal(img[b].cpu(), wi), "image of slot %d, step %d, draws %s" % (b, step, rec[b].tolist())
            assert torch.equal(msk[b].cpu(), wm), "mask of slot %d, step %d" % (b, step)
            kinds.add(int(rec[b, 32]))
            ks.add(int(rec[b, 4]))
    assert 1 in kinds and state.cpu().tolist()[1:3] == [9, 2]
    if aug.get("rot90_prob", 0) == 1.0:
        assert ks - {0}                                                   # the permuted tile axes were exercised


def scipy_elastic_reference(image, mask, rec_row, out_shape, rot_axes, P):
    """(image, mask, clean) as ``scipy_affine_reference``, at x = M (p - c + delta(p)) + o + c with the float64
    field of the test's own tensor-product sum and the float64 header matrix."""
    rec = np.asarray(rec_row, dtype=np.int32)
    m = header_matrix(rec[17:20].view(np.float32).astype(np.float64), rec[20:23].view(np.float32).astype(np.float64))
    p = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64) for n in out_shape], indexing="ij"))
    half = (np.asarray(out_shape, dtype=np.float64) - 1) / 2
    u = p - half[:, None, None, None]
    if rec[32]:
        u = u + _float64_field(P, p, P.shape[:3], out_shape)
    x = np.einsum("ac,c...->a...", m, u) + (rec[1:4].astype(np.float64) + half)[:, None, None, None]
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


@pytest.mark.parametrize("dtype,channels,src,out,axes,affine_prob", [
    (torch.float32, 1, (80, 90, 84), (64, 64, 64), (1, 2), 1.0),
    (torch.bfloat16, 2, (40, 44, 53), (32, 32, 48), (0, 1), 0.0),
])
def test_elastic_kernel_matches_scipy(dtype, channels, src, out, axes, affine_prob):
    from mslesions3d_b200.data import Augment, epoch_order
    a = Augment(seed=5, pos_ratio=0.5, flip_prob=0.5, rot90_prob=1.0, rot90_axes=axes, affine_prob=affine_prob,
                **ROT_ZOOM, elastic_prob=1.0, elastic_points=(7, 6, 8), elastic_magnitude=(3.0, 2.0, 2.5))
    a.validate(out, src)
    ds = _dataset(4, channels, src, dtype, object_size=(4, 12))
    order = epoch_order(len(ds), 0, a.seed).cuda()
    img, msk, rec = _elastic(ds, a, 4, out, order, _state(a.seed, 0))
    images, masks, rec = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy(), rec.cpu().numpy()
    for b in range(4):
        P = AEO.control_points(a.seed, 0, b, a.elastic_points, a.elastic_magnitude)
        ref_img, ref_msk, clean = scipy_elastic_reference(images[rec[b, 0]], masks[rec[b, 0]], rec[b], out, axes, P)
        assert_close_to_scipy(img[b].cpu(), msk[b].cpu(), ref_img, ref_msk, clean)


def test_in_graph_boxes_follow_the_deformed_masks():
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment, epoch_order
    src, out = (80, 72, 72), (64, 64, 64)
    a = Augment(seed=21, pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), affine_prob=0.5,
                rotate_range=(0.26, 0.26, 0.26), zoom_range=(0.1, 0.1, 0.1), elastic_prob=1.0,
                elastic_magnitude=(5.0, 5.0, 5.0))
    ds = _dataset(8, 1, src, object_size=(4, 12))
    order = epoch_order(len(ds), 0, a.seed).cuda()
    _, msk, rec = _elastic(ds, a, 8, out, order, _state(a.seed, 3))
    images, masks, rec = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy(), rec.cpu().numpy()
    want_masks = torch.stack([AEO.elastic_apply(images[r[0]], masks[r[0]], r, out,
                                                AEO.control_points(a.seed, 3, b, a.elastic_points,
                                                                   a.elastic_magnitude), a.rot90_axes)[1]
                              for b, r in enumerate(rec)])
    assert torch.equal(msk.cpu(), want_masks)
    want, want_labels = ops.gt_boxes_from_segmentation(want_masks.cuda())
    boxes, labels, meta = ops.gt_boxes_padded(msk, 0, 64)
    counts = meta[0].cpu().tolist()
    assert sum(counts) > 0
    for b in range(8):
        assert counts[b] == want[b].shape[0]
        assert torch.equal(boxes[b, :counts[b]], want[b]) and torch.equal(labels[b, :counts[b]], want_labels[b])


AUG = dict(pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1, affine_prob=0.5,
           rotate_range=(0.26, 0.26, 0.26), zoom_range=(0.1, 0.1, 0.1), elastic_prob=0.75,
           elastic_magnitude=(4.0, 4.0, 4.0))


def _epoch_plan(model, aug):
    return [p for p in model.train_engine().plans.values() if getattr(p, "augment", None) == aug][0]


def test_elastic_epoch_equals_host_fed_steps_and_is_deterministic():
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment, epoch_order
    size, epoch = (64, 64, 64), 2
    ds = _dataset(12, 1, (72, 80, 72), seed=5)
    aug = Augment(seed=17, **AUG)
    m1, m2, m3, m4 = _model(size), _model(size), _model(size), _model(size)
    losses, subjects = m1.fit_epoch(ds, 4, aug, epoch=epoch)
    assert losses.shape == (3, 2) and bool(torch.isfinite(losses).all())
    assert _epoch_plan(m1, aug).record.shape[1] == 33
    # host-fed: the same batches from ops.augment_elastic_batch at the epoch's draw state, GT on the host path
    steps = 3
    order = epoch_order(len(ds), epoch, aug.seed).cuda()
    state = _state(aug.seed, epoch * steps)
    drawn = 0
    for i in range(steps):
        img, msk, rec = _elastic(ds, aug, 4, size, order, state)
        assert torch.equal(rec[:, 0], subjects[i])
        drawn += int(rec[:, 32].sum())
        boxes, labels = ops.gt_boxes_from_segmentation(msk)
        loss = m2.fit_step({"img": img.clone(), "boxes": boxes, "labels": labels})
        assert torch.equal(loss, losses[i]), "loss of step %d" % i
    assert drawn > 0
    for x, y in zip(_train_state(m1), _train_state(m2)):
        assert torch.equal(x, y)
    again, subjects3 = m3.fit_epoch(ds, 4, aug, epoch=epoch)
    assert torch.equal(again, losses) and torch.equal(subjects3, subjects)
    for x, y in zip(_train_state(m1), _train_state(m3)):
        assert torch.equal(x, y)
    # the draw state after the epoch is that of an epoch without the field, and of the host-fed launches
    plain = dataclasses.replace(aug, elastic_prob=0.0)
    m4.fit_epoch(ds, 4, plain, epoch=epoch)
    after = _epoch_plan(m1, aug).state
    assert torch.equal(after, _epoch_plan(m4, plain).state) and torch.equal(after.cpu()[:3], state.cpu()[:3])
