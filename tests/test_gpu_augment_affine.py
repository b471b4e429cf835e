"""Rotation / zoom augmentation (ssd3d_augment_affine_batch, Augment.affine_prob, LSSD3D.fit_epoch): without the
affine and with an identity one the batches equal ssd3d_augment_batch's; with it, images, masks and records equal
the numpy oracle (oracle/augment_affine_oracle.py) bit for bit and scipy's float64 resampling within a bf16 ulp; the
in-graph ground truth follows the resampled masks; an epoch equals host-fed fit_step calls and is deterministic."""
import numpy as np
import pytest
import torch

from oracle import augment_affine_oracle as AAO
from oracle import augment_oracle as AO
from tests.test_host_augment_affine import assert_close_to_scipy, scipy_affine_reference

pytestmark = pytest.mark.gpu


def _dataset(n, channels, size, dtype=torch.float32, seed=0, num_objects=(1, 5), object_size=(6, 14)):
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import DeviceDataset
    raw, mask, _, _ = ops.generate_volumes(n, channels, size, 0, seed, num_objects, object_size)
    return DeviceDataset.from_arrays(raw, mask, dtype=dtype)


def _state(seed, counter, step=0, rank=0, world=1):
    return torch.tensor([seed, counter, step, rank, world, 0, 0, 0], dtype=torch.int64, device="cuda")


def _affine(ds, aug, n, out_size, order, state):
    from mslesions3d_b200 import ops
    return ops.augment_affine_batch(ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, n, out_size,
                                    aug.pos_ratio, aug.flip_prob, aug.rot90_prob, aug.rot90_axes, aug.scale,
                                    aug.shift, aug.affine_prob, aug.rotate_range, aug.zoom_range)


# the parametrisations of test_gpu_augment.py::test_kernel_matches_oracle
EXISTING = [
    (torch.float32, 1, (97, 120, 101), (64, 64, 64),
     dict(pos_ratio=0.5, flip_prob=0.5, rot90_prob=1.0, rot90_axes=(0, 1), scale=0.1, shift=0.2)),
    (torch.bfloat16, 2, (97, 120, 101), (64, 64, 64),
     dict(pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.75, rot90_axes=(1, 2), scale=0.3, shift=0.05)),
    (torch.float32, 2, (50, 40, 61), (48, 32, 48),
     dict(pos_ratio=0.0, flip_prob=0.5, rot90_prob=1.0, rot90_axes=(0, 2))),
    (torch.bfloat16, 1, (40, 40, 40), (32, 32, 32),
     dict(pos_ratio=0.5, flip_prob=1.0, rot90_prob=1.0, rot90_axes=(2, 0), scale=0.5)),
    (torch.float32, 1, (33, 50, 49), (32, 48, 48),
     dict(pos_ratio=1.0, flip_prob=0.25, rot90_prob=1.0, rot90_axes=(2, 1), shift=1.0)),
]


@pytest.mark.parametrize("affine_prob", [0.0, 1.0])
@pytest.mark.parametrize("dtype,channels,src,out,aug", EXISTING)
def test_without_rotation_or_zoom_equals_augment_batch(dtype, channels, src, out, aug, affine_prob):
    """affine_prob = 0, and affine_prob = 1 with zero ranges (an exact identity matrix): the batch of
    ssd3d_augment_batch, the same draws, the same state advance."""
    from mslesions3d_b200.data import Augment, epoch_order
    from mslesions3d_b200 import ops
    a = Augment(seed=12345678901, affine_prob=affine_prob, **aug)
    a.validate(out, src)
    ds = _dataset(6, channels, src, dtype, object_size=(4, 12))
    n = 4
    order = epoch_order(len(ds), 1, a.seed).cuda()
    s_old, s_new = _state(a.seed, 7), _state(a.seed, 7)
    for step in range(3):
        img0, msk0, rec0 = ops.augment_batch(ds.images, ds.masks, order, s_old, ds.boxes, ds.box_offsets, n, out,
                                             a.pos_ratio, a.flip_prob, a.rot90_prob, a.rot90_axes, a.scale, a.shift)
        img1, msk1, rec1 = _affine(ds, a, n, out, order, s_new)
        assert rec1.shape == (n, 32) and torch.equal(rec1[:, :16], rec0), "draws of step %d" % step
        words = rec1[:, 16:].cpu().numpy()
        assert (words[:, 0] == int(affine_prob > 0)).all()
        f = words[:, 1:].view(np.float32)                  # theta, z, M; zero ranges can draw theta = -0
        assert (f[:, :3] == 0).all() and (f[:, 3:6] == 1).all() and (f[:, 6:] == np.eye(3).reshape(-1)).all()
        assert torch.equal(img1, img0) and torch.equal(msk1, msk0), "batch of step %d" % step
        assert torch.equal(s_new, s_old)
    assert s_new.cpu().tolist()[1:3] == [10, 3]


AFFINE = [
    (torch.float32, 1, (97, 120, 101), (64, 64, 64),
     dict(pos_ratio=0.5, flip_prob=0.5, rot90_prob=1.0, rot90_axes=(0, 1), scale=0.1, shift=0.2)),
    (torch.bfloat16, 2, (71, 80, 77), (64, 64, 64),
     dict(pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.75, rot90_axes=(1, 2), scale=0.3, shift=0.05)),
    (torch.float32, 2, (50, 40, 61), (48, 32, 48),
     dict(pos_ratio=0.0, flip_prob=0.5, rot90_prob=1.0, rot90_axes=(0, 2))),
    (torch.bfloat16, 1, (35, 37, 35), (32, 32, 32),                      # source = crop + a few voxels: zero padding
     dict(pos_ratio=0.5, flip_prob=1.0, rot90_prob=1.0, rot90_axes=(2, 0), scale=0.5)),
]


@pytest.mark.parametrize("dtype,channels,src,out,aug", AFFINE)
def test_affine_kernel_matches_oracle(dtype, channels, src, out, aug):
    from mslesions3d_b200.data import Augment, epoch_order
    a = Augment(seed=987654321, affine_prob=0.5, rotate_range=(0.5, 0.5, 0.5), zoom_range=(0.2, 0.2, 0.2), **aug)
    a.validate(out, src)
    ds = _dataset(6, channels, src, dtype, object_size=(4, 12))
    n = 4
    order = epoch_order(len(ds), 1, a.seed).cuda()
    state = _state(a.seed, 7)
    images, masks = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy()
    boxes, offs = ds.boxes.cpu().numpy(), ds.box_offsets.cpu().numpy()
    kinds, zeros = set(), 0
    for step in range(3):
        img, msk, rec = _affine(ds, a, n, out, order, state)
        rec = rec.cpu().numpy()
        want = AO.draws(a.seed, 7 + step, step, 0, 1, n, order.cpu().numpy(), boxes, offs, src, out, a.pos_ratio,
                        a.flip_prob, a.rot90_prob, a.scale, a.shift)
        want_aff = AAO.affine_draws(a.seed, 7 + step, 0, n, a.affine_prob, a.rotate_range, a.zoom_range)
        assert np.array_equal(rec[:, :16], want) and np.array_equal(rec[:, 16:23], want_aff), "draws of step %d" % step
        for b in range(n):
            m = AAO.recorded_matrix(rec[b])
            assert np.abs(m - AAO.affine_matrix(rec[b])).max() <= 1e-6, "M of slot %d: %s" % (b, m)
            wi, wm = AAO.affine_apply(images[rec[b, 0]], masks[rec[b, 0]], rec[b], out, a.rot90_axes)
            assert torch.equal(img[b].cpu(), wi), "image of slot %d, step %d, draws %s" % (b, step, rec[b].tolist())
            assert torch.equal(msk[b].cpu(), wm), "mask of slot %d, step %d" % (b, step)
            kinds.add(int(rec[b, 16]))
            zeros += int(rec[b, 16] and (wi == 0).any())
    assert kinds == {0, 1} and state.cpu().tolist()[1:3] == [10, 3]
    if src == (35, 37, 35):
        assert zeros > 0                                                  # rotated corners outside the source


@pytest.mark.parametrize("dtype,channels,src,out,axes", [
    (torch.float32, 1, (80, 90, 84), (64, 64, 64), (1, 2)),
    (torch.bfloat16, 2, (40, 44, 53), (32, 32, 48), (0, 1)),
])
def test_affine_kernel_matches_scipy(dtype, channels, src, out, axes):
    """An independent statement: scipy's float64 trilinear / nearest resampling at coordinates built from the
    recorded theta and z with the header's matrices, rot90 and flips by numpy (no intensity step)."""
    from mslesions3d_b200.data import Augment, epoch_order
    a = Augment(seed=5, pos_ratio=0.5, flip_prob=0.5, rot90_prob=1.0, rot90_axes=axes, affine_prob=1.0,
                rotate_range=(0.5, 0.5, 0.5), zoom_range=(0.2, 0.2, 0.2))
    a.validate(out, src)
    ds = _dataset(4, channels, src, dtype, object_size=(4, 12))
    order = epoch_order(len(ds), 0, a.seed).cuda()
    img, msk, rec = _affine(ds, a, 4, out, order, _state(a.seed, 0))
    images, masks, rec = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy(), rec.cpu().numpy()
    for b in range(4):
        ref_img, ref_msk, clean = scipy_affine_reference(images[rec[b, 0]], masks[rec[b, 0]], rec[b], out, axes)
        assert_close_to_scipy(img[b].cpu(), msk[b].cpu(), ref_img, ref_msk, clean)


def test_in_graph_boxes_follow_the_resampled_masks():
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment, epoch_order
    src, out = (80, 72, 72), (64, 64, 64)
    a = Augment(seed=21, pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), affine_prob=1.0,
                rotate_range=(0.26, 0.26, 0.26), zoom_range=(0.1, 0.1, 0.1))
    ds = _dataset(8, 1, src, object_size=(4, 12))
    order = epoch_order(len(ds), 0, a.seed).cuda()
    _, msk, rec = _affine(ds, a, 8, out, order, _state(a.seed, 3))
    images, masks, rec = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy(), rec.cpu().numpy()
    want_masks = torch.stack([AAO.affine_apply(images[r[0]], masks[r[0]], r, out, a.rot90_axes)[1] for r in rec])
    want, want_labels = ops.gt_boxes_from_segmentation(want_masks.cuda())
    boxes, labels, meta = ops.gt_boxes_padded(msk, 0, 64)
    counts = meta[0].cpu().tolist()
    assert sum(counts) > 0
    for b in range(8):
        assert counts[b] == want[b].shape[0]
        assert torch.equal(boxes[b, :counts[b]], want[b]) and torch.equal(labels[b, :counts[b]], want_labels[b])


def _model(size, seed=2):
    from mslesions3d_b200.ssd3d import LSSD3D
    from oracle import ssd3d_oracle as O
    model = LSSD3D(n_classes=2, input_channels=1, input_size=size, threshold=[0.1, 0.2], lr=1e-3, min_score=0.3)
    model.load_state_dict(O.random_state_dict(1, seed=seed))
    return model.cuda().train()


def _train_state(model):
    flat = model.train_engine().flat
    return [t.clone() for t in (flat.param, flat.exp_avg, flat.exp_avg_sq, flat.status)] + \
        [b.clone() for _, b in model.named_buffers()]


AUG = dict(pos_ratio=1.0, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1, affine_prob=0.75,
           rotate_range=(0.26, 0.26, 0.26), zoom_range=(0.1, 0.1, 0.1))


def test_affine_epoch_equals_host_fed_steps_and_is_deterministic():
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment, epoch_order
    size, epoch = (64, 64, 64), 2
    ds = _dataset(12, 1, (72, 80, 72), seed=5)
    aug = Augment(seed=17, **AUG)
    m1, m2, m3 = _model(size), _model(size), _model(size)
    losses, subjects = m1.fit_epoch(ds, 4, aug, epoch=epoch)
    assert losses.shape == (3, 2) and bool(torch.isfinite(losses).all())
    # host-fed: the same batches from ops.augment_affine_batch at the epoch's draw state, GT on the host path
    steps = 3
    order = epoch_order(len(ds), epoch, aug.seed).cuda()
    state = _state(aug.seed, epoch * steps)
    for i in range(steps):
        img, msk, rec = _affine(ds, aug, 4, size, order, state)
        assert torch.equal(rec[:, 0], subjects[i])
        boxes, labels = ops.gt_boxes_from_segmentation(msk)
        loss = m2.fit_step({"img": img.clone(), "boxes": boxes, "labels": labels})
        assert torch.equal(loss, losses[i]), "loss of step %d" % i
    for x, y in zip(_train_state(m1), _train_state(m2)):
        assert torch.equal(x, y)
    again, subjects3 = m3.fit_epoch(ds, 4, aug, epoch=epoch)
    assert torch.equal(again, losses) and torch.equal(subjects3, subjects)
    for x, y in zip(_train_state(m1), _train_state(m3)):
        assert torch.equal(x, y)
