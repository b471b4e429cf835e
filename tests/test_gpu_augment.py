"""Device-resident training data (csrc/augment.cu, data.py, LSSD3D.fit_epoch): the augmentation kernel against its
numpy restatement (oracle/augment_oracle.py) bit for bit, the identity, positive crops and box geometry, the GT
packing and its overflow skip, an epoch against host-fed fit_step calls, and determinism."""
import numpy as np
import pytest
import torch

from oracle import augment_oracle as AO

pytestmark = pytest.mark.gpu


def _dataset(n, channels, size, dtype=torch.float32, seed=0, num_objects=(1, 5), object_size=(6, 14)):
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import DeviceDataset
    raw, mask, _, _ = ops.generate_volumes(n, channels, size, 0, seed, num_objects, object_size)
    return DeviceDataset.from_arrays(raw, mask, dtype=dtype)


def _state(seed, counter, step=0, rank=0, world=1):
    return torch.tensor([seed, counter, step, rank, world, 0, 0, 0], dtype=torch.int64, device="cuda")


def _augment(ds, aug, n, out_size, order, state):
    from mslesions3d_b200 import ops
    return ops.augment_batch(ds.images, ds.masks, order, state, ds.boxes, ds.box_offsets, n, out_size, aug.pos_ratio,
                             aug.flip_prob, aug.rot90_prob, aug.rot90_axes, aug.scale, aug.shift)


@pytest.mark.parametrize("dtype,channels,src,out,aug", [
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
])
def test_kernel_matches_oracle(dtype, channels, src, out, aug):
    from mslesions3d_b200.data import Augment, epoch_order
    a = Augment(seed=12345678901, **aug)
    a.validate(out, src)
    ds = _dataset(6, channels, src, dtype, object_size=(4, 12))
    n = 4
    order = epoch_order(len(ds), 1, a.seed).cuda()
    state = _state(a.seed, 7)
    images, masks = ds.images.float().cpu().numpy(), ds.masks.cpu().numpy()
    boxes, offs = ds.boxes.cpu().numpy(), ds.box_offsets.cpu().numpy()
    seen_k = set()
    for step in range(3):
        img, msk, rec = _augment(ds, a, n, out, order, state)
        want = AO.draws(a.seed, 7 + step, step, 0, 1, n, order.cpu().numpy(), boxes, offs, src, out, a.pos_ratio,
                        a.flip_prob, a.rot90_prob, a.scale, a.shift)
        assert np.array_equal(rec.cpu().numpy(), want), "draw record of step %d" % step
        for b in range(n):
            wi, wm = AO.apply(images[want[b, 0]], masks[want[b, 0]], want[b], out, a.rot90_axes)
            assert torch.equal(img[b].cpu(), wi), "image of slot %d, step %d, draws %s" % (b, step, want[b].tolist())
            assert torch.equal(msk[b].cpu(), wm), "mask of slot %d, step %d" % (b, step)
            seen_k.add(int(want[b, 4]))
    assert state.cpu().tolist()[1:3] == [10, 3]                      # the counter and the step advanced per call
    assert len(seen_k) >= 2


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_identity_augment(dtype):
    from mslesions3d_b200.data import Augment
    ds = _dataset(5, 2, (32, 48, 64), dtype)
    order = torch.arange(5, dtype=torch.int32, device="cuda").flip(0).contiguous()
    img, msk, rec = _augment(ds, Augment(), 4, (32, 48, 64), order, _state(0, 0, step=1))
    subj = [(4 + b) % 5 for b in range(4)]
    subj = [order[i].item() for i in subj]
    assert rec[:, 0].cpu().tolist() == subj
    assert torch.equal(img, ds.images[subj].to(torch.bfloat16)) and torch.equal(msk, ds.masks[subj])


def test_positive_crop_keeps_the_chosen_lesion():
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment
    ds = _dataset(8, 1, (96, 96, 96), object_size=(6, 14))
    a = Augment(pos_ratio=1.0, seed=3)
    order = torch.arange(8, dtype=torch.int32, device="cuda")
    img, msk, rec = _augment(ds, a, 8, (64, 64, 64), order, _state(a.seed, 0))
    boxes, offs = ds.boxes.cpu(), ds.box_offsets.cpu()
    got, _ = ops.gt_boxes_from_segmentation(msk)
    for b, r in enumerate(rec.cpu().tolist()):
        assert r[8] == 1
        box = boxes[offs[r[0]] + r[9]]
        shifted = (box - torch.tensor(r[1:4] * 2)).float() / 64.0
        assert ((box[3:] - box[:3] + 1) <= 64).all()
        assert any(torch.equal(row, shifted) for row in got[b].cpu()), "slot %d lost box %s" % (b, box.tolist())


@pytest.mark.parametrize("axes", [(0, 1), (1, 2), (0, 2)])
def test_boxes_follow_the_geometry(axes):
    from mslesions3d_b200 import ops
    from mslesions3d_b200.data import Augment
    ds = _dataset(8, 1, (64, 64, 64), object_size=(4, 12))
    a = Augment(flip_prob=0.5, rot90_prob=1.0, rot90_axes=axes, seed=9)
    order = torch.arange(8, dtype=torch.int32, device="cuda")
    _, msk, rec = _augment(ds, a, 8, (64, 64, 64), order, _state(a.seed, 0))
    got, _ = ops.gt_boxes_from_segmentation(msk)
    boxes, offs = ds.boxes.cpu(), ds.box_offsets.cpu()
    for b, r in enumerate(rec.cpu().tolist()):
        q, rev = AO.signed_permutation(np.array(r), axes)
        want = []
        for box in boxes[offs[r[0]]:offs[r[0] + 1]].tolist():
            lo, hi = [0] * 3, [0] * 3
            for c in range(3):
                j = q[c]
                lo[j], hi[j] = (63 - box[3 + c], 63 - box[c]) if rev[c] else (box[c], box[3 + c])
            want.append(lo + hi)
        have = torch.round(got[b].cpu().double() * 64).to(torch.int64).tolist()
        assert sorted(have) == sorted(want), "slot %d draws %s" % (b, r)


def test_gt_pack_matches_concatenated_lists_and_flags_overflow():
    from mslesions3d_b200 import ops
    ds = _dataset(6, 1, (48, 48, 48), num_objects=(2, 6), object_size=(3, 8))
    masks = ds.masks
    lists, labels = ops.gt_boxes_from_segmentation(masks)
    counts = [int(l.shape[0]) for l in lists]
    per = max(counts)
    boxes, labs, meta = ops.gt_boxes_padded(masks, 0, per)
    gb, gl, offs, status = ops.gt_pack(boxes, labs, meta, per)
    total = sum(counts)
    assert offs.cpu().tolist() == list(np.concatenate([[0], np.cumsum(counts)]))
    assert torch.equal(gb[:total], torch.cat(lists)) and torch.equal(gl[:total], torch.cat(labels))
    assert status.cpu().tolist() == [0, 0]
    # a share smaller than the largest list overflows: packed empty, counted
    boxes, labs, meta = ops.gt_boxes_padded(masks, 0, per)
    gb, gl, offs, status = ops.gt_pack(boxes, labs, meta, per - 1, status=status)
    assert status.cpu().tolist() == [1, 1] and offs.cpu().tolist() == [0] * 7
    # truncated lists (more components than max_boxes) overflow too
    boxes, labs, meta = ops.gt_boxes_padded(masks, 0, 1)
    ops.gt_pack(boxes, labs, meta, per, status=status)
    assert status.cpu().tolist() == [1, 2]


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


def test_overflowing_step_is_skipped_and_the_epoch_raises():
    from mslesions3d_b200.data import DeviceDataset
    size = (32, 32, 32)
    rs = np.random.RandomState(0)
    raw = rs.rand(4, 1, *size).astype(np.float32)
    mask = np.zeros((4,) + size, dtype=np.uint8)
    mask[:, 2:8, 2:8, 2:8] = 1                                        # two lesions per volume
    mask[:, 20:26, 20:26, 20:26] = 1
    ds = DeviceDataset.from_arrays(raw, mask)
    model = _model(size)
    model.train_engine().flatten()
    before = _train_state(model)[:3]
    with pytest.raises(RuntimeError, match="max_boxes_per_volume=1"):
        model.fit_epoch(ds, 4, max_boxes_per_volume=1)
    after = _train_state(model)[:3]
    assert all(torch.equal(x, y) for x, y in zip(before, after))
    assert model.fit_skipped_steps() == 1
    losses, _ = model.fit_epoch(ds, 4, max_boxes_per_volume=2)       # enough room: trains
    assert bool(torch.isfinite(losses).all()) and not torch.equal(model.train_engine().flat.param, before[0])


def test_epoch_equals_host_fed_steps():
    from mslesions3d_b200 import ops
    size = (64, 64, 64)
    ds = _dataset(12, 1, size, seed=5)
    m1, m2 = _model(size), _model(size)
    losses, subjects = m1.fit_epoch(ds, 4, epoch=2)
    assert losses.shape == (3, 2) and subjects.shape == (3, 4)
    subj = subjects.cpu()
    assert sorted(subj.reshape(-1).tolist()) == list(range(12))
    for i in range(3):
        idx = subj[i].long().cuda()
        boxes, labels = ops.gt_boxes_from_segmentation(ds.masks[idx])
        loss = m2.fit_step({"img": ds.images[idx].to(torch.bfloat16), "boxes": boxes, "labels": labels})
        assert torch.equal(loss, losses[i]), "loss of step %d" % i
    for x, y in zip(_train_state(m1), _train_state(m2)):
        assert torch.equal(x, y)


def test_augmented_epoch_is_deterministic():
    from mslesions3d_b200.data import Augment
    size = (64, 64, 64)
    ds = _dataset(10, 1, (80, 72, 72), seed=1)
    aug = dict(pos_ratio=0.5, flip_prob=0.5, rot90_prob=0.5, rot90_axes=(1, 2), scale=0.1, shift=0.1)
    runs = []
    for seed in (4, 4, 5):
        m = _model(size)
        losses, subjects = m.fit_epoch(ds, 4, Augment(seed=seed, **aug), epoch=1)
        runs.append((losses.cpu(), subjects.cpu(), m.train_engine().flat.param.clone()))
    assert bool(torch.isfinite(runs[0][0]).all()) and runs[0][0].shape == (3, 2)
    assert all(torch.equal(x, y) for x, y in zip(runs[0], runs[1]))
    assert not torch.equal(runs[0][0], runs[2][0]) and not torch.equal(runs[0][2], runs[2][2])
