"""CPU-only checks of the device-resident training data path: ``Augment`` / ``DeviceDataset`` validation, the
epoch sharding of ``epoch_order``, the oracle's signed-permutation statement of the geometry against numpy's own
crop / rot90 / flip, and the new C entry points' argument errors (no GPU needed)."""
import numpy as np
import pytest
import torch

from oracle import augment_oracle as AO


def test_augment_validation_errors():
    from mslesions3d_b200.data import Augment
    Augment().validate((64, 64, 64), (64, 64, 64))
    Augment(pos_ratio=1.0, flip_prob=0.5, rot90_prob=1.0, rot90_axes=(1, 2), scale=0.1, shift=0.1).validate(
        (32, 64, 64), (40, 97, 101))
    with pytest.raises(ValueError, match="smaller"):
        Augment().validate((64, 64, 64), (64, 63, 64))
    with pytest.raises(ValueError, match="equal"):
        Augment(rot90_prob=0.5, rot90_axes=(0, 2)).validate((32, 64, 64), (64, 64, 64))
    Augment(rot90_prob=0.0, rot90_axes=(0, 2)).validate((32, 64, 64), (64, 64, 64))     # never rotates
    for bad in (dict(pos_ratio=1.5), dict(flip_prob=-0.1), dict(rot90_prob=2.0)):
        with pytest.raises(ValueError, match="probability"):
            Augment(**bad).validate((64, 64, 64), (64, 64, 64))
    with pytest.raises(ValueError, match="rot90_axes"):
        Augment(rot90_prob=0.5, rot90_axes=(1, 1)).validate((64, 64, 64), (64, 64, 64))
    with pytest.raises(ValueError, match=">= 0"):
        Augment(scale=-0.1).validate((64, 64, 64), (64, 64, 64))
    with pytest.raises(Exception):
        Augment().pos_ratio = 0.5                                    # frozen


def test_dataset_validation_errors():
    from mslesions3d_b200.data import DeviceDataset
    with pytest.raises(ValueError, match="one shape"):
        DeviceDataset.from_arrays([np.zeros((1, 8, 8, 8)), np.zeros((1, 8, 8, 9))], [np.zeros((8, 8, 8))] * 2)
    with pytest.raises(ValueError, match="do not match"):
        DeviceDataset.from_arrays(np.zeros((2, 1, 8, 8, 8)), np.zeros((2, 8, 8, 9)))
    with pytest.raises(ValueError, match="do not match"):
        DeviceDataset.from_arrays(np.zeros((2, 1, 8, 8, 8)), np.zeros((3, 8, 8, 8)))
    with pytest.raises(ValueError, match="integer"):
        DeviceDataset.from_arrays(np.zeros((2, 1, 8, 8, 8)), np.full((2, 8, 8, 8), 0.5))
    with pytest.raises(ValueError, match="dtype"):
        DeviceDataset.from_arrays(np.zeros((2, 1, 8, 8, 8)), np.zeros((2, 8, 8, 8)), dtype=torch.float16)
    with pytest.raises(ValueError, match="empty"):
        DeviceDataset.from_arrays([], [])


@pytest.mark.parametrize("s,n,world", [(10, 2, 2), (7, 3, 1), (16, 4, 2), (5, 2, 3), (1, 4, 1)])
def test_epoch_order_sharding_is_disjoint_and_covers_every_subject(s, n, world):
    from mslesions3d_b200.data import epoch_order
    order = epoch_order(s, epoch=3, seed=11)
    assert order.dtype == torch.int32 and sorted(order.tolist()) == list(range(s))
    assert torch.equal(order, epoch_order(s, 3, 11)) and (s < 3 or not torch.equal(order, epoch_order(s, 4, 11)))
    steps = -(-s // (n * world))
    sub = AO.epoch_subjects(order.numpy(), n, world, steps)          # (world, steps, n)
    flat = sub.transpose(1, 0, 2).reshape(-1)                        # the global slot order of the epoch
    # the first S slots are the permutation itself: disjoint over ranks and covering every subject ...
    assert sorted(flat[:s].tolist()) == list(range(s))
    # ... and the padding of the last batch wraps around to the start of the order
    assert flat[s:].tolist() == [order[i % s].item() for i in range(s, len(flat))]
    assert len(flat) - s < n * world


@pytest.mark.parametrize("k", [0, 1, 2, 3])
@pytest.mark.parametrize("axes", [(0, 1), (1, 0), (0, 2), (2, 1)])
def test_signed_permutation_equals_numpy_rot90_flip_crop(k, axes):
    rs = np.random.RandomState(k * 10 + axes[0] * 3 + axes[1])
    out = [12, 12, 12]
    other = 3 - axes[0] - axes[1]
    out[other] = 7
    out = tuple(out)
    vol = rs.rand(2, 15, 17, 19).astype(np.float32)
    for trial in range(4):
        rec = np.zeros(16, dtype=np.int32)
        rec[1:4] = [rs.randint(0, vol.shape[1 + a] - out[a] + 1) for a in range(3)]
        rec[4] = k
        rec[5:8] = rs.randint(0, 2, size=3)
        want = AO.crop_rot_flip(vol, rec, out, axes)
        got = AO.gather(vol, rec, out, axes)
        assert want.shape == (2,) + out and np.array_equal(got, want)


def test_oracle_draws_follow_the_stated_semantics():
    order = np.array([3, 0, 2, 1])
    boxes = np.array([[2, 3, 4, 5, 6, 7], [10, 0, 0, 29, 5, 5]], dtype=np.int32)    # subject 0: a box > the window
    offs = np.array([0, 2, 2, 2, 2])
    rec = AO.draws(7, 5, 1, 0, 1, 4, order, boxes, offs, (40, 40, 40), (16, 16, 16), pos_ratio=1.0, flip_prob=0.5,
                   rot90_prob=1.0, scale=0.2, shift=0.3)
    assert rec[:, 0].tolist() == [3, 0, 2, 1]          # order[(1 * 4 + b) % 4]
    assert (rec[:, 4] >= 1).all() and (rec[:, 4] <= 3).all()
    f, o = rec[:, 10].view(np.float32), rec[:, 11].view(np.float32)
    assert (np.abs(f) <= np.float32(0.2)).all() and (np.abs(o) <= np.float32(0.3)).all()
    pos = rec[rec[:, 0] == 0][0]
    assert pos[8] == 1 and pos[15] == 2
    b = boxes[pos[9]]
    for ax in range(3):
        lo, hi = b[ax], b[3 + ax]
        if hi - lo + 1 <= 16:
            assert pos[1 + ax] <= lo and pos[1 + ax] + 15 >= hi
        else:
            assert pos[1 + ax] <= (lo + hi) // 2 <= pos[1 + ax] + 15
    assert (rec[rec[:, 0] != 0][:, 8] == 0).all()       # no lesion, no positive crop
    ident = AO.draws(7, 5, 0, 0, 1, 4, order, boxes, offs, (16, 16, 16), (16, 16, 16))
    assert (ident[:, 1:10] == np.array([0] * 8 + [-1])).all()
    assert (ident[:, 10:12].view(np.float32) == 0).all()            # f = o = 0 (either sign)


def test_new_symbols_report_argument_errors_without_a_gpu():
    from mslesions3d_b200 import _lib, build
    build.build(verbose=False)
    lib = _lib.load()
    e = _lib.SSD3D_ERR_ARG
    args = [1, 0, 1, 4, 1, 64, 64, 64, 1, 1, 1, 1, 2, 32, 32, 32, 0.0, 0.0, 0.0, 0, 1, 0.0, 0.0, 1, 1, 1, None]
    assert lib.ssd3d_augment_batch(*([None] + args[1:])) == e                      # no source
    bad = list(args); bad[13] = 65                                                 # output larger than the source
    assert lib.ssd3d_augment_batch(*bad) == e
    bad = list(args); bad[16] = 1.5                                                # pos_ratio outside [0, 1]
    assert lib.ssd3d_augment_batch(*bad) == e
    bad = list(args); bad[19] = bad[20] = 1                                        # one axis twice
    assert lib.ssd3d_augment_batch(*bad) == e
    bad = list(args); bad[13], bad[18] = 16, 1.0                                   # rot90 over unequal extents
    assert lib.ssd3d_augment_batch(*bad) == e
    bad = list(args); bad[15] = 24                                                 # W not a multiple of 16
    assert lib.ssd3d_augment_batch(*bad) == _lib.SSD3D_ERR_UNSUPPORTED
    assert lib.ssd3d_gt_pack(None, 1, 1, 1, 2, 8, 8, 1, 1, 1, 1, None) == e
    assert lib.ssd3d_gt_pack(1, 1, 1, 1, 0, 8, 8, 1, 1, 1, 1, None) == e
    assert lib.ssd3d_gt_pack(1, 1, 1, 1, 2, 8, 0, 1, 1, 1, 1, None) == e
