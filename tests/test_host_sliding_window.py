"""CPU-only checks of sliding-window inference: the window grid, its validation errors, the oracle's merge with one
window against ``detect_from_decoded``, and the argument errors of the new C entry points (no GPU needed)."""
import itertools
import math

import numpy as np
import pytest
import torch

from oracle import ssd3d_oracle as O
from oracle import window_oracle as WO


def _shapes():
    rng = np.random.default_rng(3)
    out = [((64, 64, 64), (64, 64, 64)), ((97, 120, 101), (64, 64, 64)), ((130, 64, 70), (64, 64, 64)),
           ((192, 224, 192), (96, 96, 96)), ((256, 256, 256), (128, 128, 128))]
    for _ in range(40):
        w = tuple(int(v) for v in rng.integers(1, 40, 3))
        out.append((tuple(int(x + rng.integers(0, 90)) for x in w), w))
    return out


@pytest.mark.parametrize("overlap", [0.0, 0.25, 0.5, 0.9, 0.999])
def test_window_grid_covers_every_voxel(overlap):
    from mslesions3d_b200.data import window_origins, window_strides
    for scan, win in _shapes():
        nd, nh, nw, o = window_origins(scan, win, overlap)
        assert o.shape == (nd * nh * nw, 3)
        strides = window_strides(win, overlap)
        for a, n in enumerate((nd, nh, nw)):
            st = max(1, int(math.floor(win[a] * (1 - overlap))))
            assert strides[a] == st
            assert n == math.ceil((scan[a] - win[a]) / st) + 1
            starts = sorted(set(o[:, a].tolist()))
            assert starts[0] == 0 and starts[-1] == scan[a] - win[a]
            cover = np.zeros(scan[a], dtype=bool)
            for s0 in starts:
                cover[s0:s0 + win[a]] = True
            assert cover.all()
        # W fastest: window t = (i_d * n_h + i_h) * n_w + i_w
        t = 0
        for i, j, k in itertools.product(range(nd), range(nh), range(nw)):
            assert o[t].tolist() == [o[i * nh * nw, 0], o[j * nw, 1], o[k, 2]]
            t += 1
        assert np.array_equal(WO.grid(scan, win, overlap)[1], o)


def test_window_grid_errors():
    from mslesions3d_b200.data import window_origins
    for bad in (-0.1, 1.0, 1.5):
        with pytest.raises(ValueError, match="overlap"):
            window_origins((64, 64, 64), (64, 64, 64), bad)
    with pytest.raises(ValueError, match="smaller"):
        window_origins((64, 63, 64), (64, 64, 64), 0.5)
    assert window_origins((64, 64, 64), (64, 64, 64), 0.5)[:3] == (1, 1, 1)


def test_window_oracle_with_one_window_equals_detect_from_decoded():
    g = torch.Generator().manual_seed(5)
    for n_classes in (2, 4):
        p = 300
        probs = torch.softmax(torch.randn((1, p, n_classes), generator=g) * 3, -1)
        cxcy = torch.rand((p, 3), generator=g)
        size = torch.rand((p, 3), generator=g) * 0.3 + 0.02
        boxes = torch.cat([cxcy - size / 2, cxcy + size / 2], 1)[None].float()
        ref_b, ref_l, ref_s = O.detect_from_decoded(probs, boxes, 0.3, 0.4, 20)
        # the per-window detections of the single window, then the merge over it
        ob, ol, os_ = WO.merge([ref_b[0].numpy()], [ref_l[0].numpy()], [ref_s[0].numpy()], (64, 64, 64),
                               (64, 64, 64), 0.5, n_classes, 0.3, 0.4, 20)
        eb, el, es = ref_b[0], ref_l[0], ref_s[0]
        if eb.shape[0] == 20:
            # a list that was cut to top_k is score-ordered; merged again it has exactly top_k entries, which
            # detect_objects returns as the concatenation of the classes (ssd3d.py:443-446): the same detections,
            # class by class, in the score order of the input
            order = torch.sort(el, stable=True).indices
            eb, el, es = eb[order], el[order], es[order]
        assert torch.equal(ob, eb) and torch.equal(ol, el) and torch.equal(os_, es)


def test_window_map_is_two_fp32_roundings():
    from mslesions3d_b200 import ops
    scale, off = ops.window_map((97, 120, 101), (64, 64, 64), np.array([[0, 28, 37], [33, 56, 0]]))
    assert scale == tuple(float(np.float32(64 / s)) for s in (97, 120, 101))
    assert off.dtype == torch.float32 and off[1, 0].item() == float(np.float32(33 / 97))
    x = np.array([[0.1, 0.2, 0.3, 0.6, 0.7, 0.8]], dtype=np.float32)
    m = WO.map_boxes(x, (33, 56, 0), (97, 120, 101), (64, 64, 64))
    assert m.dtype == np.float32
    assert m[0, 1] == np.float32(np.float32(0.2) * np.float32(64 / 120)) + np.float32(56 / 120)


def test_new_symbols_report_argument_errors_without_a_gpu():
    from mslesions3d_b200 import _lib, build
    build.build(verbose=False)
    lib = _lib.load()
    e = _lib.SSD3D_ERR_ARG
    args = [1, 0, 1, 1, 97, 120, 101, 64, 64, 64, 32, 32, 32, 1, None]
    assert lib.ssd3d_window_gather(*([None] + args[1:])) == e                    # no source
    bad = list(args); bad[13] = None                                             # no output
    assert lib.ssd3d_window_gather(*bad) == e
    bad = list(args); bad[8] = 121                                               # window larger than the scan
    assert lib.ssd3d_window_gather(*bad) == e
    bad = list(args); bad[11] = 0                                                # stride 0
    assert lib.ssd3d_window_gather(*bad) == e
    bad = list(args); bad[9] = 60                                                # W not a multiple of 8
    assert lib.ssd3d_window_gather(*bad) == _lib.SSD3D_ERR_UNSUPPORTED
    assert lib.ssd3d_merge_windows_workspace_bytes(1, 8, 100, 2, 100) > 0
    assert lib.ssd3d_merge_windows_workspace_bytes(0, 8, 100, 2, 100) == 0
    assert lib.ssd3d_merge_windows_workspace_bytes(1, 8, 100, 1, 100) == 0
    margs = [1, 1, 1, 1, 1, 8, 100, 1, 0.5, 0.5, 0.5, 2, 0.5, 0.45, 100, 1, 1, 1, 1, 1, 1, 1 << 30, 1, None]
    assert lib.ssd3d_merge_windows(*([None] + margs[1:])) == e                   # no window boxes
    bad = list(margs); bad[7] = None                                             # no offsets
    assert lib.ssd3d_merge_windows(*bad) == e
    bad = list(margs); bad[5] = 0                                                # no windows
    assert lib.ssd3d_merge_windows(*bad) == e
    bad = list(margs); bad[11] = 1                                               # one class
    assert lib.ssd3d_merge_windows(*bad) == e
    bad = list(margs); bad[21] = 16                                              # workspace too small
    assert lib.ssd3d_merge_windows(*bad) == e
