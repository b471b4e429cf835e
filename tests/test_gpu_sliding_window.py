"""Sliding-window inference on the GPU (csrc/windows.cu, ``LSSD3D.predict_scans``): the window gather bit for bit
against torch slicing, the merge bit for bit against ``oracle/window_oracle.py``, the identity with ``predict_step``
on one window, end-to-end parity with the per-window network + oracle merge, the window -> scan geometry, the input
kinds and step sizes, and ``predict.py --window_overlap``."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import ssd3d_oracle as O
from oracle import window_oracle as WO

pytestmark = pytest.mark.gpu


def _ops():
    from mslesions3d_b200 import ops
    return ops


def _windows_torch(scans, window, overlap):
    from mslesions3d_b200.data import window_origins
    _, _, _, o = window_origins(scans.shape[2:], window, overlap)
    d, h, w = window
    return torch.stack([s[:, a:a + d, b:b + h, c:c + w].to(torch.bfloat16) for s in scans for a, b, c in o.tolist()])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("channels", [1, 2])
@pytest.mark.parametrize("n_scans", [1, 3])
@pytest.mark.parametrize("shape,window,overlap", [((97, 120, 101), (64, 64, 64), 0.5),
                                                  ((130, 64, 70), (64, 64, 64), 0.25),
                                                  ((64, 64, 64), (64, 64, 64), 0.5),
                                                  ((70, 90, 100), (32, 48, 40), 0.3)])
def test_gather_equals_torch_slicing(dtype, channels, n_scans, shape, window, overlap):
    g = torch.Generator().manual_seed(channels * 7 + n_scans)
    scans = (torch.randn((n_scans, channels) + shape, generator=g) * 3).to(dtype).cuda()
    got = _ops().window_gather(scans, window, overlap)
    want = _windows_torch(scans, window, overlap)
    assert got.dtype == torch.bfloat16 and got.shape == want.shape
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))


def _random_windows(g, n_scans, t_count, k, n_classes, full=False, empty=(), all_empty=False, tie_levels=None):
    """Per-window padded detections: (boxes, scores, labels, count) on the device + per-scan window lists."""
    n = n_scans * t_count
    boxes = torch.zeros((n, k, 6))
    scores = torch.zeros((n, k))
    labels = torch.zeros((n, k), dtype=torch.int64)
    count = torch.zeros((n,), dtype=torch.int32)
    for i in range(n):
        if all_empty or (i % t_count) in empty:
            if i % 2:         # the placeholder of a window where nothing was found
                boxes[i, 0] = torch.tensor([0., 0., 0., 1., 1., 1.])
                count[i] = 1
            continue
        c = k if full else int(torch.randint(1, k + 1, (1,), generator=g))
        lo = torch.rand((c, 3), generator=g) * 0.7
        ext = torch.rand((c, 3), generator=g) * 0.4 + 0.05
        boxes[i, :c] = torch.cat([lo, lo + ext], 1)
        if tie_levels:
            scores[i, :c] = torch.tensor(tie_levels)[torch.randint(0, len(tie_levels), (c,), generator=g)]
        else:
            scores[i, :c] = torch.rand((c,), generator=g) * 0.5 + 0.45
        labels[i, :c] = torch.randint(1, n_classes, (c,), generator=g)
        count[i] = c
    return boxes, scores, labels, count


@pytest.mark.parametrize("n_classes", [2, 4])
@pytest.mark.parametrize("case", ["random", "ties", "empty_windows", "all_empty", "full", "tight_top_k"])
def test_merge_equals_oracle(n_classes, case):
    ops = _ops()
    g = torch.Generator().manual_seed(11 + n_classes)
    scan, window, overlap = (97, 120, 101), (64, 64, 64), 0.5
    t_count = WO.grid(scan, window, overlap)[1].shape[0]
    n_scans, k, top_k = 2, 12, 12
    kw = {}
    if case == "ties":
        kw["tie_levels"] = [0.5, 0.75, 0.875, 1.0]
    elif case == "empty_windows":
        kw["empty"] = (0, 3, 5, 6)
    elif case == "all_empty":
        kw["all_empty"] = True
    elif case == "full":
        kw["full"] = True
    boxes, scores, labels, count = _random_windows(g, n_scans, t_count, k, n_classes, **kw)
    if case == "tight_top_k":
        # 10 * top_k = 30 < the candidates of a class, and more than top_k survive the NMS
        kw["full"] = True
        boxes, scores, labels, count = _random_windows(g, n_scans, t_count, k, n_classes, full=True)
        top_k = 3
        boxes[..., 3:] = boxes[..., :3] + 0.01          # small boxes: few of them overlap
    min_score, max_overlap = ops.f32(0.45), 0.4
    out = ops.merge_windows(boxes.cuda(), scores.cuda(), labels.cuda(), count.cuda(), n_scans, scan, window,
                            overlap, n_classes, min_score, max_overlap, top_k)
    cnt = out.count.cpu().tolist()
    assert int(out.status.item()) == 0
    for s in range(n_scans):
        rows = range(s * t_count, (s + 1) * t_count)
        wb = [boxes[i, :count[i]].numpy() for i in rows]
        wl = [labels[i, :count[i]].numpy() for i in rows]
        ws = [scores[i, :count[i]].numpy() for i in rows]
        eb, el, es = WO.merge(wb, wl, ws, scan, window, overlap, n_classes, min_score, max_overlap, top_k)
        assert cnt[s] == eb.shape[0]
        assert torch.equal(out.boxes[s, :cnt[s]].cpu(), eb)
        assert torch.equal(out.labels[s, :cnt[s]].cpu(), el)
        assert torch.equal(out.scores[s, :cnt[s]].cpu(), es)
        if case == "all_empty":
            assert cnt[s] == 1 and int(el[0]) == 0
        if case == "tight_top_k":
            assert cnt[s] == top_k


def _model(n_classes, channels=1, size=(64, 64, 64), seed=3, min_score=0.35, top_k=30):
    from mslesions3d_b200.ssd3d import LSSD3D
    m = LSSD3D(n_classes=n_classes, input_channels=channels, input_size=size, min_score=min_score, top_k=top_k)
    m.load_state_dict(O.random_state_dict(channels, n_classes=n_classes, seed=seed))
    return m.cuda().eval()


def _scans(n, channels, shape, seed=0):
    from mslesions3d_b200 import synthetic
    return torch.from_numpy(synthetic.make_batch(n, channels, shape, first_idx=seed))


def _same(a, b):
    assert len(a[0]) == len(b[0])
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            assert torch.equal(u.cpu(), v.cpu())


@pytest.mark.parametrize("n_classes", [2, 3])
def test_one_window_equals_predict_step(n_classes):
    m = _model(n_classes, min_score=0.34)
    scans = _scans(2, 1, (64, 64, 64), seed=5)
    with torch.no_grad():
        for src in (scans, scans.to(torch.bfloat16)):
            got = m.predict_scans(src, overlap=0.5)
            want = m.predict_step({"img": src.to(torch.bfloat16).cuda()})
            if n_classes > 2:
                # a per-window list cut to top_k is score-ordered; merged again, exactly top_k entries come out as
                # the concatenation of the classes (ssd3d.py:443-446): the same detections, class by class
                want = list(want)
                for i in range(len(want[0])):
                    if want[1][i].shape[0] == m.top_k:
                        o = torch.sort(want[1][i], stable=True).indices
                        want[0][i], want[1][i], want[2][i] = want[0][i][o], want[1][i][o], want[2][i][o]
            for i in range(2):
                assert torch.equal(got[0][i], want[0][i])
                assert torch.equal(got[1][i], want[1][i])
                assert torch.equal(got[2][i], want[2][i])


@pytest.mark.parametrize("n_classes", [2, 3])
def test_end_to_end_equals_window_network_and_oracle_merge(n_classes):
    m = _model(n_classes, seed=7)
    scans = _scans(1, 1, (150, 128, 100), seed=9)
    window, overlap = (64, 64, 64), 0.5
    with torch.no_grad():
        got = m.predict_scans(scans, overlap=overlap)
        win = _windows_torch(scans.cuda(), window, overlap)
        wb, wl, ws = m.predict_step({"img": win})
    wb = [b.cpu().numpy() for b in wb]
    wl = [l.cpu().numpy() for l in wl]
    ws = [s.cpu().numpy() for s in ws]
    eb, el, es = WO.merge(wb, wl, ws, (150, 128, 100), window, overlap, n_classes, _ops().f32(m.min_score),
                          m.max_overlap, m.top_k)
    assert torch.equal(got[0][0].cpu(), eb) and torch.equal(got[1][0].cpu(), el) and torch.equal(got[2][0].cpu(), es)
    assert (el > 0).any()                     # the random network does detect something here


def test_geometry_of_lesion_cubes():
    ops = _ops()
    scan, window, overlap = (90, 75, 110), (48, 40, 64), 0.5
    _, origins = WO.grid(scan, window, overlap)
    t_count = origins.shape[0]
    g = np.random.default_rng(4)
    for case in range(12):
        size = g.integers(2, 12, 3)
        o = origins[g.integers(0, t_count)]
        lo = np.array([o[a] + g.integers(0, window[a] - size[a]) for a in range(3)])
        mask = torch.zeros(scan, dtype=torch.uint8)
        mask[lo[0]:lo[0] + size[0], lo[1]:lo[1] + size[1], lo[2]:lo[2] + size[2]] = 1
        want, _ = ops.gt_boxes_from_segmentation(mask[None].cuda())
        boxes = torch.zeros((t_count, 1, 6))
        count = torch.zeros((t_count,), dtype=torch.int32)
        holders = 0
        for t, (a, b, c) in enumerate(origins.tolist()):
            if all(lo[i] >= (a, b, c)[i] and lo[i] + size[i] <= (a, b, c)[i] + window[i] for i in range(3)):
                wm = mask[a:a + window[0], b:b + window[1], c:c + window[2]]
                wbox, _ = ops.gt_boxes_from_segmentation(wm.contiguous()[None].cuda())
                boxes[t, 0] = wbox[0][0].cpu()
                count[t] = 1
                holders += 1
        assert holders >= 1
        out = ops.merge_windows(boxes.cuda(), torch.ones((t_count, 1)).cuda(),
                                torch.ones((t_count, 1), dtype=torch.int64).cuda(), count.cuda(), 1, scan, window,
                                overlap, 2, 0.5, 0.5, 10)
        assert int(out.count.item()) == 1 and int(out.labels[0, 0]) == 1
        got, ref = out.boxes[0, 0].cpu().numpy(), want[0][0].cpu().numpy()
        assert np.all(np.abs(got.astype(np.float64) - ref) <= 2 * np.spacing(np.abs(ref))), (case, got, ref)


def test_inputs_and_steps():
    from mslesions3d_b200.data import DeviceDataset
    m = _model(2, seed=11)
    scans = _scans(5, 1, (96, 80, 72), seed=13)
    masks = np.zeros((5, 96, 80, 72), dtype=np.uint8)
    with torch.no_grad():
        single = [m.predict_scans(scans[i:i + 1], overlap=0.5) for i in range(5)]
        single = tuple([r[j][0] for r in single] for j in range(3))
        for per in (1, 2):
            _same(m.predict_scans(scans, overlap=0.5, scans_per_step=per), single)
        _same(m.predict_scans(scans.cuda(), overlap=0.5, scans_per_step=2), single)
        _same(m.predict_scans(scans, overlap=0.5, scans_per_step=2, to_host=True), single)
        ds = DeviceDataset(scans.cuda(), torch.from_numpy(masks).cuda(), torch.zeros((1, 6), dtype=torch.int32).cuda(),
                           torch.zeros((6,), dtype=torch.int32).cuda())
        _same(m.predict_scans(ds, overlap=0.5, scans_per_step=2), single)
        _same(m.predict_scans(scans, overlap=0.5, scans_per_step=2), m.predict_scans(scans, overlap=0.5,
                                                                                    scans_per_step=2))
    with pytest.raises(ValueError, match="channels"):
        m.predict_scans(torch.zeros((1, 2, 64, 64, 64)))
    with pytest.raises(ValueError, match="smaller"):
        m.predict_scans(torch.zeros((1, 1, 64, 63, 64)))


def test_predict_py_window_overlap(tmp_path):
    from mslesions3d_b200 import predict, synthetic
    from mslesions3d_b200.nifti import load_nifti
    data = synthetic.write_dataset(str(tmp_path / "data"), 2, image_size=(96, 80, 72), random_seed=3)
    m = _model(2, seed=17)
    out_dir = str(tmp_path / "out")
    predict.predict_example(None, out_dir, data, None, min_score=0.35, top_k=30, model=m, window_overlap=0.5)
    sub = os.path.join(out_dir, "train_set", "min_score_0.35")
    names = sorted(os.listdir(sub))
    assert any(n.endswith("_preds.nii.gz") for n in names) and any(n.endswith("_preds.csv") for n in names)
    for n in names:
        if n.endswith("_preds.nii.gz"):
            vol, _ = load_nifti(os.path.join(sub, n))
            assert tuple(vol.shape) == (96, 80, 72)
    for iou in (0.5, 0.1):
        with open(os.path.join(sub, "aa_metrics_per_subject_(min_IoU=%s).json" % iou)) as f:
            assert len(json.load(f)) == 2
