"""The CPU oracle replayed against golden outputs of the UNMODIFIED reference
(tests/golden/*.pt, produced by tests/golden/make_golden.py).  Runs anywhere."""
import pytest
import torch

from oracle import ssd3d_oracle as O
from tests.conftest import load_golden
from tests.golden import golden_inputs as GI

torch.set_num_threads(1)


@pytest.mark.parametrize("name", list(GI.PRIOR_CASES))
def test_priors_match_reference(name):
    case, gold = GI.PRIOR_CASES[name], load_golden("priors.pt")[name]
    p = O.prior_boxes(case["size"], case.get("aspect_ratios"), in_channels=case["channels"])
    assert p.shape[0] == gold["n"]
    assert torch.equal(p[:4], gold["first"]) and torch.equal(p[-4:], gold["last"])
    assert float(p.double().sum()) == gold["sum64"]
    assert torch.equal(p.double().sum(0), gold["colsum64"])
    if gold["full"] is not None:
        assert torch.equal(p, gold["full"])
    assert torch.equal(p, O.prior_boxes_fast(case["size"], case.get("aspect_ratios"), in_channels=case["channels"]))


def test_prior_known_answers():
    # SURVEY.md section 8a row F6 (64^3 probe of the reference)
    p = O.prior_boxes((64, 64, 64))
    assert p.shape == (1168, 6)
    assert p[0].tolist() == [.0625, .0625, .0625, .09375, .09375, .09375]
    assert p[1].tolist() == [.0625, .0625, .0625, .1875, .1875, .1875]
    assert p[-1].tolist() == [.75, .75, .75, .4375, .4375, .4375]
    assert float(p.sum()) == 2289.75
    assert O.prior_boxes((96, 96, 96)).shape[0] == 3942
    assert O.prior_boxes_fast((128, 128, 128), in_channels=2).shape[0] == 9344
    assert O.prior_boxes_fast((160, 192, 160), in_channels=2).shape[0] == 43800
    assert O.prior_boxes_fast((160, 192, 160), {0: [1.], 3: [1.], 5: [1.], 7: [1.]}, in_channels=2).shape[0] == 2501400


@pytest.mark.parametrize("name", list(GI.FORWARD_CASES))
def test_forward_matches_reference(name):
    case, gold = GI.FORWARD_CASES[name], load_golden("forward.pt")[name]
    sd, x = GI.forward_inputs(case)
    assert GI.checksum_matches(x, gold["x_sum"]), "synthetic input drifted from the golden run"
    assert GI.checksum_matches(torch.cat([v.flatten().float() for v in sd.values()]), gold["w_sum"])
    assert set(sd.keys()) == set(gold["keys"])
    with torch.no_grad():
        locs, scores = O.forward(sd, x, case.get("aspect_ratios"), case.get("n_classes", 2))
    # same torch ops in the same order; only conv algorithm selection may differ by batch shape
    torch.testing.assert_close(locs, gold["locs"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(scores, gold["scores"], rtol=1e-5, atol=1e-5)


def test_box_functions_match_reference():
    g = load_golden("boxes.pt")
    a, b, gc = g["a"], g["b"], g["gc"]
    pri = O.xyz_to_cxcycz(b)
    assert torch.equal(O.find_intersection3d(a, b), g["inter"])
    assert torch.equal(O.find_jaccard_overlap3d(a, b), g["iou"])
    assert torch.equal(O.xyz_to_cxcycz(a), g["cxcycz"])
    assert torch.equal(O.cxcycz_to_xyz(pri), g["xyz"])
    assert torch.equal(O.gcxgcygcz_to_cxcycz(gc, pri), g["decoded"])
    assert torch.equal(O.cxcycz_to_gcxgcygcz(O.xyz_to_cxcycz(b.flip(0)), pri), g["encoded"])


@pytest.mark.parametrize("name", list(GI.DETECT_CASES))
def test_detect_matches_reference(name):
    case, gold = GI.DETECT_CASES[name], load_golden("detect.pt")[name]
    priors = O.prior_boxes(case["size"], in_channels=case["channels"])
    locs, scores = GI.detect_inputs(case, priors.shape[0])
    assert GI.checksum_matches(torch.cat([locs.flatten(), scores.flatten()]), gold["in_sum"])
    b, l, s, idx = O.detect_objects(locs, scores, priors, case["min_score"], case["max_overlap"], case["top_k"],
                                    return_indices=True)
    for i in range(case["batch"]):
        assert torch.equal(l[i], gold["labels"][i])
        assert torch.equal(s[i], gold["scores"][i])
        assert torch.equal(b[i], gold["boxes"][i])
        assert idx[i].shape == l[i].shape


@pytest.mark.parametrize("name", list(GI.DETECT_LONG_CASES))
def test_detect_long_lists_match_reference(name):
    """detect_objects of the unmodified reference beyond the fused kernel's limits (25 016 priors, 9 000 candidates
    through the greedy NMS, top-k cut of the kept list): pins the oracle that the any-length GPU path is tested
    against (tests/test_gpu_nms_long.py)."""
    case, gold = GI.DETECT_LONG_CASES[name], load_golden("detect_long.pt")[name]
    priors = O.prior_boxes_fast(case["size"], case["aspect_ratios"], in_channels=case["channels"])
    assert priors.shape[0] == gold["n_priors"] > 16384 and 10 * case["top_k"] > 8192
    assert torch.equal(priors, O.prior_boxes(case["size"], case["aspect_ratios"], in_channels=case["channels"]))
    locs, scores = GI.detect_long_inputs(case, priors.shape[0])
    assert GI.checksum_matches(torch.cat([locs.flatten(), scores.flatten()]), gold["in_sum"])
    b, l, s, idx = O.detect_objects(locs, scores, priors, case["min_score"], case["max_overlap"], case["top_k"],
                                    return_indices=True)
    for i in range(case["batch"]):
        assert l[i].shape[0] == case["top_k"]
        assert torch.equal(l[i], gold["labels"][i])
        assert torch.equal(s[i], gold["scores"][i])
        assert torch.equal(b[i], gold["boxes"][i])


@pytest.mark.parametrize("name", list(GI.MATCH_CASES))
def test_multibox_loss_matches_reference(name):
    case, gold = GI.MATCH_CASES[name], load_golden("match.pt")[name]
    priors = O.prior_boxes(case["size"], in_channels=case["channels"])
    locs, scores, boxes, labels = GI.match_inputs(case, priors.shape[0])
    conf, loc, tc, tl = O.multibox_loss(locs, scores, boxes, labels, priors, case["threshold"], return_targets=True)
    assert torch.equal(tc.clamp(min=0), gold["tc"])
    assert int((tc > 0).sum()) == gold["n_pos"]
    assert torch.equal(tl[tc > 0], gold["true_locs_pos"])
    assert torch.equal(conf, gold["conf_loss"])
    assert torch.equal(loc, gold["loc_loss"])


def test_bf16_emulation_is_close_to_fp32():
    case = GI.FORWARD_CASES["c2_48"]
    sd, x = GI.forward_inputs(case)
    with torch.no_grad():
        l32, s32 = O.forward(sd, x)
        l16, s16 = O.forward(sd, x, emulate_bf16=True)
    assert (l32 - l16).abs().max() < 0.15 and (s32 - s16).abs().max() < 0.15
    assert (l32 - l16).abs().mean() < 0.02


@pytest.mark.parametrize("name", list(GI.MAP_CASES))
def test_map_matches_reference(name):
    case, gold = GI.MAP_CASES[name], load_golden("map.pt")[name]
    db, dl, ds, tb, tl, td = GI.map_inputs(case)
    assert GI.checksum_matches(torch.cat([torch.cat(db).flatten(), torch.cat(ds)]), gold["in_sum"])
    o = O.calculate_map(db, dl, ds, tb, tl, td, case["min_overlap"])
    d = gold["detail"]
    assert o["mAP"] == d["mAP"] == gold["simple"][1]
    if sum(case["n_det"]) and 1 in o:
        assert torch.equal(o[1]["tp"], d["TP"]) and torch.equal(o[1]["fp"], d["FP"])
        assert torch.equal(o[1]["sorted_scores"], d["sorted_det_scores"][1])
        assert float(o[1]["AP"]) == d["APs"]
        for a, b in ((o[1]["recall"], d["recall"]), (o[1]["precision"], d["precision"]), (o[1]["f1"], d["f1_score"])):
            assert float(a) == float(b) or (float(a) != float(a) and float(b) != float(b))   # NaN when 0/0
        assert int(o[1]["detected"].numel()) == d["n_true_boxes"]
        assert torch.equal(o[1]["volumes"][o[1]["detected"] == 1], d["found_boxes_volumes_per_class"])
        assert torch.equal(o[1]["volumes"][o[1]["detected"] == 0], d["not_found_boxes_volumes_per_class"])


@pytest.mark.parametrize("name", list(GI.TRAIN_CASES))
def test_train_step_matches_reference(name):
    """Train-mode forward + MultiBox loss + autograd backward of the oracle vs the unmodified reference."""
    case, gold = GI.TRAIN_CASES[name], load_golden("train.pt")[name]
    sd, x, boxes, labels = GI.train_inputs(case)
    assert GI.checksum_matches(x, gold["x_sum"])
    pri = O.prior_boxes(case["size"], in_channels=case["channels"])
    r = O.train_step_grads(sd, x, boxes, labels, pri, case["threshold"])
    torch.testing.assert_close(r["conf"], gold["conf"], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(r["loc"], gold["loc"], rtol=1e-5, atol=1e-5)
    assert abs(GI.checksum(r["locs"]) - gold["locs_sum"]) <= 1e-3 * max(1.0, abs(gold["locs_sum"]))
    for k, g in gold["grads"].items():
        got = r["grads"][k]
        if g is None:
            assert got is None, k
            continue
        flat = got.flatten()
        assert abs(float(flat.double().norm()) - g["norm"]) <= 2e-3 * g["norm"] + 1e-7, k
        torch.testing.assert_close(flat[:8], g["head"], rtol=5e-3, atol=1e-5 * max(1.0, g["norm"]), msg=k)
        torch.testing.assert_close(flat[-8:], g["tail"], rtol=5e-3, atol=1e-5 * max(1.0, g["norm"]), msg=k)
    for k, v in gold["buffers"].items():
        got = r["running"][k]
        if k.endswith("num_batches_tracked"):
            assert int(got) == int(v)
        else:
            torch.testing.assert_close(got, v, rtol=1e-4, atol=1e-5, msg=k)


@pytest.mark.parametrize("name", list(GI.GTBOX_CASES))
def test_gt_boxes_match_reference(name):
    """Oracle connected-component box extraction vs BoundingBoxesGeneratord.converter of the unmodified reference
    (boxes bit-exact, same order, same zero-volume filter)."""
    case, gold = GI.GTBOX_CASES[name], load_golden("gtbox.pt")[name]
    segs = GI.gtbox_inputs(case)
    assert float(segs.astype("float64").sum()) == gold["in_sum"]
    for v in range(segs.shape[0]):
        b, l = O.gt_boxes_from_segmentation(segs[v], case["n_classes"])
        if gold["boxes"][v] is None:           # the reference raises on a volume without objects
            assert b.shape == (0, 6) and l.shape == (0,)
            continue
        assert torch.equal(b, gold["boxes"][v]) and torch.equal(l, gold["labels"][v])


@pytest.mark.parametrize("name", list(GI.GTBOX_INSTANCE_CASES))
def test_gt_boxes_instances_match_reference(name):
    """Oracle "instances" mode vs BoundingBoxesGeneratord.converter(segmentation_mode="instances") of the unmodified
    reference: boxes bit-exact, class-then-id order, ids outside the ranges ignored, zero-volume filter."""
    case, gold = GI.GTBOX_INSTANCE_CASES[name], load_golden("gtbox_instances.pt")[name]
    segs = GI.gtbox_instance_inputs(case)
    assert float(segs.astype("float64").sum()) == gold["in_sum"]
    for v in range(segs.shape[0]):
        b, l = O.gt_boxes_from_instances(segs[v], case["thresholds"])
        if gold["boxes"][v] is None:           # the reference raises on a volume without objects
            assert b.shape == (0, 6) and l.shape == (0,)
            continue
        assert torch.equal(b, gold["boxes"][v]) and torch.equal(l, gold["labels"][v])


def test_synthetic_ground_truth_is_what_the_extractor_finds():
    """The in-memory generator's GT boxes (synthetic.boxes_from_mask, scipy labelling as the reference) equal the
    oracle's flood-fill extraction on the generator's own masks, touching cubes included."""
    import numpy as np
    from mslesions3d_b200 import synthetic
    for idx in range(8):
        _, mask, _ = synthetic.generate_volume(idx, (40, 40, 40), (1, 5), (6, 14), 0)
        b, l = O.gt_boxes_from_segmentation(mask, 0)
        want = synthetic.boxes_from_mask(mask)
        assert np.array_equal(b.numpy(), want) and int(l.sum()) == want.shape[0]


@pytest.mark.parametrize("n,thr,extent,dup,scale", [(1, 0.5, 0.3, 0, 1.0), (500, 0.5, 0.1, 20, 1.0), (3000, 0.5, 0.3, 50, 1.0),
                                                    (3000, 0.0, 0.3, 0, 1.0), (4000, 0.3, 0.25, 10, 37.0),
                                                    (2500, 0.7, 0.15, 0, 1.0)])
def test_grid_nms_oracle_equals_the_reference_loop(n, thr, extent, dup, scale):
    """The spatially hashed CPU oracle used for the 120 k-candidate GPU parity test gives exactly the keep mask of
    the n x n restatement of ssd3d.py:407-426 (which is itself pinned by the reference's golden detections)."""
    import numpy as np
    g = torch.Generator().manual_seed(n + int(thr * 10))
    c = extent * torch.rand(n, 3, generator=g)
    s = (0.03 + 0.05 * torch.rand(n, 1, generator=g)).expand(n, 3)
    b = torch.cat([c - s / 2, c + s / 2], 1).contiguous()
    if dup:
        b[n - dup:] = b[:dup]
    if scale != 1.0:
        b = b * scale - 11.0
    t = float(np.float32(thr))
    want = O.greedy_nms(b, t)
    assert torch.equal(O.greedy_nms_grid(b, t), want)
    if n >= 500:
        assert 0 < int((~want).sum()) < n


# ---- the C restatement of the greedy NMS (oracle/nms_oracle.c), used for the 1 M / 2.5 M GPU comparisons -------
def _nms_boxes(n, seed, lo=0.02, hi=0.1, spread=0.4, cubic=True):
    g = torch.Generator().manual_seed(seed)
    c = spread * torch.rand(n, 3, generator=g)
    s = lo + (hi - lo) * torch.rand(n, 1 if cubic else 3, generator=g)
    return torch.cat([c - s / 2, c + s / 2], 1).contiguous()


@pytest.mark.parametrize("n,thr,cubic", [(3000, 0.5, True), (5000, 0.3, True), (4000, 0.0, True), (3500, 0.7, False),
                                         (2500, 0.45, False)])
def test_c_nms_oracle_matches_nxn_restatement(n, thr, cubic):
    import numpy as np
    from oracle import nms_oracle
    b = _nms_boxes(n, 900 + n, cubic=cubic)
    b[n // 2:n // 2 + 200] = b[:200]                 # exact duplicates (IoU = 1)
    b[7] = torch.tensor([.1, .1, .1, .1, .2, .2])    # zero-volume box: IoU 0 or NaN, never suppresses / suppressed
    want = O.greedy_nms(b, np.float32(thr))
    got = torch.from_numpy(nms_oracle.greedy_nms(b.numpy(), thr))
    assert torch.equal(got, want)
    assert 0 < int(want.sum()) < n


def test_c_nms_oracle_voxel_units_and_preconditions():
    import numpy as np
    from oracle import nms_oracle
    b = _nms_boxes(3000, 77, lo=4.0, hi=30.0, spread=200.0, cubic=False)
    assert torch.equal(torch.from_numpy(nms_oracle.greedy_nms(b.numpy(), 0.5)), O.greedy_nms(b, np.float32(0.5)))
    with pytest.raises(ValueError):
        nms_oracle.greedy_nms(b.numpy(), -0.1)
    bad = b.clone()
    bad[3, 0] = float("nan")
    with pytest.raises(ValueError):
        nms_oracle.greedy_nms(bad.numpy(), 0.5)
    assert nms_oracle.greedy_nms(np.zeros((0, 6), np.float32), 0.5).shape == (0,)
