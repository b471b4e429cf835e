"""Seeded inputs shared by ``make_golden.py`` (reference side, build container) and the
tests that replay the golden outputs (any machine).  Everything here is deterministic
CPU RNG (numpy MT19937 / torch CPU generator), so inputs are regenerated, not stored.
"""
import numpy as np
import torch

from oracle import ssd3d_oracle as O
from mslesions3d_b200 import synthetic

PRIOR_CASES = {
    "cube64": dict(channels=1, size=(64, 64, 64)),
    "cube96": dict(channels=1, size=(96, 96, 96)),
    "cube128": dict(channels=2, size=(128, 128, 128)),
    "noncube": dict(channels=2, size=(32, 64, 48)),
    "odd40": dict(channels=1, size=(40, 40, 40)),
    "layer0": dict(channels=2, size=(16, 32, 32), aspect_ratios={0: [1.], 3: [1.]}),
}

FORWARD_CASES = {
    "c1_64": dict(channels=1, size=(64, 64, 64), batch=1, seed=0),
    "c2_48": dict(channels=2, size=(48, 48, 48), batch=2, seed=1),
    "noncube": dict(channels=2, size=(32, 64, 48), batch=2, seed=2),
    "odd40": dict(channels=1, size=(40, 40, 40), batch=1, seed=3),
    "layer0": dict(channels=2, size=(16, 32, 32), batch=1, seed=4, aspect_ratios={0: [1.], 3: [1.]}),
}

DETECT_CASES = {
    "default": dict(channels=1, size=(64, 64, 64), batch=3, seed=10, min_score=0.5, max_overlap=0.5, top_k=100),
    "all_topk50": dict(channels=1, size=(64, 64, 64), batch=2, seed=11, min_score=0.0, max_overlap=0.5, top_k=50),
    "loose": dict(channels=1, size=(64, 64, 64), batch=2, seed=12, min_score=0.3, max_overlap=0.3, top_k=200),
    "empty": dict(channels=1, size=(64, 64, 64), batch=2, seed=13, min_score=0.9999999, max_overlap=0.5, top_k=100),
    "three_class": dict(channels=1, size=(64, 64, 64), batch=2, seed=14, min_score=0.4, max_overlap=0.45,
                        top_k=60, n_classes=3),
    "cube96": dict(channels=1, size=(96, 96, 96), batch=1, seed=15, min_score=0.2, max_overlap=0.5, top_k=300),
}

# detect_objects beyond the fused kernel's limits (P > 16384 priors and 10*top_k > 8192): a layer-0 head on a
# non-cubic volume gives 25 016 priors; min_score keeps ~12 000 of them, top_k = 900 truncates the list to 9 000
# candidates that ALL go through the greedy NMS (the reference builds a 9 000 x 9 000 IoU matrix here)
DETECT_LONG_CASES = {
    "layer0_topk900": dict(channels=1, size=(32, 48, 32), batch=1, seed=16, min_score=0.45, max_overlap=0.5, top_k=900,
                           aspect_ratios={0: [1.], 3: [1.], 5: [1.], 7: [1.]}),
}

MATCH_CASES = {
    "hard05": dict(channels=1, size=(64, 64, 64), seed=20, threshold=0.5, n_obj=[3, 1, 6, 0]),
    "soft": dict(channels=1, size=(64, 64, 64), seed=21, threshold=[0.1, 0.2], n_obj=[2, 5, 4, 3]),
    "hardlist": dict(channels=1, size=(64, 64, 64), seed=22, threshold=[0.3], n_obj=[1, 2]),
    "chunked": dict(channels=1, size=(64, 64, 64), seed=23, threshold=[0.1, 0.2], n_obj=[230, 100, 7]),
    "three_class": dict(channels=1, size=(96, 96, 96), seed=24, threshold=[0.1, 0.2], n_obj=[4, 9], n_classes=3),
}


def checksum(t: torch.Tensor) -> float:
    return float(t.double().sum())


def checksum_matches(t: torch.Tensor, gold: float) -> bool:
    """``checksum(t) == gold`` up to the rounding of the float64 sum itself: the order in which torch adds on the
    CPU (vector width, thread count) moves the last bits from one machine to another.  1e-13 of the sum of
    magnitudes is far above that rounding and far below what a drifted random stream or input recipe changes."""
    t = t.double()
    return abs(float(t.sum()) - gold) <= 1e-13 * max(1.0, float(t.abs().sum()))


def forward_inputs(case):
    """(state_dict, image) for a FORWARD case."""
    sd = O.random_state_dict(case["channels"], case.get("aspect_ratios"), case.get("n_classes", 2),
                             seed=100 + case["seed"])
    x = synthetic.make_batch(case["batch"], case["channels"], case["size"], first_idx=7 * case["seed"])
    return sd, torch.from_numpy(x)


def detect_long_inputs(case, n_priors):
    """Like ``detect_inputs`` for tens of thousands of priors, where random fp32 probabilities would collide: the
    class-1 probabilities are a random permutation of (k + 0.5) / P (spacing far above an fp32 ulp), so the
    reference's unstable sort has a unique answer."""
    g = torch.Generator().manual_seed(case["seed"])
    n = case["batch"]
    locs = torch.randn(n, n_priors, 6, generator=g) * 0.7
    p = torch.stack([(torch.randperm(n_priors, generator=g).double() + 0.5) / n_priors for _ in range(n)])
    scores = torch.stack([torch.zeros_like(p), torch.log(p / (1.0 - p))], 2).float()
    probs = torch.softmax(scores, 2)
    for i in range(n):
        if torch.unique(probs[i, :, 1]).numel() != n_priors:
            raise AssertionError("tie in golden scores; change the seed of case %r" % (case,))
    return locs, scores


def detect_inputs(case, n_priors):
    """(predicted_locs (N,P,6), predicted_scores (N,P,C)) with tie-free class probabilities."""
    g = torch.Generator().manual_seed(case["seed"])
    n, c = case["batch"], case.get("n_classes", 2)
    locs = torch.randn(n, n_priors, 6, generator=g) * 0.7
    scores = torch.randn(n, n_priors, c, generator=g) * 1.5
    # nudge exact duplicates so that the (unstable) reference sort has a unique answer
    probs = torch.softmax(scores, 2)
    for i in range(n):
        for k in range(1, c):
            col = probs[i, :, k]
            if torch.unique(col).numel() != col.numel():
                raise AssertionError("tie in golden scores; change the seed of case %r" % (case,))
    return locs, scores


def random_gt_boxes(g, n_obj, lo=0.06, hi=0.30):
    side = lo + (hi - lo) * torch.rand(n_obj, 1, generator=g)
    side = side.expand(n_obj, 3) * (0.8 + 0.4 * torch.rand(n_obj, 3, generator=g))
    corner = torch.rand(n_obj, 3, generator=g) * (1.0 - side)
    return torch.cat([corner, corner + side], 1).float()


def match_inputs(case, n_priors):
    """(predicted_locs, predicted_scores, boxes list, labels list) for a MATCH case."""
    g = torch.Generator().manual_seed(case["seed"])
    n = len(case["n_obj"])
    c = case.get("n_classes", 2)
    locs = torch.randn(n, n_priors, 6, generator=g) * 0.5
    scores = torch.randn(n, n_priors, c, generator=g)
    boxes, labels = [], []
    for k in case["n_obj"]:
        boxes.append(random_gt_boxes(g, k))
        labels.append(torch.randint(1, c, (k,), generator=g))
    return locs, scores, boxes, labels


MAP_CASES = {
    "typical": dict(seed=40, n_obj=[3, 0, 5, 2, 1], n_det=[12, 4, 20, 7, 9], min_overlap=0.1),
    "strict": dict(seed=41, n_obj=[6, 6, 6], n_det=[30, 25, 40], min_overlap=0.5),
    "no_objects": dict(seed=42, n_obj=[0, 0], n_det=[5, 3], min_overlap=0.5),
    "crowded": dict(seed=43, n_obj=[40, 35], n_det=[100, 100], min_overlap=0.1),
}


def map_inputs(case):
    """(det_boxes, det_labels, det_scores, true_boxes, true_labels, true_difficulties): lists of per-image
    tensors; detections are jittered copies of the objects plus random boxes, scores tie-free."""
    g = torch.Generator().manual_seed(case["seed"])
    tb, tl, td, db, dl, ds = [], [], [], [], [], []
    for n_obj, n_det in zip(case["n_obj"], case["n_det"]):
        t = random_gt_boxes(g, n_obj)
        reps = []
        while sum(r.shape[0] for r in reps) < n_det:          # several detections per object, then clutter
            reps.append(t if (n_obj and len(reps) < 2) else random_gt_boxes(g, max(1, n_det // 3)))
        d = torch.cat(reps)[:n_det]
        d = d + 0.03 * torch.randn(d.shape, generator=g)
        d = torch.cat([torch.minimum(d[:, :3], d[:, 3:] - 0.01), d[:, 3:]], 1).float()
        tb.append(t)
        tl.append(torch.ones(n_obj, dtype=torch.long))
        td.append(torch.zeros(n_obj, dtype=torch.bool))
        db.append(d)
        dl.append(torch.ones(n_det, dtype=torch.long))
        ds.append(torch.rand(n_det, generator=g))
    allsc = torch.cat(ds)
    assert torch.unique(allsc).numel() == allsc.numel(), "tie in golden scores"
    return db, dl, ds, tb, tl, td


TRAIN_CASES = {
    "c1_64_b2": dict(channels=1, size=(64, 64, 64), batch=2, seed=50, threshold=[0.1, 0.2]),
    "c2_48_b3": dict(channels=2, size=(48, 48, 48), batch=3, seed=51, threshold=0.5),
}


def train_inputs(case):
    """(state_dict, image, gt boxes list, gt labels list) for a TRAIN case (synthetic cube volumes + their boxes)."""
    sd = O.random_state_dict(case["channels"], seed=200 + case["seed"])
    x, b, l = synthetic.make_batch(case["batch"], case["channels"], case["size"], first_idx=3 * case["seed"],
                                   with_boxes=True)
    return sd, torch.from_numpy(x), [torch.from_numpy(v) for v in b], [torch.from_numpy(v) for v in l]


# ---- ground-truth boxes from segmentations (utils.py:438-513) --------------------------------------------------
GTBOX_CASES = {
    # binary: cubes that may touch / overlap (merge into one component), a one-voxel-thick plate and a lone voxel
    # (zero volume, dropped), two cubes touching only along an edge (separate under face connectivity)
    "binary_cubes": dict(seed=50, mode="binary", n_classes=0, size=(48, 40, 56), n_volumes=3, kind="cubes"),
    # classes: values 0..3 with n_classes = 2 (3 is not a class and is ignored); same-class blobs across a class
    # boundary stay separate, output is ordered by class first
    "classes2": dict(seed=51, mode="classes", n_classes=2, size=(40, 48, 36), n_volumes=2, kind="classes"),
    # sparse noise: hundreds of irregular components, many of them flat
    "binary_noise": dict(seed=52, mode="binary", n_classes=0, size=(20, 18, 22), n_volumes=2, kind="noise"),
    # non-convex shapes: a spiral / L / U that need several union rounds, and an empty volume
    "binary_shapes": dict(seed=53, mode="binary", n_classes=0, size=(32, 32, 32), n_volumes=2, kind="shapes"),
}


def gtbox_inputs(case):
    """-> float32 array (n_volumes, D, H, W) of segmentation values."""
    rng = np.random.RandomState(case["seed"])
    D, H, W = case["size"]
    out = np.zeros((case["n_volumes"], D, H, W), dtype=np.float32)
    for v in range(case["n_volumes"]):
        seg = out[v]
        if case["kind"] in ("cubes", "classes"):
            for _ in range(rng.randint(4, 9)):
                side = rng.randint(3, 12)
                c = [rng.randint(0, dim - side) for dim in (D, H, W)]
                val = 1 if case["kind"] == "cubes" else rng.randint(1, 4)
                seg[c[0]:c[0] + side, c[1]:c[1] + side, c[2]:c[2] + side] = val
            seg[2, 3:9, 4:11] = 1                      # plate: zero extent along axis 0
            seg[D - 1, H - 1, W - 1] = 1               # lone voxel in the last corner
            seg[10:13, 20:23, 30:33] = 1               # two cubes sharing one edge only
            seg[13:16, 23:26, 30:33] = 1
            if case["kind"] == "classes":
                seg[20:24, 5:9, 5:9] = 1               # class 1 | class 2 face to face: two components
                seg[24:28, 5:9, 5:9] = 2
        elif case["kind"] == "noise":
            seg[:] = (rng.rand(D, H, W) < 0.22).astype(np.float32)
        elif case["kind"] == "shapes" and v == 0:
            seg[4, 4:28, 4] = 1                        # U shape in one plane, 1 voxel thick -> dropped
            seg[4:20, 4, 4] = 1
            seg[8:12, 8:28, 8:12] = 1                  # L shape, thick
            seg[8:24, 24:28, 8:12] = 1
            for k in range(40):                        # staircase: connected through faces only step by step
                seg[16 + k // 4, 10 + (k % 4), 16 + k // 3] = 1
                seg[16 + k // 4, 10 + (k % 4), min(31, 17 + k // 3)] = 1
                seg[min(31, 17 + k // 4), 10 + (k % 4), 16 + k // 3] = 1
    return out


# ---------------------------------------------------------------------------------------------------
# BoundingBoxesGeneratord "instances" mode (utils.py:439-441,483-513): volumes that already hold one id per object
# ---------------------------------------------------------------------------------------------------
GTBOX_INSTANCE_CASES = {
    # two classes by id range; ids outside every range (5, 3500) are ignored; id 1003 is split over two far-apart
    # blobs (one box around both); id 2002 is one voxel thick (zero volume, dropped); class-2 ids are painted
    # before class-1 ids so that the output order (class, then id) differs from the voxel order
    "two_ranges": dict(seed=60, size=(40, 36, 44), n_volumes=2, thresholds=[(1000, 2000), (2000, 3000)]),
    # one open range (1, inf), small ids, the last volume is empty
    "open_range": dict(seed=61, size=(24, 28, 20), n_volumes=3, thresholds=[(1, float("inf"))]),
}


def gtbox_instance_inputs(case):
    """-> float32 array (n_volumes, D, H, W) of instance ids."""
    rng = np.random.RandomState(case["seed"])
    D, H, W = case["size"]
    out = np.zeros((case["n_volumes"], D, H, W), dtype=np.float32)
    two = len(case["thresholds"]) == 2
    for v in range(case["n_volumes"]):
        if not two and v == case["n_volumes"] - 1:
            continue                                    # empty volume
        seg = out[v]
        ids = ([2000 + k for k in range(1, 5)] + [1000 + k for k in range(1, 7)] + [5, 3500]) if two \
            else [int(k) for k in rng.permutation(np.arange(1, 12))]
        for i in ids:
            side = rng.randint(2, 9)
            c = [rng.randint(0, dim - side) for dim in (D, H, W)]
            seg[c[0]:c[0] + side, c[1]:c[1] + side, c[2]:c[2] + side] = i
        if two:
            seg[1:4, 1:4, 1:4] = 1003                   # second blob of id 1003
            seg[D - 4:D - 1, H - 4:H - 1, W - 4:W - 1] = 1003
            seg[seg == 2002] = 0
            seg[7, 3:9, 5:12] = 2002                    # plate: zero extent along axis 0
    return out
