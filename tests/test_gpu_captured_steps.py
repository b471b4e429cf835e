"""The captured steps against their uncaptured forms: the eager ``fit_step`` runs the same step body as the graph, and
the read-back check of every captured inference step raises on NaN and recovers on the next clean input."""
import pytest
import torch

from oracle import ssd3d_oracle as O
from mslesions3d_b200 import synthetic

pytestmark = pytest.mark.gpu


def _bit_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    """torch.equal on the bits (a NaN loss of a skipped step equals itself)."""
    return (a.dtype == b.dtype and a.shape == b.shape and
            torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8)))


def _same(a, b) -> bool:
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and _bit_equal(a, b)
    return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))


def test_eager_fit_step_equals_captured():
    """Three ``fit_step``s with ``use_cuda_graph = False`` and three with ``True``, from one state dict over the same
    batches: bit-identical losses, parameters, Adam moments and step counters, and BatchNorm buffers."""
    from mslesions3d_b200.ssd3d import LSSD3D
    size, channels = (64, 64, 64), 1
    sd = O.random_state_dict(channels, seed=5)
    batches = []
    for k in range(3):
        x, b, l = synthetic.make_batch(8, channels, size, first_idx=11 + 8 * k, with_boxes=True)
        batches.append({"img": torch.from_numpy(x).cuda(), "boxes": [torch.from_numpy(v).cuda() for v in b],
                        "labels": [torch.from_numpy(v).cuda() for v in l]})
    runs = []
    for graph in (False, True):
        model = LSSD3D(n_classes=2, input_channels=channels, input_size=size, threshold=[0.1, 0.2], lr=1e-3)
        model.load_state_dict(sd)
        model = model.cuda().train()
        model.use_cuda_graph = graph
        losses = torch.stack([model.fit_step(batch) for batch in batches])
        flat = model.train_engine().flat
        runs.append([losses, flat.param, flat.exp_avg, flat.exp_avg_sq, flat.status,
                     *(b for _, b in sorted(model.named_buffers()))])
    eager, captured = runs
    assert torch.isfinite(eager[0]).all()
    for name, e, c in zip(["losses", "param", "exp_avg", "exp_avg_sq", "status", "buffers"], eager, captured):
        assert _bit_equal(e, c), name


def test_nan_through_captured_inference_steps():
    """A NaN voxel raises the reference's NaN exception through the captured ``predict_step``, ``predict_batches`` and
    ``predict_scans``; the next clean call on the same plans returns the detections of before."""
    from mslesions3d_b200.ssd3d import LSSD3D
    size = (48, 48, 48)
    model = LSSD3D(n_classes=2, input_channels=1, input_size=size, min_score=0.35, top_k=30)
    model.load_state_dict(O.random_state_dict(1, seed=5))
    model = model.cuda().eval()
    x = torch.from_numpy(synthetic.make_batch(2, 1, size, first_idx=3))
    scans = torch.from_numpy(synthetic.make_batch(2, 1, (64, 56, 64), first_idx=7))
    bad_x, bad_scans = x.clone(), scans.clone()
    bad_x[1, 0, 20, 21, 22] = float("nan")
    bad_scans[0, 0, 40, 30, 20] = float("nan")
    steps = {
        "predict_step": lambda v: model.predict_step({"img": v.cuda()}),
        "predict_batches": lambda v: list(model.predict_batches([{"img": v.pin_memory()}, {"img": v.cuda()}])),
        "predict_scans": lambda v: model.predict_scans(v, overlap=0.5),
    }
    inputs = {"predict_step": (x, bad_x), "predict_batches": (x, bad_x), "predict_scans": (scans, bad_scans)}
    with torch.no_grad():
        before = {name: run(inputs[name][0]) for name, run in steps.items()}
        for name, run in steps.items():
            clean, bad = inputs[name]
            with pytest.raises(Exception, match="NaN error again in the base network"):
                run(bad)
            assert _same(run(clean), before[name]), name
