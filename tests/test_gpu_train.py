"""GPU parity of the training-step kernels (train-mode BatchNorm, conv weight / data gradients, Adam) and of
the whole ``LSSD3D.training_step`` / ``fit_step`` against torch-CPU autograd (the reference's own mechanism,
ssd3d.py:467-531) on identical inputs.

Tolerances (floating point; stated per BASELINE.json north_star):
  * one kernel vs fp32 autograd on the SAME bf16-rounded inputs: bf16 outputs within one bf16 ulp of the fp32
    result (accumulation order may flip the last bit), fp32 reductions (weight / BN-parameter gradients)
    within 2e-3 relative L2 error;
  * whole network gradients vs the oracle that emulates the product path's bf16 storage points (forward
    activations AND activation gradients): relative L2 error of the whole gradient (all parameters
    concatenated) <= 0.12; per parameter cosine >= 0.90, and <= 2 % relative error where nothing has been
    amplified yet (class heads, the BatchNorm right under each head).  The step is ill-conditioned by construction: batch-statistic BN over the few voxels of the deep maps amplifies
    a 1-ulp bf16 flip of an activation ~70x, and the fp32 and the bf16-emulating oracle differ from EACH OTHER
    by 25-40 % on the same inputs; the L1 localisation gradient is a sign function, so with a handful of
    positive priors one flipped sign moves a loc-head gradient by tens of percent.  The kernels are therefore
    held to the emulating oracle (same rounding points) and the per-kernel tests above carry the tight bounds;
  * vs the fp32 oracle: cosine >= 0.85 per parameter, losses within 2 %.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import ssd3d_oracle as O
from mslesions3d_b200 import synthetic
from tests import bench_shapes as S

pytestmark = pytest.mark.gpu


def _ops():
    from mslesions3d_b200 import ops
    return ops


def bf16r(t):
    return t.to(torch.bfloat16).float()


def to_cl(x):
    return x.cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)


def assert_bf16_close(got, want, what, ulps=1.0, frac_limit=0.03):
    got, want = got.float().cpu(), want.float().cpu()
    assert got.shape == want.shape, "%s: shape %s vs %s" % (what, tuple(got.shape), tuple(want.shape))
    diff = (got - want).abs()
    scale = float(want.abs().max())
    tol = ulps * (2.0 ** -7) * torch.clamp(want.abs(), min=scale * 2.0 ** -6)
    bad = diff > tol
    assert not bool(bad.any()), "%s: %d/%d beyond %.1f bf16 ulp, max diff %.4g at ref %.4g" % (
        what, int(bad.sum()), bad.numel(), ulps, float(diff.max()), float(want.flatten()[diff.argmax()]))


def rel_l2(got, want):
    got, want = got.float().cpu().flatten(), want.float().cpu().flatten()
    return float((got - want).norm() / want.norm().clamp(min=1e-20))


# ---------------------------------------------------------------------------------------------------
# train-mode BatchNorm + ReLU, forward and backward
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,c,size", S.extend(
    [(2, 32, (9, 10, 11)), (3, 64, (8, 8, 8)), (1, 128, (5, 6, 7)), (2, 512, (2, 2, 2)), (4, 256, (3, 3, 3)),
     (2, 32, (24, 24, 24)),
     # the cluster kernel takes up to 8192 rows (csrc/bn_unit.cu:634-636): the C3 tail, 4096 and 4352 rows
     (16, 256, (6, 6, 6)), (1, 32, (16, 16, 16)), (1, 32, (16, 16, 17))],
    # every BatchNorm input of the benchmarked training step (1.77 M rows of the stem down to the 432 of f7), then
    # both sides of the cluster / tile and register-kept / streamed switches
    S.bn_shapes(S.TRAIN), S.BN_BOUNDARY, S.BN_BOUNDARY_PASSES))
def test_bn_train_relu_forward_backward(n, c, size):
    ops = _ops()
    g = torch.Generator().manual_seed(c + n)
    z = bf16r(torch.randn((n, c) + size, generator=g) * 1.5 + 0.3 * torch.randn(1, c, 1, 1, 1, generator=g))
    bn = torch.nn.BatchNorm3d(c)
    with torch.no_grad():
        bn.weight.copy_(0.5 + torch.rand(c, generator=g))
        bn.bias.copy_(0.2 * torch.randn(c, generator=g))
        bn.running_mean.copy_(0.1 * torch.randn(c, generator=g))
        bn.running_var.copy_(0.5 + torch.rand(c, generator=g))
    ref = torch.nn.BatchNorm3d(c)
    ref.load_state_dict(bn.state_dict())
    ref.train()
    zr = z.clone().requires_grad_(True)
    want = F.relu(ref(zr))
    ga = bf16r(torch.randn(want.shape, generator=g))
    want.backward(ga)

    bn = bn.cuda().train()
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    a, st = ops.bn_train_relu(to_cl(z), bn, flag)
    assert a.dtype == torch.bfloat16 and a.is_contiguous(memory_format=torch.channels_last_3d)
    assert_bf16_close(a, bf16r(want.detach()), "bn forward")
    torch.testing.assert_close(bn.running_mean.cpu(), ref.running_mean, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(bn.running_var.cpu(), ref.running_var, rtol=1e-5, atol=1e-6)
    assert int(bn.num_batches_tracked) == 1 and int(flag) == 0

    dgamma = torch.empty(c, device="cuda")
    dbeta = torch.empty(c, device="cuda")
    dz = ops.bn_relu_backward(to_cl(z), to_cl(ga), st, dgamma, dbeta)
    assert rel_l2(dgamma, ref.weight.grad) < 2e-3 and rel_l2(dbeta, ref.bias.grad) < 2e-3
    assert_bf16_close(dz, bf16r(zr.grad), "bn backward dz", ulps=2.0)
    # bit-reproducible: the two-stage reductions have a fixed order
    dg2, db2 = torch.empty_like(dgamma), torch.empty_like(dbeta)
    ops.bn_relu_backward(to_cl(z), to_cl(ga), st, dg2, db2)
    assert torch.equal(dg2, dgamma) and torch.equal(db2, dbeta)


@pytest.mark.parametrize("n,c,size", S.extend(
    [(16, 32, (24, 24, 24)), (4, 32, (48, 48, 48)), (16, 64, (12, 12, 12)), (16, 1024, (3, 3, 3)), (16, 512, (6, 6, 6)),
     (16, 128, (6, 6, 6)), (1, 32, (1, 1, 3)), (3, 128, (7, 5, 3)), (16, 256, (12, 12, 12)),
     # more than 32768 rows: the grid-barrier kernel, C/8 = 32, 64, 128
     (1, 256, (34, 33, 31)), (1, 512, (33, 32, 32)), (2, 1024, (17, 32, 32))],
    S.bn_shapes(S.TRAIN), S.BN_BOUNDARY))
def test_bn_single_launch_matches_three_launch_passes(n, c, size):
    """csrc/bn_unit.cu (one launch, grid barriers) against the three-launch passes of train.cu on the same inputs:
    same statistics to fp32 rounding, same activations / gradients to 1 bf16 ulp; repeated launches (the barrier
    words are reused) are bit-identical; the launch counter shows which path ran."""
    ops = _ops()
    g = torch.Generator().manual_seed(7 * c + n)
    z = to_cl(bf16r(torch.randn((n, c) + size, generator=g) * 1.3 + 0.4 * torch.randn(1, c, 1, 1, 1, generator=g)))
    ga = to_cl(bf16r(torch.randn((n, c) + size, generator=g)))
    res = {}
    for mode in ("0", "1", "1"):
        fwd, bwd = (ops.bn_train_relu, ops.bn_relu_backward) if mode == "1" else \
            (ops._bn_train_relu_passes, ops._bn_relu_backward_passes)
        bn = torch.nn.BatchNorm3d(c)
        with torch.no_grad():
            bn.weight.copy_(0.5 + torch.rand(c, generator=torch.Generator().manual_seed(c)))
            bn.bias.copy_(0.2 * torch.randn(c, generator=torch.Generator().manual_seed(c + 1)))
        bn = bn.cuda().train()
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        before = ops.LAUNCHES[0]
        a, st = fwd(z, bn, flag)
        assert ops.LAUNCHES[0] - before == (1 if mode == "1" else 3)
        dgamma, dbeta = torch.empty(c, device="cuda"), torch.empty(c, device="cuda")
        dz = bwd(z, ga.clone(), st, dgamma, dbeta)
        torch.cuda.synchronize()
        cur = dict(a=a, dz=dz, dgamma=dgamma, dbeta=dbeta, scale=st.scale, shift=st.shift, mean=st.mean,
                   invstd=st.invstd, rm=bn.running_mean.clone(), rv=bn.running_var.clone(), flag=int(flag),
                   nbt=int(bn.num_batches_tracked))
        if mode == "1" and "1" in res:
            for k in ("a", "dz", "dgamma", "dbeta", "scale", "shift", "mean", "invstd", "rm", "rv"):
                assert torch.equal(cur[k], res["1"][k]), "single-launch path not reproducible: " + k
        res[mode] = cur
    three, one = res["0"], res["1"]
    assert one["flag"] == 0 and one["nbt"] == 1
    for k in ("scale", "shift", "mean", "invstd", "rm", "rv"):
        torch.testing.assert_close(one[k], three[k], rtol=2e-6, atol=1e-6)
    assert rel_l2(one["dgamma"], three["dgamma"]) < 1e-5 and rel_l2(one["dbeta"], three["dbeta"]) < 1e-5
    assert_bf16_close(one["a"], three["a"], "single-launch bn forward")
    assert_bf16_close(one["dz"], three["dz"], "single-launch bn backward")


def test_bn_train_nan_sets_flag():
    ops = _ops()
    z = torch.randn(1, 32, 4, 4, 4)
    z[0, 3, 1, 1, 1] = float("nan")
    bn = torch.nn.BatchNorm3d(32).cuda().train()
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.bn_train_relu(to_cl(z), bn, flag)
    assert int(flag) & 1


# ---------------------------------------------------------------------------------------------------
# pointwise conv: raw forward, data gradient, weight gradient
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout,n,size", S.extend(
    [(32, 64, 2, (12, 12, 12)), (64, 128, 2, (6, 7, 5)), (128, 128, 1, (6, 6, 6)), (128, 256, 3, (3, 3, 3)),
     (256, 512, 2, (2, 2, 2)), (512, 512, 1, (3, 2, 2)), (32, 64, 1, (37, 5, 3))],
    # every pointwise unit of the benchmarked training step (f1: M = 221184)
    [(u.cin, u.cout, u.n, u.size) for u in S.table(S.TRAIN)["pw"]]))
def test_pointwise_raw_dgrad_wgrad(cin, cout, n, size):
    ops = _ops()
    g = torch.Generator().manual_seed(cin + cout)
    x = bf16r(torch.randn((n, cin) + size, generator=g)).requires_grad_(True)
    w = bf16r(torch.randn((cout, cin, 1, 1, 1), generator=g) * (cin ** -0.5)).requires_grad_(True)
    y = F.conv3d(x, w)
    gy = bf16r(torch.randn(y.shape, generator=g))
    y.backward(gy)
    wp = ops.pack_pw_weight(w.detach().cuda())
    got = ops.pwconv_raw(to_cl(x.detach()), wp)
    assert_bf16_close(got, bf16r(y.detach()), "pw raw")
    m = n * size[0] * size[1] * size[2]
    dx = torch.empty_like(to_cl(x.detach()))
    ops.pw_gemm_raw(m, to_cl(gy), wp.t().contiguous(), dx)
    assert_bf16_close(dx, bf16r(x.grad), "pw dgrad")
    dw = torch.empty((cout, cin, 1, 1, 1), device="cuda")
    ops.pwconv_wgrad(to_cl(gy), to_cl(x.detach()), dw)
    assert rel_l2(dw, w.grad) < 2e-3, rel_l2(dw, w.grad)
    dw2 = torch.empty_like(dw)
    ops.pwconv_wgrad(to_cl(gy), to_cl(x.detach()), dw2)
    assert torch.equal(dw, dw2)


# ---------------------------------------------------------------------------------------------------
# depthwise conv
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,n,size,stride", S.extend(
    [(32, 2, (12, 12, 12), 2), (64, 1, (9, 7, 11), 2), (128, 2, (6, 6, 6), 1), (256, 1, (5, 4, 3), 2),
     (512, 2, (2, 2, 2), 1), (128, 1, (7, 8, 9), 1), (32, 1, (24, 24, 24), 2),
     # large enough for the TMA halo-tile forward / weight-gradient kernels
     (32, 2, (32, 32, 32), 2), (64, 1, (24, 20, 28), 2), (128, 1, (16, 16, 16), 1), (32, 1, (19, 21, 17), 2),
     (96, 2, (9, 12, 10), 1)],
    # every depthwise unit of the benchmarked training step (f1-f3 halo tiles, f4-f7 the CUDA-core weight gradient),
    # then both sides of the halo-tile / CUDA-core switch and the ends of the CUDA-core plan
    [(u.c, u.n, u.size, u.stride) for u in S.table(S.TRAIN)["dw"]], S.DW_BOUNDARY))
def test_depthwise_raw_dgrad_wgrad(c, n, size, stride):
    ops = _ops()
    g = torch.Generator().manual_seed(c + stride)
    x = bf16r(torch.randn((n, c) + size, generator=g)).requires_grad_(True)
    w = bf16r(torch.randn((c, 1, 3, 3, 3), generator=g) * 0.3).requires_grad_(True)
    y = F.conv3d(x, w, None, stride, 1, 1, c)
    gy = bf16r(torch.randn(y.shape, generator=g))
    y.backward(gy)
    wd = ops.pack_dw_weight(w.detach().cuda())
    got = ops.dwconv3d_raw(to_cl(x.detach()), wd, stride)
    assert_bf16_close(got, bf16r(y.detach()), "dw raw")
    dx = ops.dwconv3d_dgrad(to_cl(gy), wd, to_cl(x.detach()), stride)
    assert_bf16_close(dx, bf16r(x.grad), "dw dgrad")
    dw = torch.empty((c, 1, 3, 3, 3), device="cuda")
    ops.dwconv3d_wgrad(to_cl(gy), to_cl(x.detach()), stride, dw)
    assert rel_l2(dw, w.grad) < 2e-3, rel_l2(dw, w.grad)


# ---------------------------------------------------------------------------------------------------
# stem conv
# ---------------------------------------------------------------------------------------------------
# the benchmarked training step's stem (fit_step on fp32 batches, fit_epoch on bf16 ones)
BENCH_STEM = [(u.cin, u.n, u.size, u.stride_d, dt) for u in S.table(S.TRAIN)["stem"]
              for dt in (torch.float32, torch.bfloat16)]


@pytest.mark.parametrize("cin,n,size,sd,dtype", S.extend(
    [(1, 2, (16, 16, 16), 2, torch.float32), (2, 1, (12, 16, 24), 1, torch.bfloat16), (1, 1, (9, 11, 13), 2, torch.float32),
     (3, 2, (8, 8, 8), 2, torch.float32), (4, 1, (8, 16, 8), 1, torch.bfloat16), (1, 2, (48, 48, 48), 2, torch.float32),
     # large enough for the halo-tile kernel (>= 148 tiles of 128 voxels)
     (2, 2, (40, 44, 48), 1, torch.bfloat16), (3, 2, (33, 50, 56), 2, torch.float32),
     (4, 3, (32, 48, 40), 2, torch.bfloat16), (1, 3, (31, 45, 72), 1, torch.bfloat16),
     (2, 1, (64, 64, 64), 2, torch.float32)],
    BENCH_STEM, S.STEM_WGRAD_BOUNDARY))
def test_stem_raw_wgrad(cin, n, size, sd, dtype):
    ops = _ops()
    g = torch.Generator().manual_seed(cin * 7 + sd)
    x = bf16r(torch.randn((n, cin) + size, generator=g))
    w = bf16r(torch.randn((32, cin, 3, 3, 3), generator=g) * 0.2).requires_grad_(True)
    y = F.conv3d(x, w, None, (sd, 2, 2), 1)
    gy = bf16r(torch.randn(y.shape, generator=g))
    y.backward(gy)
    xd = x.to(dtype).cuda()
    got = ops.stem_conv_raw(xd, ops.pack_stem_weight(w.detach().cuda()), sd)
    assert_bf16_close(got, bf16r(y.detach()), "stem raw")
    dw = torch.empty((32, cin, 3, 3, 3), device="cuda")
    ops.stem_wgrad(to_cl(gy), xd, sd, dw)
    assert rel_l2(dw, w.grad) < 2e-3, rel_l2(dw, w.grad)


@pytest.mark.parametrize("cin,n,size,sd,dtype", S.extend(
    [(1, 2, (64, 64, 64), 2, torch.float32), (2, 1, (48, 64, 80), 2, torch.bfloat16), (1, 3, (40, 48, 56), 1, torch.float32)],
    BENCH_STEM, S.STEM_WGRAD_BOUNDARY))
def test_stem_unit_backward_fused_equals_two_step(cin, n, size, sd, dtype):
    """ssd3d_bn_unit_bwd(dz = NULL) + ssd3d_stem_wgrad_bn (the BatchNorm + ReLU backward applied to the gradient rows
    inside the weight-gradient kernel, dz never written) against bn_relu_backward + stem_wgrad: bit-identical.  Below
    M = 128 * 148 output voxels the fused path declines without launching anything."""
    ops = _ops()
    g = torch.Generator().manual_seed(11 * cin + n)
    x = bf16r(torch.randn((n, cin) + size, generator=g)).to(dtype).cuda()
    w = bf16r(torch.randn((32, cin, 3, 3, 3), generator=g) * 0.2).cuda()
    z = ops.stem_conv_raw(x, ops.pack_stem_weight(w), sd)
    bn = torch.nn.BatchNorm3d(32)
    with torch.no_grad():
        bn.weight.copy_(0.5 + torch.rand(32, generator=g))
        bn.bias.copy_(0.2 * torch.randn(32, generator=g))
    bn = bn.cuda().train()
    a, st = ops.bn_train_relu(z, bn, None)
    ga = to_cl(bf16r(torch.randn(tuple(z.shape), generator=g)))
    dg1, db1, dw1 = torch.empty(32, device="cuda"), torch.empty(32, device="cuda"), torch.empty_like(w)
    before = ops.LAUNCHES[0]
    fused = ops.stem_unit_backward(z, ga, st, dg1, db1, x, sd, dw1)
    # the fused path runs on the TMA tile kernel, which takes M >= 128 * 148 rows (csrc/train.cu:1507, ops.py:858)
    m = z.numel() // 32
    if m < S.STEM_WGRAD_TILE_ROWS:
        assert not fused and ops.LAUNCHES[0] == before, "fused path took M = %d rows" % m
        return
    assert fused, "fused path refused a shape it should take"
    dg2, db2, dw2 = torch.empty(32, device="cuda"), torch.empty(32, device="cuda"), torch.empty_like(w)
    dz = ops.bn_relu_backward(z, ga.clone(), st, dg2, db2)
    ops.stem_wgrad(dz, x, sd, dw2)
    assert torch.equal(dg1, dg2) and torch.equal(db1, db2)
    assert torch.equal(dw1, dw2), float((dw1 - dw2).abs().max())
    assert bool(torch.isfinite(dw1).all()) and float(dw1.abs().max()) > 0


# ---------------------------------------------------------------------------------------------------
# SSD heads: gradient rows, bias / weight / data gradients
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,n,size,ncls", S.extend(
    [(128, 2, (6, 6, 6), 2), (256, 2, (3, 3, 3), 2), (512, 3, (2, 2, 2), 2), (128, 1, (5, 7, 4), 2),
     (128, 1, (12, 12, 12), 2),
     # n_classes >= 3: bpl*(6+n_classes) > 16 -> several 16-column groups
     (128, 2, (6, 6, 6), 3), (256, 1, (4, 3, 5), 5), (128, 1, (5, 5, 5), 11),
     # batches whose maps hold a 64-voxel box: the tcgen05 weight gradient
     # (the C3 heads at batch 16; C = 64: half-empty channel tile; ragged boxes)
     (256, 16, (3, 3, 3), 2), (256, 16, (6, 6, 6), 2), (512, 16, (3, 3, 3), 2), (64, 2, (8, 8, 8), 2),
     (192, 5, (5, 3, 7), 3)],
    # every head of the benchmarked training step (two boxes per location, as the body below assumes)
    [(u.c, u.n, u.size, 2) for u in S.table(S.TRAIN)["head"]]))
def test_head_backward(c, n, size, ncls):
    ops = _ops()
    bpl = 2
    g = torch.Generator().manual_seed(c + size[0])
    x = bf16r(torch.randn((n, c) + size, generator=g)).requires_grad_(True)
    lw = bf16r(torch.randn((bpl * 6, c, 3, 3, 3), generator=g) * 0.05).requires_grad_(True)
    cw = bf16r(torch.randn((bpl * ncls, c, 3, 3, 3), generator=g) * 0.05).requires_grad_(True)
    lb = torch.zeros(bpl * 6, requires_grad=True)
    cb = torch.zeros(bpl * ncls, requires_grad=True)
    v = size[0] * size[1] * size[2]
    p_total, off = v * bpl + 10, 6          # this layer's priors sit at an offset inside a longer prior list
    locs = F.conv3d(x, lw, lb, 1, 1).permute(0, 2, 3, 4, 1).reshape(n, -1, 6)
    scores = F.conv3d(x, cw, cb, 1, 1).permute(0, 2, 3, 4, 1).reshape(n, -1, ncls)
    dlocs = torch.randn((n, p_total, 6), generator=g)
    dscores = torch.randn((n, p_total, ncls), generator=g)
    # the kernels round the head gradient rows to bf16; give autograd the same values
    dl_used = bf16r(dlocs[:, off:off + v * bpl])
    ds_used = bf16r(dscores[:, off:off + v * bpl])
    torch.autograd.backward([locs, scores], [dl_used, ds_used])

    dbl, dbc = torch.empty(bpl * 6, device="cuda"), torch.empty(bpl * ncls, device="cuda")
    dO = ops.head_grad_pack(dlocs.cuda(), dscores.cuda(), n, size[0], size[1], size[2], bpl, ncls, off, dbl, dbc)
    # bias gradients are column sums of the UNROUNDED fp32 rows
    torch.testing.assert_close(dbl.cpu(), dlocs[:, off:off + v * bpl].reshape(-1, bpl * 6).sum(0), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dbc.cpu(), dscores[:, off:off + v * bpl].reshape(-1, bpl * ncls).sum(0), rtol=1e-4,
                               atol=1e-4)
    want_rows = torch.cat([dl_used.reshape(n * v, bpl * 6), ds_used.reshape(n * v, bpl * ncls)], 1)
    groups = (want_rows.shape[1] + 15) // 16
    want_rows = F.pad(want_rows, (0, groups * 16 - want_rows.shape[1]))
    assert tuple(dO.shape) == (groups, n * v, 16)
    assert torch.equal(dO.float().cpu().permute(1, 0, 2).reshape(n * v, groups * 16), want_rows)
    dwl, dwc = torch.empty_like(lw, device="cuda"), torch.empty_like(cw, device="cuda")
    ops.head_wgrad(dO, to_cl(x.detach()), bpl * 6, bpl * ncls, dwl, dwc)
    assert rel_l2(dwl, lw.grad) < 2e-3 and rel_l2(dwc, cw.grad) < 2e-3, (rel_l2(dwl, lw.grad), rel_l2(dwc, cw.grad))
    wpk, _ = ops.pack_head_weight(lw.detach().cuda(), lb.detach().cuda(), cw.detach().cuda(), cb.detach().cuda())
    # all 16-column groups accumulate in fp32 inside one launch: one rounding, whatever n_classes
    dx = ops.head_dgrad(dO, wpk, to_cl(x.detach()), n_cols=bpl * (6 + ncls))
    assert_bf16_close(dx, bf16r(x.grad), "head dgrad")
    add = bf16r(torch.randn(x.shape, generator=g))
    dx2 = ops.head_dgrad(dO, wpk, to_cl(x.detach()), addend=to_cl(add), n_cols=bpl * (6 + ncls))
    assert_bf16_close(dx2, bf16r(x.grad + add), "head dgrad + addend", ulps=1.5)


# ---------------------------------------------------------------------------------------------------
# Adam
# ---------------------------------------------------------------------------------------------------
def test_adam_matches_torch():
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    n, bias_start = 10007, 8000
    p0 = torch.randn(n, generator=g)
    pw = p0[:bias_start].clone().requires_grad_(True)
    pb = p0[bias_start:].clone().requires_grad_(True)
    lr = 1e-3
    opt = torch.optim.Adam([{"params": [pb], "lr": 2 * lr}, {"params": [pw]}], lr=lr, weight_decay=0.0005)
    p = p0.clone().cuda()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for step in range(1, 6):
        grad = torch.randn(n, generator=g) * (0.1 if step % 2 else 3.0)
        pw.grad, pb.grad = grad[:bias_start].clone(), grad[bias_start:].clone()
        opt.step()
        ops.adam_step(p, (grad * 4).cuda(), m, v, bias_start, lr, 2 * lr, step, weight_decay=0.0005, grad_scale=0.25)
        want = torch.cat([pw.detach(), pb.detach()])
        torch.testing.assert_close(p.cpu(), want, rtol=2e-6, atol=2e-7)


def test_adam_dev_state_schedule_and_skip():
    """The graph-capturable step (ssd3d_adam_step_dev): step counter, bias correction and the reference's
    CosineAnnealingLR(T_max=40) (scheduler stepped BEFORE the optimizer step of the same batch, ssd3d.py:525-527)
    all on the device; a non-finite gradient skips the update and advances neither counter nor schedule."""
    ops = _ops()
    g = torch.Generator().manual_seed(4)
    n, bias_start = 5003, 4000
    p0 = torch.randn(n, generator=g)
    pw = p0[:bias_start].clone().requires_grad_(True)
    pb = p0[bias_start:].clone().requires_grad_(True)
    lr = 1e-3
    opt = torch.optim.Adam([{"params": [pb], "lr": 2 * lr}, {"params": [pw]}], lr=lr, weight_decay=0.0005)
    sch = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=40)
    p = p0.clone().cuda()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    state = torch.zeros(4, dtype=torch.int32, device="cuda")
    scal = torch.zeros(8, dtype=torch.float32, device="cuda")
    import warnings
    for step in range(1, 46):
        grad = torch.randn(n, generator=g)
        if step in (3, 17):                  # a batch without positives: NaN gradient -> skipped, nothing advances
            bad = grad.clone()
            bad[11] = float("nan")
            before = p.clone()
            ops.adam_step_dev(p, bad.cuda(), m, v, bias_start, lr, state, scal, t_max=40, weight_decay=0.0005)
            assert torch.equal(p, before)
        pw.grad, pb.grad = grad[:bias_start].clone(), grad[bias_start:].clone()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sch.step()                       # ssd3d.py:525-527: before the optimizer step
        opt.step()
        ops.adam_step_dev(p, (grad * 2).cuda(), m, v, bias_start, lr, state, scal, t_max=40, weight_decay=0.0005,
                          grad_scale=0.5)
        want = torch.cat([pw.detach(), pb.detach()])
        torch.testing.assert_close(p.cpu(), want, rtol=3e-6, atol=3e-7, msg="step %d" % step)
    assert state.cpu().tolist()[:3] == [0, 2, 45]


# ---------------------------------------------------------------------------------------------------
# whole network
# ---------------------------------------------------------------------------------------------------
def _train_case(channels=1, size=(64, 64, 64), batch=4, seed=5):
    sd = O.random_state_dict(channels, seed=seed)
    x, b, l = synthetic.make_batch(batch, channels, size, first_idx=11, with_boxes=True)
    boxes = [torch.from_numpy(v) for v in b]
    labels = [torch.from_numpy(v) for v in l]
    return sd, torch.from_numpy(x), boxes, labels


def _model(sd, channels, size, **kw):
    from mslesions3d_b200.ssd3d import LSSD3D
    model = LSSD3D(n_classes=2, input_channels=channels, input_size=size, **kw)
    model.load_state_dict(sd)
    return model.cuda().train()


@pytest.mark.parametrize("channels,size,batch", [(1, (64, 64, 64), 8), (2, (64, 64, 64), 6)])
def test_training_step_gradients(channels, size, batch):
    sd, x, boxes, labels = _train_case(channels, size, batch)
    thr = [0.1, 0.2]
    model = _model(sd, channels, size, threshold=thr, alpha=1.0)
    out = model.training_step({"img": x, "boxes": boxes, "labels": labels, "subject": list(range(batch))})
    loss = out["loss"]
    loss.backward()
    pri = O.prior_boxes(size, in_channels=channels)
    emu = O.train_step_grads(sd, x, boxes, labels, pri, thr, emulate_bf16=True)
    f32 = O.train_step_grads(sd, x, boxes, labels, pri, thr)
    # losses
    conf, loc = float(out["log"]["train_conf_loss"]), float(out["log"]["train_loc_loss"])
    assert abs(conf - float(emu["conf"])) <= 5e-3 * abs(float(emu["conf"])), (conf, float(emu["conf"]))
    assert abs(loc - float(emu["loc"])) <= 5e-3 * abs(float(emu["loc"])), (loc, float(emu["loc"]))
    assert abs(conf - float(f32["conf"])) <= 2e-2 * abs(float(f32["conf"]))
    # BN buffers after the step
    for k, v in emu["running"].items():
        got = model.state_dict()[k].cpu()
        if k.endswith("num_batches_tracked"):
            assert int(got) == int(v) == 1
        else:
            torch.testing.assert_close(got, v, rtol=2e-2, atol=2e-3, msg=k)
    worst, num, den = (0.0, None), 0.0, 0.0
    params = dict(model.named_parameters())
    assert params["rescale_factors"].grad is None
    for k, want in emu["grads"].items():
        if want is None:
            continue
        got = params[k].grad
        assert got is not None and got.shape == want.shape, k
        if float(want.norm()) == 0.0:
            assert float(got.norm()) == 0.0, k
            continue
        r = rel_l2(got, want)
        cos = float((got.cpu().flatten() * want.flatten()).sum() / (got.norm().cpu() * want.norm()))
        worst = max(worst, (r, k))
        num += float((got.cpu() - want).norm()) ** 2
        den += float(want.norm()) ** 2
        print("%-40s rel L2 %.4f cos %.5f" % (k, r, cos))
        # Two bf16 pipelines (this one and the emulating oracle) differ where a rounded pre-activation lands on the
        # other side of a ReLU or an L1 residual changes sign; measured on B200 (profiles/r02_train_parity.txt):
        # backbone tensors <= 0.25, the loc head of a layer with a handful of positives <= 0.38, class heads
        # <= 0.006.  The exact per-stage check (<= 2e-3 everywhere) is tests/test_gpu_train_insitu.py.
        limit = 0.45 if k.startswith("pred_convs.loc_convs") else 0.35
        assert r <= limit and cos >= 0.92, "%s: rel L2 %.4f cos %.5f" % (k, r, cos)
        if k.startswith("pred_convs.cl_convs") or k.endswith(("3.bn2.weight", "5.bn2.weight", "7.bn2.weight")):
            # before any amplification: class-head gradients and the BN right under a head
            assert r <= 0.02, "%s: rel L2 %.4f" % (k, r)
        w32 = f32["grads"][k]
        cos32 = float((got.cpu().flatten() * w32.flatten()).sum() / (got.norm().cpu() * w32.norm()))
        assert cos32 >= 0.85, "%s: cosine vs fp32 oracle %.4f" % (k, cos32)
    print("worst rel L2 vs emulating oracle: %.4f (%s); whole gradient: %.4f" % (worst + ((num / den) ** 0.5,)))
    assert (num / den) ** 0.5 <= 0.02          # measured 0.0014 / 0.0022


def test_training_step_is_reproducible_and_eval_still_works():
    sd, x, boxes, labels = _train_case(1, (64, 64, 64), 2)
    grads = []
    for _ in range(2):
        model = _model(sd, 1, (64, 64, 64), threshold=[0.1, 0.2])
        out = model.training_step({"img": x, "boxes": boxes, "labels": labels})
        out["loss"].backward()
        grads.append({k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None})
    for k in grads[0]:
        assert torch.equal(grads[0][k], grads[1][k]), k
    model.eval()
    with torch.no_grad():
        b, l, s = model.predict_step({"img": x}, 0)
    assert len(b) == 2


@pytest.mark.parametrize("graph", [False, True])
def test_fit_step_follows_reference_optimizer(graph):
    """Three fused steps (forward, loss, backward, Adam with cosine schedule) vs the fp32 oracle driven the way
    pytorch-lightning drives the reference.  Adam normalises the gradient, so a parameter moves by about lr
    per step whatever the gradient's scale: compare the parameter DELTAS."""
    size, channels, lr = (64, 64, 64), 1, 1e-3
    sd, x, boxes, labels = _train_case(channels, size, 8)
    thr = [0.1, 0.2]
    model = _model(sd, channels, size, threshold=thr, lr=lr)
    model.use_cuda_graph = graph
    batch = {"img": x, "boxes": boxes, "labels": labels}
    losses = [model.fit_step(batch).cpu() for _ in range(3)]
    pri = O.prior_boxes(size, in_channels=channels)
    want_sd, want_losses = O.fit_steps(sd, [(x, boxes, labels)] * 3, pri, thr, lr)
    for got, want in zip(losses, want_losses):
        assert abs(float(got[0]) - want[0]) <= 0.05 * abs(want[0]), (got, want)
        assert abs(float(got[1]) - want[1]) <= 0.05 * abs(want[1]), (got, want)
    assert float(losses[2][0]) < float(losses[0][0])       # the confidence loss goes down
    got_sd = model.state_dict()
    assert torch.equal(got_sd["rescale_factors"].cpu(), sd["rescale_factors"])
    for k, v0 in sd.items():
        if not v0.is_floating_point() or k == "rescale_factors" or "running" in k:
            continue
        d_got = got_sd[k].cpu().float() - v0
        d_want = want_sd[k] - v0
        cos = float((d_got.flatten() * d_want.flatten()).sum() / (d_got.norm() * d_want.norm()).clamp(min=1e-30))
        assert cos >= 0.70, "%s: update direction cosine %.3f" % (k, cos)
        assert 0.5 <= float(d_got.norm() / d_want.norm().clamp(min=1e-30)) <= 2.0, k
    # eval-mode inference after training uses the updated weights and running statistics
    model.eval()
    with torch.no_grad():
        locs, scores = model(x)
        el, es = O.forward({k: v.cpu() for k, v in got_sd.items()}, x, emulate_bf16=True)
    assert float((locs.cpu() - el).abs().max()) < 0.1 and float((scores.cpu() - es).abs().max()) < 0.1


def test_fit_step_skips_a_batch_without_positives():
    """No ground-truth box in the whole batch -> n_pos = 0 -> the MultiBox loss is 0/0 (the reference raises
    "Loss is NaN", ssd3d.py:938-940): the fused step must leave parameters and Adam moments untouched and count it."""
    sd, x, boxes, labels = _train_case(1, (64, 64, 64), 2)
    model = _model(sd, 1, (64, 64, 64), threshold=[0.1, 0.2], lr=1e-3)
    empty = {"img": x, "boxes": [torch.zeros((0, 6)) for _ in boxes], "labels": [torch.zeros((0,), dtype=torch.long) for _ in labels]}
    model.fit_step({"img": x, "boxes": boxes, "labels": labels})
    before = {k: v.clone() for k, v in model.state_dict().items() if "running" not in k and "num_batches" not in k}
    loss = model.fit_step(empty)
    assert not bool(torch.isfinite(loss).all())
    assert model.fit_skipped_steps() == 1
    after = model.state_dict()
    for k, v in before.items():
        assert torch.equal(after[k], v), k
    loss2 = model.fit_step({"img": x, "boxes": boxes, "labels": labels})
    assert bool(torch.isfinite(loss2).all()) and model.fit_skipped_steps() == 1
    assert any(not torch.equal(after[k], before[k]) for k in before)


def test_training_step_noncube_input_and_bf16_images():
    """Non-cubic volumes use stem stride (1,2,2) (ssd3d.py:60) and the x/y-swapped prior axes (SURVEY.md B3); the
    fused step also accepts bf16 images.  Losses against the bf16-emulating oracle, gradients by cosine."""
    size, channels = (32, 64, 48), 2
    sd = O.random_state_dict(channels, seed=8)
    x, b, l = synthetic.make_batch(4, channels, size, first_idx=3, with_boxes=True)
    x = torch.from_numpy(x)
    boxes, labels = [torch.from_numpy(v) for v in b], [torch.from_numpy(v) for v in l]
    thr = [0.1, 0.2]
    model = _model(sd, channels, size, threshold=thr)
    out = model.training_step({"img": x, "boxes": boxes, "labels": labels})
    out["loss"].backward()
    pri = O.prior_boxes(size, in_channels=channels)
    emu = O.train_step_grads(sd, x, boxes, labels, pri, thr, emulate_bf16=True)
    assert abs(float(out["log"]["train_conf_loss"]) - float(emu["conf"])) <= 5e-3 * abs(float(emu["conf"]))
    assert abs(float(out["log"]["train_loc_loss"]) - float(emu["loc"])) <= 5e-3 * abs(float(emu["loc"]))
    params = dict(model.named_parameters())
    num = den = 0.0
    for k, want in emu["grads"].items():
        if want is None or float(want.norm()) == 0.0:
            continue
        got = params[k].grad.cpu()
        num += float((got - want).norm()) ** 2
        den += float(want.norm()) ** 2
    assert (num / den) ** 0.5 <= 0.15, (num / den) ** 0.5
    # fused step on bf16 images: same first loss as on the fp32 images (the stem rounds fp32 inputs to bf16 itself)
    m1 = _model(sd, channels, size, threshold=thr, lr=1e-4)
    m2 = _model(sd, channels, size, threshold=thr, lr=1e-4)
    l1 = m1.fit_step({"img": x, "boxes": boxes, "labels": labels}).cpu()
    l2 = m2.fit_step({"img": x.to(torch.bfloat16), "boxes": boxes, "labels": labels}).cpu()
    assert torch.equal(l1, l2)
