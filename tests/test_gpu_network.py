"""GPU parity of the network kernels (stem, depthwise, pointwise tcgen05 GEMM, fused tcgen05 head) and of the
whole ``LSSD3D.forward`` against the CPU oracle and the golden outputs of the unmodified reference.

Tolerances (floating point, stated per BASELINE.json north_star "within a stated bf16/fp32 tolerance"):
  * single kernel vs oracle on identical bf16-rounded inputs, fp32 accumulate, bf16 stored output:
    |a - b| <= 2^-7 * max(|b|, 2^-6)  (one bf16 ulp; accumulation order may flip the last bit), and fewer
    than 2 % of elements may differ at all;
  * fp32 head outputs vs oracle on identical inputs: |a - b| <= 2e-3 * max(1, |b|) (K up to 13824 products);
  * whole network vs the bf16-emulating oracle: max abs error <= 0.06, mean abs error <= 6e-3;
  * whole network vs the fp32 reference golden: max abs error <= 0.25, mean abs error <= 0.03
    (bf16 storage of 16 activations deep; the oracle's own bf16 emulation differs from fp32 by the same amount).
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import ssd3d_oracle as O
from tests import bench_shapes as S
from tests.conftest import load_golden
from tests.golden import golden_inputs as GI

pytestmark = pytest.mark.gpu


def _ops():
    from mslesions3d_b200 import ops
    return ops


def bf16r(t):
    return t.to(torch.bfloat16).float()


def assert_bf16_close(got, want, what):
    got, want = got.float().cpu(), want.float().cpu()
    assert got.shape == want.shape, "%s: shape %s vs %s" % (what, tuple(got.shape), tuple(want.shape))
    diff = (got - want).abs()
    tol = (2.0 ** -7) * torch.clamp(want.abs(), min=2.0 ** -6)
    bad = diff > tol
    frac = float((diff > 0).float().mean())
    assert not bool(bad.any()), "%s: %d/%d beyond one bf16 ulp, max diff %.4g at ref %.4g" % (
        what, int(bad.sum()), bad.numel(), float(diff.max()), float(want.flatten()[diff.argmax()]))
    assert frac < 0.02, "%s: %.2f%% of elements differ" % (what, 100 * frac)


def to_cl(x_ncdhw):
    """CPU fp32 NCDHW -> CUDA channels-last-3d bf16 (logical NCDHW)."""
    return x_ncdhw.cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)


def rand_bn(c, g):
    scale = 0.5 + torch.rand(c, generator=g)
    shift = 0.2 * torch.randn(c, generator=g)
    return scale, shift


# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,size,sd,dtype,batch", [
    (1, (64, 64, 64), 2, torch.float32, 1),
    (2, (32, 48, 40), 1, torch.bfloat16, 2),
    (2, (17, 19, 23), 2, torch.float32, 2),
    (1, (40, 40, 40), 2, torch.bfloat16, 3),
    (3, (9, 16, 31), 1, torch.float32, 1),
    (2, (128, 128, 128), 2, torch.bfloat16, 1),    # the benchmark shape: tcgen05 path, 64-wide tiles
    (1, (96, 96, 96), 2, torch.float32, 1),        # fp32 TMA tile, 16-wide tiles
    (4, (16, 32, 24), 1, torch.float32, 2),        # K = 108 -> two k-blocks
    (3, (24, 24, 24), 2, torch.bfloat16, 1),
    (2, (6, 8, 8), 2, torch.bfloat16, 3),          # tile larger than the volume
    (2, (10, 22, 72), 2, torch.bfloat16, 2),       # banded-B kernel: ragged second row slot (Wo = 36), ragged H / D tiles
    (1, (12, 6, 128), 1, torch.bfloat16, 1),       # banded-B kernel: Ho = 3 -> 4 x 4 row slots, stride 1 along D
    (2, (33, 40, 96), 2, torch.bfloat16, 1),       # the training shape's row width (Wo = 48), odd depth
] + [(u.cin, u.size, u.stride_d, u.dtype, u.n) for u in S.table(S.INFER)["stem"]]     # the benchmark's batch of 8
  + S.STEM_FWD_BOUNDARY)                                                              # banded-B vs gather at W = 64k
def test_stem_conv(cin, size, sd, dtype, batch):
    ops = _ops()
    g = torch.Generator().manual_seed(cin * 100 + size[0])
    x = torch.randn((batch, cin) + size, generator=g)
    w = torch.randn((32, cin, 3, 3, 3), generator=g) * 0.2
    scale, shift = rand_bn(32, g)
    want = F.conv3d(bf16r(x), bf16r(w), None, (sd, 2, 2), 1)
    want = bf16r(F.relu(want * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1)))
    lib = ops._lib.load()
    kernels = [None, "simt"]             # None = the library's own choice
    if lib.ssd3d_stem_tc_supported(int(dtype == torch.bfloat16), cin, size[2]):
        kernels.append("tc")             # gather-based tcgen05 implicit GEMM
    if lib.ssd3d_stem_tz_supported(int(dtype == torch.bfloat16), cin, size[2]):
        kernels.append("tz")             # banded-B tcgen05 GEMM on raw TMA rows
    got = {}
    for kernel in kernels:
        got[kernel] = ops.stem_conv_bn_relu(x.to(dtype).cuda(), ops.pack_stem_weight(w.cuda()), scale.cuda(), shift.cuda(),
                                            sd, kernel=kernel)
        assert got[kernel].dtype == torch.bfloat16 and got[kernel].is_contiguous(memory_format=torch.channels_last_3d)
        assert_bf16_close(got[kernel], want, "stem %s" % (kernel or "auto"))
    # the library's own choice is the kernel the shape selects, bit for bit
    assert torch.equal(got[None], got[S.stem_kernel(dtype, cin, size[2])])


@pytest.mark.parametrize("c,size,stride,batch", [
    (32, (16, 16, 16), 2, 2),
    (32, (9, 11, 13), 2, 1),
    (64, (8, 8, 8), 2, 2),
    (128, (8, 8, 8), 1, 2),
    (128, (5, 6, 7), 1, 1),
    (256, (4, 4, 4), 2, 3),
    (512, (2, 2, 2), 1, 2),
    (512, (3, 3, 3), 1, 1),
    (40, (6, 5, 9), 1, 1),
    # maps large enough for the TMA halo-tile kernel (Wo >= 8): full and ragged tiles, several channel chunks
    (32, (32, 32, 32), 2, 2),
    (32, (17, 19, 21), 2, 1),
    (64, (16, 16, 16), 2, 3),
    (128, (8, 16, 12), 1, 2),
    (128, (9, 10, 11), 1, 1),
    (96, (7, 9, 17), 2, 2),
    (32, (64, 64, 64), 2, 1),
])
def test_depthwise_conv(c, size, stride, batch):
    ops = _ops()
    g = torch.Generator().manual_seed(c + size[0] + stride)
    x = bf16r(torch.randn((batch, c) + size, generator=g))
    w = torch.randn((c, 1, 3, 3, 3), generator=g) * 0.3
    scale, shift = rand_bn(c, g)
    want = F.conv3d(x, bf16r(w), None, stride, 1, 1, c)
    want = bf16r(F.relu(want * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1)))
    got = ops.dwconv3d_bn_relu(to_cl(x), ops.pack_dw_weight(w.cuda()), scale.cuda(), shift.cuda(), stride)
    assert_bf16_close(got, want, "depthwise")
    direct = ops.dwconv3d_bn_relu(to_cl(x), ops.pack_dw_weight(w.cuda()), scale.cuda(), shift.cuda(), stride,
                                  force_direct=True)
    assert_bf16_close(direct, want, "depthwise (direct kernel)")
    # both kernels accumulate the 27 taps in the same order in fp32: identical bits
    assert torch.equal(got, direct)


@pytest.mark.parametrize("cin,cout,size,batch", [
    (32, 64, (16, 16, 16), 2),     # BK = 32 (64-byte swizzle), one k-block
    (64, 128, (8, 8, 8), 2),       # BK = 64, one k-block
    (128, 128, (8, 8, 8), 1),
    (128, 256, (4, 4, 4), 2),      # M = 128
    (256, 256, (3, 3, 3), 2),      # M = 54: partial tile
    (256, 512, (2, 2, 2), 3),      # M = 24, several N tiles
    (512, 512, (4, 4, 4), 8),      # 8 k-blocks through a 4-deep ring
    (512, 1024, (3, 3, 3), 1),
    (96, 48, (5, 5, 5), 1),        # BK = 32, three k-blocks, Cout % 16 == 0 only
    # enough tiles for the persistent kernel (gemm_pw.cu): several tiles per CTA, ragged last tile, 1-8 k-blocks
    (32, 64, (40, 40, 40), 1),
    (64, 128, (32, 32, 32), 1),
    (64, 128, (31, 33, 17), 2),
    (128, 128, (16, 16, 16), 8),
    (256, 256, (24, 24, 24), 1),
    (512, 512, (16, 16, 16), 2),
    (128, 32, (30, 30, 30), 1),
])
def test_pointwise_conv_tcgen05(cin, cout, size, batch):
    ops = _ops()
    g = torch.Generator().manual_seed(cin + cout)
    x = bf16r(torch.randn((batch, cin) + size, generator=g))
    w = torch.randn((cout, cin, 1, 1, 1), generator=g) / (cin ** 0.5)
    scale, shift = rand_bn(cout, g)
    want = F.conv3d(x, bf16r(w))
    want = bf16r(F.relu(want * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1)))
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    got = ops.pwconv_bn_relu(to_cl(x), ops.pack_pw_weight(w.cuda()), scale.cuda(), shift.cuda(), flag)
    assert_bf16_close(got, want, "pointwise")
    assert int(flag.item()) == 0


def test_pointwise_nan_flag():
    ops = _ops()
    x = torch.zeros((1, 64, 4, 4, 4))
    x[0, 3, 1, 2, 3] = float("nan")
    w = torch.ones((64, 64, 1, 1, 1))
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.pwconv_bn_relu(to_cl(x), ops.pack_pw_weight(w.cuda()), torch.ones(64).cuda(), torch.zeros(64).cuda(), flag)
    assert int(flag.item()) == 1


@pytest.mark.parametrize("c,size,batch,n_classes", [
    (128, (8, 8, 8), 2, 2),
    (256, (4, 4, 4), 3, 2),
    (512, (2, 2, 2), 1, 2),
    (128, (12, 12, 12), 1, 2),
    (256, (6, 6, 6), 2, 2),
    (512, (3, 3, 3), 2, 2),
    (128, (5, 6, 10), 1, 3),       # NPAD = 32
    (32, (16, 12, 20), 1, 2),      # layer-0 head: BK = 32
    (512, (4, 4, 4), 8, 2),
    (128, (16, 16, 16), 2, 2),     # several 4x8x8 tiles, J = 3 row blocks, no K split
    (256, (8, 8, 8), 8, 2),        # K split across CTAs + ordered reduction
    (64, (9, 7, 20), 1, 2),        # one chunk, ragged tiles
    (128, (16, 16, 16), 8, 2),     # the benchmark's f3 head: kw-GEMM + stencil territory (M = 32768)
    (64, (21, 19, 23), 2, 2),      # M = 18354, ragged tiles on every axis
    (256, (16, 16, 16), 4, 2),
] + S.HEAD_KW_BOUNDARY)           # the kw-GEMM's 48- and 144-column tilings, at 147 and 148 tiles of 128 voxels
@pytest.mark.parametrize("algo", [1, 2, 3])
def test_head_conv_tcgen05(c, size, batch, n_classes, algo):
    ops = _ops()
    if algo == 2 and c % 64:
        pytest.skip("halo-tile kernel needs C % 64 == 0 (the per-tap kernel covers C = 32)")
    if algo == 3 and (c % 64 or n_classes != 2 or batch * size[0] * size[1] * size[2] < 256):
        pytest.skip("kw-GEMM + stencil needs C % 64 == 0, NPAD == 16 and at least 256 voxels")
    if algo == 3:
        assert ops.head_kw_supported(torch.empty((batch, c) + size, device="meta"), 16)
    g = torch.Generator().manual_seed(c + size[2] + n_classes)
    bpl = 2
    x = bf16r(torch.randn((batch, c) + size, generator=g))
    lw = torch.randn((bpl * 6, c, 3, 3, 3), generator=g) / ((27 * c) ** 0.5)
    cw = torch.randn((bpl * n_classes, c, 3, 3, 3), generator=g) / ((27 * c) ** 0.5)
    lb = torch.randn(bpl * 6, generator=g)
    cb = torch.randn(bpl * n_classes, generator=g)
    want_l = F.conv3d(x, bf16r(lw), lb, 1, 1).permute(0, 2, 3, 4, 1).reshape(batch, -1, 6)
    want_s = F.conv3d(x, bf16r(cw), cb, 1, 1).permute(0, 2, 3, 4, 1).reshape(batch, -1, n_classes)
    here = want_l.shape[1]
    pad_front, pad_back = 10, 6   # the layer writes a slice of the concatenated prior axis
    P = pad_front + here + pad_back
    locs = torch.full((batch, P, 6), -77.0, device="cuda")
    scores = torch.full((batch, P, n_classes), -77.0, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    wp, bp = ops.pack_head_weight(lw.cuda(), lb.cuda(), cw.cuda(), cb.cuda())
    ops.head_conv(to_cl(x), wp, bp, locs, scores, bpl, n_classes, pad_front, flag, algo=algo)
    locs, scores = locs.cpu(), scores.cpu()
    assert bool((locs[:, :pad_front] == -77).all()) and bool((locs[:, pad_front + here:] == -77).all())
    assert bool((scores[:, :pad_front] == -77).all()) and bool((scores[:, pad_front + here:] == -77).all())
    for got, want, what in ((locs[:, pad_front:pad_front + here], want_l, "locs"),
                            (scores[:, pad_front:pad_front + here], want_s, "scores")):
        err = (got - want).abs()
        tol = 2e-3 * torch.clamp(want.abs(), min=1.0)
        assert bool((err <= tol).all()), "%s: max err %.4g (%d beyond tol)" % (what, float(err.max()), int((err > tol).sum()))
    assert int(flag.item()) == 0


# ---------------------------------------------------------------------------------------------------
def _model_for(case, sd):
    from mslesions3d_b200.ssd3d import LSSD3D
    m = LSSD3D(n_classes=case.get("n_classes", 2), input_channels=case["channels"], input_size=tuple(case["size"]),
               aspect_ratios=case.get("aspect_ratios", {}))
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval()


@pytest.mark.parametrize("name", list(GI.FORWARD_CASES))
def test_forward_vs_oracle_and_reference_golden(name):
    case, gold = GI.FORWARD_CASES[name], load_golden("forward.pt")[name]
    sd, x = GI.forward_inputs(case)
    model = _model_for(case, sd)
    with torch.no_grad():
        locs, scores = model(x.cuda())
        el, es = O.forward(sd, x, case.get("aspect_ratios"), case.get("n_classes", 2), emulate_bf16=True)
    locs, scores = locs.cpu(), scores.cpu()
    assert locs.shape == gold["locs"].shape and scores.shape == gold["scores"].shape
    for got, emu, ref, what in ((locs, el, gold["locs"], "locs"), (scores, es, gold["scores"], "scores")):
        d_emu = (got - emu).abs()
        d_ref = (got - ref).abs()
        assert float(d_emu.max()) <= 0.06 and float(d_emu.mean()) <= 6e-3, \
            "%s vs bf16 oracle: max %.4g mean %.4g" % (what, float(d_emu.max()), float(d_emu.mean()))
        assert float(d_ref.max()) <= 0.25 and float(d_ref.mean()) <= 0.03, \
            "%s vs fp32 reference: max %.4g mean %.4g" % (what, float(d_ref.max()), float(d_ref.mean()))


def test_forward_feature_maps_match_oracle():
    case = GI.FORWARD_CASES["c2_48"]
    sd, x = GI.forward_inputs(case)
    model = _model_for(case, sd)
    with torch.no_grad():
        feats = model.base(x.cuda())
        _, _, efeats = O.forward(sd, x, emulate_bf16=True, return_features=True)
    assert list(feats.keys()) == list(efeats.keys())
    for k in feats:
        got, want = feats[k].float().cpu(), efeats[k]
        assert got.shape == want.shape
        err = (got - want).abs()
        # a one-ulp bf16 flip early in the stack propagates through up to 15 layers: allow 8 bf16 ulps on
        # any single element, and a small mean
        tol = (2.0 ** -4) * torch.clamp(want.abs(), min=0.5)
        assert bool((err <= tol).all()), "fmap %d: max err %.4g" % (k, float(err.max()))
        assert float(err.mean()) < 3e-3


def test_forward_bf16_input_and_nan_exception():
    case = GI.FORWARD_CASES["c2_48"]
    sd, x = GI.forward_inputs(case)
    model = _model_for(case, sd)
    with torch.no_grad():
        a = model(x.cuda())
        b = model(x.cuda().to(torch.bfloat16))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])   # fp32 input is rounded to bf16 on load
    bad = x.clone()
    bad[0, 0, 5, 5, 5] = float("nan")
    with torch.no_grad(), pytest.raises(Exception, match="NaN"):
        model(bad.cuda())
    with torch.no_grad():   # the sticky flag was cleared
        c = model(x.cuda())
    assert torch.equal(a[0], c[0])


def test_cpu_tensor_is_an_error_not_a_fallback():
    ops = _ops()
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.dwconv3d_bn_relu(torch.zeros(1, 32, 4, 4, 4), torch.zeros(27, 32), torch.ones(32), torch.zeros(32), 1)
