"""The fused Block kernel (csrc/conv_dwpw.cu: depthwise -> shared memory -> tcgen05 pointwise, mobilenet.py:34-49)
against (a) the two stand-alone kernels it replaces -- same arithmetic, so the outputs must be IDENTICAL -- and
(b) the torch-CPU fp32 oracle on bf16-rounded inputs (<= 1 bf16 ulp after each rounding point), on full tiles,
ragged edges, odd sizes and every (Cin, Cout, stride) the kernel is built for; NaN propagation into the flag."""
import pytest
import torch
import torch.nn.functional as F

from tests import bench_shapes as S

pytestmark = pytest.mark.gpu

CASES = [
    # (cin, cout, stride, n, (d, h, w))
    (32, 64, 2, 2, (32, 32, 32)),
    (32, 64, 2, 1, (20, 18, 26)),        # ragged tiles on every axis
    (32, 64, 2, 3, (9, 11, 17)),         # odd input sizes
    (64, 128, 2, 2, (16, 16, 16)),
    (64, 128, 2, 1, (12, 22, 18)),
    (128, 128, 1, 2, (8, 8, 8)),
    (128, 128, 1, 1, (5, 9, 12)),
    (128, 128, 1, 8, (16, 16, 16)),      # the benchmark's f3
]
# the benchmark's f1 and f2 (batch 8, 64^3 and 32^3 inputs): the other blocks the fused kernel is built for
# (csrc/conv_dwpw.cu:483-490)
CASES = S.extend(CASES, [(b.cin, b.cout, b.stride, b.n, b.size) for b in S.table(S.INFER)["block"]
                         if b.unit in ("f1", "f2", "f3")])


def bf16r(t):
    return t.to(torch.bfloat16).float()


def _inputs(cin, cout, n, size, seed):
    g = torch.Generator().manual_seed(seed)
    x = bf16r(torch.randn((n, cin) + size, generator=g))
    w1 = bf16r(torch.randn((cin, 1, 3, 3, 3), generator=g) * 0.25)
    w2 = bf16r(torch.randn((cout, cin, 1, 1, 1), generator=g) * (1.5 / cin ** 0.5))
    s1, b1 = 0.5 + torch.rand(cin, generator=g), 0.2 * torch.randn(cin, generator=g)
    s2, b2 = 0.5 + torch.rand(cout, generator=g), 0.2 * torch.randn(cout, generator=g)
    return x, w1, w2, s1, b1, s2, b2


@pytest.mark.parametrize("cin,cout,stride,n,size", CASES)
def test_fused_block_equals_the_two_kernels_and_the_oracle(cin, cout, stride, n, size):
    from mslesions3d_b200 import ops
    x, w1, w2, s1, b1, s2, b2 = _inputs(cin, cout, n, size, cin + stride + size[0])
    xc = x.cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
    wd, wp = ops.pack_dw_weight(w1.cuda()), ops.pack_pw_weight(w2.cuda())
    dev = [t.cuda() for t in (s1, b1, s2, b2)]
    assert ops.block_fused_supported(xc, cout, stride)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    got = ops.block_dwpw_bn_relu(xc, wd, dev[0], dev[1], wp, dev[2], dev[3], stride, flag)
    mid = ops.dwconv3d_bn_relu(xc, wd, dev[0], dev[1], stride)
    want = ops.pwconv_bn_relu(mid, wp, dev[2], dev[3], flag)
    assert got.shape == want.shape and int(flag.item()) == 0
    assert torch.equal(got, want), "fused vs stand-alone kernels: %d of %d elements differ, max |diff| %g" % (
        int((got != want).sum()), got.numel(), float((got.float() - want.float()).abs().max()))
    # oracle: fp32 convs on the CPU, bf16 rounding where the kernels store bf16
    a1 = bf16r(F.relu(F.conv3d(x, w1, None, stride, 1, 1, cin) * s1.view(1, -1, 1, 1, 1) + b1.view(1, -1, 1, 1, 1)))
    ref = F.relu(F.conv3d(a1, w2) * s2.view(1, -1, 1, 1, 1) + b2.view(1, -1, 1, 1, 1))
    diff = (got.float().cpu() - bf16r(ref)).abs()
    tol = 2.0 ** -7 * torch.clamp(ref.abs(), min=float(ref.abs().max()) * 2.0 ** -6)
    # the intermediate is rounded to bf16 on both sides from sums taken in a different order: a 1-ulp flip of one
    # intermediate element moves an output by up to |w2| ulps -- allow a small fraction beyond 1 ulp, none beyond 3
    assert float((diff > tol).float().mean()) < 2e-3 and not bool((diff > 3 * tol).any())


def test_fused_block_sets_the_nan_flag_and_skips_unsupported_shapes():
    from mslesions3d_b200 import _lib, ops
    x, w1, w2, s1, b1, s2, b2 = _inputs(32, 64, 1, (16, 16, 16), 5)
    x[0, 3, 4, 5, 6] = float("nan")
    xc = x.cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    y = ops.block_dwpw_bn_relu(xc, ops.pack_dw_weight(w1.cuda()), s1.cuda(), b1.cuda(), ops.pack_pw_weight(w2.cuda()),
                               s2.cuda(), b2.cuda(), 2, flag)
    assert int(flag.item()) & _lib.NAN_BACKBONE and bool(torch.isnan(y.float()).any())
    small = torch.zeros((1, 32, 8, 8, 8), dtype=torch.bfloat16, device="cuda")
    assert not ops.block_fused_supported(small, 64, 2)          # Wo = 4 < 8: the stand-alone kernels take it
    assert not ops.block_fused_supported(torch.zeros((1, 256, 16, 16, 16), device="cuda"), 256, 1)


def test_block_forward_fuse_uses_the_fused_kernel_and_matches_unfused():
    """Block.forward (eval) picks the fused kernel for the three large blocks; the whole network's outputs are
    identical with fuse=False."""
    from mslesions3d_b200 import synthetic
    from mslesions3d_b200.ssd3d import LSSD3D
    from oracle import ssd3d_oracle as O
    size = (64, 64, 64)
    model = LSSD3D(n_classes=2, input_channels=2, input_size=size)
    model.load_state_dict(O.random_state_dict(2, seed=6))
    model = model.cuda().eval()
    x = torch.from_numpy(synthetic.make_batch(2, 2, size)).cuda()
    from mslesions3d_b200 import ops
    with torch.no_grad():
        before = ops.LAUNCHES[0]
        l1, s1 = model(x)
        fused_launches = ops.LAUNCHES[0] - before
        before = ops.LAUNCHES[0]
        l0, s0 = model.pred_convs(model.base(x, fuse=False), model.base.nan_flag(x.device))
        plain_launches = ops.LAUNCHES[0] - before
    assert fused_launches < plain_launches            # 64^3: blocks f1 (32^3 -> 16^3) and f2/f3 (8^3) qualify
    assert torch.equal(l0, l1) and torch.equal(s0, s1)

