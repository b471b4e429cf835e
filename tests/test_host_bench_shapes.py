"""The benchmark's kernel shapes (tests/bench_shapes.py) against a hand-written list, and the boundary cases against
the kernel switches they sit on.  A change to the model, to bench.py's configuration or to a switch fails here instead
of leaving the GPU parity tests on shapes the benchmark no longer runs."""
import ast
import os

import torch

from tests import bench_shapes as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, BF16 = torch.float32, torch.bfloat16


def test_configs_mirror_bench_py():
    tree = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    consts = {}
    for node in tree.body:
        if isinstance(node, ast.Assign) and isinstance(node.targets[0], ast.Tuple):
            names = [t.id for t in node.targets[0].elts]
            consts.update(zip(names, ast.literal_eval(node.value)))
    assert (consts["CHANNELS"], consts["SIZE"], consts["BATCH"]) == (S.INFER.channels, S.INFER.size, S.INFER.batch)
    assert (consts["TRAIN_CHANNELS"], consts["TRAIN_SIZE"], consts["TRAIN_BATCH"]) == \
        (S.TRAIN.channels, S.TRAIN.size, S.TRAIN.batch)


def _strip(records):
    return [tuple(r)[1:] for r in records]


def test_training_step_shapes():
    t = S.table(S.TRAIN)
    assert _strip(t["stem"]) == [(1, 16, (96, 96, 96), 2, F32)]
    assert S.bn_shapes(S.TRAIN) == [
        (16, 32, (48, 48, 48)), (16, 32, (24, 24, 24)), (16, 64, (24, 24, 24)), (16, 64, (12, 12, 12)),
        (16, 128, (12, 12, 12)), (16, 128, (6, 6, 6)), (16, 256, (6, 6, 6)), (16, 256, (3, 3, 3)), (16, 512, (3, 3, 3))]
    assert [S.rows(n, size) for n, _, size in S.bn_shapes(S.TRAIN)] == [
        1769472, 221184, 221184, 27648, 27648, 3456, 3456, 432, 432]
    # (c, n, input size, stride)
    assert _strip(t["dw"]) == [
        (32, 16, (48, 48, 48), 2), (64, 16, (24, 24, 24), 2), (128, 16, (12, 12, 12), 1), (128, 16, (12, 12, 12), 2),
        (256, 16, (6, 6, 6), 1), (256, 16, (6, 6, 6), 2), (512, 16, (3, 3, 3), 1)]
    # (cin, cout, n, size)
    assert _strip(t["pw"]) == [
        (32, 64, 16, (24, 24, 24)), (64, 128, 16, (12, 12, 12)), (128, 128, 16, (12, 12, 12)),
        (128, 256, 16, (6, 6, 6)), (256, 256, 16, (6, 6, 6)), (256, 512, 16, (3, 3, 3)), (512, 512, 16, (3, 3, 3))]
    assert S.rows(16, t["pw"][0].size) == 221184
    # (c, n, size, boxes per location): test_head_backward assumes two
    assert _strip(t["head"]) == [(128, 16, (12, 12, 12), 2), (256, 16, (6, 6, 6), 2), (512, 16, (3, 3, 3), 2)]


def test_inference_shapes():
    t = S.table(S.INFER)
    assert _strip(t["stem"]) == [(2, 8, (128, 128, 128), 2, BF16)]
    # (cin, cout, stride, n, input size)
    assert _strip(t["block"])[:3] == [(32, 64, 2, 8, (64, 64, 64)), (64, 128, 2, 8, (32, 32, 32)),
                                      (128, 128, 1, 8, (16, 16, 16))]
    assert _strip(t["head"]) == [(128, 8, (16, 16, 16), 2), (256, 8, (8, 8, 8), 2), (512, 8, (4, 4, 4), 2)]


def test_benchmark_shapes_reach_the_large_kernel_variants():
    kinds = [S.bn_kernel(S.rows(n, size), c) for n, c, size in S.bn_shapes(S.TRAIN)]
    assert kinds == ["tile32-stream", "tile32-stream", "tile64-stream", "tile64-keep", "tile64-keep",
                     "cluster", "cluster", "cluster", "cluster"]
    dw = [S.dw_wgrad_kernel(u.c, u.n, u.size, u.stride) for u in S.table(S.TRAIN)["dw"]]
    assert dw[:3] == [("tma",)] * 3 and [k[0] for k in dw[3:]] == ["simt"] * 4
    stem = S.table(S.TRAIN)["stem"][0]
    assert S.stem_kernel(F32, stem.cin, stem.size[2]) == "tc"
    assert S.stem_kernel(BF16, stem.cin, stem.size[2]) == "tc"
    assert S.rows(stem.n, tuple(s // 2 for s in stem.size)) >= S.STEM_WGRAD_TILE_ROWS
    istem = S.table(S.INFER)["stem"][0]
    assert S.stem_kernel(istem.dtype, istem.cin, istem.size[2]) == "tz"
    for h in S.table(S.TRAIN)["head"][:1] + S.table(S.INFER)["head"][:1]:
        assert S.head_kw_columns(h.c, h.n, h.size) == 144


def test_bn_boundaries_sit_on_both_sides():
    got = [(S.rows(n, size), c, S.bn_kernel(S.rows(n, size), c)) for n, c, size in S.BN_BOUNDARY]
    assert got == [(8192, 32, "cluster"), (8193, 32, "tile32-keep"), (8192, 128, "cluster"), (8193, 128, "tile64-keep"),
                   (151552, 32, "tile32-keep"), (151553, 32, "tile32-stream"),
                   (75776, 64, "tile64-keep"), (75777, 64, "tile64-stream")]
    assert [S.bn_kernel(S.rows(n, size), c) for n, c, size in S.BN_BOUNDARY_PASSES] == ["passes"]
    # the restated plan follows the switch points it names
    assert S.bn_kernel(8192, 96) == "cluster" and S.bn_kernel(10 ** 6, 512) == "tile64-stream"
    assert S.bn_kernel(10 ** 6, 24) == "passes" and S.bn_kernel(10 ** 6, 8192) == "passes"
    assert S.bn_kernel(10 ** 6, 4096, sms=32) == "unit"          # more 64-channel groups than SMs


def test_depthwise_boundaries_sit_on_both_sides():
    got = [S.dw_wgrad_kernel(*case) for case in S.DW_BOUNDARY]
    assert [k[0] for k in got[:4]] == ["tma", "simt", "tma", "simt"]
    # Wo = 8 / 7 (stride 2), then Do = 4 / 3 (stride 1)
    assert [(s[2] - 1) // st + 1 for _, _, s, st in S.DW_BOUNDARY[:2]] == [8, 7]
    assert [(s[0] - 1) // st + 1 for _, _, s, st in S.DW_BOUNDARY[2:4]] == [4, 3]
    assert got[4:] == [("simt", 2, 21, False), ("simt", 8, 404, False), ("simt", 8, 592, True)]


def test_stem_and_head_boundaries_sit_on_both_sides():
    m = [S.rows(n, ((size[0] - 1) // sd + 1, (size[1] - 1) // 2 + 1, (size[2] - 1) // 2 + 1))
         for _, n, size, sd, _ in S.STEM_WGRAD_BOUNDARY]
    assert m == [18942, 18944, 18940, 18944] and S.STEM_WGRAD_TILE_ROWS == 18944
    # every case has rows the TMA tile kernel can address, so only M decides
    assert all(S.stem_kernel(dt, cin, size[2]) != "simt" for cin, _, size, _, dt in S.STEM_WGRAD_BOUNDARY)
    assert [S.stem_kernel(dt, cin, size[2]) for cin, size, _, dt, _ in S.STEM_FWD_BOUNDARY] == \
        ["tz", "tc", "tc", "tz", "tc", "tc"]
    assert [S.head_kw_columns(c, n, size) for c, size, n, _ in S.HEAD_KW_BOUNDARY] == [48, 144]
