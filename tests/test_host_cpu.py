"""CPU-only checks (no GPU, no compute through the library): the C-ABI library builds/loads and exports every
symbol ``include/ssd3d_b200.h`` declares with matching arity; the host-side mirror of the reference's classes
(constructor, state_dict keys, priors, hyper-parameters, checkpoints, weight packing layouts) behaves."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import ssd3d_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "ssd3d_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(?:int|int64_t|const char\*)\s+(ssd3d_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    return out


@pytest.fixture(scope="module")
def lib():
    from mslesions3d_b200 import build, _lib
    build.build(verbose=False)
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from mslesions3d_b200 import _lib
    declared = _header_functions()
    assert len(declared) >= 14
    assert set(declared) == set(_lib.SIGNATURES), "header and ctypes table disagree"
    for name, n_args in declared.items():
        assert hasattr(lib, name), "libssd3d_b200.so does not export %s" % name
        assert len(_lib.SIGNATURES[name][1]) == n_args, "%s: header has %d params" % (name, n_args)
    assert lib.ssd3d_version().decode().startswith("ssd3d_b200 sm_100a")


def test_library_is_sm100a_tcgen05_code():
    import shutil
    import subprocess
    from mslesions3d_b200 import _lib
    # the toolkit under CUDA_HOME (where the build looks for nvcc), whether or not its bin directory is on PATH
    cuda_bin = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")
    cuobjdump = shutil.which("cuobjdump", path=cuda_bin) or shutil.which("cuobjdump")
    if not cuobjdump:
        pytest.skip("cuobjdump not found")
    elf = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in elf and "sm_90" not in elf and "sm_80" not in elf
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, "%s missing from the GEMM SASS" % mnemonic


def test_workspace_size_queries_need_no_gpu(lib):
    assert lib.ssd3d_detect_workspace_bytes(8, 9344, 2, 100) > 8 * 9344 * 24
    assert lib.ssd3d_detect_workspace_bytes(0, 9344, 2, 100) == 0
    assert lib.ssd3d_multibox_workspace_bytes(16, 3942) > 16 * 3942 * 5


def test_argument_errors_are_reported_without_a_gpu(lib):
    from mslesions3d_b200 import _lib
    assert lib.ssd3d_dwconv3d_bn_relu(None, None, None, None, None, 1, 32, 4, 4, 4, 1, None) == _lib.SSD3D_ERR_ARG
    assert lib.ssd3d_pwconv_bn_relu(1, 1, 1, 1, 1, 128, 33, 64, None, None) == _lib.SSD3D_ERR_ARG
    with pytest.raises(RuntimeError, match="invalid argument"):
        _lib.check(_lib.SSD3D_ERR_ARG, "x")


def test_model_surface_matches_reference_names():
    from mslesions3d_b200.ssd3d import LSSD3D, SSD3D, MultiBoxLoss, MobileNetBase, PredictionConvolutions
    assert SSD3D is LSSD3D
    torch.manual_seed(0)
    m = LSSD3D(n_classes=2, input_channels=1, input_size=(64, 64, 64))
    sd = m.state_dict()
    ref = O.random_state_dict(1)
    assert set(sd.keys()) == set(ref.keys()) and len(sd) == 103
    assert all(sd[k].shape == ref[k].shape for k in ref)
    assert sum(p.numel() for p in m.parameters()) == 949936
    assert torch.equal(m.priors_cxcycz.cpu(), O.prior_boxes((64, 64, 64)))
    assert float(m.rescale_factors.mean()) == 20.0
    assert m.hparams["input_size"] == (64, 64, 64) and m.boxes_per_location == 2
    assert isinstance(m.base, MobileNetBase) and isinstance(m.pred_convs, PredictionConvolutions)
    assert isinstance(m.loss_fn, MultiBoxLoss) and m.loss_fn.thresholding_mode == "hard"
    opt, sch = m.configure_optimizers()
    assert opt[0].param_groups[0]["lr"] == 2 * m.lr and opt[0].param_groups[1]["weight_decay"] == 0.0005
    for case in (dict(channels=2, size=(32, 64, 48)), dict(channels=2, size=(16, 32, 32),
                                                           aspect_ratios={0: [1.], 3: [1.]})):
        mm = LSSD3D(n_classes=2, input_channels=case["channels"], input_size=case["size"],
                    aspect_ratios=case.get("aspect_ratios", {}))
        assert torch.equal(mm.priors_cxcycz.cpu(), O.prior_boxes(case["size"], case.get("aspect_ratios"),
                                                                 in_channels=case["channels"]))
    with pytest.raises(Exception, match="Type error"):
        MultiBoxLoss(m.priors_cxcycz, threshold=1)


def test_no_cpu_path_and_train_mode_is_loud():
    from mslesions3d_b200.ssd3d import LSSD3D
    from mslesions3d_b200 import ops
    m = LSSD3D(n_classes=2, input_channels=1, input_size=(32, 32, 32)).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(1, 1, 32, 32, 32))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.iou3d_pairwise(torch.zeros(2, 6), torch.zeros(2, 6))


def test_checkpoint_round_trip(tmp_path):
    from mslesions3d_b200.ssd3d import LSSD3D
    m = LSSD3D(n_classes=3, input_channels=2, input_size=(32, 32, 32), top_k=7)
    path = os.path.join(tmp_path, "m.ckpt")
    torch.save({"state_dict": m.state_dict(), "hyper_parameters": dict(m.hparams)}, path)   # PL checkpoint layout
    m2 = LSSD3D.load_from_checkpoint(path, min_score=0.25)
    assert m2.n_classes == 3 and m2.top_k == 7 and m2.min_score == 0.25
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))


def test_weight_packing_layouts():
    """The packed matrices reproduce the convs as plain matmuls (layout check, CPU)."""
    from mslesions3d_b200 import ops
    g = torch.Generator().manual_seed(0)
    # head: (NPAD, 27*C) with K index tap*C + c
    c, bpl, ncls = 8, 2, 3
    x = torch.randn(1, c, 4, 5, 6, generator=g)
    lw, lb = torch.randn(bpl * 6, c, 3, 3, 3, generator=g), torch.randn(bpl * 6, generator=g)
    cw, cb = torch.randn(bpl * ncls, c, 3, 3, 3, generator=g), torch.randn(bpl * ncls, generator=g)
    wp, bp = ops.pack_head_weight(lw, lb, cw, cb)
    assert wp.shape == (32, 27 * c) and wp.dtype == torch.bfloat16
    xp = F.pad(x, (1, 1, 1, 1, 1, 1))
    cols = []
    for kd in range(3):
        for kh in range(3):
            for kw in range(3):
                cols.append(xp[0, :, kd:kd + 4, kh:kh + 5, kw:kw + 6].permute(1, 2, 3, 0).reshape(-1, c))
    a = torch.cat(cols, 1)                                           # (voxels, 27*C), tap-major
    out = a @ wp.float().t() + bp
    want_l = F.conv3d(x, lw.to(torch.bfloat16).float(), lb, 1, 1).permute(0, 2, 3, 4, 1).reshape(-1, bpl * 6)
    want_c = F.conv3d(x, cw.to(torch.bfloat16).float(), cb, 1, 1).permute(0, 2, 3, 4, 1).reshape(-1, bpl * ncls)
    torch.testing.assert_close(out[:, :bpl * 6], want_l, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(out[:, bpl * 6:bpl * (6 + ncls)], want_c, rtol=1e-4, atol=1e-4)
    assert float(out[:, bpl * (6 + ncls):].abs().max()) == 0.0
    # stem: (32, KPAD) bf16, k = cin*27 + tap, zero padded
    w = torch.randn(32, 2, 3, 3, 3, generator=g)
    ps = ops.pack_stem_weight(w)
    assert ps.shape == (32, 64) and ps.dtype == torch.bfloat16
    assert float(ps[5, 1 * 27 + 1 * 9 + 2 * 3 + 0]) == float(w[5, 1, 1, 2, 0].to(torch.bfloat16))
    assert float(ps[:, 54:].abs().max()) == 0.0
    assert ops.pack_stem_weight(torch.randn(32, 3, 3, 3, 3)).shape == (32, 128)
    # depthwise: (27, C)
    wd = torch.randn(16, 1, 3, 3, 3, generator=g)
    pd = ops.pack_dw_weight(wd)
    assert pd.shape == (27, 16) and float(pd[2 * 9 + 0 * 3 + 1, 7]) == float(wd[7, 0, 2, 0, 1].to(torch.bfloat16))
    # BN fold
    bn = torch.nn.BatchNorm3d(4).eval()
    bn.running_mean.normal_(generator=g), bn.running_var.uniform_(0.5, 1.5, generator=g)
    bn.weight.data.normal_(generator=g), bn.bias.data.normal_(generator=g)
    s, b = ops.fold_bn(bn)
    xx = torch.randn(2, 4, 3, 3, 3, generator=g)
    torch.testing.assert_close(xx * s.view(1, -1, 1, 1, 1) + b.view(1, -1, 1, 1, 1), bn(xx), rtol=1e-5, atol=1e-5)


def test_synthetic_volumes_follow_the_generator_spec():
    from mslesions3d_b200 import synthetic
    vols, boxes, labels = synthetic.make_batch(2, 2, (32, 32, 32), with_boxes=True, object_size=(4, 9))
    assert vols.shape == (2, 2, 32, 32, 32) and vols.dtype.name == "float32"
    assert abs(float(vols[0, 0].mean())) < 1e-3 and abs(float(vols[0, 0].std()) - 1) < 1e-2   # z-scored
    assert all(b.shape[1] == 6 and (b[:, 3:] > b[:, :3]).all() for b in boxes)
    v2 = synthetic.make_batch(2, 2, (32, 32, 32), object_size=(4, 9))
    assert (vols == v2).all()


def test_box_outline_segmentation_known_answer():
    """predict.py:181-216: a box paints its outline with its 1-based index; placeholder / low scores are skipped."""
    import torch
    from mslesions3d_b200.predict import box_outline_segmentation
    boxes = torch.tensor([[0.25, 0.25, 0.25, 0.5, 0.5, 0.5], [0., 0., 0., 1., 1., 1.], [0.1, 0.1, 0.1, 0.2, 0.2, 0.2]])
    labels = torch.tensor([1, 0, 1])
    scores = torch.tensor([0.9, 0.8, 0.2])
    seg, scores_map, infos = box_outline_segmentation(boxes, labels, scores, (16, 16, 16), 0.5)
    assert [m[0] for m in scores_map] == [1, 2, 3] and list(infos) == [1]
    assert infos[1][1] == [4, 4, 4, 8, 8, 8] and infos[1][2] == 1
    assert seg.max() == 1 and seg[4, 4, 4] == 1 and seg[9, 9, 9] == 1 and seg[6, 6, 6] == 0 and seg[4, 6, 6] == 1
    assert int((seg == 1).sum()) == 6 * 6 * 6 - 4 * 4 * 4      # the shell of the 6^3 block [4, 9]^3


def test_nifti_writer_known_answer_header_and_round_trip(tmp_path):
    """NIfTI-1 single-file layout (what nib.save writes for predict.py:225-226 / generate_artificial_dataset.py:
    106-111): 348-byte header, magic n+1, vox_offset 352, Fortran-ordered voxels, affine in the sform."""
    import gzip
    import struct
    import numpy as np
    from mslesions3d_b200 import nifti
    rs = np.random.RandomState(0)
    vol = rs.rand(5, 6, 7)
    aff = np.array([[2., 0, 0, -10], [0, 3., 0, 5], [0, 0, 4., 1], [0, 0, 0, 1]])
    path = str(tmp_path / "v.nii.gz")
    nifti.save_nifti(path, vol, aff)
    blob = gzip.open(path, "rb").read()
    assert len(blob) == 352 + vol.size * 8
    assert struct.unpack_from("<i", blob, 0)[0] == 348 and blob[344:348] == b"n+1\x00"
    assert struct.unpack_from("<8h", blob, 40) == (3, 5, 6, 7, 1, 1, 1, 1)
    assert struct.unpack_from("<2h", blob, 70) == (64, 64)                      # float64, 64 bits
    assert struct.unpack_from("<4f", blob, 76) == (1.0, 2.0, 3.0, 4.0)          # qfac, voxel sizes
    assert struct.unpack_from("<f", blob, 108)[0] == 352.0
    assert struct.unpack_from("<2h", blob, 252) == (0, 2)                       # qform_code, sform_code
    assert struct.unpack_from("<4f", blob, 280) == (2.0, 0.0, 0.0, -10.0)
    first = np.frombuffer(blob, dtype="<f8", count=6, offset=352)
    assert (first[:5] == vol[:, 0, 0]).all() and first[5] == vol[0, 1, 0]       # first axis fastest
    back, aff2 = nifti.load_nifti(path)
    assert back.dtype == np.float64 and (back == vol).all() and (aff2 == aff).all()
    for dt in ("uint8", "int16", "uint16", "int32", "float32"):
        a = (rs.rand(3, 4, 2, 2) * 100).astype(dt)
        p2 = str(tmp_path / ("a_%s.nii" % dt))
        nifti.save_nifti(p2, a)
        b, eye = nifti.load_nifti(p2)
        assert b.dtype == a.dtype and (b == a).all() and (eye == np.eye(4)).all()


def test_dataset_directory_round_trip(tmp_path):
    """write_dataset / load_dataset_dir reproduce make_batch (same generator stream, normalisation and GT boxes)."""
    import numpy as np
    from mslesions3d_b200 import synthetic
    d = synthetic.write_dataset(str(tmp_path / "ds"), 3, (32, 32, 32))
    import os
    assert sorted(os.listdir(os.path.join(d, "images"))) == ["sub-000%d_image.nii.gz" % i for i in range(3)]
    assert sorted(os.listdir(os.path.join(d, "labels"))) == ["sub-000%d_seg.nii.gz" % i for i in range(3)]
    subjects, vols, boxes, labels = synthetic.load_dataset_dir(d, with_boxes=True)
    want, wb, wl = synthetic.make_batch(3, 1, (32, 32, 32), with_boxes=True)
    assert subjects == ["0000", "0001", "0002"] and (vols == want).all()
    for a, b, la, lb in zip(boxes, wb, labels, wl):
        assert (a == b).all() and (la == lb).all()


def test_long_list_detect_routing_and_key_decoding():
    """Host logic of the any-length detect path: which (P, top_k) leave the fused kernel (ssd3d_b200.h: P > SORT_MAX
    and 10*top_k > SORT_MAX/2), and the {~orderable(score) << 32 | prior} key layout the device kernels emit."""
    import torch
    from mslesions3d_b200 import _lib, ops
    assert not ops.detect_needs_long_lists(9344, 100)               # C2
    assert not ops.detect_needs_long_lists(9344, 50000)             # P <= SORT_MAX: one block sorts everything
    assert not ops.detect_needs_long_lists(2501400, 800)            # 8000 candidates through the fused NMS
    assert ops.detect_needs_long_lists(2501400, 820)
    assert ops.detect_needs_long_lists(_lib.SORT_MAX + 1, 50000)    # model_insight.py:146
    score = torch.tensor([1.0, 0.75, 0.5, 1e-30, 0.0, 0.2500001])
    bits = score.view(torch.int32).to(torch.int64) | 0x80000000      # orderable() of a non-negative float
    keys = (((~bits) & 0xFFFFFFFF) << 32) | torch.arange(6)
    assert bool((keys >= 0).all())                                   # compare equal as signed and unsigned
    assert torch.equal(ops._key_scores(keys), score)
    order = torch.argsort(keys)                                      # ascending key = descending score
    assert order.tolist() == [0, 1, 2, 5, 3, 4]
    with __import__("pytest").raises(RuntimeError):
        ops.nms3d_sorted_chunked(torch.zeros(4, 6), 0.5)             # CPU tensors are refused: no CPU path
