"""CPU: C-ABI surface, host-side packing logic, frame sharding over gloo (world_size 2)."""
import os
import re
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    from sessd_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "sessd_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)                                   # declarations only, not the prose
    declared = set(re.findall(r"\b(sessd_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    for name in declared:
        assert name in _lib.SIGNATURES, name             # the binding declares its signature
        assert hasattr(_lib.lib._prod, name), name       # and dlsym succeeds in the PRODUCT library
    assert "sm_100a" in _lib.version()
    # no compute calls here (no GPU in this container): argument validation only
    assert _lib.lib.sessd_voxelize_workspace_bytes(20000, 1, None) == 0
    assert _lib.lib.sessd_nms_workspace_bytes(1000) == 8 * (1000 * 16 + 64)
    # importing / using the product does not load the lab library: checked in a fresh interpreter, since GPU tests that run earlier in
    # the same session load it on purpose
    code = ("import sys; sys.path.insert(0, %r); from sessd_b200 import _lib; _lib.version(); "
            "_lib.lib.sessd_voxelize_workspace_bytes(20000, 1, None); _lib.lib.sessd_nms_workspace_bytes(1000); "
            "assert not _lib.lib.lab_loaded; assert 'libsessd_b200_lab' not in open('/proc/self/maps').read()") % os.path.join(ROOT, "se-ssd_b200")
    subprocess.check_call([sys.executable, "-c", code])


def test_lab_library_exports_every_declared_symbol_and_nothing_of_the_product():
    """include/sessd_b200_lab.h (non-default kernel variants + probes) lives in its own library; the product library exports none of it."""
    import ctypes
    from sessd_b200 import _lib
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "sessd_b200_lab.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(sessd_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.LAB_SIGNATURES)
    prod = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert not hasattr(prod, name), name
        assert hasattr(_lib.lib, name), name             # resolves through the lazily loaded lab library
    assert _lib.lib.lab_loaded


def test_shared_library_is_sm100a_sass():
    out = subprocess.run(["cuobjdump", "-lelf", os.path.join(ROOT, "se-ssd_b200", "libsessd_b200.so")], capture_output=True, text=True)
    if out.returncode != 0:
        return
    assert "sm_100a" in out.stdout


def test_product_anchors_equal_reference_golden(golden_dir):
    from cases import sha
    from sessd_b200 import weights
    g = np.load(os.path.join(golden_dir, "anchors_assign.npz"))
    anc = weights.kitti_car_anchors()
    assert anc.shape == (70400, 7) and (sha(anc) == g["anchors_sha"]).all()


def _tap_conv(x_nhwc, wp, taps, in_stride, grid_hw):
    """numpy/torch emulation of the tap-list contract of sessd_bev_conv (zero outside the input)."""
    b, h, w, cin = x_nhwc.shape
    out = torch.zeros((b, grid_hw[0], grid_hw[1], wp.shape[2]), dtype=x_nhwc.dtype)
    for t, (dy, dx) in enumerate(taps):
        for oy in range(grid_hw[0]):
            iy = oy * in_stride + dy
            if iy < 0 or iy >= h:
                continue
            for ox in range(grid_hw[1]):
                ix = ox * in_stride + dx
                if 0 <= ix < w:
                    out[:, oy, ox] += x_nhwc[:, iy, ix] @ wp[t]
    return out


def test_conv_and_deconv_tap_packing_equals_torch():
    from sessd_b200.runners import _deconv_classes, _pack_conv
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 6, 5, 7, generator=g, dtype=torch.float64)          # NCHW
    xn = x.permute(0, 2, 3, 1).contiguous()
    for stride in (1, 2):
        w = torch.randn(4, 6, 3, 3, generator=g, dtype=torch.float64)
        ref = F.conv2d(x, w, None, stride, 1)
        wp, taps = _pack_conv(w)
        got = _tap_conv(xn, wp, [(dy - 1, dx - 1) for dy, dx in taps], stride, ref.shape[2:])
        assert torch.allclose(got.permute(0, 3, 1, 2), ref, atol=1e-12)
    wt = torch.randn(6, 4, 3, 3, generator=g, dtype=torch.float64)
    ref = F.conv_transpose2d(x, wt, None, 2, 1, output_padding=1)          # [1,4,10,14]
    full = torch.zeros_like(ref).permute(0, 2, 3, 1).contiguous()
    for py, px, wp, taps in _deconv_classes(wt):
        full[:, py::2, px::2] = _tap_conv(xn, wp, taps, 1, (5, 7))
    assert torch.allclose(full.permute(0, 3, 1, 2), ref, atol=1e-12)


def test_weight_split_and_bn_fold():
    from sessd_b200 import weights
    from sessd_b200.runners import SPMIDDLE_LAYERS, fold_bn
    sd = weights.random_detector_state(1)
    layers, ssfa, head = weights.split_detector_state(sd)
    assert len(layers) == len(SPMIDDLE_LAYERS) == 14
    assert tuple(layers[0]["weight"].shape) == (3, 3, 3, 4, 16) and tuple(layers[13]["weight"].shape) == (3, 1, 1, 64, 64)
    assert "bottom_up_block_0.1.weight" in ssfa and "tasks.0.conv_box.weight" in head
    x = torch.randn(10, 16)
    sc, sh = fold_bn(layers[0]["gamma"], layers[0]["beta"], layers[0]["mean"], layers[0]["var"])
    ref = F.batch_norm(x, layers[0]["mean"], layers[0]["var"], layers[0]["gamma"], layers[0]["beta"], False, 0.0, 1e-3)
    assert torch.allclose(x * sc + sh, ref, atol=1e-6)


def test_frame_sharding_two_ranks_gloo(tmp_path):
    """world_size-2 CPU run of the N>1 host path: f -> rank f mod world, one fixed-size all_gather, no other collective."""
    script = tmp_path / "w.py"
    script.write_text(
        "import os, sys, numpy as np, torch, torch.distributed as dist\n"
        "sys.path.insert(0, %r)\n"
        "from sessd_b200 import shard\n"
        "dist.init_process_group('gloo')\n"
        "r, w = dist.get_rank(), dist.get_world_size()\n"
        "F = 7\n"
        "mine = shard.frames_for_rank(F, r, w)\n"
        "local = {f: (np.full((f + 1, 7), f, np.float32), np.full((f + 1,), 0.5 + f, np.float32)) for f in mine}\n"
        "allr = shard.gather_detections(local, F, 100, r, w)\n"
        "assert sorted(allr) == list(range(F)), sorted(allr)\n"
        "for f, (b, s) in allr.items():\n"
        "    assert b.shape == (f + 1, 7) and (b == f).all() and (s == 0.5 + f).all()\n"
        "assert set(mine) == set(range(r, F, w))\n"
        "print('rank', r, 'ok')\n" % os.path.join(ROOT, "se-ssd_b200"))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29731", str(script)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("ok") == 2


def test_sparse_fp16_split_weight_packing_layout_and_precision():
    """ops.pack_weight_sp_h2: tile layouts the TMA maps of spconv_h2.cu assume, per-channel power-of-two scales, hi + lo == scaled weight
    to fp16-split precision (22+ significand bits)."""
    from sessd_b200 import ops
    g = torch.Generator().manual_seed(3)
    for cin, cout, cp, layout in ((64, 64, 64, "cg"), (32, 32, 32, "cg"), (32, 64, 32, "cg"), (32, 32, 32, "h2"), (16, 32, 32, "h2")):
        w = torch.randn(27, cin, cout, generator=g) * torch.logspace(-3, 1, cout)[None, None, :]      # channel scales over 4 decades
        tiles, inv = ops.pack_weight_sp_h2(w, cp, layout=layout)
        assert tiles.dtype == torch.float16 and inv.shape == (cout,)
        ex = torch.log2(inv)
        assert torch.equal(ex, ex.round())                                   # exact powers of two
        scaled = w.permute(0, 2, 1) / inv[None, :, None]                     # [kvol, cout, cin] * 2^e
        assert float(scaled.abs().amax()) < 2048.0 and float(scaled.abs().amax(dim=(0, 2)).min()) >= 1024.0
        if cp == 64 or layout == "cg":                                       # [kvol, 2 (hi | lo), Cout, Cin]: the pair-gather kernel's tiles
            assert tuple(tiles.shape) == (27, 2, cout, cin)
            hi, lo = tiles[:, 0].float(), tiles[:, 1].float()
        else:
            assert tuple(tiles.shape) == (27, cout, 64)
            hi, lo = tiles[:, :, :cin].float(), tiles[:, :, 32:32 + cin].float()
            assert not tiles[:, :, cin:32].any() and not tiles[:, :, 32 + cin:].any()     # zero padding of the 16-channel layers
        err = (hi + lo - scaled).abs().max() / scaled.abs().max()
        assert float(err) < 2.0 ** -21


def test_checkpoint_reads_reference_written_file(golden_dir):
    """Files written by the REFERENCE's own save_checkpoint (tests/golden/make_checkpoint_golden.py, which also verified that the
    reference's load_checkpoint reads OUR files): {'meta','state_dict','optimizer'} and a bare 'module.'-prefixed OrderedDict."""
    import os
    import torch
    from cases import checkpoint_model
    from det3d.torchie.trainer.checkpoint import load_checkpoint
    want = checkpoint_model(seed=7).state_dict()
    for name in ("ref_checkpoint.pth", "ref_checkpoint_module_prefix.pth"):
        m = checkpoint_model(seed=1)
        ck = load_checkpoint(m, os.path.join(golden_dir, name), map_location="cpu", strict=True)
        for k, v in m.state_dict().items():
            assert torch.equal(v, want[k]), (name, k)
    assert ck is not None
    ck = load_checkpoint(checkpoint_model(seed=1), os.path.join(golden_dir, "ref_checkpoint.pth"), map_location="cpu")
    assert ck["meta"] == {"epoch": 3, "iter": 1234} and "optimizer" in ck


def test_voxelization_train_mode_filters_gt_outside_range():
    """reference preprocess.py:199-205 + sampler/preprocess.py:138-148: a labeled training frame loses the GT boxes that have NO BEV
    corner strictly inside [0,-40,70.4,40]; a straddling box (one corner inside) stays."""
    from det3d.datasets.pipelines.preprocess import filter_gt_box_outside_range
    rng = [0.0, -40.0, 70.4, 40.0]
    boxes = np.array([
        [30.0, 0.0, -1.0, 1.6, 3.9, 1.5, 0.3],      # inside
        [-5.0, 0.0, -1.0, 1.6, 3.9, 1.5, 0.0],      # fully outside (x < 0)
        [0.5, 0.0, -1.0, 1.6, 3.9, 1.5, 0.0],       # straddles x = 0: corners at x = -0.3 and 1.3
        [71.2, 39.0, -1.0, 1.6, 3.9, 1.5, 0.0],     # corners x in [70.4, 72.0]: x = 70.4 is ON the boundary -> outside
        [35.0, 41.0, -1.0, 1.6, 1.9, 1.5, 0.0],     # y in [40.05, 41.95]: outside
    ], np.float64)
    m = filter_gt_box_outside_range(boxes, rng)
    assert m.tolist() == [True, False, True, False, False]
    assert filter_gt_box_outside_range(np.zeros((0, 7)), rng).shape == (0,)


def test_bench_weights_are_quiet_calibrated_and_library_free():
    """bench / parity workload parameters: exact silence over empty space, committed calibration, and importable without the
    CUDA library (the CPU reference arm must not load libsessd_b200.so)."""
    import subprocess
    import sys
    import torch
    from oracle import frame as oframe
    from sessd_data import weights
    layers, ssfa, head = weights.bench_detector_state("ring", 0)
    assert np.all(oframe.empty_space_logits(ssfa, head) == weights.EMPTY_LOGIT)
    cal = weights.load_bench_calibration()
    for kind in ("ring", "uniform"):
        assert 300 <= cal[kind]["candidates_on_seed0"] <= 500 and cal[kind]["distinct_in_top1000"] == 1000
    code = ("import sys; sys.path[:0] = %r; import sessd_data.weights as w, sessd_data.synth as s, oracle.frame; "
            "w.bench_detector_state('ring', 0); s.ring_cloud(0, 100); "
            "import ctypes; assert not any('sessd_b200' in m for m in sys.modules), 'product package imported'; "
            "maps = open('/proc/self/maps').read(); assert 'libsessd_b200' not in maps, 'product library loaded'") % (sys.path[:3],)
    subprocess.check_call([sys.executable, "-c", code])
    assert isinstance(head["tasks.0.conv_cls.bias"], torch.Tensor)


def test_bench_parity_matcher_by_anchor_index():
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    ref_boxes = np.arange(21, dtype=np.float32).reshape(3, 7)
    ref_scores = np.array([0.9, 0.8, 0.7], np.float32)
    got = {"anchor_index": np.array([5, 9, 11]), "box3d_lidar": ref_boxes[[0, 1]].tolist() + [[0] * 7], "scores": np.array([0.9, 0.8, 0.31], np.float32)}
    got["box3d_lidar"] = np.array(got["box3d_lidar"], np.float32)
    m = b.match_detections(got, ref_boxes, ref_scores, np.array([5, 9, 13]))
    assert m["n_matched"] == 2 and m["max_abs_box_diff"] == 0.0 and m["same_order"]
    assert sorted((u["side"], u["anchor"]) for u in m["unmatched"]) == [("gpu", 11), ("oracle", 13)]


def test_c_abi_rejects_null_arguments_before_touching_the_device():
    """INTEGRATION.md §C: every compute entry point validates its arguments first and returns SESSD_EINVAL (-1) -- it never exits the
    process (the reference's CHECK_ERROR does, iou3d.cpp:13-21) and needs no GPU to say so.  All-null / all-zero calls; the pairwise IoU
    entries and the host ODIoU evaluator treat n = m = 0 as an empty, successful call (like the reference on empty box sets)."""
    import ctypes as C
    from sessd_b200._lib import SIGNATURES, lib
    empty_ok = {"sessd_boxes_overlap_bev", "sessd_boxes_aligned_overlap_bev", "sessd_boxes_iou_bev", "sessd_boxes_iou3d", "sessd_odiou_pairs_host"}
    not_compute = {"sessd_launch_count", "sessd_tile_list_stride"}
    checked = 0
    for name, (ret, args) in SIGNATURES.items():
        if ret is not C.c_int or name in not_compute:
            continue
        vals = []
        for a in args:
            if a is C.c_void_p:
                vals.append(C.c_void_p(0))
            elif a in (C.c_int, C.c_long, C.c_longlong, C.c_size_t, C.c_uint):
                vals.append(0)
            elif a in (C.c_float, C.c_double):
                vals.append(0.0)
            elif isinstance(a, type) and issubclass(a, C.Structure):
                vals.append(a())
            else:
                vals.append(None)                      # typed pointer
        rc = getattr(lib, name)(*vals)
        assert rc == (0 if name in empty_ok else -1), (name, rc)
        checked += 1
    assert checked >= 30
