"""Drop-in boundary: the det3d / spconv / iou3d_cuda API surface (SURVEY.md 8b).  CPU part: config + registries + builders;
GPU part: VoxelNet.forward(example, return_loss=False) through the reference's own pipeline transforms and collate format."""
import json
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUR_CFG = os.path.join(ROOT, "examples", "second", "configs", "config.py")


def _build(cfg_path):
    from det3d.models import build_detector
    from det3d.torchie import Config
    cfg = Config.fromfile(cfg_path)
    model = build_detector(cfg.model, train_cfg=cfg.train_cfg, test_cfg=cfg.test_cfg)
    return cfg, model


@pytest.mark.parametrize("against_reference", [False, True], ids=["repo-config", "reference-config-unchanged"])
def test_config_loads_and_detector_builds(against_reference, golden_dir):
    """The repo's config builds the detector.  `reference-config-unchanged`: it is also the detector this package builds from the
    reference's examples/second config file, unchanged (tests/golden/reference_config_detector.json, written by make_golden.py):
    same state-dict names, shapes and dtypes, parameter count, test_cfg and assigner output stride."""
    cfg, model = _build(OUR_CFG)
    assert cfg.model.type == "VoxelNet" and cfg.test_cfg.nms.nms_iou_threshold == 0.01
    assert cfg.assigner.out_size_factor == 8
    from sessd_b200 import weights
    sd = weights.random_detector_state(0)
    missing = model.load_state_dict(sd, strict=True)          # reference state-dict key names
    assert not missing.missing_keys and not missing.unexpected_keys
    n_params = sum(p.numel() for p in model.parameters())
    assert 3.7e6 < n_params < 3.9e6                            # ~3.8 M parameters (SURVEY.md 2.2)
    if against_reference:
        with open(os.path.join(golden_dir, "reference_config_detector.json")) as f:
            g = json.load(f)
        assert [[k, list(v.shape), str(v.dtype)] for k, v in model.state_dict().items()] == g["state_dict"]
        assert n_params == g["n_params"] and cfg.model.type == g["model_type"] and cfg.assigner.out_size_factor == g["out_size_factor"]
        assert json.loads(json.dumps(cfg.test_cfg)) == g["test_cfg"]


def test_registry_semantics():
    from det3d.models.registry import BACKBONES
    from det3d.utils import Registry, build_from_cfg
    with pytest.raises(KeyError):
        build_from_cfg(dict(type="NoSuchBackbone"), BACKBONES)
    r = Registry("x")

    @r.register_module
    class A(object):
        def __init__(self, v=1):
            self.v = v

    with pytest.raises(KeyError):
        r.register_module(A)                                   # duplicates are an error, like the reference
    assert build_from_cfg(dict(type="A"), r, dict(v=3)).v == 3
    with pytest.raises(TypeError):
        r.register_module(3)


def test_anchor_assigner_pipeline_matches_reference_golden(golden_dir):
    """AssignTarget (config #1, CPU): anchors + labels + regression targets equal the reference's assign_v2 output."""
    from det3d.datasets.pipelines import AssignTarget
    from det3d.torchie import Config
    from sessd_b200 import synth
    cfg = Config.fromfile(OUR_CFG)
    at = AssignTarget(cfg=cfg.train_cfg.assigner)
    gt, _ = synth.random_boxes(21, 12)
    gt[:, 2] = -1.0
    res = dict(mode="train", labeled=True, lidar=dict(annotations=dict(gt_boxes=gt.copy(), gt_classes=np.ones(12, np.int32),
                                                                            gt_names=np.array(["Car"] * 12))))
    res, _ = at(res, None)
    g = np.load(os.path.join(golden_dir, "anchors_assign.npz"))
    t = res["lidar"]["targets"]
    assert np.array_equal(t["anchors"][0][:704], g["anchors_head"])
    assert np.array_equal(t["labels"][0].astype(np.int8), g["labels"])
    pos = np.nonzero(t["labels"][0] > 0)[0]
    assert np.array_equal(pos, g["pos_idx"]) and np.array_equal(t["reg_targets"][0][pos], g["pos_targets"])


def test_host_assigner_mirror_matches_reference_on_all_golden_cases(golden_dir):
    """Host TargetAssigner.assign_v2 (numpy) == the reference on empty / single / many GT, GT without overlap, forced-only positives, ties."""
    from cases import assign_cases
    from det3d.datasets.pipelines import AssignTarget
    from det3d.torchie import Config
    at = AssignTarget(cfg=Config.fromfile(OUR_CFG).train_cfg.assigner)
    ta, ad = at.target_assigners[0], at.anchor_dicts_by_task[0]
    g = np.load(os.path.join(golden_dir, "assign_cases.npz"))
    for name, gt in assign_cases():
        m = len(gt)
        r = ta.assign_v2(ad, gt, None, gt_classes=np.ones(m, np.int32), gt_names=np.array(["Car"] * m), enable_similar_type=True)
        assert np.array_equal(r["labels"].astype(np.int8), g[name + "_labels"]), name
        pos = np.nonzero(r["labels"] > 0)[0]
        assert np.array_equal(pos, g[name + "_pos_idx"]) and np.array_equal(r["bbox_targets"][pos], g[name + "_pos_targets"]), name
        assert np.array_equal(np.asarray(r["positive_gt_id"][0], np.int32), g[name + "_positive_gt_id"]), name


def _example_from_clouds(cfg, clouds):
    from det3d.datasets.pipelines import AssignTarget, Reformat, Voxelization
    from det3d.torchie.parallel import collate_kitti
    tf = [Voxelization(cfg=cfg.voxel_generator), AssignTarget(cfg=cfg.train_cfg.assigner), Reformat()]
    frames = []
    for i, c in enumerate(clouds):
        res = dict(mode="val", metadata=dict(token=i), lidar=dict(points=c))
        for t in tf:
            res, _ = t(res, None)
        frames.append(res)
    return collate_kitti(frames)


@pytest.mark.gpu
def test_voxelnet_dropin_matches_oracle_and_engine():
    """The reference's config builds the drop-in VoxelNet; its detections on the bench workload's weights equal the CPU oracle's
    (kept sets identical, boxes / scores within 1e-4)."""
    from oracle import frame as oframe
    from sessd_b200 import synth, weights
    cfg, model = _build(OUR_CFG)
    anchors = weights.kitti_car_anchors()
    clouds = [synth.ring_cloud(31, 20000), synth.ring_cloud(32, 15000)]
    layers, ssfa, head = weights.bench_detector_state("ring", 0)
    sd = {}
    for i, l in enumerate(layers):
        sd["backbone.middle_conv.%d.weight" % (3 * i)] = l["weight"]
        for k, nm in (("gamma", "weight"), ("beta", "bias"), ("mean", "running_mean"), ("var", "running_var")):
            sd["backbone.middle_conv.%d.%s" % (3 * i + 1, nm)] = l[k]
    sd.update({"neck." + k: v for k, v in ssfa.items()})
    sd.update({"bbox_head." + k: v for k, v in head.items()})
    missing = model.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all(k.endswith("num_batches_tracked") for k in missing.missing_keys), missing
    model = model.cuda().eval()
    example = _example_from_clouds(cfg, clouds)
    assert example["coordinates"].shape[1] == 4 and example["anchors"][0].shape == (2, 70400, 7)
    dev = {k: (v.cuda() if isinstance(v, torch.Tensor) else [t.cuda() for t in v] if k == "anchors" else v) for k, v in example.items()}
    with torch.no_grad():
        dets = model(dev, return_loss=False)
    assert len(dets) == 2
    lnp = oframe.layers_to_numpy(layers)
    for f, cloud in enumerate(clouds):
        boxes, scores, _l, aux = oframe.frame_detections(cloud, lnp, ssfa, head, anchors)
        assert boxes.shape[0] > 3
        d = dets[f]
        assert d["metadata"]["token"] == f and d["label_preds"].dtype == torch.int64
        assert d["box3d_lidar"].shape[0] == boxes.shape[0]
        np.testing.assert_allclose(d["box3d_lidar"].cpu().numpy(), boxes.numpy(), rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(d["scores"].cpu().numpy(), scores.numpy(), rtol=1e-4, atol=1e-6)


@pytest.mark.gpu
def test_spconv_module_api_matches_oracle():
    """spconv.SparseConvTensor / SubMConv3d / SparseConv3d / SparseSequential / dense() used stand-alone."""
    import spconv
    from oracle import cpu as ocpu, spconv_ref as S
    from sessd_b200 import synth
    from torch import nn
    v, c, n = ocpu.points_to_voxel(synth.ring_cloud(9, 5000), synth.VOXEL_SIZE, synth.PC_RANGE, 5, 20000)
    coors = np.concatenate([np.zeros((len(c), 1), np.int32), c], 1).astype(np.int32)
    feat = (v.sum(1) / n[:, None]).astype(np.float32)
    torch.manual_seed(0)
    net = spconv.SparseSequential(spconv.SubMConv3d(4, 16, 3, bias=False, indice_key="k0"), nn.ReLU(),
                                  spconv.SparseConv3d(16, 32, 3, 2, padding=1, bias=True)).cuda()
    x = spconv.SparseConvTensor(torch.from_numpy(feat).cuda(), torch.from_numpy(coors).cuda(), [41, 1600, 1408], 1)
    y = net(x)
    w0 = net[0].weight.detach().cpu().numpy().reshape(27, 4, 16)
    w1 = net[2].weight.detach().cpu().numpy().reshape(27, 16, 32)
    nbr0 = S.neighbor_table(coors, (41, 1600, 1408), coors, (3, 3, 3), (1, 1, 1), (1, 1, 1))
    f0 = np.maximum(S.conv_from_nbr(feat, nbr0, w0), 0)
    oc, osh = S.strided_out_coors(coors, (41, 1600, 1408), (3, 3, 3), (2, 2, 2), (1, 1, 1))
    nbr1 = S.neighbor_table(coors, (41, 1600, 1408), oc, (3, 3, 3), (2, 2, 2), (1, 1, 1))
    f1 = S.conv_from_nbr(f0, nbr1, w1) + net[2].bias.detach().cpu().numpy()[None]
    assert y.spatial_shape == list(osh) and np.array_equal(y.indices.cpu().numpy(), oc)
    assert np.abs(y.features.cpu().numpy() - f1).max() / np.abs(f1).max() < 1e-5
    dense = y.dense()
    assert tuple(dense.shape) == (1, 32, 21, 800, 704)
    assert float(dense.abs().sum()) == pytest.approx(float(y.features.abs().sum()), rel=1e-4)


@pytest.mark.gpu
def test_iou3d_utils_api():
    from det3d.core.iou3d import iou3d_utils
    from oracle import cpu as ocpu
    from sessd_b200 import synth
    import iou3d_cuda
    b1, s1 = synth.random_boxes(3, 200, spread=0.3)
    b2, _ = synth.random_boxes(4, 150, spread=0.3)
    a, b = torch.from_numpy(b1).cuda(), torch.from_numpy(b2).cuda()
    iou = iou3d_utils.boxes_iou_bev_gpu(a, b)
    ref = ocpu.boxes_iou_bev(ocpu.boxes3d_to_bev(b1), ocpu.boxes3d_to_bev(b2))
    np.testing.assert_allclose(iou.cpu().numpy(), ref, rtol=2e-5, atol=2e-5)
    i3 = iou3d_utils.boxes_iou3d_gpu(a, b)
    assert i3.shape == (200, 150) and float(i3.max()) <= 1.0 + 1e-5
    al = iou3d_utils.boxes_aligned_iou3d_gpu(a[:150], b)
    np.testing.assert_allclose(al.cpu().numpy()[:, 0], np.diag(i3.cpu().numpy()[:150]), rtol=1e-4, atol=1e-5)
    keep = iou3d_utils.nms_gpu(a, torch.from_numpy(s1).cuda(), 0.1)
    order = np.argsort(-s1, kind="stable")
    bev = torch.zeros(200, 5)
    bev[:, 0], bev[:, 1] = torch.from_numpy(b1[:, 0] - b1[:, 4] / 2), torch.from_numpy(b1[:, 2] - b1[:, 3] / 2)   # rect=True layout
    bev[:, 2], bev[:, 3] = torch.from_numpy(b1[:, 0] + b1[:, 4] / 2), torch.from_numpy(b1[:, 2] + b1[:, 3] / 2)
    bev[:, 4] = torch.from_numpy(b1[:, 6])
    ref_keep = order[ocpu.nms_sorted(bev.numpy()[order], 0.1, 0)]
    assert np.array_equal(keep.cpu().numpy(), ref_keep)
    with pytest.raises(RuntimeError):
        iou3d_cuda.boxes_iou_bev_gpu(torch.zeros(2, 5), torch.zeros(2, 5).cuda(), torch.zeros(2, 2).cuda())


@pytest.mark.gpu
def test_voxel_generator_and_rotate_nms_api(golden_dir):
    from cases import sha
    from det3d.core.bbox import box_torch_ops
    from det3d.core.input.voxel_generator import VoxelGenerator
    from det3d.ops.nms.nms_cpu import rotate_nms_cc
    from oracle import cpu as ocpu
    from sessd_b200 import synth
    vg = VoxelGenerator([0.05, 0.05, 0.1], [0, -40.0, -3.0, 70.4, 40.0, 1.0], 5, 20000)
    assert list(vg.grid_size) == [1408, 1600, 40]
    v, c, n = vg.generate(synth.uniform_cloud(0, 20000))
    g = np.load(os.path.join(golden_dir, "voxel_cases.npz"))
    assert np.array_equal(c, g["uniform20k_coors"]) and (sha(v) == g["uniform20k_voxels_sha"]).all() and c.dtype == np.int32
    boxes, scores = synth.random_boxes(8, 600, spread=0.3)
    b5 = boxes[:, [0, 1, 3, 4, 6]]
    sel = box_torch_ops.rotate_nms(torch.from_numpy(b5).cuda(), torch.from_numpy(scores).cuda(), 1000, 100, 0.01)
    order = np.lexsort((np.arange(600), -scores.astype(np.float64)))
    ref = order[ocpu.rotate_nms_cc(np.concatenate([b5[order], scores[order, None]], 1), 0.01)[:100]]
    assert sel.dtype == torch.int64 and np.array_equal(sel.cpu().numpy(), ref)
    lst = rotate_nms_cc(np.concatenate([b5, scores[:, None]], 1), 0.01)
    assert isinstance(lst, list) and lst[:100] == list(ref)


def test_kitti_wire_format_loaders_match_reference_golden(golden_dir, tmp_path):
    """LoadPointCloudFromFile / LoadPointCloudAnnotations: .bin points, calib frustum and camera->lidar GT boxes equal the reference's
    box_np_ops outputs (tests/golden/kitti_wire.npz); the frustum feeds the detector's post-processing filter."""
    from cases import kitti_wire_case
    from det3d.core.bbox.geometry import frustum_planes
    from det3d.datasets.pipelines import LoadPointCloudAnnotations, LoadPointCloudFromFile
    from sessd_b200 import synth
    g = np.load(os.path.join(golden_dir, "kitti_wire.npz"))
    info = kitti_wire_case()
    pts = synth.ring_cloud(3, 5000)
    (tmp_path / "training" / "velodyne").mkdir(parents=True)
    pts.tofile(str(tmp_path / "training" / "velodyne" / "000007.bin"))
    res = dict(metadata=dict(image_prefix=str(tmp_path), num_point_features=4), lidar={}, mode="val")
    res, _ = LoadPointCloudFromFile(dataset="KittiDataset")(res, info)
    assert np.array_equal(res["lidar"]["points"], pts)
    (tmp_path / "training" / "velodyne_reduced").mkdir()
    pts[:100].tofile(str(tmp_path / "training" / "velodyne_reduced" / "000007.bin"))      # the reduced file wins when it exists
    res, _ = LoadPointCloudFromFile(dataset="KittiDataset")(res, info)
    assert res["lidar"]["points"].shape == (100, 4)
    res, _ = LoadPointCloudAnnotations(with_bbox=True)(res, info)
    assert res["calib"]["frustum"].shape == (1, 6, 4, 3) and np.array_equal(res["calib"]["frustum"], g["frustum"])
    ann = res["lidar"]["annotations"]
    assert list(ann["names"]) == ["Car", "Pedestrian", "Car", "Cyclist"]
    assert ann["boxes"].dtype == g["gt_boxes"].dtype and np.array_equal(ann["boxes"], g["gt_boxes"])
    planes = frustum_planes(res["calib"]["frustum"])            # what MultiGroupHead.predict hands to sessd_postprocess
    assert planes.shape[-2:] == (6, 4) and np.isfinite(planes).all()


def test_checkpoint_wire_format_roundtrip(tmp_path):
    """{"meta", "state_dict"} files, bare state dicts and DataParallel `module.` prefixes load into the config-built detector."""
    from collections import OrderedDict
    from det3d.torchie.trainer import load_checkpoint, save_checkpoint
    from sessd_b200 import weights
    cfg, model = _build(OUR_CFG)
    sd = weights.random_detector_state(11)
    model.load_state_dict(sd, strict=True)
    f1 = str(tmp_path / "epoch_1.pth")
    save_checkpoint(model, f1, meta=dict(epoch=1))
    ck = torch.load(f1, weights_only=False)
    assert set(ck.keys()) == {"meta", "state_dict"} and set(ck["state_dict"].keys()) == set(sd.keys())
    assert tuple(ck["state_dict"]["backbone.middle_conv.0.weight"].shape) == (3, 3, 3, 4, 16)      # spconv layout kz,ky,kx,Cin,Cout
    cfg2, fresh = _build(OUR_CFG)
    load_checkpoint(fresh, f1, map_location="cpu", strict=True)
    for k, v in fresh.state_dict().items():
        assert torch.equal(v, sd[k]), k
    f2 = str(tmp_path / "dp.pth")
    torch.save({"state_dict": OrderedDict(("module." + k, v) for k, v in sd.items())}, f2)
    cfg3, fresh2 = _build(OUR_CFG)
    load_checkpoint(fresh2, f2, map_location="cpu", strict=True)
    assert torch.equal(fresh2.state_dict()["neck.conv_0.0.weight"], sd["neck.conv_0.0.weight"])
    with pytest.raises(IOError):
        load_checkpoint(fresh2, str(tmp_path / "missing.pth"))


def test_voxelnet_forward_control_flow_with_stub_stages():
    """VoxelNet.forward wiring (CPU, stub stages): which example keys reach which stage, `_raw` twins for the teacher branch,
    predict vs loss dispatch -- the call contract of det3d/models/detectors/voxelnet_sessd.py."""
    from det3d.models.detectors import VoxelNet
    calls = []

    class Stage:
        def __init__(self, name):
            self.name = name

        def __call__(self, *a):
            calls.append((self.name, a))
            return (self.name,) + tuple(x if isinstance(x, (str, int)) else type(x).__name__ for x in a)

    class HeadStub(Stage):
        def predict(self, example, preds, test_cfg):
            return ("predict", preds, test_cfg)

        def loss(self, example, preds, preds_ema):
            return ("loss", preds, preds_ema)

    net = object.__new__(VoxelNet)
    net.reader, net.backbone, net.neck, net.bbox_head = Stage("reader"), Stage("backbone"), Stage("neck"), HeadStub("head")
    net.test_cfg = "TEST_CFG"
    ex = dict(voxels="V", num_points="NP", coordinates="C", num_voxels=[1, 2, 3], shape=["SHAPE"],
              voxels_raw="Vr", num_points_raw="NPr", coordinates_raw="Cr", num_voxels_raw=[1, 2], shape_raw=["SHAPEr"])
    out = net.forward(ex, return_loss=False)
    assert out[0] == "predict" and out[2] == "TEST_CFG"
    assert calls[0] == ("reader", ("V", "NP")) and calls[1][0] == "backbone" and calls[1][1][1:] == ("C", 3, "SHAPE")
    assert [c[0] for c in calls] == ["reader", "backbone", "neck", "head"]
    calls.clear()
    out = net.forward(ex, is_ema=[True, None])                       # teacher branch: raw copy in, head outputs back
    assert out[0] == "head" and calls[0] == ("reader", ("Vr", "NPr")) and calls[1][1][1:] == ("Cr", 2, "SHAPEr")
    calls.clear()
    out = net.forward(ex, is_ema=[False, "EMA_PREDS"], return_loss=True)
    assert out[0] == "loss" and out[2] == "EMA_PREDS"
