"""Generate the committed golden fixtures by running the REFERENCE's own code in this container.

Run once here (``python tests/golden/make_golden.py``); /root/reference does not exist on the GPU box, so
tests only ever read the ``.npz`` files this script writes.  Nothing from the reference is copied: its files
are imported *where they lie* through ``sys.modules`` shims (recipe: SURVEY.md Appendix A).

Fixtures (all inputs are re-derivable from seeds through ``sessd_b200.synth`` / the ``*_random_state`` helpers,
so only outputs -- or their hashes when large -- are stored):
  voxel_cases.npz      reference numba voxeliser (point_cloud_ops_v2.py) on 7 seeded / edge-case clouds
  iou_cases.npz        reference iou3d_cpu.cpp (compiled in place -> oracle/_ref): overlap / IoU matrices
  anchors_assign.npz   reference AnchorGeneratorRange + TargetAssigner.assign_v2 (12 seeded GT boxes)
  decode_case.npz      reference box_torch_ops.second_box_decode
  ssfa_head_case.npz   reference SSFA + Head modules (rpn_v1.py, mg_head_sessd.py) with seeded state dicts
  vfe_case.npz         reference VoxelFeatureExtractorV3
  iou_self_case.npz    reference iou3d_cpu.cpp: BEV IoU of 150 seeded boxes against themselves
  reference_config_detector.json
                       the detector this repo's det3d builds from the reference's unchanged examples/second config:
                       state-dict layout, parameter count, test_cfg and assigner output stride
"""
import hashlib
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "se-ssd_b200"))

from sessd_b200 import synth  # noqa: E402
from oracle import bev_ref, build as obuild, cpu as ocpu  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))
from cases import assign_cases, head_loss_case, iou_inputs, kitti_wire_case, odiou_pairs, sha, voxel_cases  # noqa: E402  (seeded inputs shared with the tests)


def _pkg(name):
    m = types.ModuleType(name)
    m.__path__ = [os.path.join(REF, *name.split("."))]
    sys.modules[name] = m
    return m


def _stub(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def _load(name, rel):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


# --------------------------------------------------------------------------------------------
def gen_voxel():
    pc = _load("pc_v2_ref", "det3d/ops/point_cloud/point_cloud_ops_v2.py")
    out = {}
    for name, pts, mp, mv in voxel_cases():
        v, c, n = pc.points_to_voxel(pts, np.float32(synth.VOXEL_SIZE), np.float32(synth.PC_RANGE), mp, True, mv)
        ov, oc, on = ocpu.points_to_voxel(pts, synth.VOXEL_SIZE, synth.PC_RANGE, mp, mv)
        assert (v == ov).all() and (c == oc).all() and (n == on).all(), name
        out[name + "_coors"] = c.astype(np.int32)
        out[name + "_num"] = n.astype(np.int32)
        out[name + "_voxels_sha"] = sha(v)
        out[name + "_points_sha"] = sha(pts)
        if v.shape[0] <= 2500:
            out[name + "_voxels"] = v
        print("voxel", name, v.shape)
    np.savez_compressed(os.path.join(HERE, "voxel_cases.npz"), **out)


# --------------------------------------------------------------------------------------------
def gen_iou():
    ref = obuild.load_ref() or (obuild.build_ref() and obuild.load_ref())
    b1, b2 = iou_inputs()
    a5, c5 = ocpu.boxes3d_to_bev(b1), ocpu.boxes3d_to_bev(b2)
    ov = torch.zeros(len(a5), len(c5))
    iou = torch.zeros(len(a5), len(c5))
    ref.boxes_overlap_bev_cpu(torch.from_numpy(a5), torch.from_numpy(c5), ov)
    ref.boxes_iou_bev_cpu(torch.from_numpy(a5), torch.from_numpy(c5), iou)
    assert (ocpu.boxes_overlap_bev(a5, c5) == ov.numpy()).all()
    assert (ocpu.boxes_iou_bev(a5, c5) == iou.numpy()).all()
    np.savez_compressed(os.path.join(HERE, "iou_cases.npz"), overlap=ov.numpy(), iou=iou.numpy())
    print("iou", ov.shape, float(ov.max()), int((ov > 0).sum()))


def gen_iou_self():
    ref = obuild.load_ref() or (obuild.build_ref() and obuild.load_ref())
    b, _ = synth.random_boxes(99, 150, spread=0.2)
    a5 = ocpu.boxes3d_to_bev(b)
    iou = torch.zeros(150, 150)
    ref.boxes_iou_bev_cpu(torch.from_numpy(a5), torch.from_numpy(a5), iou)
    assert (ocpu.boxes_iou_bev(a5, a5) == iou.numpy()).all()
    np.savez_compressed(os.path.join(HERE, "iou_self_case.npz"), iou=iou.numpy())
    print("iou self", iou.shape, int((iou > 0).sum()))


# --------------------------------------------------------------------------------------------
def gen_config():
    """Build the detector from the reference's examples/second config file, unchanged, through this repo's det3d (run before the
    reference shims replace `det3d` in sys.modules)."""
    from det3d.models import build_detector
    from det3d.torchie import Config
    cfg = Config.fromfile(os.path.join(REF, "examples", "second", "configs", "config.py"))
    model = build_detector(cfg.model, train_cfg=cfg.train_cfg, test_cfg=cfg.test_cfg)
    out = dict(model_type=cfg.model.type, out_size_factor=cfg.assigner.out_size_factor, test_cfg=json.loads(json.dumps(cfg.test_cfg)),
               n_params=sum(p.numel() for p in model.parameters()))
    sd = [[k, list(v.shape), str(v.dtype)] for k, v in model.state_dict().items()]
    with open(os.path.join(HERE, "reference_config_detector.json"), "w") as f:       # one state-dict entry per line
        f.write(json.dumps(out)[:-1] + ', "state_dict": [\n' + ",\n".join(json.dumps(e) for e in sd) + "\n]}\n")
    print("config: %s, %d state-dict entries, %d parameters" % (out["model_type"], len(sd), out["n_params"]))


# --------------------------------------------------------------------------------------------
def install_det3d_shims():
    for p in ("det3d", "det3d.core", "det3d.core.bbox", "det3d.core.anchor", "det3d.ops", "det3d.ops.nms",
              "det3d.models", "det3d.models.necks", "det3d.models.bbox_heads", "det3d.models.readers",
              "det3d.torchie", "det3d.utils", "det3d.core.iou3d", "det3d.core.sampler", "det3d.models.losses"):
        _pkg(p)
    _stub("spconv")
    _stub("spconv.utils", rbbox_iou=None, rbbox_intersection=None)
    _stub("det3d.ops.nms.nms_cpu", rotate_nms_cc=None, rotate_weighted_nms_cc=None)
    _stub("det3d.ops.nms.nms_gpu", nms_gpu=None, rotate_iou_gpu=None, rotate_nms_gpu=None)
    _stub("matplotlib")
    _stub("matplotlib.pyplot")
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    _orig_meshgrid = np.meshgrid
    np.meshgrid = lambda *a, **k: list(_orig_meshgrid(*a, **k))   # box_np_ops.py:814 item-assigns into it

    class _Reg:
        def register_module(self, cls):
            return cls

    reg = _Reg()
    _stub("det3d.models.registry", READERS=reg, BACKBONES=reg, NECKS=reg, HEADS=reg, LOSSES=reg, DETECTORS=reg)
    _stub("det3d.torchie.cnn", constant_init=None, kaiming_init=None, xavier_init=None)
    _stub("det3d.torchie.trainer", load_checkpoint=None)
    _stub("det3d.models.builder", build_loss=None)
    sys.modules["det3d.models"].builder = sys.modules["det3d.models.builder"]
    _stub("det3d.models.losses.metrics")
    sys.modules["det3d.models.losses"].metrics = sys.modules["det3d.models.losses.metrics"]
    sys.modules["det3d.models.losses"].accuracy = None
    _stub("det3d.core.iou3d.iou3d_utils")
    sys.modules["det3d.core.iou3d"].iou3d_utils = sys.modules["det3d.core.iou3d.iou3d_utils"]
    _stub("det3d.core.sampler.preprocess")
    sys.modules["det3d.core.sampler"].preprocess = sys.modules["det3d.core.sampler.preprocess"]
    # real norm builder needs syncbn/dist: provide the two norm types the config uses (norm.py:60-111)
    from torch import nn

    def build_norm_layer(cfg, num_features, postfix=""):
        cfg = dict(cfg)
        t = cfg.pop("type")
        cfg.setdefault("eps", 1e-5)
        layer = {"BN": nn.BatchNorm2d, "BN1d": nn.BatchNorm1d}[t](num_features, **cfg)
        return "bn" + str(postfix), layer

    misc = _load("det3d.models.utils.misc", "det3d/models/utils/misc.py")
    _stub("det3d.models.utils", Empty=misc.Empty, GroupNorm=misc.GroupNorm, Sequential=misc.Sequential,
          change_default_args=misc.change_default_args, build_norm_layer=build_norm_layer,
          get_paddings_indicator=misc.get_paddings_indicator)
    sys.modules["det3d.models"].utils = sys.modules["det3d.models.utils"]


def gen_anchors_assign():
    bn = _load("det3d.core.bbox.box_np_ops", "det3d/core/bbox/box_np_ops.py")
    sys.modules["det3d.core.bbox"].box_np_ops = bn
    bt = _load("det3d.core.bbox.box_torch_ops", "det3d/core/bbox/box_torch_ops.py")
    sys.modules["det3d.core.bbox"].box_torch_ops = bt
    rs = _load("det3d.core.bbox.region_similarity", "det3d/core/bbox/region_similarity.py")
    bc = _load("det3d.core.bbox.box_coders", "det3d/core/bbox/box_coders.py")
    ag_mod = _load("det3d.core.anchor.anchor_generator", "det3d/core/anchor/anchor_generator.py")
    _load("det3d.core.anchor.target_ops_v2", "det3d/core/anchor/target_ops_v2.py")
    ta_mod = _load("det3d.core.anchor.target_assigner", "det3d/core/anchor/target_assigner.py")
    ag = ag_mod.AnchorGeneratorRange(anchor_ranges=[0, -40.0, -1.0, 70.4, 40.0, -1.0], sizes=[1.6, 3.9, 1.56],
                                     rotations=[0, 1.57], velocities=None, class_name="Car",
                                     match_threshold=0.6, unmatch_threshold=0.45)
    ta = ta_mod.TargetAssigner(box_coder=bc.GroundBox3dCoderTorch(linear_dim=False, vec_encode=False, n_dim=7),
                               anchor_generators=[ag], region_similarity_calculator=rs.NearestIouSimilarity(),
                               positive_fraction=None, sample_size=512)
    ad = ta.generate_anchors_dict([1, 200, 176])
    anchors = ad["Car"]["anchors"]
    gt, _ = synth.random_boxes(21, 12)
    gt[:, 2] = -1.0
    res = ta.assign_v2(ad, gt, None, gt_classes=np.ones(12, np.int32), gt_names=np.array(["Car"] * 12),
                       enable_similar_type=True)
    from oracle import anchors as oa
    mine = oa.create_anchors_3d_range()
    assert (mine.reshape(-1, 7) == anchors.reshape(-1, 7)).all()
    om = oa.assign_targets(anchors.reshape(-1, 7), gt)
    assert (om["labels"] == res["labels"]).all()
    assert np.array_equal(om["bbox_targets"], res["bbox_targets"])
    pos = np.nonzero(res["labels"] > 0)[0]
    np.savez_compressed(os.path.join(HERE, "anchors_assign.npz"),
                        anchors_sha=sha(anchors), anchors_head=anchors.reshape(-1, 7)[:704].copy(),
                        anchors_tail=anchors.reshape(-1, 7)[-704:].copy(),
                        labels=res["labels"].astype(np.int8), pos_idx=pos.astype(np.int32),
                        pos_targets=res["bbox_targets"][pos], weights_sum=np.float64(res["bbox_outside_weights"].sum()))
    print("anchors", anchors.shape, "pos", len(pos), "neg", int((res["labels"] == 0).sum()))
    # more assigner cases (empty / single / many GT, GT without any overlap, forced-only positives, ties)
    cases = {}
    for name, g in assign_cases():
        m = len(g)
        r = ta.assign_v2(ad, g, None, gt_classes=np.ones(m, np.int32), gt_names=np.array(["Car"] * m), enable_similar_type=True)
        o = oa.assign_targets(anchors.reshape(-1, 7), g)
        assert (o["labels"] == r["labels"]).all(), name
        assert np.array_equal(o["bbox_targets"], r["bbox_targets"]), name
        assert np.array_equal(o["bbox_outside_weights"], r["bbox_outside_weights"]), name
        assert np.array_equal(o["positive_gt_id"], r["positive_gt_id"][0]), name
        p_ = np.nonzero(r["labels"] > 0)[0]
        cases[name + "_labels"] = r["labels"].astype(np.int8)
        cases[name + "_pos_idx"] = p_.astype(np.int32)
        cases[name + "_pos_targets"] = r["bbox_targets"][p_]
        cases[name + "_positive_gt_id"] = np.asarray(r["positive_gt_id"][0], np.int32)
        print("assign", name, "gt", m, "pos", len(p_), "neg", int((r["labels"] == 0).sum()), "ignore", int((r["labels"] < 0).sum()))
    np.savez_compressed(os.path.join(HERE, "assign_cases.npz"), **cases)
    # decode fixture from the reference torch op
    g = torch.Generator().manual_seed(5)
    enc = torch.randn(2048, 7, generator=g) * 0.3
    anc = torch.from_numpy(anchors.reshape(-1, 7)[::34][:2048].copy())
    dec = bt.second_box_decode(enc, anc)
    assert torch.equal(dec, bev_ref.box_decode(enc, anc))
    np.savez_compressed(os.path.join(HERE, "decode_case.npz"), decoded=dec.numpy())
    print("decode", dec.shape)


def gen_wire():
    """KITTI wire format: reference box_np_ops.get_valid_frustum / box_camera_to_lidar / change_box3d_center_ on a synthetic calibration."""
    bn = sys.modules.get("det3d.core.bbox.box_np_ops") or _load("det3d.core.bbox.box_np_ops", "det3d/core/bbox/box_np_ops.py")
    info = kitti_wire_case()
    c = info["calib"]
    fr = bn.get_valid_frustum(c["R0_rect"], c["Tr_velo_to_cam"], c["P2"], info["image"]["image_shape"])
    a = info["annos"]
    keep = [i for i, x in enumerate(a["name"]) if x != "DontCare"]
    gt = np.concatenate([a["location"][keep], a["dimensions"][keep], a["rotation_y"][keep][..., np.newaxis]], axis=1).astype(np.float32)
    gt = bn.box_camera_to_lidar(gt, c["R0_rect"], c["Tr_velo_to_cam"])
    bn.change_box3d_center_(gt, [0.5, 0.5, 0], [0.5, 0.5, 0.5])
    np.savez_compressed(os.path.join(HERE, "kitti_wire.npz"), frustum=fr, gt_boxes=gt)
    print("wire: frustum", fr.shape, fr.dtype, "gt", gt.shape, gt.dtype)


def gen_loss():
    """Supervised head loss terms from the REFERENCE's own loss classes (losses.py) and head helpers (mg_head_sessd.py)."""
    from oracle import loss_ref
    _stub("det3d.models.losses.utils", weight_reduce_loss=None)
    losses = _load("det3d.models.losses.losses", "det3d/models/losses/losses.py")
    mg = sys.modules.get("det3d.models.bbox_heads.mg_head_sessd") or _load("det3d.models.bbox_heads.mg_head_sessd",
                                                                           "det3d/models/bbox_heads/mg_head_sessd.py")
    head_np, anc_np, labels_np, targets_np = head_loss_case()
    head = torch.from_numpy(head_np).clone().requires_grad_(True)
    anchors, labels, reg_targets = torch.from_numpy(anc_np), torch.from_numpy(labels_np).long(), torch.from_numpy(targets_np)
    box, cls, dr = loss_ref.split_head(head)
    B = 2
    loss_norm = dict(type="NormByNumPositives", pos_cls_weight=1.0, neg_cls_weight=1.0)
    cls_w, reg_w, cared = mg.MultiGroupHead.prepare_loss_weights(None, labels, loss_norm=loss_norm, dtype=torch.float32)
    cls_targets = (labels * cared.type_as(labels)).unsqueeze(-1)
    enc_p, enc_t = mg.add_sin_difference(box, reg_targets)
    loc = losses.WeightedSmoothL1Loss(sigma=3.0, code_weights=[1.0] * 7, codewise=True, loss_weight=2.0)(enc_p, enc_t, weights=reg_w)
    cl = losses.SigmoidFocalLoss(alpha=0.25, gamma=2.0, loss_weight=1.0)(cls.unsqueeze(-1), cls_targets, weights=cls_w)
    dir_t = mg.get_direction_target(anchors.unsqueeze(0).expand(B, -1, -1).contiguous(), reg_targets, dir_offset=0.0)
    w = (labels > 0).type_as(dr)
    w = w / torch.clamp(w.sum(-1, keepdim=True), min=1.0)
    dl = losses.WeightedSoftmaxClassificationLoss(name="direction_classifier", loss_weight=0.2)(dr, dir_t, weights=w)
    cls_pos, cls_neg = mg._get_pos_neg_loss(cl, labels)
    total = 1.0 * cl.sum() / B + 2.0 * loc.sum() / B + 0.2 * dl.sum() / B
    total.backward()
    grad = head.grad.numpy()
    # oracle == reference
    o = loss_ref.head_supervised_loss(*loss_ref.split_head(torch.from_numpy(head_np)), anchors, labels, reg_targets)
    for k, ref in (("cls", cl.sum((1, 2))), ("loc", loc.sum((1, 2))), ("dir", dl.sum(1))):
        assert torch.allclose(o[k], ref.detach(), rtol=1e-6, atol=1e-7), (k, o[k], ref)
    pos = np.nonzero(labels_np.reshape(-1) > 0)[0]
    sample = np.arange(0, labels_np.size, 97)
    np.savez_compressed(os.path.join(HERE, "head_loss_case.npz"), cls=cl.sum((1, 2)).detach().numpy(), loc=loc.sum((1, 2)).detach().numpy(),
                        dir=dl.sum(1).detach().numpy(), cls_pos=np.float32(cls_pos.item()), cls_neg=np.float32(cls_neg.item()),
                        total=np.float32(total.item()), grad_sha=sha(grad), grad_abs_sum=np.float64(np.abs(grad).sum()),
                        grad_pix_idx=np.unique(np.concatenate([pos // 2, sample // 2])).astype(np.int32),
                        grad_pix=grad.reshape(-1, 24)[np.unique(np.concatenate([pos // 2, sample // 2]))])
    print("loss: cls", cl.sum((1, 2)).tolist(), "loc", loc.sum((1, 2)).tolist(), "dir", dl.sum(1).tolist(), "total", float(total))


def gen_consistency():
    """SE-SSD consistency loss of the REFERENCE (mg_head_sessd.py:573-703: nn_distance + consistency_loss, run unmodified on the CPU): the
    rotated BEV IoU inside comes from the reference's own iou3d_cpu.cpp (oracle/_ref) behind the reference's boxes3d_to_bev_torch, `.cuda()`
    is a no-op here.  Stores the loss and d(loss)/d(student predictions)."""
    import types
    from cases import consistency_case
    _stub("det3d.models.losses.utils", weight_reduce_loss=None)
    losses = sys.modules.get("det3d.models.losses.losses") or _load("det3d.models.losses.losses", "det3d/models/losses/losses.py")
    mg = sys.modules.get("det3d.models.bbox_heads.mg_head_sessd") or _load("det3d.models.bbox_heads.mg_head_sessd",
                                                                           "det3d/models/bbox_heads/mg_head_sessd.py")
    bt = sys.modules.get("det3d.core.bbox.box_torch_ops") or _load("det3d.core.bbox.box_torch_ops", "det3d/core/bbox/box_torch_ops.py")
    iu = _load("det3d.core.iou3d.utils", "det3d/core/iou3d/utils.py")
    ref = obuild.load_ref() or (obuild.build_ref() and obuild.load_ref())

    def boxes_iou_bev_gpu(a, b):
        a5, b5 = iu.boxes3d_to_bev_torch(a.detach(), "wlh", False).contiguous(), iu.boxes3d_to_bev_torch(b.detach(), "wlh", False).contiguous()
        out = torch.zeros(a5.shape[0], b5.shape[0])
        ref.boxes_iou_bev_cpu(a5, b5, out)
        return out

    mg.iou3d_utils = types.SimpleNamespace(boxes_iou_bev_gpu=boxes_iou_bev_gpu)
    mg.box_torch_ops = bt
    torch.Tensor.cuda = lambda self, *a, **k: self
    stu_np, tea_np, anc, trans = consistency_case()
    stu = {k: torch.from_numpy(v).clone().requires_grad_(True) for k, v in stu_np.items()}
    tea = {k: torch.from_numpy(v).clone() for k, v in tea_np.items()}
    head = types.SimpleNamespace(
        box_coder=types.SimpleNamespace(decode_torch=lambda enc, a: bt.second_box_decode(enc, a, False, False)),
        post_center_range=torch.tensor([0, -40.0, -5.0, 70.4, 40.0, 5.0]),
        loss_reg=losses.WeightedSmoothL1Loss(sigma=3.0, code_weights=[1.0] * 7, codewise=True, loss_weight=2.0),
        loss_iou_consistency=losses.WeightedSmoothL1Loss(sigma=3.0, code_weights=None, codewise=True, loss_weight=1.0),
        loss_score_consistency=losses.WeightedSmoothL1Loss(sigma=3.0, code_weights=None, codewise=True, loss_weight=1.0),
        loss_dir_consistency=torch.nn.MSELoss(reduction="mean"))
    head.nn_distance = types.MethodType(mg.MultiGroupHead.nn_distance, head)
    example = dict(transformation=trans, annos_raw=[None, None], anchors=[torch.from_numpy(anc)[None, None].expand(1, 2, -1, -1)])
    # example["anchors"][0][0] must be the [A, 7] anchor table
    example["anchors"] = [[torch.from_numpy(anc)]]
    loss = mg.MultiGroupHead.consistency_loss(head, [stu], [tea], example)
    loss.sum().backward()
    g = {k: v.grad.numpy() for k, v in stu.items() if v.grad is not None}
    nz = np.nonzero(np.abs(g["box_preds"]).sum(-1).reshape(-1))[0]
    np.savez_compressed(os.path.join(HERE, "consistency_case.npz"), loss=loss.detach().numpy().astype(np.float32),
                        grad_rows=nz.astype(np.int32), grad_box=g["box_preds"].reshape(-1, 7)[nz], grad_cls=g["cls_preds"].reshape(-1)[nz],
                        grad_iou=g["iou_preds"].reshape(-1)[nz], grad_box_abs_sum=np.float64(np.abs(g["box_preds"]).sum()),
                        grad_cls_abs_sum=np.float64(np.abs(g["cls_preds"]).sum()), grad_iou_abs_sum=np.float64(np.abs(g["iou_preds"]).sum()),
                        grad_dir_is_none=np.bool_("dir_cls_preds" not in g or not np.abs(g.get("dir_cls_preds", 0)).sum()))
    print("consistency: loss", loss.tolist(), "rows with gradient", len(nz), "grad sums", float(np.abs(g["box_preds"]).sum()),
          float(np.abs(g["cls_preds"]).sum()), float(np.abs(g["iou_preds"]).sum()))


def gen_odiou():
    """ODIoU loss of the REFERENCE (det3d/models/losses/odious.py, imported where it lies; runs on the CPU): per-pair value and the gradient
    w.r.t. the predicted box through the reference's own custom autograd Functions."""
    od = _load("odious_ref", "det3d/models/losses/odious.py")
    g, q = odiou_pairs()
    vals, grads = [], []
    for i in range(len(g)):
        gi = torch.from_numpy(g[i:i + 1].copy())
        qi = torch.from_numpy(q[i:i + 1].copy()).requires_grad_(True)
        loss = od.odiou_3D()(gi, qi, torch.ones(1), 2)            # = 2.0 * odiou / 2
        loss.backward()
        vals.append(float(loss.detach()))
        grads.append(qi.grad.numpy()[0].copy())
    np.savez_compressed(os.path.join(HERE, "odiou_case.npz"), odiou=np.float32(vals), grad_q=np.stack(grads, 0).astype(np.float32))
    print("odiou:", np.round(np.float32(vals), 4).tolist()[:8], "...", np.round(np.float32(vals)[-6:], 4).tolist())


def gen_models():
    import logging

    rpn = _load("det3d.models.necks.rpn_v1", "det3d/models/necks/rpn_v1.py")
    ssfa = rpn.SSFA(layer_nums=[5], ds_layer_strides=[1], ds_num_filters=[128], us_layer_strides=[1],
                    us_num_filters=[128], num_input_features=128, norm_cfg=None, logger=logging.getLogger("RPN"))
    sd = bev_ref.ssfa_random_state(7)
    missing = ssfa.load_state_dict(sd, strict=True)
    print("ssfa load:", missing)
    ssfa.eval()
    g = torch.Generator().manual_seed(8)
    x = torch.relu(torch.randn(1, 128, 24, 16, generator=g))
    with torch.no_grad():
        y = ssfa(x)
        y_or = bev_ref.ssfa_forward(x, sd)
    err = float((y - y_or).abs().max() / y.abs().max())
    print("ssfa ref vs oracle rel err", err)
    assert err < 1e-5
    # Head (mg_head_sessd.py:195-230)
    mg = _load("det3d.models.bbox_heads.mg_head_sessd", "det3d/models/bbox_heads/mg_head_sessd.py")
    head = mg.Head(128, 14, 2, use_dir=True, num_dir=4, header=False)
    hsd = bev_ref.head_random_state(9, prefix="")
    head.load_state_dict(hsd, strict=True)
    with torch.no_grad():
        h = head(y)
    h_or = bev_ref.head_forward(y, hsd, prefix="")
    for k in h:
        assert torch.allclose(h[k], h_or[k], rtol=1e-5, atol=1e-6), k
    np.savez_compressed(os.path.join(HERE, "ssfa_head_case.npz"), ssfa_out=y.numpy(),
                        **{k: v.numpy() for k, v in h.items()})
    # VFE V3
    ve = _load("det3d.models.readers.voxel_encoder", "det3d/models/readers/voxel_encoder.py")
    vfe = ve.VoxelFeatureExtractorV3(num_input_features=4)
    pts = synth.uniform_cloud(1, 2000)
    v, c, n = ocpu.points_to_voxel(pts, synth.VOXEL_SIZE, synth.PC_RANGE, 5, 20000)
    m = vfe(torch.from_numpy(v), torch.from_numpy(n))
    assert torch.equal(m, bev_ref.vfe_mean(torch.from_numpy(v), torch.from_numpy(n)))
    np.savez_compressed(os.path.join(HERE, "vfe_case.npz"), mean=m.numpy())
    print("vfe", m.shape)


if __name__ == "__main__":
    only = sys.argv[1:]           # e.g. `make_golden.py assign` regenerates only the anchor / assigner fixtures
    if not only or "voxel" in only:
        gen_voxel()
    if not only or "iou" in only:
        gen_iou()
        gen_iou_self()
    if "config" in only:             # imports this repo's det3d, which the shims below replace: run on its own (`make_golden.py config`)
        gen_config()
    install_det3d_shims()
    if not only or "assign" in only:
        gen_anchors_assign()
    if not only or "odiou" in only:
        gen_odiou()
    if not only or "loss" in only:
        gen_loss()
    if not only or "wire" in only:
        gen_wire()
    if "consistency" in only:        # patches torch.Tensor.cuda: run on its own (`make_golden.py consistency`)
        gen_consistency()
    if not only or "models" in only:
        gen_models()
