"""CPU: the oracle restatements against the committed golden vectors produced by the REFERENCE's own code
(tests/golden/make_golden.py) -- this is what pins the oracle."""
import os

import numpy as np
import pytest
import torch

from cases import iou_inputs, sha, voxel_cases


def test_oracle_voxeliser_equals_reference_golden(golden_dir):
    from oracle import cpu as ocpu
    from sessd_b200 import synth
    g = np.load(os.path.join(golden_dir, "voxel_cases.npz"))
    for name, pts, mp, mv in voxel_cases():
        assert (sha(pts) == g[name + "_points_sha"]).all()
        v, c, n = ocpu.points_to_voxel(pts, synth.VOXEL_SIZE, synth.PC_RANGE, mp, mv)
        assert np.array_equal(c, g[name + "_coors"]) and np.array_equal(n, g[name + "_num"])
        assert (sha(v) == g[name + "_voxels_sha"]).all()
    # semantic edge cases of the sequential loop
    assert g["cut300_coors"].shape[0] == 300 and g["clustered_num"].max() == 5 and g["empty_coors"].shape[0] == 0


def test_oracle_rotated_iou_equals_reference_golden_bit_exact(golden_dir):
    from oracle import cpu as ocpu
    g = np.load(os.path.join(golden_dir, "iou_cases.npz"))
    b1, b2 = iou_inputs()
    a5, c5 = ocpu.boxes3d_to_bev(b1), ocpu.boxes3d_to_bev(b2)
    assert np.array_equal(ocpu.boxes_overlap_bev(a5, c5), g["overlap"])
    assert np.array_equal(ocpu.boxes_iou_bev(a5, c5), g["iou"])


def test_oracle_matches_compiled_reference_when_present(golden_dir):
    """The reference's iou3d_cpu.cpp on 150 seeded boxes against themselves, bit-exact: always against its recorded output
    (tests/golden/iou_self_case.npz), and live as well when oracle/_ref holds the reference compiled in place."""
    from oracle import build as obuild, cpu as ocpu
    from sessd_b200 import synth
    b, _ = synth.random_boxes(99, 150, spread=0.2)
    a5 = ocpu.boxes3d_to_bev(b)
    got = ocpu.boxes_iou_bev(a5, a5)
    assert np.array_equal(got, np.load(os.path.join(golden_dir, "iou_self_case.npz"))["iou"])
    ref = obuild.load_ref()
    if ref is None:
        return
    out = torch.zeros(150, 150)
    ref.boxes_iou_bev_cpu(torch.from_numpy(a5), torch.from_numpy(a5), out)
    assert np.array_equal(out.numpy(), got)


def test_oracle_anchors_and_assigner_equal_reference_golden(golden_dir):
    from oracle import anchors as oa
    from sessd_b200 import synth
    g = np.load(os.path.join(golden_dir, "anchors_assign.npz"))
    anc = oa.create_anchors_3d_range().reshape(-1, 7)
    assert (sha(anc) == g["anchors_sha"]).all()
    assert np.array_equal(anc[:704], g["anchors_head"]) and np.array_equal(anc[-704:], g["anchors_tail"])
    gt, _ = synth.random_boxes(21, 12)
    gt[:, 2] = -1.0
    res = oa.assign_targets(anc, gt)
    assert np.array_equal(res["labels"].astype(np.int8), g["labels"])
    pos = np.nonzero(res["labels"] > 0)[0]
    assert np.array_equal(pos, g["pos_idx"])
    assert np.array_equal(res["bbox_targets"][pos], g["pos_targets"])
    assert float(res["bbox_outside_weights"].sum()) == float(g["weights_sum"])


def test_oracle_assigner_equals_reference_on_all_golden_cases(golden_dir):
    """Empty / single / 40 GT, GT without any overlap, forced-only positives, duplicate GT, ties, near-bbox swap boundary."""
    from cases import assign_cases
    from oracle import anchors as oa
    g = np.load(os.path.join(golden_dir, "assign_cases.npz"))
    anc = oa.create_anchors_3d_range().reshape(-1, 7)
    for name, gt in assign_cases():
        res = oa.assign_targets(anc, gt)
        assert np.array_equal(res["labels"].astype(np.int8), g[name + "_labels"]), name
        pos = np.nonzero(res["labels"] > 0)[0]
        assert np.array_equal(pos, g[name + "_pos_idx"]), name
        assert np.array_equal(res["bbox_targets"][pos], g[name + "_pos_targets"]), name
        assert np.array_equal(res["positive_gt_id"], g[name + "_positive_gt_id"]), name


def test_oracle_decode_ssfa_head_vfe_equal_reference_golden(golden_dir):
    from oracle import anchors as oa, bev_ref, cpu as ocpu
    from sessd_b200 import synth
    g = np.load(os.path.join(golden_dir, "decode_case.npz"))
    gen = torch.Generator().manual_seed(5)
    enc = torch.randn(2048, 7, generator=gen) * 0.3
    anc = torch.from_numpy(oa.create_anchors_3d_range().reshape(-1, 7)[::34][:2048].copy())
    assert np.array_equal(bev_ref.box_decode(enc, anc).numpy(), g["decoded"])
    np.testing.assert_allclose(ocpu.box_decode(enc.numpy(), anc.numpy()), g["decoded"], rtol=2e-6, atol=1e-6)
    g2 = np.load(os.path.join(golden_dir, "ssfa_head_case.npz"))
    x = torch.relu(torch.randn(1, 128, 24, 16, generator=torch.Generator().manual_seed(8)))
    y = bev_ref.ssfa_forward(x, bev_ref.ssfa_random_state(7))
    np.testing.assert_allclose(y.numpy(), g2["ssfa_out"], rtol=1e-5, atol=1e-6)
    h = bev_ref.head_forward(y, bev_ref.head_random_state(9, prefix=""), prefix="")
    for k in ("box_preds", "cls_preds", "dir_cls_preds", "iou_preds"):
        np.testing.assert_allclose(h[k].numpy(), g2[k], rtol=1e-5, atol=1e-6)
    g3 = np.load(os.path.join(golden_dir, "vfe_case.npz"))
    v, _c, n = ocpu.points_to_voxel(synth.uniform_cloud(1, 2000), synth.VOXEL_SIZE, synth.PC_RANGE, 5, 20000)
    assert np.array_equal(bev_ref.vfe_mean(torch.from_numpy(v), torch.from_numpy(n)).numpy(), g3["mean"])


def test_oracle_sparse_shapes_match_reference_comments():
    """scn.py:113,122,134,146 pin the output-shape rule; SURVEY.md 8(d) pins the active-site / pair counts."""
    from oracle import cpu as ocpu, spconv_ref as S
    from sessd_b200 import synth
    v, c, n = ocpu.points_to_voxel(synth.uniform_cloud(0, 20000), synth.VOXEL_SIZE, synth.PC_RANGE, 5, 20000)
    cur = np.concatenate([np.zeros((len(c), 1), np.int32), c], 1)
    shape = (41, 1600, 1408)
    counts, pairs, shapes = [], [], []
    for kind, _ci, _co, ks, st, pd, _key in S.SPMIDDLE_FHD_LAYERS:
        if kind != "spconv":
            continue
        oc, oshape = S.strided_out_coors(cur, shape, ks, st, pd)
        pairs.append(int((S.neighbor_table(cur, shape, oc, ks, st, pd) >= 0).sum()))
        cur, shape = oc, oshape
        counts.append(len(oc))
        shapes.append(oshape)
    assert shapes == [(21, 800, 704), (11, 400, 352), (5, 200, 176), (2, 200, 176)]
    assert counts == [67955, 103374, 85774, 52169]
    assert pairs == [68148, 228309, 323785, 104137]


def test_rotate_nms_second_opinion_exact_polygon_clip():
    """The oracle swaps boost::geometry for iou3d_cpu arithmetic (boost is absent): cross-check the keep set against
    an exact fp64 convex-polygon clip.  Differences are only allowed for pairs within 1e-4 of the threshold."""
    from oracle import cpu as ocpu
    from sessd_b200 import synth

    def corners(b):
        x, y, w, l, r = [float(v) for v in b]
        c, s = np.cos(r), np.sin(r)
        pts = np.array([[-w / 2, -l / 2], [-w / 2, l / 2], [w / 2, l / 2], [w / 2, -l / 2]])
        return np.stack([pts[:, 0] * c + pts[:, 1] * s + x, -pts[:, 0] * s + pts[:, 1] * c + y], 1)

    def area(p):
        return 0.5 * abs(np.dot(p[:, 0], np.roll(p[:, 1], -1)) - np.dot(p[:, 1], np.roll(p[:, 0], -1))) if len(p) >= 3 else 0.0

    def cross2(u, v):
        return u[0] * v[1] - u[1] * v[0]

    def clip(subj, clipper):
        out = subj
        sign = np.sign(cross2(clipper[1] - clipper[0], clipper[2] - clipper[1]))
        for i in range(4):
            a, b = clipper[i], clipper[(i + 1) % 4]
            inp, out = out, []
            if len(inp) == 0:
                break
            for j in range(len(inp)):
                p, q = inp[j], inp[(j + 1) % len(inp)]
                sp = sign * cross2(b - a, p - a)
                sq = sign * cross2(b - a, q - a)
                if sp >= 0:
                    out.append(p)
                if sp * sq < 0:
                    t = sp / (sp - sq)
                    out.append(p + t * (q - p))
            out = np.array(out) if len(out) else np.zeros((0, 2))
        return out

    boxes, scores = synth.random_boxes(5, 400, spread=0.3)
    b5 = boxes[:, [0, 1, 3, 4, 6]].astype(np.float64)
    order = np.argsort(-scores, kind="stable")
    cs = [corners(b) for b in b5]
    dead = np.zeros(len(b5), bool)
    keep = []
    near = False
    for ii, i in enumerate(order):
        if dead[i]:
            continue
        keep.append(i)
        for j in order[ii + 1:]:
            if dead[j]:
                continue
            inter = area(clip(cs[i], cs[j]))
            iou = inter / (b5[i, 2] * b5[i, 3] + b5[j, 2] * b5[j, 3] - inter)
            near |= abs(iou - 0.01) < 1e-4
            if iou >= 0.01:
                dead[j] = True
    dets = np.concatenate([b5[order], scores[order, None]], 1).astype(np.float32)
    ref = order[ocpu.rotate_nms_cc(dets, 0.01, ge=True)]
    if not near:
        assert np.array_equal(np.array(keep), ref)


def test_oracle_head_loss_equals_reference_golden(golden_dir):
    """Supervised head loss (focal + sin-difference smooth-L1 + direction CE) and its autograd gradient vs the reference's loss classes."""
    import torch
    from cases import head_loss_case, sha
    from oracle import loss_ref
    g = np.load(os.path.join(golden_dir, "head_loss_case.npz"))
    head_np, anc, labels, targets = head_loss_case()
    head = torch.from_numpy(head_np).clone().requires_grad_(True)
    o = loss_ref.head_supervised_loss(*loss_ref.split_head(head), torch.from_numpy(anc), torch.from_numpy(labels).long(), torch.from_numpy(targets))
    for k in ("cls", "loc", "dir"):
        np.testing.assert_allclose(o[k].detach().numpy(), g[k], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(float(o["cls_pos"].detach().sum() / 2), float(g["cls_pos"]), rtol=1e-6)
    np.testing.assert_allclose(float(o["cls_neg"].detach().sum() / 2), float(g["cls_neg"]), rtol=1e-6)
    total = (o["cls"].sum() + 2.0 * o["loc"].sum() + 0.2 * o["dir"].sum()) / 2
    np.testing.assert_allclose(float(total.detach()), float(g["total"]), rtol=1e-6)
    total.backward()
    grad = head.grad.numpy().reshape(-1, 24)
    np.testing.assert_allclose(grad[g["grad_pix_idx"]], g["grad_pix"], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(np.abs(grad).sum(), float(g["grad_abs_sum"]), rtol=1e-5)


# ---------------------------------------------------------------------------------------------------- second opinion for spconv_ref
@pytest.mark.parametrize("kind,ks,st,pd", [("subm", (3, 3, 3), (1, 1, 1), (1, 1, 1)), ("spconv", (3, 3, 3), (2, 2, 2), (1, 1, 1)),
                                           ("spconv", (3, 3, 3), (2, 2, 2), (0, 1, 1)), ("spconv", (3, 1, 1), (2, 1, 1), (0, 0, 0))])
def test_spconv_restatement_equals_dense_conv3d(kind, ks, st, pd):
    """spconv 1.x is absent (parity unpinned), so the restatement in oracle/spconv_ref.py is cross-checked against an INDEPENDENT
    implementation: torch.nn.functional.conv3d on the densified (cropped) volume.
      * SparseConv3d: the output set is every position reached by at least one active input, and the values equal the dense
        cross-correlation there (everywhere else the dense result is exactly 0);
      * SubMConv3d: the output set is the input set; values = dense cross-correlation (padding k//2) sampled at the active sites.
    Covers the four (kernel, stride, padding) combinations of scn.py:106-149, 2 frames, ~12 % occupancy."""
    import torch
    import torch.nn.functional as F
    from oracle import spconv_ref as S
    rng = np.random.default_rng(11)
    B, shape, cin, cout = 2, (9, 20, 18), 5, 7
    occ = rng.random((B,) + shape) < 0.12
    coors = np.argwhere(occ).astype(np.int32)                       # ascending (b, z, y, x) = canonical order
    feat = rng.standard_normal((len(coors), cin))
    w = rng.standard_normal(ks + (cin, cout))                       # spconv layout [kz,ky,kx,Cin,Cout]
    dense = np.zeros((B, cin) + shape)
    dense[coors[:, 0], :, coors[:, 1], coors[:, 2], coors[:, 3]] = feat
    wt = torch.from_numpy(w).permute(4, 3, 0, 1, 2).contiguous()    # conv3d layout [Cout,Cin,kz,ky,kx]
    if kind == "subm":
        out_coors, oshape = coors, shape
        nbr = S.neighbor_table(coors, shape, coors, ks, (1, 1, 1), tuple(k // 2 for k in ks))
        ref = F.conv3d(torch.from_numpy(dense), wt, None, 1, tuple(k // 2 for k in ks)).numpy()
    else:
        out_coors, oshape = S.strided_out_coors(coors, shape, ks, st, pd)
        nbr = S.neighbor_table(coors, shape, out_coors, ks, st, pd)
        ref = F.conv3d(torch.from_numpy(dense), wt, None, st, pd).numpy()
        assert tuple(ref.shape[2:]) == oshape
        # output set == positions reached by an active input == support of conv3d(occupancy, ones)
        reach = F.conv3d(torch.from_numpy(occ[:, None].astype(np.float64)), torch.ones((1, 1) + ks, dtype=torch.float64), None, st, pd).numpy()[:, 0] > 0
        assert np.array_equal(np.argwhere(reach).astype(np.int32), out_coors)
        mask = np.zeros_like(reach)
        mask[out_coors[:, 0], out_coors[:, 1], out_coors[:, 2], out_coors[:, 3]] = True
        assert np.abs(ref[~np.broadcast_to(mask[:, None], ref.shape)]).max() == 0.0
    got = S.conv_from_nbr(feat, nbr, w.reshape(-1, cin, cout), np.float64)
    want = ref[out_coors[:, 0], :, out_coors[:, 1], out_coors[:, 2], out_coors[:, 3]]
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    # canonical pairs: every (in, out) pair satisfies pos_in = pos_out * stride - pad + k
    for k, (pi, po) in enumerate(S.pairs_from_nbr(nbr)):
        kz, r = divmod(k, ks[1] * ks[2])
        ky, kx = divmod(r, ks[2])
        s3 = (1, 1, 1) if kind == "subm" else st
        p3 = tuple(q // 2 for q in ks) if kind == "subm" else pd
        exp = out_coors[po, 1:] * np.array(s3) - np.array(p3) + np.array([kz, ky, kx])
        assert np.array_equal(coors[pi, 1:], exp) and np.array_equal(coors[pi, 0], out_coors[po, 0])


@pytest.mark.parametrize("kind,ks,st,pd", [("subm", (3, 3, 3), (1, 1, 1), (1, 1, 1)), ("spconv", (3, 3, 3), (2, 2, 2), (1, 1, 1)),
                                           ("spconv", (3, 3, 3), (2, 2, 2), (0, 1, 1)), ("spconv", (3, 1, 1), (2, 1, 1), (0, 0, 0))])
def test_spconv_backward_restatement_equals_dense_autograd(kind, ks, st, pd):
    """oracle/spconv_grad_ref.py (oracle of the not-yet-built backward kernels) against an INDEPENDENT implementation: torch autograd
    through F.conv3d on the densified volume, loss = <out sampled at the output set, G>.  Also the two identities the device design
    rests on: dgrad == the FORWARD gather run with (G, transposed table, W^T), and for SubM layers the transposed table is the
    offset-reversed table (no second rulebook).  + eval-mode BN / ReLU backward vs autograd."""
    import torch
    import torch.nn.functional as F
    from oracle import spconv_grad_ref as SG, spconv_ref as S
    rng = np.random.default_rng(23)
    B, shape, cin, cout = 2, (9, 14, 12), 4, 6
    occ = rng.random((B,) + shape) < 0.15
    coors = np.argwhere(occ).astype(np.int32)
    feat = rng.standard_normal((len(coors), cin))
    w = rng.standard_normal(ks + (cin, cout))
    if kind == "subm":
        out_coors, s3, p3 = coors, (1, 1, 1), tuple(k // 2 for k in ks)
    else:
        out_coors, _ = S.strided_out_coors(coors, shape, ks, st, pd)
        s3, p3 = st, pd
    nbr = S.neighbor_table(coors, shape, out_coors, ks, s3, p3)
    G = rng.standard_normal((len(out_coors), cout))
    dense = torch.zeros((B, cin) + shape, dtype=torch.float64)
    dense[coors[:, 0], :, coors[:, 1], coors[:, 2], coors[:, 3]] = torch.from_numpy(feat)
    dense.requires_grad_(True)
    wt = torch.from_numpy(w).permute(4, 3, 0, 1, 2).contiguous().requires_grad_(True)
    out = F.conv3d(dense, wt, None, s3, p3)
    sampled = out[out_coors[:, 0], :, out_coors[:, 1], out_coors[:, 2], out_coors[:, 3]]
    (sampled * torch.from_numpy(G)).sum().backward()
    want_gfeat = dense.grad[coors[:, 0], :, coors[:, 1], coors[:, 2], coors[:, 3]].numpy()
    want_gw = wt.grad.permute(2, 3, 4, 1, 0).reshape(-1, cin, cout).numpy()
    wk = w.reshape(-1, cin, cout)
    gfeat, gw = SG.conv_backward_from_nbr(feat, nbr, wk, G)
    np.testing.assert_allclose(gfeat, want_gfeat, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(gw, want_gw, rtol=1e-12, atol=1e-12)
    # dgrad as a forward gather over the transposed table with transposed weights
    nbr_t = SG.transpose_nbr(nbr, len(coors))
    np.testing.assert_allclose(S.conv_from_nbr(G, nbr_t, np.ascontiguousarray(wk.transpose(0, 2, 1)), np.float64), want_gfeat, rtol=1e-12, atol=1e-12)
    if kind == "subm":
        assert np.array_equal(nbr_t, nbr[:, ::-1])
    # eval-mode BatchNorm1d + ReLU behind the conv
    gamma, beta, mean, var = rng.uniform(0.5, 1.5, cout), rng.standard_normal(cout), rng.standard_normal(cout), rng.uniform(0.5, 2.0, cout)
    x = torch.from_numpy(S.conv_from_nbr(feat, nbr, wk, np.float64)).requires_grad_(True)
    y = torch.relu((x - torch.from_numpy(mean)) / torch.sqrt(torch.from_numpy(var) + 1e-3) * torch.from_numpy(gamma) + torch.from_numpy(beta))
    (y * torch.from_numpy(G)).sum().backward()
    np.testing.assert_allclose(SG.bn_relu_backward(x.detach().numpy(), G, gamma, beta, mean, var), x.grad.numpy(), rtol=1e-12, atol=1e-12)


def test_neck_dgrad_restatement_equals_autograd():
    """oracle/bev_grad_ref.py: the data gradient of every conv family of the SSFA neck written as a FORWARD conv / deconv with re-packed
    weights (what the device kernels would run) equals torch autograd, the reference's own mechanism."""
    import torch
    import torch.nn.functional as F
    from oracle import bev_grad_ref as BG
    g = torch.Generator().manual_seed(3)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)      # noqa: E731
    for (k, stride, pad, cin, cout) in [(3, 1, 1, 6, 5), (1, 1, 0, 6, 4), (3, 2, 1, 5, 7)]:
        x = rnd(2, cin, 12, 10).requires_grad_(True)
        w = rnd(cout, cin, k, k)
        y = F.conv2d(x, w, None, stride, pad)
        G = rnd(*y.shape)
        (y * G).sum().backward()
        got = BG.conv_dgrad(G, w, stride, pad)
        assert got.shape == x.shape
        torch.testing.assert_close(got, x.grad, rtol=1e-12, atol=1e-12)
    x = rnd(2, 7, 6, 5).requires_grad_(True)
    wd = rnd(7, 4, 3, 3)
    y = F.conv_transpose2d(x, wd, None, 2, 1, output_padding=1)
    assert tuple(y.shape[2:]) == (12, 10)
    G = rnd(*y.shape)
    (y * G).sum().backward()
    torch.testing.assert_close(BG.deconv_dgrad(G, wd), x.grad, rtol=1e-12, atol=1e-12)
