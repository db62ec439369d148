"""GPU twins of the operators added last: the device side of bbox_target, the test-time mask paste and the other
late additions.  Their host logic and, for kernels, the kernel source itself also run on the CPU in
tests/test_bbox_target_host.py and tests/test_mask_paste_host.py."""
import os

import numpy as np
import pytest
import torch

from simpledet_b200 import ops

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


# ---- CustomOp 'bbox_target' --------------------------------------------------------------------------------------------
def test_bbox_target_against_the_reference_operator(cuda):
    from test_bbox_target_host import G, check_case, kwargs_of

    for name in (str(n) for n in G["names"]):
        np.random.seed(int(G[f"{name}_seed"]))                      # the operator draws from the global numpy RNG
        out = ops.OPS["bbox_target"](torch.from_numpy(G[f"{name}_prop"]).to(cuda),
                                     torch.from_numpy(G[f"{name}_gt"]).to(cuda), **kwargs_of(name))
        check_case(name, out)


# ---- test-time mask paste (models/maskrcnn/utils.py:26-67) ----------------------------------------------------------
def test_segm_results_against_the_reference_function(cuda):
    """ops.segm_results on the device against the reference's own segm_results run on cv2
    (tests/golden/make_golden_mask_paste.py); numpy inputs, like the reference's host arrays."""
    from test_mask_paste_host import NAMES, case

    for name in NAMES:
        im_h, im_w, box, cls, masks, want = case(name)
        got = ops.OPS["segm_results"](box, cls, masks, im_h, im_w)
        assert [g["counts"] for g in got] == want, name
        assert all(g["size"] == [im_h, im_w] for g in got)


def test_segm_results_at_test_size_against_the_oracle(cuda):
    """100 detections on an 800 x 1333 image (mask_r50v1_fpn_1x's test size), CUDA tensors in."""
    from oracle import np_ops

    rng = np.random.default_rng(9)
    im_h, im_w, n, k, m = 800, 1333, 100, 80, 28
    xy = rng.uniform(-10, [im_w - 40, im_h - 40], (n, 2))
    wh = rng.uniform(12, [700, 500], (n, 2))
    box = np.concatenate([xy, xy + wh], 1).astype(np.float32)
    box[0] = [-3.0, -2.0, im_w + 2.0, im_h + 1.0]
    z = rng.standard_normal((n, 7, 7)).astype(np.float32)
    one = (1 / (1 + np.exp(-2 * np.kron(z, np.ones((4, 4), np.float32))))).astype(np.float32)
    cls = rng.integers(0, k, n).astype(np.int32)
    masks = np.zeros((n, k, m, m), np.float32)
    masks[np.arange(n), cls] = one
    got = ops.segm_results(torch.from_numpy(box).to(cuda), torch.from_numpy(cls).to(cuda),
                           torch.from_numpy(masks).to(cuda), im_h, im_w)
    want = np_ops.segm_results(box, cls, masks, im_h, im_w)
    for i in range(n):
        assert got[i]["counts"] == want[i]["counts"], (i, box[i])


def test_coco_records_from_final_detections(cuda):
    from oracle import np_ops

    rng = np.random.default_rng(4)
    B, N, K = 2, 300, 6
    score = rng.random((B, N, K)).astype(np.float32) * (rng.random((B, N, K)) < 0.2)
    xy = rng.uniform(0, 500, (B, N, K, 2))
    bbox = np.concatenate([xy, xy + rng.uniform(10, 200, (B, N, K, 2))], -1).reshape(B, N, K * 4).astype(np.float32)
    out, cnt = ops.final_detections(torch.from_numpy(score).to(cuda), torch.from_numpy(bbox).to(cuda), 0.5, 0.05, 100)
    cats = [1, 2, 3, 5, 8, 13]
    recs = ops.coco_records_from_final_detections([11, 12], out, cnt, cats)
    want = []
    for b, iid in enumerate((11, 12)):
        per = np_ops.do_nms(score[b], bbox[b], 0.5, 0.05)
        want += ops.coco_bbox_records(iid, {cats[c]: d for c, d in per.items()}, 100)
    assert recs == want


# ---- the reference's TRAIN graphs through the façade Trainer, real operators --------------------------------------------
def test_faster_rcnn_fpn_train_step_on_the_device(cuda):
    """config/faster_r50v1_fpn_1x.py's train symbol (fixture written by the reference's own builders on the façade):
    forward + backward + MXNet SGD update on the device - Proposal_v3 x 5, get_top_proposal, ProposalTarget, the fused
    FPN RoIAlign (autograd), SoftmaxOutput / smooth_l1 / MakeLoss with MXNet's gradients."""
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "faster_r50v1_fpn_1x_train_symbol.json")).read())
    B, H, W = 2, 256, 384
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5))
    labels = ("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight")
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=labels)
    s_total = sum((H // st) * (W // st) for st in (4, 8, 16, 32, 64))
    g = torch.Generator().manual_seed(0)
    gt = torch.full((B, 100, 5), -1.0)
    for b in range(B):
        xy = torch.rand(6, 2, generator=g) * torch.tensor([W - 120.0, H - 120.0])
        gt[b, :6, :4] = torch.cat([xy, xy + 30 + torch.rand(6, 2, generator=g) * 80], 1)
        gt[b, :6, 4] = torch.randint(1, 81, (6,), generator=g).float()
    feed = dict(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B), gt_bbox=gt,
                rpn_cls_label=torch.randint(-1, 2, (B, 3, s_total), generator=g).float(),
                rpn_reg_target=torch.randn(B, 12, s_total, generator=g),
                rpn_reg_weight=(torch.rand(B, 12, s_total, generator=g) < 0.1).float())
    before = tr.ex.params["bbox_fc1_weight"].detach().clone()
    for _ in range(2):
        outs = tr.forward_backward(**feed)
        assert all(torch.isfinite(o).all() for o in outs)
        grads = tr.grads()
        assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())
        assert float(grads["stage2_unit1_conv1_weight"].abs().sum()) > 0 and float(grads["P2_lateral_weight"].abs().sum()) > 0
        tr.update(lr=0.001, momentum=0.9, wd=1e-4, rescale_grad=1.0)
    assert tuple(outs[3].shape) == (B * 512, 81) and tuple(outs[5].shape) == (B, 512)
    assert not torch.equal(before, tr.ex.params["bbox_fc1_weight"].detach())


def test_retinanet_train_step_on_the_device(cuda):
    from simpledet_b200.facade import executor as E
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "retina_r50v1_fpn_1x_train_symbol.json")).read())
    B, H, W = 2, 256, 384
    shapes = dict(data=(B, 3, H, W))
    byname = dict(zip(sym.list_arguments(), E.infer_shapes(sym, shapes)[0]))
    labels = ("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight")
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=labels)
    g = torch.Generator().manual_seed(0)
    n_anchor = byname["rpn_cls_label"][1]
    cls = torch.zeros(byname["rpn_cls_label"])
    cls[:, torch.randperm(n_anchor, generator=g)[:60]] = torch.randint(1, 81, (60,), generator=g).float()
    cls[:, torch.randperm(n_anchor, generator=g)[:200]] = -1.0
    feed = dict(data=torch.randn(shapes["data"], generator=g), rpn_cls_label=cls,
                rpn_reg_target=torch.randn(byname["rpn_reg_target"], generator=g),
                rpn_reg_weight=(torch.rand(byname["rpn_reg_weight"], generator=g) < 0.02).float())
    outs = tr.forward_backward(**feed)
    grads = tr.grads()
    assert all(torch.isfinite(o).all() for o in outs) and set(grads) == set(tr.trainable)
    assert all(torch.isfinite(v).all() for v in grads.values())
    assert sum(float(v.abs().sum()) > 0 for v in grads.values()) > 0.9 * len(grads)


def test_mask_rcnn_train_step_on_the_device(cuda):
    """config/mask_r50v1_fpn_1x.py's train symbol: as the Faster R-CNN step plus ProposalMaskTarget (polygon
    rasteriser on the device), the 14x14 RoIAlign on the 128 foreground slots, the class-channel gather and
    SigmoidCrossEntropy."""
    from simpledet_b200 import synth
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "mask_r50v1_fpn_1x_train_symbol.json")).read())
    B, H, W = 2, 512, 832
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5), gt_poly=(B, 100, 2500))
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight"))
    s_total = sum((H // st) * (W // st) for st in (4, 8, 16, 32, 64))
    _, gt, polys = synth.mask_scene(np.random.default_rng(3), B, 64, 100, 2500)
    g = torch.Generator().manual_seed(0)
    feed = dict(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B),
                gt_bbox=torch.from_numpy(gt), gt_poly=torch.from_numpy(polys),
                rpn_cls_label=torch.randint(-1, 2, (B, 3, s_total), generator=g).float(),
                rpn_reg_target=torch.randn(B, 12, s_total, generator=g),
                rpn_reg_weight=(torch.rand(B, 12, s_total, generator=g) < 0.1).float())
    outs = tr.forward_backward(**feed)
    grads = tr.grads()
    assert all(torch.isfinite(o).all() for o in outs) and tuple(outs[-1].shape) == (1,)
    assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())
    assert float(grads["mask_fcn_logit_weight"].abs().sum()) > 0


def test_dcn_c4_train_step_on_the_device(cuda):
    """config/dcn/faster_dcn_r50v1bc4_c5_512roi_1x.py's train symbol: legacy Proposal, ROIAlign_v2 forward + backward
    on C4, three DeformableConvolution blocks (im2col / col2im kernels) inside the C5 head."""
    from simpledet_b200.facade import executor as E
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "faster_dcn_r50v1bc4_c5_512roi_1x_train_symbol.json")).read())
    B, H, W = 2, 256, 384
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5))
    byname = dict(zip(sym.list_arguments(), E.infer_shapes(sym, shapes)[0]))
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight"))
    g = torch.Generator().manual_seed(0)
    gt = torch.full((B, 100, 5), -1.0)
    for b in range(B):
        xy = torch.rand(5, 2, generator=g) * torch.tensor([W - 150.0, H - 150.0])
        gt[b, :5, :4] = torch.cat([xy, xy + 40 + torch.rand(5, 2, generator=g) * 100], 1)
        gt[b, :5, 4] = torch.randint(1, 81, (5,), generator=g).float()
    feed = dict(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B), gt_bbox=gt,
                rpn_cls_label=torch.randint(-1, 2, byname["rpn_cls_label"], generator=g).float(),
                rpn_reg_target=torch.randn(byname["rpn_reg_target"], generator=g),
                rpn_reg_weight=(torch.rand(byname["rpn_reg_weight"], generator=g) < 0.1).float())
    outs = tr.forward_backward(**feed)
    grads = tr.grads()
    assert all(torch.isfinite(o).all() for o in outs)
    assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())
    offs = [n for n in grads if "offset" in n and n.endswith("weight")]
    assert len(offs) == 3


def test_crowdhuman_train_step_with_bbox_target_on_the_device(cuda):
    """config/crowdhuman/faster_r50v1b_fpn_1x.py's train symbol: the CustomOp 'bbox_target' inside the graph, between
    get_top_proposal and the fused FPN RoIAlign."""
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "crowdhuman_faster_r50v1b_fpn_1x_train_symbol.json")).read())
    B, H, W = 2, 256, 384
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5))
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight"))
    s_total = sum((H // st) * (W // st) for st in (4, 8, 16, 32, 64))
    g = torch.Generator().manual_seed(0)
    gt = torch.full((B, 100, 5), -1.0)
    for b in range(B):
        xy = torch.rand(8, 2, generator=g) * torch.tensor([W - 150.0, H - 150.0])
        gt[b, :8, :4] = torch.cat([xy, xy + 40 + torch.rand(8, 2, generator=g) * 100], 1)
        gt[b, :8, 4] = 1.0
    np.random.seed(0)
    outs = tr.forward_backward(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B),
                               gt_bbox=gt, rpn_cls_label=torch.randint(-1, 2, (B, 3, s_total), generator=g).float(),
                               rpn_reg_target=torch.randn(B, 12, s_total, generator=g),
                               rpn_reg_weight=(torch.rand(B, 12, s_total, generator=g) < 0.1).float())
    grads = tr.grads()
    assert all(torch.isfinite(o).all() for o in outs) and tuple(outs[3].shape) == (B * 512, 2)
    assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())
    lab = outs[5]
    assert ((lab == 0) | (lab == 1)).all() and int((lab == 1).sum()) >= 2 * 8      # at least the gt boxes themselves


def test_mask_test_records_on_the_device(cuda):
    """mask_test.py's per-image loop with the masks left on the device (CUDA tensor in, records out)."""
    from oracle import np_ops

    rng = np.random.default_rng(8)
    D, K, M, im_h, im_w = 40, 6, 28, 300, 400
    info = np.array([600.0, 800.0, 2.0], np.float32)
    post_cls = rng.integers(0, K, D).astype(np.float32)
    post_cls[[3, 11, 19]] = -1
    xy = rng.uniform(0, [600, 400], (D, 2))
    post_box = np.concatenate([xy, xy + rng.uniform(30, 200, (D, 2))], 1).astype(np.float32)
    post_score = rng.random(D).astype(np.float32)
    z = rng.standard_normal((D, 1 + K, 7, 7)).astype(np.float32)
    mask = np.ascontiguousarray(1 / (1 + np.exp(-2 * np.kron(z, np.ones((4, 4), np.float32)))), np.float32)
    cats = [1, 2, 3, 5, 8, 13]
    got = ops.mask_test_records(9, info, im_h, im_w, post_score, post_box, post_cls, torch.from_numpy(mask).to(cuda), cats, 100)
    cls = post_cls.astype(np.int32)
    valid = np.where(cls > -1)[0]
    want_segm = np_ops.segm_results((post_box / info[2])[valid], cls[valid], mask[:, 1:][valid], im_h, im_w)
    by_score = {float(post_score[v]): s["counts"].decode("utf8") for v, s in zip(valid, want_segm)}
    assert len(got) == len(valid) and [r["score"] for r in got] == sorted(r["score"] for r in got)
    for r in got:
        assert r["segmentation"]["counts"] == by_score[r["score"]] and r["segmentation"]["size"] == [im_h, im_w]


def test_tridentnet_inference_graph_on_the_device(cuda):
    """config/tridentnet_r50v1c4_c5_1x.py's test symbol (fixture from the reference's own builders): three
    weight-sharing dilation branches stacked into the batch axis, ONE legacy Proposal over the 3-image batch, ROIAlign_v2
    on C4, the C5 head on 3 x 300 rois, DecodeBBox."""
    from simpledet_b200 import facade
    from simpledet_b200.facade import symbol as S

    sym = S.fromjson(open(os.path.join(GOLD, "tridentnet_r50v1c4_c5_1x_test_symbol.json")).read())
    shapes = dict(data=(1, 3, 800, 1333), im_info=(1, 3), im_id=(1,), rec_id=(1,))
    gen = torch.Generator(device=cuda).manual_seed(5)
    feed = dict(data=torch.randn(shapes["data"], device=cuda, generator=gen), im_info=torch.tensor([[800.0, 1333.0, 1.0]], device=cuda),
                im_id=torch.ones(1, device=cuda), rec_id=torch.ones(1, device=cuda))
    ex = facade.Executor(sym, cuda).init_params(shapes, rng_std=0.02)
    with torch.no_grad():
        got = ex.forward(**feed)
    torch.cuda.synchronize()
    assert [tuple(o.shape) for o in got[3:]] == [(900, 81), (900, 4)]
    assert all(torch.isfinite(o).all() for o in got)
    np.testing.assert_allclose(got[3].sum(-1).cpu().numpy(), 1.0, rtol=1e-4)


def test_cascade_rcnn_inference_and_train_step_on_the_device(cuda):
    """config/cascade_r50v1_fpn_1x.py: the test graph (three fused FPN RoIAlign stages chained through DecodeBBox) and
    one training step (three ProposalTarget stages, nine loss heads) with the real operators."""
    from simpledet_b200 import facade
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "cascade_r50v1_fpn_1x_test_symbol.json")).read())
    shapes = dict(data=(1, 3, 800, 1333), im_info=(1, 3), im_id=(1,), rec_id=(1,))
    gen = torch.Generator(device=cuda).manual_seed(5)
    ex = facade.Executor(sym, cuda).init_params(shapes, rng_std=0.02)
    with torch.no_grad():
        got = ex.forward(data=torch.randn(shapes["data"], device=cuda, generator=gen),
                         im_info=torch.tensor([[800.0, 1333.0, 1.0]], device=cuda), im_id=torch.ones(1, device=cuda),
                         rec_id=torch.ones(1, device=cuda))
    assert [tuple(o.shape) for o in got[3:]] == [(1, 1000, 81), (1, 1000, 4)] and all(torch.isfinite(o).all() for o in got)

    sym = S.fromjson(open(os.path.join(GOLD, "cascade_r50v1_fpn_1x_train_symbol.json")).read())
    B, H, W = 2, 256, 384
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5))
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight"))
    s_total = sum((H // st) * (W // st) for st in (4, 8, 16, 32, 64))
    g = torch.Generator().manual_seed(0)
    gt = torch.full((B, 100, 5), -1.0)
    for b in range(B):
        xy = torch.rand(6, 2, generator=g) * torch.tensor([W - 120.0, H - 120.0])
        gt[b, :6, :4] = torch.cat([xy, xy + 30 + torch.rand(6, 2, generator=g) * 80], 1)
        gt[b, :6, 4] = torch.randint(1, 81, (6,), generator=g).float()
    outs = tr.forward_backward(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B),
                               gt_bbox=gt, rpn_cls_label=torch.randint(-1, 2, (B, 3, s_total), generator=g).float(),
                               rpn_reg_target=torch.randn(B, 12, s_total, generator=g),
                               rpn_reg_weight=(torch.rand(B, 12, s_total, generator=g) < 0.1).float())
    grads = tr.grads()
    assert len(outs) == 12 and all(torch.isfinite(o).all() for o in outs)
    assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())


def test_tridentnet_train_step_on_the_device(cuda):
    """config/tridentnet_r50v1c4_c5_1x.py's train symbol: `_contrib_Proposal_v2` and `ProposalTarget_v2` (valid_ranges,
    filter_scales) inside the graph, three weight-sharing branches in the batch axis."""
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "tridentnet_r50v1c4_c5_1x_train_symbol.json")).read())
    B, H, W, NB = 2, 256, 384, 3
    fh, fw = H // 16, W // 16
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5), valid_ranges=(B, NB, 2),
                  rpn_cls_label=(B, NB, 15, fh, fw), rpn_reg_target=(B, NB, 60, fh, fw), rpn_reg_weight=(B, NB, 60, fh, fw))
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02)
    g = torch.Generator().manual_seed(0)
    gt = torch.full((B, 100, 5), -1.0)
    for b in range(B):
        xy = torch.rand(6, 2, generator=g) * torch.tensor([W - 150.0, H - 150.0])
        gt[b, :6, :4] = torch.cat([xy, xy + 20 + torch.rand(6, 2, generator=g) * 120], 1)
        gt[b, :6, 4] = torch.randint(1, 81, (6,), generator=g).float()
    outs = tr.forward_backward(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B),
                               gt_bbox=gt, valid_ranges=torch.tensor([[[0.0, 90.0], [30.0, 160.0], [90.0, -1.0]]] * B),
                               rpn_cls_label=torch.randint(-1, 2, shapes["rpn_cls_label"], generator=g).float(),
                               rpn_reg_target=torch.randn(shapes["rpn_reg_target"], generator=g),
                               rpn_reg_weight=(torch.rand(shapes["rpn_reg_weight"], generator=g) < 0.1).float())
    grads = tr.grads()
    assert all(torch.isfinite(o).all() for o in outs) and tuple(outs[4].shape) == (B * NB, 128)
    assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())


def test_maskiou_compute_against_the_reference_operator(cuda):
    g = np.load(os.path.join(GOLD, "reference_maskiou_compute.npz"))
    iou, w = ops.OPS["maskiou_compute"](*[torch.from_numpy(g[k]).to(cuda) for k in ("logits", "target", "ratio", "inds")])
    assert np.array_equal(iou.cpu().numpy(), g["iou"]) and np.array_equal(w.cpu().numpy(), g["weight"])


def test_mask_scoring_rcnn_train_step_on_the_device(cuda):
    """config/ms_r50v1_fpn_1x.py's train symbol: ProposalMaskTarget(output_ratio=True) (the mask_ratio kernel) feeding
    the CustomOp 'maskiou_compute' and the MaskIoU head."""
    from simpledet_b200 import synth
    from simpledet_b200.facade import symbol as S
    from simpledet_b200.facade import train as T

    sym = S.fromjson(open(os.path.join(GOLD, "ms_r50v1_fpn_1x_train_symbol.json")).read())
    B, H, W = 2, 512, 832
    shapes = dict(data=(B, 3, H, W), im_info=(B, 3), gt_bbox=(B, 100, 5), gt_poly=(B, 100, 2500))
    tr = T.Trainer(sym, shapes, device=cuda, fixed_param=("conv0", "stage1", "gamma", "beta"), rng_std=0.02,
                   label_names=("rpn_cls_label", "rpn_reg_target", "rpn_reg_weight"))
    s_total = sum((H // st) * (W // st) for st in (4, 8, 16, 32, 64))
    _, gt, polys = synth.mask_scene(np.random.default_rng(3), B, 64, 100, 2500)
    g = torch.Generator().manual_seed(0)
    outs = tr.forward_backward(data=torch.randn(shapes["data"], generator=g), im_info=torch.tensor([[H, W, 1.0]] * B),
                               gt_bbox=torch.from_numpy(gt), gt_poly=torch.from_numpy(polys),
                               rpn_cls_label=torch.randint(-1, 2, (B, 3, s_total), generator=g).float(),
                               rpn_reg_target=torch.randn(B, 12, s_total, generator=g),
                               rpn_reg_weight=(torch.rand(B, 12, s_total, generator=g) < 0.1).float())
    grads = tr.grads()
    assert len(outs) == 8 and all(torch.isfinite(o).all() for o in outs)
    assert set(grads) == set(tr.trainable) and all(torch.isfinite(v).all() for v in grads.values())
