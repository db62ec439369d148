#!/usr/bin/env python
"""bench.py — the benchmark of the simpledet_b200 hot path.

  python bench.py --gpus N --steps K --warmup W            (our CUDA path; K timed steps)
  python bench.py ... --dump-outputs DIR                   (also writes the last timed step's outputs as .npy)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU path = oracle)
  python bench.py --workload retina_train|mask_train|dcn_softnms ...   (BASELINE.json configs 3-5)

Default workload `infer` (BASELINE.json configs[1]): one "step" = one pass of the detection-specific hot path of
`faster_r50v1_fpn_1x` inference (detection_infer_speed.py's graph + detection_test.py's NMS) over a batch of
synthetic 800x1333 images per GPU:

   5 x _contrib_Proposal_v3 (strides 4..64) -> get_top_proposal(1000) -> fused FPN RoIAlign_v2 7x7
   (1000 rois x 256 ch) -> _contrib_DecodeBBox (81 classes) -> per-class NMS (80 classes)

The backbone / RoI-head GEMMs are not on this path (tensor-core library work); their outputs (FPN features, RPN
maps, head logits/deltas) are the synthetic inputs.  The training workloads add the ONE collective of the
reference's data-parallel step: an fp32 all-reduce of the flat gradient bucket (166 MB, scaled by 1/G,
core/detection_module.py:680-690, detection_train.py:266) overlapped with the step on a second stream.
Prints ONE JSON line.  `roofline` = the dominant kernel of the step; `roofline_target` (infer, N=1) = the
north-star shape 512 rois x 256 ch x 14x14 timed in the same process.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STRIDES_RPN = (4, 8, 16, 32, 64)
STRIDES_ROI = (4, 8, 16, 32)
IMG_H, IMG_W = 800, 1333
C_FEAT, N_ROI, K_CLS, POOLED = 256, 1000, 81, 7
GRAD_BUCKET_FLOATS = 41_500_000  # ~41.5 M parameters of faster_r50v1_fpn -> 166 MB fp32 (SURVEY §8e)


def level_shapes(strides):
    return [(-(-IMG_H // s), -(-IMG_W // s)) for s in strides]


# ================================================================================================
# workloads: make_inputs(rng, B) -> dict of numpy arrays; step(ops, d, ev) on device tensors;
#            cpu(d, n_images) = the oracle on host arrays; roofline(...) -> (kernel name, algorithmic bytes)
# ================================================================================================
class Infer:
    name = "infer"
    text = ("faster_r50v1_fpn_1x inference hot path, synthetic 800x1333: 5x Proposal_v3 -> get_top_proposal(1000)"
            " -> FPN RoIAlign_v2 7x7 (1000 rois x 256 ch) -> DecodeBBox(81) -> per-class NMS(80)")
    train = False
    kernel = ("roi_align_cl_kernel (fused FPN RoIAlign 7x7 over channels-last FPN features, %d rois x 256 ch; "
              "whole operator: plan + order + gather kernels)")

    @staticmethod
    def make_inputs(rng, B):
        d = {}
        for s, (h, w) in zip(STRIDES_RPN, level_shapes(STRIDES_RPN)):
            logit = rng.standard_normal((B, 3, h, w)).astype(np.float32) * 2 - 3
            fg = 1 / (1 + np.exp(-logit))
            d[f"cls_prob{s}"] = np.concatenate([1 - fg, fg], 1).astype(np.float32)
            d[f"bbox_pred{s}"] = (rng.standard_normal((B, 12, h, w)) * 0.3).astype(np.float32)
        for s, (h, w) in zip(STRIDES_ROI, level_shapes(STRIDES_ROI)):
            # FPN features in the layout the tensor-core convolutions that produce them emit: channels-last (B,H,W,C)
            d[f"feat{s}"] = rng.standard_normal((B, h, w, C_FEAT)).astype(np.float32)
        d["im_info"] = np.tile(np.array([[IMG_H, IMG_W, 1.0]], np.float32), (B, 1))
        z = rng.standard_normal((B, N_ROI, K_CLS)).astype(np.float32) * 2
        z[..., 0] += 3  # mostly background, a few confident classes
        e = np.exp(z - z.max(-1, keepdims=True))
        d["cls_score"] = (e / e.sum(-1, keepdims=True)).astype(np.float32)
        d["head_bbox_pred"] = (rng.standard_normal((B, N_ROI, 4 * K_CLS)) * 0.5).astype(np.float32)
        return d

    @staticmethod
    def step(ops, d, ev=None):
        boxes, scores = ops.Proposal_v3_fpn([d[f"cls_prob{s}"] for s in STRIDES_RPN],
                                            [d[f"bbox_pred{s}"] for s in STRIDES_RPN], d["im_info"], STRIDES_RPN,
                                            rpn_pre_nms_top_n=1000, rpn_post_nms_top_n=1000, threshold=0.7,
                                            rpn_min_size=0, scales=(8,), ratios=(0.5, 1.0, 2.0))
        rois, _ = ops.get_top_proposal(boxes, scores, N_ROI)
        feats = [d[f"feat{s}"] for s in STRIDES_ROI]
        if ev:
            ev[0].record()
        roi_feat = ops.fpn_roi_align_nhwc(feats, rois, STRIDES_ROI, POOLED, 224, 4)[0]  # (B, N, C, 7, 7)
        if ev:
            ev[1].record()
        # (RoI head: 2 fc + cls/reg fc on tensor cores — library GEMMs, not on this path)
        bbox = ops.DecodeBBox(rois, d["head_bbox_pred"], d["im_info"], (0, 0, 0, 0), (0.1, 0.1, 0.2, 0.2),
                              class_agnostic=False)
        dets, counts, keep, nkeep, src = ops.multiclass_nms(d["cls_score"], bbox, 0.5, 0.05, first_class=1)
        return {"rois": rois, "result": (dets, counts, keep, nkeep),
                "outputs": {"rois": rois, "decoded_bbox": bbox, **nms_outputs(dets, counts, keep, nkeep, src)}}

    @staticmethod
    def roofline_bytes(out, d, B):
        """SURVEY.md §8(d): sz(out) + sum_l min(sz(feat_l), sum of window bytes on l) + sz(rois)."""
        return roialign_algorithmic_bytes(out["rois"].cpu().numpy(), B, POOLED, False)

    @staticmethod
    def prepare_cpu(d):
        """The reference's operators read NCHW: re-lay the features once, outside the timed region."""
        d = dict(d)
        for s in STRIDES_ROI:
            d[f"feat{s}"] = np.ascontiguousarray(d[f"feat{s}"].transpose(0, 3, 1, 2))
        return d

    @staticmethod
    def cpu(d, n_images):
        import oracle
        from oracle import np_ops

        for b in range(n_images):
            sl = slice(b, b + 1)
            boxes, scores = [], []
            for s in STRIDES_RPN:
                r, sc = oracle.proposal_v3(d[f"cls_prob{s}"][sl], d[f"bbox_pred{s}"][sl], d["im_info"][sl],
                                           feature_stride=s, scales=(8,), ratios=(0.5, 1, 2), rpn_pre_nms_top_n=1000,
                                           rpn_post_nms_top_n=1000, threshold=0.7, rpn_min_size=0)
                boxes.append(r)
                scores.append(sc)
            rois, _ = np_ops.get_top_proposal(np.concatenate(boxes, 1), np.concatenate(scores, 1), N_ROI)
            oracle.fpn_roi_align_v2_forward([d[f"feat{s}"][sl] for s in STRIDES_ROI], rois, STRIDES_ROI,
                                            (POOLED, POOLED))
            bbox = oracle.decode_bbox(rois, d["head_bbox_pred"][sl], d["im_info"][sl], (0, 0, 0, 0),
                                      (0.1, 0.1, 0.2, 0.2), False)
            np_ops.do_nms(d["cls_score"][b][:, 1:], bbox[0][:, 4:], 0.5, 0.05)

    cpu_note = ("RoIAlign/decode/proposal C restatement with OpenMP over all host cores, NMS numpy "
                "(single thread) as in the reference")


class RetinaTrain:
    """BASELINE configs[2]: retina_r50v1_fpn_1x training step, per GPU B=2: FocalLoss fwd+bwd on (B,200700,80) logits,
    BBoxNorm bwd on (B,36,22300), the test-branch decode GenProposalRetina on P3..P7 + per-class NMS; one gradient
    all-reduce."""
    name = "retina_train"
    text = ("retina_r50v1_fpn_1x training-step hot path, synthetic COCO-shape batch: FocalLoss fwd+bwd (200700 anchors x "
            "80 classes per image, valid-normalised) + BBoxNorm bwd + GenProposalRetina(P3-P7, top-800 per level) + per-class "
            "NMS(80) + fp32 gradient all-reduce (166 MB)")
    train = True
    kernel = "focal_backward_kernel (FocalLoss backward, %d x 200700 x 80)"
    N_ANCH, K = 200700, 80
    STRIDES = (8, 16, 32, 64, 128)

    @classmethod
    def make_inputs(cls, rng, B):
        d = {"logits": (rng.standard_normal((B, cls.N_ANCH, cls.K), dtype=np.float32) * 0.5 - 4.6)}
        lab = np.zeros((B, cls.N_ANCH), np.float32)
        for b in range(B):
            lab[b, rng.choice(cls.N_ANCH, 100, replace=False)] = rng.integers(1, cls.K + 1, 100)
            lab[b, rng.choice(cls.N_ANCH, cls.N_ANCH // 50, replace=False)] = -1
        d["label"] = lab
        d["bbox_loss"] = rng.standard_normal((B, 36, 22300), dtype=np.float32)
        d["reg_label"] = lab[:, :22300].copy()
        for s, (h, w) in zip(cls.STRIDES, level_shapes(cls.STRIDES)):
            # class probabilities of a freshly initialised head (bias -4.6, models/retinanet/builder.py prior 0.01)
            # with unit-variance logits: ~5 % of the 720*H*W pairs clear the 0.05 threshold
            z = rng.standard_normal((B, 9 * cls.K, h, w), dtype=np.float32) - np.float32(4.6)
            d[f"cls{s}"] = (1.0 / (1.0 + np.exp(-z))).astype(np.float32)
            d[f"reg{s}"] = rng.standard_normal((B, 36, h, w), dtype=np.float32) * 0.3
        d["im_info"] = np.tile(np.array([[IMG_H, IMG_W, 1.0]], np.float32), (B, 1))
        return d

    @classmethod
    def step(cls, ops, d, ev=None):
        import torch

        logits = d["logits"].detach().requires_grad_(True)
        out = ops.FocalLoss(logits, d["label"], alpha=0.25, gamma=2.0, normalization="valid", grad_scale=1.0)
        if ev:
            ev[0].record()
        out.backward(torch.ones_like(out))
        if ev:
            ev[1].record()
        bl = d["bbox_loss"].detach().requires_grad_(True)
        bn = ops.BBoxNorm(bl, d["reg_label"])
        bn.backward(d["bbox_loss"])
        scales = tuple(4 * 2 ** (i / 3) for i in range(3))
        boxes, scores = [], []
        for s in cls.STRIDES:
            anchors = ops.GenAnchor(d[f"cls{s}"][:1, :9], scales=scales, ratios=(0.5, 1, 2), feature_stride=s)
            b_, s_ = ops.GenProposalRetina(d[f"cls{s}"], d[f"reg{s}"], d["im_info"], anchors, num_anchors=9,
                                           feature_stride=s, rpn_pre_nms_top_n=800, rpn_min_size=0, thresh=0.05,
                                           anchor_mean=(0, 0, 0, 0), anchor_std=(1, 1, 1, 1))
            boxes.append(b_)
            scores.append(s_)
        boxes, scores = torch.cat(boxes, 1), torch.cat(scores, 1)
        dets, counts, keep, nkeep, src = ops.multiclass_nms(scores, boxes, 0.5, 0.05, first_class=1)
        return {"result": (logits.grad[:, :1024, :].contiguous(), bl.grad[:, :, :256].contiguous(), nkeep),
                "outputs": {"focal_prob": out, "focal_grad": logits.grad, "bbox_norm": bn, "bbox_norm_grad": bl.grad,
                            "retina_boxes": boxes, "retina_scores": scores,
                            **nms_outputs(dets, counts, keep, nkeep, src)}}

    @classmethod
    def roofline_bytes(cls, out, d, B):
        return 2 * B * cls.N_ANCH * cls.K * 4 + B * cls.N_ANCH * 4   # 2 sz(data) + sz(label), SURVEY §8d

    @classmethod
    def cpu(cls, d, n_images):
        import oracle
        from oracle import np_ops

        sl = slice(0, n_images)
        p = oracle.sigmoid(d["logits"][sl])
        oracle.focal_loss_backward(p, d["label"][sl], 0.25, 2.0, 1.0, "valid", None)
        oracle.bbox_norm_backward(d["bbox_loss"][sl], d["reg_label"][sl])
        scales = tuple(4 * 2 ** (i / 3) for i in range(3))
        for b in range(n_images):
            bs, ss = [], []
            for s, (h, w) in zip(cls.STRIDES, level_shapes(cls.STRIDES)):
                anchors = oracle.gen_anchor(h, w, s, scales, (0.5, 1, 2))
                b_, s_ = oracle.gen_proposal_retina(d[f"cls{s}"][b:b + 1], d[f"reg{s}"][b:b + 1], d["im_info"][b:b + 1], anchors,
                                                    num_anchors=9, rpn_pre_nms_top_n=800, rpn_min_size=0, thresh=0.05,
                                                    anchor_mean=(0, 0, 0, 0), anchor_std=(1, 1, 1, 1))
                bs.append(b_[0])
                ss.append(s_[0])
            np_ops.do_nms(np.concatenate(ss)[:, 1:], np.concatenate(bs), 0.5, 0.05)

    cpu_note = "focal / bbox-norm / retina decode C restatements (OpenMP where the reference's mxnet_op::Kernel is), numpy NMS"


class MaskTrain:
    """BASELINE configs[3]: mask_r50v1_fpn_1x training step, per GPU B=2: ProposalMaskTarget on 2000 rois/img (512 kept,
    28x28 masks), RoIAlign 7x7 on the 512 rois/img and 14x14 on the 128 fg rois/img, forward WITH argmax planes and
    backward, SigmoidCrossEntropy on the mask logits; one gradient all-reduce."""
    name = "mask_train"
    text = ("mask_r50v1_fpn_1x training-step hot path: ProposalMaskTarget(2000 rois/img -> 512, 28x28 masks) + FPN "
            "RoIAlign 7x7 (512 rois/img) fwd+bwd + FPN RoIAlign 14x14 (128 rois/img) fwd+bwd + SigmoidCrossEntropy "
            "fwd+bwd + fp32 gradient all-reduce (166 MB)")
    train = True
    kernel = "roi_align_v2_fwd_kernel with argmax planes (FPN RoIAlign 7x7 training forward, %d rois x 256 ch)"

    @staticmethod
    def make_inputs(rng, B):
        from simpledet_b200 import synth

        rois, gt, polys = synth.mask_scene(rng, B, 2000, 100, 2500)
        d = {"rois": rois, "gt": gt, "polys": polys}
        for s, (h, w) in zip(STRIDES_ROI, level_shapes(STRIDES_ROI)):
            d[f"feat{s}"] = rng.standard_normal((B, C_FEAT, h, w)).astype(np.float32)
        d["g7"] = rng.standard_normal((B, 512, C_FEAT, 7, 7), dtype=np.float32)
        d["g14"] = rng.standard_normal((B, 128, C_FEAT, 14, 14), dtype=np.float32)
        d["mask_logit"] = rng.standard_normal((B * 128, 28 * 28), dtype=np.float32)
        return d

    @staticmethod
    def step(ops, d, ev=None):
        B = d["rois"].shape[0]
        r = ops.ProposalMaskTarget(d["rois"], d["gt"], d["polys"], 81, B, 512, 28, 0.5, 0.5, 0.0, False, seed=7)
        rois512, mask_t = r[0], r[4]
        feats = [d[f"feat{s}"].detach().requires_grad_(True) for s in STRIDES_ROI]
        if ev:
            ev[0].record()
        o7 = ops.fpn_roi_align(feats, rois512, STRIDES_ROI, 7)
        if ev:
            ev[1].record()
        o7.backward(d["g7"])
        o14 = ops.fpn_roi_align(feats, rois512[:, :128].contiguous(), STRIDES_ROI, 14)
        o14.backward(d["g14"])
        ml = d["mask_logit"].detach().requires_grad_(True)
        loss = ops.SigmoidCrossEntropy(ml, mask_t.reshape(B * 128, 28 * 28))
        loss.backward(loss.new_ones(loss.shape))
        names = ("rois", "label", "bbox_target", "bbox_weight", "mask_target")
        return {"rois": rois512, "result": (loss, feats[3].grad, ml.grad[:64].contiguous()),
                "outputs": {**{"target_" + n: t for n, t in zip(names, r)}, "roi_feat7": o7, "roi_feat14": o14,
                            **{f"feat{s}_grad": f.grad for s, f in zip(STRIDES_ROI, feats)},
                            "mask_loss": loss, "mask_logit_grad": ml.grad}}

    @staticmethod
    def roofline_bytes(out, d, B):
        return roialign_algorithmic_bytes(out["rois"].cpu().numpy(), B, 7, True, n_roi=512)

    @staticmethod
    def cpu(d, n_images):
        import oracle

        sl = slice(0, n_images)
        rng = np.random.default_rng(0)
        pr = rng.integers(0, 2 ** 32, (n_images, 4, 2100), dtype=np.uint64).astype(np.uint32)
        r = oracle.proposal_mask_target(d["rois"][sl], d["gt"][sl], d["polys"][sl], pr, 81, 512, 28, fg_fraction=0.25,
                                        fg_thresh=0.5, bg_thresh_hi=0.5, bg_thresh_lo=0.0)
        rois = r[0]
        lv = oracle.fpn_assign_levels(rois, STRIDES_ROI).reshape(rois.shape[:2])
        for pooled, nr, g in ((7, 512, d["g7"]), (14, 128, d["g14"])):
            for i, s in enumerate(STRIDES_ROI):
                lr = np.where((lv[:, :nr] == i)[..., None], rois[:, :nr], np.float32(0))
                o, ax, ay = oracle.roi_align_v2_forward(d[f"feat{s}"][sl], lr, (pooled, pooled), 1.0 / s)
                oracle.roi_align_v2_backward(g[sl], ax, ay, d[f"feat{s}"][sl].shape)
        oracle.sigmoid_ce_forward(d["mask_logit"][:n_images * 128], r[5].reshape(n_images * 128, -1))
        oracle.sigmoid_ce_backward(d["mask_logit"][:n_images * 128], r[5].reshape(n_images * 128, -1))

    cpu_note = ("C restatements: ProposalMaskTarget single thread (as the reference), the reference graph's 4-level "
                "RoIAlign_v2 fwd (OpenMP) + GPU-order bwd, SigmoidCE")


class DcnSoftNms:
    """BASELINE configs[4]: dcn faster_r50v1_fpn + soft-NMS at bs=2/GPU: the DCNv1 C4 block (256 -> 256, 3x3, 4
    deformable groups) on (2,256,50,84) - deformable im2col + library GEMM - x3 blocks, and batched linear soft-NMS
    over 80 classes x <=1000 boxes per image.  Inference: no collective."""
    name = "dcn_softnms"
    text = ("dcn faster_r50v1_fpn + soft-NMS hot path, bs=2/GPU: 3 x DeformableConvolution(256->256, 3x3, dg=4) on "
            "(2,256,50,84) channels-last [deformable im2col + cuBLAS GEMM] + batched linear soft-NMS (80 classes x <=1000 "
            "boxes/img)")
    train = False
    kernel = "deform_im2col_cl_kernel (DCNv1 sampling over channels-last features, %d x 256 x 50 x 84, dg=4)"

    @staticmethod
    def make_inputs(rng, B):
        d = {"data": rng.standard_normal((B, 50, 84, 256), dtype=np.float32),  # channels-last (B,H,W,C)
             "offset": rng.standard_normal((B, 72, 50, 84), dtype=np.float32) * 2,
             "weight": rng.standard_normal((256, 256, 3, 3), dtype=np.float32) * 0.02}
        P, m = B * 80, 1000
        dets = np.zeros((P, m, 5), np.float32)
        for p in range(P):
            xy = rng.uniform(0, 1100, (m, 2))
            dets[p] = np.concatenate([xy, xy + rng.uniform(8, 300, (m, 2)), rng.permutation(m)[:, None] / m + 1e-3], 1)
        d["dets"] = dets
        d["counts"] = rng.integers(0, m + 1, P).astype(np.int32)
        return d

    @staticmethod
    def step(ops, d, ev=None):
        import torch
        from simpledet_b200 import _lib

        x = d["data"]
        B, H, W, C = x.shape
        L = _lib.lib()
        st = torch.cuda.current_stream().cuda_stream
        wp = d["weight"].permute(2, 3, 1, 0).reshape(9 * C, C)   # W'[(tap, c)][f]
        col_t = torch.empty((B, H * W, 9 * C), device=x.device)
        for blk in range(3):
            if ev and blk == 0:
                ev[0].record()
            _lib.check(L.sdet_deformable_im2col_nhwc(x.data_ptr(), d["offset"].data_ptr(), col_t.data_ptr(), B, C, H, W, 3, 3,
                                                     1, 1, 1, 1, 1, 1, 4, st))
            if ev and blk == 0:
                ev[1].record()
            x = torch.matmul(col_t, wp).view(B, H, W, C)   # dense contraction: cuBLAS (library work); output channels-last
        ob, oi, oc = ops.soft_nms_batched(d["dets"], 0.5, 0.5, 0.001, 1, counts=d["counts"])
        return {"result": (x[..., :8].contiguous(), oc),
                "outputs": {"dcn_out": x, "soft_nms_boxes": (ob, oc), "soft_nms_inds": (oi, oc), "soft_nms_counts": oc}}

    @staticmethod
    def roofline_bytes(out, d, B):
        return 4 * (B * 256 * 50 * 84 + B * 72 * 50 * 84 + B * 256 * 9 * 50 * 84)   # sz(data)+sz(offset)+sz(col)

    @staticmethod
    def prepare_cpu(d):
        """The numpy restatement reads NCHW: the 16 channels it samples, re-laid once outside the timed region."""
        d = dict(d)
        d["data_nchw16"] = np.ascontiguousarray(d["data"][..., :16].transpose(0, 3, 1, 2))
        return d

    @staticmethod
    def cpu(d, n_images):
        import oracle
        from oracle import np_ops

        for b in range(n_images):
            # the numpy restatement of deformable_im2col is slow: one deformable group's worth of channels per image
            np_ops.deformable_im2col(d["data_nchw16"][b:b + 1], d["offset"][b:b + 1, :18], (3, 3), (1, 1), (1, 1), (1, 1), 1)
            for p in range(b * 80, (b + 1) * 80):
                oracle.soft_nms(d["dets"][p, :d["counts"][p]], 0.5, 0.5, 0.001, 1)

    cpu_note = ("numpy deformable_im2col restatement on 16 of the 256 channels of ONE block (scaled x16 x3 is not applied: "
                "the figure is an upper bound on the CPU arm's speed), compiled soft_nms restatement over all 80 classes")


WORKLOADS = {w.name: w for w in (Infer, RetinaTrain, MaskTrain, DcnSoftNms)}
DUMP_SAMPLE = 1 << 20  # --dump-outputs: larger outputs are written as this many elements at fixed, seeded positions


def nms_outputs(dets, counts, keep, nkeep, src):
    """multiclass_nms's arrays; a (tensor, counts) pair marks rows past counts[p] of problem p as unspecified."""
    return {"nms_dets": (dets, counts), "nms_counts": counts, "nms_keep": (keep, nkeep), "nms_nkeep": nkeep,
            "nms_src": (src, counts)}


def dump_outputs(outputs, out_dir):
    """Write each output of a step as out_dir/<name>.npy: floating point as float32, integers as float64 (exact).
    Rows an operator leaves unspecified are written as 0; an output of more than DUMP_SAMPLE elements is written as
    the elements at DUMP_SAMPLE flat positions drawn with a fixed seed, in increasing order."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, x in outputs.items():
        if isinstance(x, tuple):
            x, n = x
            valid = torch.arange(x.shape[1], device=x.device)[None, :] < n.reshape(-1, 1).to(x.device)
            x = torch.where(valid.reshape(valid.shape + (1,) * (x.dim() - 2)), x, torch.zeros((), dtype=x.dtype,
                                                                                               device=x.device))
        x = x.detach()
        if x.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(x.numel(), DUMP_SAMPLE, replace=False))
            x = x.reshape(-1)[torch.from_numpy(idx).to(x.device)]
        a = x.cpu().numpy().astype(np.float32 if x.is_floating_point() else np.float64)
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= 64 << 20, f"--dump-outputs wrote {total} bytes"


def roialign_algorithmic_bytes(rois_np, B, pooled, with_argmax, n_roi=None, C=C_FEAT):
    """SURVEY.md §8(d): sz(out) [x3 with argmax planes] + sum_l min(sz(feat_l), sum of window bytes on l) + sz(rois)."""
    import oracle

    n_roi = n_roi or rois_np.shape[1]
    lv = oracle.fpn_assign_levels(rois_np, STRIDES_ROI).reshape(rois_np.shape[:2])
    total = B * n_roi * C * pooled * pooled * 4 * (3 if with_argmax else 1) + rois_np.size * 4
    for l, ((h, w), s) in enumerate(zip(level_shapes(STRIDES_ROI), STRIDES_ROI)):
        m = lv == l
        if not m.any():
            continue
        r = rois_np[m] / s
        x1 = np.clip(np.floor(r[:, 0]), 0, w - 1)
        x2 = np.clip(np.ceil(r[:, 2]), 0, w - 1)
        y1 = np.clip(np.floor(r[:, 1]), 0, h - 1)
        y2 = np.clip(np.ceil(r[:, 3]), 0, h - 1)
        total += min(float(((x2 - x1 + 1) * (y2 - y1 + 1)).sum()) * C * 4, B * C * h * w * 4)
    return int(total)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md): one
    `nvidia-smi -lms 20` child streams samples while the region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.idx, self.proc = [], gpu_index, None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.proc.stdout.readline()  # first sample = the child is up; region starts after it
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.03)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 6 and f[0].replace(".", "").isdigit():
                self.rows.append(f)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and the pinned buffers it allocates next) to the CPUs of its GPU's NUMA node: 8 ranks pushing
    ~200 MB/step of pinned H2D across the socket interconnect is what bent the end-to-end curve at N=4/8.
    The CPU list comes from sysfs (`local_cpulist` of the GPU's PCI device); nothing is bound unless the list holds
    at least 8 CPUs this process may use (a wrong, tiny set would serialise the launch thread)."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if not bus:
            return None
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/local_cpulist"
        cpus = open(path).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if len(ids) >= 8:
            os.sched_setaffinity(0, ids)
            return cpus
    except Exception:
        pass
    return None


def time_cpu(wl, d, budget_s=12.0):
    import oracle

    oracle.build()
    oracle.set_threads()
    if hasattr(wl, "prepare_cpu"):
        d = wl.prepare_cpu(d)
    t0 = time.perf_counter()
    wl.cpu(d, 1)
    one = time.perf_counter() - t0
    nimg = next(iter(d.values())).shape[0] if wl is not DcnSoftNms else d["data"].shape[0]
    n = max(1, min(nimg * 4, int(budget_s / max(one, 1e-3))))
    t0 = time.perf_counter()
    done = 0
    while done < n:
        m = min(nimg, n - done)
        wl.cpu(d, m)
        done += m
    dt = time.perf_counter() - t0
    return done / dt, done


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The operator_cxx pieces that compile
    here (oracle/_ref/libref_cxx.so: RoIAlign_v2, DecodeBBox, ProposalTarget, ...) pin the oracle port bit for bit
    (tests/test_oracle_ref_cxx.py); the port is what is timed because it is the one with the OpenMP loop of
    mxnet_op::Kernel<...,cpu>::Launch (the shim build is serial).  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import oracle

    wl = WORKLOADS[args.workload]
    oracle.build()
    rng = np.random.default_rng(0)
    d = wl.make_inputs(rng, 1)
    if hasattr(wl, "prepare_cpu"):
        d = wl.prepare_cpu(d)
    cores = oracle.set_threads() or 1  # (torchrun exports OMP_NUM_THREADS=1: undo it for the CPU arm)
    for _ in range(min(args.warmup, 1)):
        wl.cpu(d, 1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        wl.cpu(d, 1)  # one step = a bounded sample: 1 image of the workload
    dt = time.perf_counter() - t0
    v = args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "images/sec", "value": round(v, 3), "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * dt / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl.text, "images_per_step": 1},
        "cpu_baseline": {"value": round(v, 3), "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": "1 image per step; " + wl.cpu_note},
        "e2e": {"value": round(v, 3), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_ours(args):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as g
    from simpledet_b200 import _lib, ops, shard

    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: there is no CPU fallback for the product path")
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        g.build()
    if world > 1:
        dist.barrier()
    _lib.lib()

    B, K, W = args.images_per_gpu, args.steps, max(args.warmup, 3)
    rng = np.random.default_rng(1234 + rank)
    probe = wl.make_inputs(rng, B)
    set_mb = sum(v.nbytes for v in probe.values()) / 1e6
    R = max(2, -(-300 // max(1, int(set_mb))))  # rotating input sets: footprint >> 126 MB L2
    host_sets = [probe] + [wl.make_inputs(rng, B) for _ in range(R - 1)]
    dev_sets = [{k: torch.from_numpy(v).to(dev) for k, v in hs.items()} for hs in host_sets]
    pinned = [{k: torch.from_numpy(v).pin_memory() for k, v in hs.items()} for hs in host_sets]
    h2d_bytes = sum(v.numel() * v.element_size() for v in pinned[0].values())

    main = torch.cuda.current_stream()
    comm_s = torch.cuda.Stream()
    bucket = torch.zeros(GRAD_BUCKET_FLOATS, device=dev) if wl.train else None
    ar_events = []

    def grad_allreduce():
        """The step's one collective, on its own stream so that it overlaps the step's kernels."""
        if bucket is None:
            return
        comm_s.wait_stream(main)
        with torch.cuda.stream(comm_s):
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if world > 1:
                dist.all_reduce(bucket)
            bucket.mul_(1.0 / world)  # rescale_grad = 1/G (detection_train.py:266)
            b_.record()
            ar_events.append((a, b_))

    def one_step(d, ev=None):
        grad_allreduce()
        out = wl.step(ops, d, ev)
        main.wait_stream(comm_s)
        return out

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident throughput (`value`) ----
    for i in range(W):
        out = one_step(dev_sets[i % R])
    ar_events.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sync_all()
    n0 = _lib.launch_count()
    gc.disable()  # as timeit does: a collector pass landing in some windows of K steps and not in others is noise
    with ClockSampler(local) as clk:
        e0.record()
        # only the final step's outputs are kept: holding each step's into the next would make the caching
        # allocator grow (cudaMalloc) inside the timed region
        for i in range(K - 1):
            one_step(dev_sets[i % R], kev[i])
        last = one_step(dev_sets[(K - 1) % R], kev[K - 1])
        e1.record()
        sync_all()
    gc.enable()
    launches = _lib.launch_count() - n0
    ms = shard.max_over_ranks(e0.elapsed_time(e1), dev)
    k_us = float(np.mean([a.elapsed_time(b) for a, b in kev])) * 1e3
    ar_ms = float(np.median([a.elapsed_time(b) for a, b in ar_events])) if ar_events else None
    if args.dump_outputs and rank == 0:
        dump_outputs(last["outputs"], args.dump_outputs)
    del last

    # ---- end to end through the public API with HOST buffers (`e2e`) ----
    # Every step copies its inputs from pinned host memory and reads its result back into pinned host memory; all
    # of it is inside the timed region.  Steps are independent, so the copy of step i+1 runs on a second stream
    # while step i computes (two device input slots, event-ordered).
    copy_s, back_s = torch.cuda.Stream(), torch.cuda.Stream()
    slots = [{k: torch.empty_like(v, device=dev) for k, v in pinned[0].items()} for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    host_out = [None, None]
    done_ev = [torch.cuda.Event() for _ in range(2)]

    def e2e_upload(i):
        j = i % 2
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(consumed[j])  # the step that last read this slot has finished
            for k, v in pinned[i % R].items():
                slots[j][k].copy_(v, non_blocking=True)
            copied[j].record(copy_s)

    def e2e_compute(i):
        j = i % 2
        main.wait_event(copied[j])
        res = one_step(slots[j])["result"]
        consumed[j].record(main)
        if host_out[j] is None:
            host_out[j] = [torch.empty(x.shape, dtype=x.dtype).pin_memory() for x in res]
        done_ev[j].record(main)
        with torch.cuda.stream(back_s):
            back_s.wait_event(done_ev[j])
            for h, x in zip(host_out[j], res):
                x.record_stream(back_s)
                h.copy_(x, non_blocking=True)
        return host_out[j]

    def e2e_run(n):
        for ev in consumed:
            ev.record(main)
        e2e_upload(0)
        for i in range(n):
            if i + 1 < n:
                e2e_upload(i + 1)
            res_ = e2e_compute(i)
        main.wait_stream(back_s)
        main.wait_stream(copy_s)
        return res_

    res = e2e_run(3)
    d2h_bytes = sum(x.numel() * x.element_size() for x in res)
    sync_all()
    with ClockSampler(local) as clk2:
        e0.record()
        e2e_run(K)
        e1.record()
        sync_all()
    clk.rows += clk2.rows  # clocks are reported over both timed regions
    e2e_local = e0.elapsed_time(e1)
    e2e_ms = shard.max_over_ranks(e2e_local, dev)
    h2d_gbs = h2d_bytes * K / (e2e_local * 1e-3) / 1e9
    if world > 1:
        t = torch.tensor([h2d_gbs], device=dev, dtype=torch.float64)
        gl = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gl, t)
        h2d_per_rank = [round(float(x.item()), 1) for x in gl]
    else:
        h2d_per_rank = [round(h2d_gbs, 1)]

    # ---- north-star shape (infer, rank 0 of a 1-GPU run): 512 rois x 256 ch x 14x14 on the same pyramid ----
    target = None
    if wl is Infer and world == 1 and not args.no_target:
        from simpledet_b200 import synth

        trng = np.random.default_rng(0)
        feats_cl = [torch.randn((1, h, w, C_FEAT), device=dev) for h, w in level_shapes(STRIDES_ROI)]
        feats_nchw = [f.permute(0, 3, 1, 2).contiguous() for f in feats_cl]
        rois_np = synth.random_rois(trng, 1, 512)
        rois = torch.from_numpy(rois_np).to(dev)
        flush = torch.empty(128 * 1024 * 1024, device=dev)

        def timed(fn):
            tev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(30)]
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            for a, b_ in tev:
                flush.fill_(1.0)  # 512 MB write: evicts the 126 MB L2
                a.record()
                fn()
                b_.record()
            torch.cuda.synchronize()
            ts = sorted(a.elapsed_time(b_) for a, b_ in tev)
            return ts[len(ts) // 2] * 1e3

        t_alg = roialign_algorithmic_bytes(rois_np, 1, 14, False)
        target = (timed(lambda: ops.fpn_roi_align_nhwc(feats_cl, rois, STRIDES_ROI, 14)),
                  timed(lambda: ops.fpn_roi_align_raw(feats_nchw, rois, STRIDES_ROI, 14, with_argmax=False)), t_alg)
        del flush

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * B * K / (ms / 1e3)
    e2e_value = world * B * K / (e2e_ms / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)"
    alg = wl.roofline_bytes(out, host_sets[0], B)
    achieved = alg / (k_us * 1e-6) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get(wl.name)
    except Exception:
        pass
    out_json = {
        "metric": "images/sec", "value": round(value, 2), "unit": "images/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl.text, "images_per_gpu_per_step": B, "global_images_per_step": B * world,
                   "parallelism": f"dp{world} (sharded by image" + (", one fp32 gradient all-reduce per step)" if wl.train
                                                                      else ", no data-path collective)"),
                   "l2": f"{R} rotating input sets ({int(R * set_mb)} MB) larger than L2, no flush",
                   "timed_region": f"{K} steps, e2e {K} steps",
                   "numa_binding": numa, "weights": "random synthetic activations (seeded)"},
        "clocks": clk.summary(),
        "e2e": {"value": round(e2e_value, 2), "unit": "images/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": round(e2e_ms / K, 4), "h2d_gbs_per_rank": h2d_per_rank},
        "gpu_launches": int(launches),
        "roofline": {"kernel": wl.kernel % (B * (N_ROI if wl is Infer else 512) if wl in (Infer, MaskTrain) else B),
                     "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic,
                     "algorithmic_bytes_per_launch": alg, "us_per_launch": round(k_us, 2),
                     "timed": "CUDA events around the operator inside the step (for RoIAlign: plan + layout + main "
                              "kernels together)", "peak_source": peak_src,
                     "share_of_step": round(k_us / (1e3 * ms / K), 4)},
    }
    if target is not None:
        t_cl, t_nchw, t_alg = target

        def entry(us, what):
            return {"kernel": what, "bound": "hbm", "achieved": round(t_alg / (us * 1e-6) / 1e9, 1), "peak": peak,
                    "unit": "GB/s", "frac": round(t_alg / (us * 1e-6) / 1e9 / peak, 4),
                    "algorithmic_bytes_per_launch": t_alg, "us_per_launch": round(us, 2), "peak_source": peak_src}

        out_json["roofline_target"] = entry(
            t_cl, "fused FPN RoIAlign_v2 forward, north-star shape 512 rois x 256 ch x 14x14, channels-last features "
                  "(whole operator: plan + order + roi_align_cl_kernel), L2 flushed before every launch")
        out_json["roofline_target_nchw"] = entry(
            t_nchw, "same shape through the NCHW operator contract (sdet_fpn_roi_align_v2_forward_ex, automatic path: "
                    "plan + order + per-roi kernel), L2 flushed before every launch")
    if wl.train:
        nbytes = GRAD_BUCKET_FLOATS * 4
        out_json["allreduce"] = {"bytes": nbytes, "ms": None if ar_ms is None else round(ar_ms, 3), "ranks": world,
                                 "bus_gbs": None if (ar_ms is None or world == 1) else
                                 round(2 * (world - 1) / world * nbytes / (ar_ms * 1e-3) / 1e9, 1),
                                 "note": "fp32 flat gradient bucket, ncclAllReduce(sum) + 1/G scale on a second stream, "
                                         "overlapped with the step's kernels; timed with events on that stream"}
    if world == 1 and not args.no_cpu_baseline:
        v, n = time_cpu(wl, host_sets[0])
        out_json["cpu_baseline"] = {"value": round(v, 3), "unit": "images/s", "cores": os.cpu_count() or 1,
                                    "kind": "port", "sample": f"{n} image(s) of the same workload; " + wl.cpu_note}
    print(json.dumps(out_json))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="infer", choices=sorted(WORKLOADS))
    ap.add_argument("--images-per-gpu", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-target", action="store_true", help="skip the north-star-shape measurement (keeps an ncu launch "
                    "list of the step free of its launches)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy "
                    "(float32, integers as float64; outputs over %d elements as a fixed seeded sample), so that two "
                    "builds can be compared on identical inputs" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
