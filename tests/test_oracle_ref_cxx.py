"""Pins the oracle (oracle/*.c restatements) to the REFERENCE ITSELF: the reference's own operator_cxx sources,
compiled unmodified against oracle/shim (oracle/build_ref_cxx.py -> oracle/_ref/libref_cxx.so), are run on the
same inputs and every output is compared BIT FOR BIT.

CPU-only.  Where the compiled library is absent, each call is answered from the digests of what the library
returned (tests/reference_replay.py, tests/golden/reference_calls.json) and the comparisons are made against those."""
import numpy as np
import pytest

import oracle
from oracle import ref_cxx as _ref_cxx
from reference_replay import Reference, same
from simpledet_b200 import synth

ref_cxx = Reference(_ref_cxx if _ref_cxx.available() else None)
K_WRITE, K_ADD = _ref_cxx.K_WRITE, _ref_cxx.K_ADD

EDGE_ROIS = np.array([[
    [0, 0, 0, 0], [-500, -400, -100, -50], [5000, 4000, 6000, 5000], [0, 0, 1343, 799],
    [96, 96, 96 + 7 * 48, 96 + 7 * 48], [100, 100, 100.2, 100.2], [100, 100, 101.5, 250],
    [64, 64, 64.96, 64.96], [300, 200, 100, 50], [1200, 700, 1400, 900], [-30, -30, 60, 60],
]], np.float32)


# ------------------------------------------------------------------------------------------------ RoIAlign_v2
def _ra(data, rois, pooled, scale):
    kw = dict(pooled_size=pooled, spatial_scale=scale)
    shapes, nvis = ref_cxx.infer_shape("_contrib_ROIAlign_v2", kw, [data.shape, rois.shape])
    assert nvis == 1 and len(shapes) == 3  # roi_align_v2.cc:175-178: only `output` is visible
    B, N = rois.shape[:2]
    assert shapes[0] == (B, N, data.shape[1], pooled[0], pooled[1])
    out, ax, ay = ref_cxx.forward("_contrib_ROIAlign_v2", kw, [data, rois])
    ro, rx, ry = oracle.roi_align_v2_forward(data, rois, pooled, scale)
    assert same(out, ro) and same(ax, rx) and same(ay, ry)
    return out, ax, ay


def test_roi_align_forward_config1_and_shapes():
    data, rois, pooled, scale = synth.config1(0)
    _ra(data, rois, pooled, scale)
    _ra(data[:, :8], rois, (14, 14), scale)
    _ra(data[:, :5], rois[:, :40], (3, 5), scale)


def test_roi_align_forward_edge_cases():
    """SURVEY Appendix A 1-6: zero roi, rois outside, whole map, integer-aligned samples, sub-0.01 strides
    (3 samples per axis), inverted roi, border straddling; ties (first max wins)."""
    rng = np.random.default_rng(7)
    data = rng.standard_normal((1, 6, 25, 42)).astype(np.float32)
    _ra(data, EDGE_ROIS, (7, 7), 1 / 32)
    _ra(data, EDGE_ROIS, (14, 14), 1 / 32)
    const = np.ones((1, 4, 50, 50), np.float32)
    const[:, 1] = 0.0
    const[:, 2, ::2] = 2.0
    const[:, 3] = -1.0
    _ra(const, synth.random_rois(np.random.default_rng(2), 1, 64, 800, 800), (7, 7), 1 / 16)


def test_roi_align_two_images():
    rng = np.random.default_rng(3)
    data = rng.standard_normal((2, 4, 30, 40)).astype(np.float32)
    rois = synth.random_rois(rng, 2, 20, 480, 640)
    _ra(data, rois, (7, 7), 1 / 16)   # image index = n / num_rois_per_batch (roi_align_v2-inl.h:77)


def test_roi_align_backward_gpu_functor():
    """ROIAlignBackwardKernelGPU_v2 (roi_align_v2.cu:17-85) through the driver (:88-143), serial atomicAdd order;
    kWriteTo zero-fills, kAddTo accumulates, grad_rois is zero."""
    data, rois, pooled, scale = synth.config1(1)
    data = data[:, :16]
    kw = dict(pooled_size=pooled, spatial_scale=scale)
    out, ax, ay = ref_cxx.forward("_contrib_ROIAlign_v2", kw, [data, rois])
    g = np.random.default_rng(1).standard_normal(out.shape).astype(np.float32)
    rx, ry = oracle.roi_align_v2_forward(data, rois, pooled, scale)[1:]
    assert same(ax, rx) and same(ay, ry)
    gd, gr = ref_cxx.forward("_backward_ROIAlign_v2", kw, [g, rois, ax, ay], out_shapes=[data.shape, rois.shape], dev="gpu")
    assert same(gd, oracle.roi_align_v2_backward(g, rx, ry, data.shape))
    assert same(gr, np.zeros_like(rois))
    acc = np.full(data.shape, 0.5, np.float32)
    acc_ref, _ = ref_cxx.forward("_backward_ROIAlign_v2", kw, [g, rois, ax, ay], outputs=[acc.copy(), np.zeros_like(rois)],
                                 dev="gpu", reqs=[K_ADD, K_WRITE])
    assert same(acc_ref, oracle.roi_align_v2_backward(g, rx, ry, data.shape, accumulate_into=acc))


def test_roi_align_param_checks():
    """ROIAlignParam_v2 (roi_align_v2-inl.h:27-38): spatial_scale in [0,1], pooled_size 2-D and non-zero."""
    d, r = (1, 4, 10, 10), (1, 3, 4)
    for kw in (dict(pooled_size=(7, 7), spatial_scale=1.5), dict(pooled_size=(7, 7), spatial_scale=-0.1),
               dict(pooled_size=(7, 0), spatial_scale=0.5), dict(pooled_size=(7,), spatial_scale=0.5),
               dict(pooled_size=(7, 7))):
        with pytest.raises(RuntimeError):
            ref_cxx.infer_shape("_contrib_ROIAlign_v2", kw, [d, r])
    with pytest.raises(RuntimeError):  # bbox must be (B, N, 4)
        ref_cxx.infer_shape("_contrib_ROIAlign_v2", dict(pooled_size=(7, 7), spatial_scale=0.5), [d, (1, 3, 5)])


# ------------------------------------------------------------------------------------------------ ROIPooling_v1
@pytest.mark.parametrize("dev", ["cpu", "gpu"])   # gpu: roi_pooling_v1.cu's kernels run serially on the host
def test_roi_pooling_v1(dev):
    rng = np.random.default_rng(4)
    data = rng.standard_normal((2, 5, 30, 40)).astype(np.float32)
    r = synth.random_rois(rng, 1, 50, 480, 640)[0]
    rois = np.concatenate([rng.integers(0, 2, (50, 1)).astype(np.float32), r], 1)
    rois[0, 1:] = 0
    rois[1, 1:] = [700, 500, 800, 600]  # outside: empty bins
    for pooled, scale in (((7, 7), 1 / 16), ((2, 3), 1 / 16), ((6, 6), 0.7 / 16)):
        kw = dict(pooled_size=pooled, spatial_scale=scale)
        out, idx = ref_cxx.forward("ROIPooling_v1", kw, [data, rois], dev=dev)
        ro, ri = oracle.roi_pool_v1_forward(data, rois, pooled, scale)
        assert same(out, ro) and same(idx, ri)
        # Backward (ROIPoolBackwardAcc_v1: the .cc gathers per input pixel, the .cu likewise - no atomics)
        og = rng.standard_normal(out.shape).astype(np.float32)
        gd, _ = ref_cxx.backward("ROIPooling_v1", kw, [og], [data, rois], [out, idx], dev=dev)
        assert same(gd, oracle.roi_pool_v1_backward(og, ri, rois, data.shape))
    # the docstring vector of the reference (roi_pooling_v1.cc:265-285)
    x = np.arange(48, dtype=np.float32).reshape(1, 1, 8, 6)
    y = np.array([[0, 0, 0, 4, 4]], np.float32)
    out, _ = ref_cxx.forward("ROIPooling_v1", dict(pooled_size=(2, 2), spatial_scale=1.0), [x, y], dev=dev)
    assert same(out, np.array([14, 16, 26, 28], np.float32).reshape(1, 1, 2, 2))
    out, _ = ref_cxx.forward("ROIPooling_v1", dict(pooled_size=(2, 2), spatial_scale=0.7), [x, y], dev=dev)
    assert same(out, np.array([7, 9, 19, 21], np.float32).reshape(1, 1, 2, 2))


# ------------------------------------------------------------------------------------------------ DecodeBBox
@pytest.mark.parametrize("agnostic", [True, False])
@pytest.mark.parametrize("dtype", ["xywh", "xyxy"])
def test_decode_bbox(agnostic, dtype):
    rng = np.random.default_rng(5)
    B, N, K = 2, 300, 5
    rois = synth.random_rois(rng, B, N)
    deltas = (rng.standard_normal((B, N, 4 * K)) * np.array([1, 1, 2.5, 2.5] * K)).astype(np.float32)
    im_info = np.array([[800, 1333, 1.0], [600, 901, 1.5]], np.float32)
    kw = dict(class_agnostic=agnostic, bbox_decode_type=dtype, bbox_mean=(0.0, 0.1, 0.0, -0.1), bbox_std=(0.1, 0.1, 0.2, 0.2))
    (out,) = ref_cxx.forward("_contrib_DecodeBBox", kw, [rois, deltas, im_info])
    ref = oracle.decode_bbox(rois, deltas, im_info, kw["bbox_mean"], kw["bbox_std"], agnostic, dtype)
    assert same(out, ref)


def test_decode_bbox_defaults():
    """DecodeBBoxParam defaults (decodebbox-inl.h:55-67): class_agnostic=True, xywh, mean 0, std (.1,.1,.2,.2)."""
    rng = np.random.default_rng(6)
    rois = synth.random_rois(rng, 1, 50)
    deltas = rng.standard_normal((1, 50, 8)).astype(np.float32)
    im_info = np.array([[800, 1333, 1.0]], np.float32)
    shapes, _ = ref_cxx.infer_shape("_contrib_DecodeBBox", {}, [rois.shape, deltas.shape, im_info.shape])
    assert shapes == [(1, 50, 4)]
    (out,) = ref_cxx.forward("_contrib_DecodeBBox", {}, [rois, deltas, im_info])
    assert same(out, oracle.decode_bbox(rois, deltas, im_info))


# ------------------------------------------------------------------------------------------------ GenAnchor
@pytest.mark.parametrize("stride,scales,ratios,hw", [(16, (8.0,), (0.5, 1.0, 2.0), (13, 21)), (8, (4.0, 5.04, 6.35), (0.5, 1.0, 2.0), (10, 17)),
                                                     (32, (2.0, 4.0), (0.33, 1.7), (7, 9))])
def test_gen_anchor(stride, scales, ratios, hw):
    cls_prob = np.zeros((1, 2 * len(scales) * len(ratios), hw[0], hw[1]), np.float32)
    ref = oracle.gen_anchor(hw[0], hw[1], stride, scales, ratios)
    for dev in ("cpu", "gpu"):                    # generate_anchor.cc and generate_anchor.cu's kernel
        (out,) = ref_cxx.forward("_contrib_GenAnchor", dict(feature_stride=stride, scales=scales, ratios=ratios), [cls_prob],
                                 dev=dev)
        assert same(out, ref.reshape(out.shape)), dev


# ------------------------------------------------------------------------------------------------ ProposalTarget
def _rot(lst, k):
    lst = list(lst)
    for _ in range(k):
        lst = [lst[-1]] + lst[:-1] if lst else lst
    return lst


def _pt_inputs(rng, B, R, G, n_gt, n_fg_like):
    """rois = jittered copies of the gt boxes (many foreground) + random boxes, some zero-padded rows;
    gt (B,G,5) with class -1 padding."""
    gt = np.full((B, G, 5), -1, np.float32)
    rois = np.zeros((B, R, 4), np.float32)
    for b in range(B):
        g = synth.random_rois(rng, 1, n_gt, min_side=40, max_side=300)[0]
        gt[b, :n_gt, :4] = g
        gt[b, :n_gt, 4] = rng.integers(1, 81, n_gt)
        jit = g[rng.integers(0, n_gt, n_fg_like)] + rng.uniform(-12, 12, (n_fg_like, 4)).astype(np.float32)
        rnd = synth.random_rois(rng, 1, R - n_fg_like - 3)[0]
        rois[b, :n_fg_like] = jit
        rois[b, n_fg_like:R - 3] = rnd
    return rois, gt


def oracle_under_constant_rand(rois, gt, kw, rand_const, v2=False, valid_ranges=None, polys=None, mask_size=None,
                               output_ratio=False):
    """The oracle's ProposalTarget with the priorities that reproduce what libstdc++'s std::random_shuffle does
    when every rand() returns `rand_const` (0: rotate right by one; 27719: identity for lists <= 12)."""
    B, R, _ = rois.shape
    G = gt.shape[1]
    IR = kw["image_rois"]
    # the oracle's candidate lists, to express the reference's shuffles as priorities: run the oracle with
    # image_rois large enough to keep every candidate in index order (priority = index), read max-overlaps back
    T = R + G
    okw = dict(num_classes=kw["num_classes"], fg_fraction=kw.get("fg_fraction", 0.25), fg_thresh=kw["fg_thresh"],
               bg_thresh_hi=kw["bg_thresh_hi"], bg_thresh_lo=kw["bg_thresh_lo"],
               proposal_without_gt=kw["proposal_without_gt"], class_agnostic=kw.get("class_agnostic", False),
               bbox_mean=kw.get("bbox_mean", (0, 0, 0, 0)), bbox_std=kw.get("bbox_std", (0.1, 0.1, 0.2, 0.2)),
               bbox_weight=kw.get("bbox_weight", (1, 1, 1, 1)))
    if v2:
        okw.update(valid_ranges=valid_ranges, filter_scales=kw.get("filter_scales", False))
    ident = np.tile(np.arange(T, dtype=np.uint32), (B, 3, 1))
    probe = oracle.proposal_target(rois, gt, ident, image_rois=T, **dict(okw, fg_fraction=1.0, bg_thresh_lo=-1.0,
                                                                           bg_thresh_hi=kw["fg_thresh"]))
    # probe keeps [all fg in index order, then all non-fg in index order]: recover per-candidate max overlap
    fgq = int(IR * kw.get("fg_fraction", 0.25))
    rounds = 8
    pr = np.zeros((B, 2 + rounds, T), np.uint32)
    for b in range(B):
        kept, iou = probe[5][b], probe[4][b]
        n = int(kept.max()) + 1   # rows beyond the n distinct candidates are the probe's own negative padding
        ov = np.zeros(n, np.float32)
        ov[kept[:n]] = iou[:n]
        fg = [i for i in range(n) if ov[i] >= kw["fg_thresh"]]
        neg = [i for i in range(n) if not ov[i] >= kw["fg_thresh"]]
        bg = [i for i in range(n) if kw["bg_thresh_lo"] <= ov[i] < kw["bg_thresh_hi"]]
        if rand_const == 0:      # libstdc++ random_shuffle with rand() == 0: rotate right by one
            sh = lambda l, k: _rot(l, k)
        else:                     # rand() % (i+1) == i for every i <= 11: identity
            assert max(len(fg), len(bg), len(neg)) <= 12
            sh = lambda l, k: list(l)
        for d, lst in ((0, sh(fg, 1)), (1, sh(bg, 1))):
            pr[b, d] = T  # anything not in the list sorts last
            for pos, i in enumerate(lst):
                pr[b, d, i] = pos
        for r in range(rounds):
            pr[b, 2 + r] = T
            for pos, i in enumerate(sh(neg, r + 1)):
                pr[b, 2 + r, i] = pos
    if polys is not None:
        return oracle.proposal_mask_target(rois, gt, polys, pr, image_rois=IR, mask_size=mask_size,
                                           output_ratio=output_ratio, **okw)
    return oracle.proposal_target(rois, gt, pr, image_rois=IR, **okw)


def _run_pair(rois, gt, kw, rand_const, v2=False, valid_ranges=None):
    op = "ProposalTarget_v2" if v2 else "ProposalTarget"
    ref_cxx.set_rand_const(rand_const)
    ins = [rois, gt] + ([valid_ranges] if v2 else [])
    r_rois, r_lab, r_tgt, r_wgt, r_iou = ref_cxx.forward(op, dict(kw, batch_images=rois.shape[0]), ins)
    o = oracle_under_constant_rand(rois, gt, kw, rand_const, v2, valid_ranges)
    assert same(r_rois, o[0]), "rois"
    assert same(r_lab, o[1]), "labels"
    assert same(r_tgt, o[2]), "bbox_target"
    assert same(r_wgt, o[3]), "bbox_weight"
    assert same(r_iou, o[4]), "match_gt_iou"
    return o


BASE = dict(num_classes=81, image_rois=64, fg_thresh=0.5, bg_thresh_hi=0.5, bg_thresh_lo=0.0, proposal_without_gt=False)


def test_proposal_target_truncating_shuffles():
    """Plenty of fg and bg: both shuffles truncate (proposal_target.cc:81-85, 100-104); gt appended after the
    rois (-inl.h:177-185); zero-padded rois dropped by y2 > 0 (:174); padding gt by cls != -1 (:158)."""
    rng = np.random.default_rng(10)
    rois, gt = _pt_inputs(rng, 2, 300, 20, 6, 90)
    o = _run_pair(rois, gt, BASE, 0)
    assert (o[1][:, :16] > 0).all() and (o[1][:, 16:] == 0).all()   # labels only for the first fg_n rows
    _run_pair(rois, gt, dict(BASE, class_agnostic=True, num_classes=2), 0)
    _run_pair(rois, gt, dict(BASE, proposal_without_gt=True), 0)
    _run_pair(rois, gt, dict(BASE, bg_thresh_lo=0.1, fg_fraction=0.5, bbox_mean=(0.0, 0.0, 0.1, 0.1),
                             bbox_std=(0.2, 0.2, 0.3, 0.3), bbox_weight=(1.0, 2.0, 3.0, 4.0)), 0)


def test_proposal_target_negative_padding_rounds():
    """Few candidates: kept < image_rois, padded by re-shuffled negatives over several rounds (:116-122)."""
    rng = np.random.default_rng(11)
    rois, gt = _pt_inputs(rng, 2, 16, 6, 2, 5)
    _run_pair(rois, gt, dict(BASE, image_rois=64), 0)       # rotations
    _run_pair(rois, gt, dict(BASE, image_rois=48), 27719)   # identity shuffles (lists <= 12)


def test_proposal_target_v2():
    """ProposalTarget_v2: valid_ranges + filter_scales (proposal_target_v2-inl.h:186-203)."""
    rng = np.random.default_rng(12)
    rois, gt = _pt_inputs(rng, 2, 200, 12, 6, 60)
    vr = np.array([[0, 120], [100, 1000]], np.float32)
    _run_pair(rois, gt, dict(BASE, filter_scales=True), 0, v2=True, valid_ranges=vr)
    _run_pair(rois, gt, dict(BASE, filter_scales=False), 0, v2=True, valid_ranges=vr)


def test_proposal_target_shapes_and_visible_outputs():
    shapes, nvis = ref_cxx.infer_shape("ProposalTarget", dict(BASE, batch_images=2), [(2, 300, 4), (2, 20, 5)])
    assert shapes == [(2, 64, 4), (2, 64), (2, 64, 324), (2, 64, 324), (2, 64)] and nvis == 4
    _, nvis = ref_cxx.infer_shape("ProposalTarget", dict(BASE, batch_images=2, output_iou=True), [(2, 300, 4), (2, 20, 5)])
    assert nvis == 5


# ------------------------------------------------------------------------------------------------ FocalLoss / BBoxNorm
# focal_loss-inl.h / bbox_norm-inl.h are written as mshadow expression templates; the shim evaluates the same
# expression trees element by element (oracle/shim/mxnet_shim.h, namespace mshadow::expr).
def focal_case(seed, B=2, N=60, K=7):
    rng = np.random.default_rng(seed)
    data = (rng.standard_normal((B, N, K)) * 2.5 - 2).astype(np.float32)
    label = rng.integers(-1, K + 1, (B, N)).astype(np.float32)   # -1 ignore, 0 background, 1..K foreground
    ograd = rng.standard_normal((B, N, K)).astype(np.float32)
    return data, label, ograd


FOCAL_MODES = [dict(alpha=0.25, gamma=2.0, normalization="valid", grad_scale=1.0, out_grad=False),
               dict(alpha=0.5, gamma=1.5, normalization="batch", grad_scale=0.3, out_grad=True),
               dict(alpha=0.1, gamma=0.0, normalization="null", grad_scale=2.0, out_grad=False)]


@pytest.mark.parametrize("mode", range(len(FOCAL_MODES)))
def test_focal_loss_forward_backward(mode):
    kw = FOCAL_MODES[mode]
    data, label, ograd = focal_case(30 + mode)
    shapes, nvis = ref_cxx.infer_shape("_contrib_FocalLoss", dict(kw, workspace=8), [data.shape, label.shape])
    assert shapes == [data.shape] and nvis == 1
    (out,) = ref_cxx.forward("_contrib_FocalLoss", dict(kw, workspace=8), [data, label])
    prob = oracle.sigmoid(data)
    assert same(out, prob)
    gd, gl = ref_cxx.backward("_contrib_FocalLoss", dict(kw, workspace=8), [ograd], [data, label], [out])
    want = oracle.focal_loss_backward(prob, label, kw["alpha"], kw["gamma"], kw["grad_scale"], kw["normalization"],
                                      ograd if kw["out_grad"] else None)
    assert same(gd, want)
    assert np.abs(want).max() > 0 and not (want[label == -1] != 0).any()


def test_bbox_norm_backward():
    rng = np.random.default_rng(41)
    B, A4, P = 2, 12, 35
    data = rng.standard_normal((B, A4, P)).astype(np.float32)
    label = rng.integers(-1, 3, (B, (A4 // 4) * P)).astype(np.float32)
    gout = rng.standard_normal((B, A4, P)).astype(np.float32)
    (out,) = ref_cxx.forward("_contrib_BBoxNorm", {}, [data, label])
    assert same(out, data)                                             # identity forward (bbox_norm-inl.h:96)
    gd, gl = ref_cxx.backward("_contrib_BBoxNorm", {}, [gout], [data, label], [out])
    assert same(gd, oracle.bbox_norm_backward(gout, label)) and same(gl, np.zeros_like(label))
    zero = np.zeros_like(label)                                        # no positive label: divisor max(0 + 1, 1) = 1
    gd0, _ = ref_cxx.backward("_contrib_BBoxNorm", {}, [gout], [data, zero], [out])
    assert same(gd0, oracle.bbox_norm_backward(gout, zero))


# ------------------------------------------------------------------------------------------------ SigmoidCrossEntropy
def sigmoid_ce_case(seed=43, R=9, D=50):
    rng = np.random.default_rng(seed)
    data = (rng.standard_normal((R, D)) * 3).astype(np.float32)
    label = rng.integers(-1, 2, (R, D)).astype(np.float32)   # -1 ignore, 0 / 1 targets
    label[4] = -1                                             # a row with no valid target: loss 0 / (0 + 1e-5)
    return data, label


def test_sigmoid_cross_entropy_gpu_path_on_the_host():
    """The operator exists for the GPU only; its kernels (sigmoid_cross_entropy.cu:43-83) and the mshadow reductions
    around them run serially on the host (the build strips the `<<<...>>>` launch configurations, nothing else)."""
    data, label = sigmoid_ce_case()
    shapes, nvis = ref_cxx.infer_shape("_contrib_SigmoidCrossEntropy", dict(grad_scale=1.0), [data.shape, label.shape])
    assert nvis == 1 and shapes == [(9,), (9, 50), (9,), (9, 50), (9,)]
    with pytest.raises(RuntimeError):                         # sigmoid_cross_entropy.cc:41: the CPU operator is a stub
        ref_cxx.forward("_contrib_SigmoidCrossEntropy", dict(grad_scale=1.0), [data, label], dev="cpu")
    for scale in (1.0, 0.37):
        outs = ref_cxx.forward("_contrib_SigmoidCrossEntropy", dict(grad_scale=scale), [data, label], dev="gpu")
        loss = oracle.sigmoid_ce_forward(data, label)
        assert same(outs[0], loss) and loss[4] == 0
        (gd, _) = ref_cxx.backward("_contrib_SigmoidCrossEntropy", dict(grad_scale=scale), [np.ones_like(loss)],
                                   [data, label], outs, dev="gpu")
        assert same(gd, oracle.sigmoid_ce_backward(data, label, scale))


# ------------------------------------------------------------------------------------------------ Proposal_v3 (GPU operator)
# proposal_v3.cu is the operator SimpleDet runs (its CPU twin in proposal_v3.cc:372 reads the scores out of range).
# The build turns its launches into serial loops over every thread (oracle/build_ref_cxx.py, shim_launch) and gives it
# CUDA's float math overloads; thrust::stable_sort_by_key is std::stable_sort.
def rpn_case(seed, B=2, A=3, H=20, W=30, stride=16, shrink=(7, 20)):
    rng = np.random.default_rng(seed)
    logit = rng.standard_normal((B, A, H, W)).astype(np.float32) * 2 - 1
    fg = 1 / (1 + np.exp(-logit))
    cls = np.concatenate([1 - fg, fg], 1).astype(np.float32)
    cls[0, A:, 3, 4:9] = cls[0, A, 3, 4]                      # equal scores: the stable sort keeps index order
    reg = (rng.standard_normal((B, 4 * A, H, W)) * 0.3).astype(np.float32)
    reg[0, 2, 5, 5] = 9.0                                      # dw above the exp clip
    info = np.array([[H * stride - shrink[0], W * stride - shrink[1], 1.0], [H * stride, W * stride, 1.5]], np.float32)[:B]
    return cls, reg, info


PROPOSAL_V3_CASES = [
    dict(seed=0, kw=dict(rpn_pre_nms_top_n=300, rpn_post_nms_top_n=100, threshold=0.7, rpn_min_size=8, scales=(8,),
                         ratios=(0.5, 1, 2), feature_stride=16)),
    dict(seed=1, kw=dict(rpn_pre_nms_top_n=6000, rpn_post_nms_top_n=300, threshold=0.5, rpn_min_size=40, scales=(4, 8),
                         ratios=(0.5, 1, 2), feature_stride=16), A=6),          # pre > count, many boxes filtered
    dict(seed=2, kw=dict(rpn_pre_nms_top_n=200, rpn_post_nms_top_n=200, threshold=0.3, rpn_min_size=0, scales=(8,),
                         ratios=(1,), feature_stride=32), A=1, H=9, W=13, stride=32, shrink=(40, 70)),  # padded cells
]


@pytest.mark.parametrize("case", range(len(PROPOSAL_V3_CASES)))
@pytest.mark.parametrize("is_train", [False, True])
@pytest.mark.parametrize("iou_loss", [False, True])
def test_proposal_v3_gpu_operator(case, is_train, iou_loss):
    c = dict(PROPOSAL_V3_CASES[case])
    kw = dict(c.pop("kw"), is_train=is_train, iou_loss=iou_loss)
    cls, reg, info = rpn_case(**c)
    out, score = ref_cxx.forward("_contrib_Proposal_v3", dict(kw, output_score=True, workspace=64), [cls, reg, info], dev="gpu")
    r, sc = oracle.proposal_v3(cls, reg, info, **kw)
    n = r.shape[1]
    if n == out.shape[1]:
        assert same(out, r)
        assert same(score, sc)
    else:
        # is_train with fewer anchors than rpn_post_nms_top_n (P6 of an FPN in training: 819 < 2000).  The operator's
        # output keeps rpn_post_nms_top_n rows per image, but the loop shrinks its row count to n = min(post, pre)
        # and ALSO uses n as the per-image stride (proposal_v3.cu:471-476, :629-631): image b's n rows land at flat
        # row b*n of the (B, post) buffer, the rest is never written (stays zero).  The oracle returns (B, n) rows;
        # they must be the rows the reference wrote, wherever it put them.
        assert same(out, placed(out.shape, r, n, 4))
        assert same(score, placed(score.shape, sc, n, 1))


# ------------------------------------------------------------------------- the rest of the proposal family (GPU operators)
# proposal.cu, proposal_v2.cu, nms.cu, generate_proposal.cu, generate_proposal_retina.cu: same build treatment as
# proposal_v3.cu.  All of them shrink `rpn_post_nms_top_n` to min(post, pre) and then use the shrunken value as the
# per-image stride of the (B, post_param, .) output (proposal.cu / nms.cu PrepareOutput call sites), so when
# pre < post the rows of image b land at flat row b*n: `placed()` puts the oracle's rows where the reference puts
# them, in a zero buffer of the operator's output shape (the rows it never writes stay zero); `written()` reads them
# back from there (tests/golden/make_golden_cxx.py).
def written(buf, n, last):
    B = buf.shape[0]
    return buf.reshape(-1, last)[:B * n].reshape(B, n, last)


def placed(shape, rows, n, last):
    buf = np.zeros(shape, np.float32)
    B = shape[0]
    buf.reshape(-1, last)[:B * n] = np.asarray(rows)[:, :n].reshape(-1, last)
    return buf


@pytest.mark.parametrize("case", range(len(PROPOSAL_V3_CASES)))
@pytest.mark.parametrize("iou_loss", [False, True])
def test_proposal_v1_v2_gpu_operators(case, iou_loss):
    c = dict(PROPOSAL_V3_CASES[case])
    kw = dict(c.pop("kw"), iou_loss=iou_loss)
    cls, reg, info = rpn_case(**c)
    for is_train in (False, True):
        out, score = ref_cxx.forward("_contrib_Proposal", dict(kw, is_train=is_train, output_score=True, workspace=64),
                                     [cls, reg, info], dev="gpu")
        r, sc = oracle.proposal_legacy(cls, reg, info, version=1, is_train=is_train, **kw)
        assert same(out, placed(out.shape, r, r.shape[1], 4)), (is_train,)
        assert same(score, placed(score.shape, sc, r.shape[1], 1))
    vr = np.array([[0, 64], [32, 1e5]], np.float32)[:cls.shape[0]]
    for filt in (False, True):
        out, score = ref_cxx.forward("_contrib_Proposal_v2", dict(kw, filter_scales=filt, output_score=True, workspace=64),
                                     [cls, reg, info, vr], dev="gpu")
        r, sc = oracle.proposal_legacy(cls, reg, info, version=2, valid_ranges=vr, filter_scales=filt, **kw)
        assert same(out, placed(out.shape, r, r.shape[1], 4)), (filt,)
        assert same(score, placed(score.shape, sc, r.shape[1], 1))


def nms_case(seed=3, B=2, count=500):
    from simpledet_b200 import synth
    rng = np.random.default_rng(seed)
    sc = rng.uniform(0, 1, (B, count, 1)).astype(np.float32)
    sc[0, 10:20] = sc[0, 10]                                  # equal scores: stable order
    return np.concatenate([synth.random_rois(rng, B, count), sc], 2)


NMS_CASES = [(300, 100), (6000, 300), (200, 400)]             # pre < count; pre > count; post > pre (shrunken stride)


@pytest.mark.parametrize("already_sorted", [False, True])
@pytest.mark.parametrize("pre,post", NMS_CASES)
def test_contrib_nms_gpu_operator(already_sorted, pre, post):
    data = nms_case()
    if already_sorted:
        data = np.stack([x[np.argsort(-x[:, 4], kind="stable")] for x in data])
    kw = dict(rpn_pre_nms_top_n=pre, rpn_post_nms_top_n=post, threshold=0.6, already_sorted=already_sorted)
    out, score = ref_cxx.forward("_contrib_NMS", dict(kw, output_score=True, workspace=64), [data], dev="gpu")
    r, sc = oracle.contrib_nms(data, **kw)
    n = min(post, pre, data.shape[1])
    assert same(out, placed(out.shape, r, n, 4)) and same(score, placed(score.shape, sc, n, 1))


@pytest.mark.parametrize("case", range(len(PROPOSAL_V3_CASES)))
@pytest.mark.parametrize("iou_loss", [False, True])
def test_gen_proposal_gpu_operator(case, iou_loss):
    c = dict(PROPOSAL_V3_CASES[case])
    kw = c.pop("kw")
    cls, reg, info = rpn_case(**c)
    B, A2, H, W = cls.shape
    anchors = oracle.gen_anchor(H, W, kw["feature_stride"], kw["scales"], kw["ratios"])
    for pre in (150, A2 // 2 * H * W + 40):                   # more rows than anchors: the tail is never written
        k = dict(feature_stride=kw["feature_stride"], rpn_pre_nms_top_n=pre, rpn_min_size=kw["rpn_min_size"], iou_loss=iou_loss)
        (out,) = ref_cxx.forward("_contrib_GenProposal", dict(k, workspace=64), [cls, reg, info, anchors], dev="gpu")
        n = min(pre, A2 // 2 * H * W)
        want = np.zeros(out.shape, np.float32)
        want[:, :n] = oracle.gen_proposal(cls, reg, info, anchors, **k)[:, :n]
        assert same(out, want)


RETINA_CASES = [(80, 0.05, 1000, True), (80, 0.0, 300, True), (1, 0.3, 1000, True), (8, 0.05, 100, False)]


def retina_case(K, seed=52, B=2, A=9, H=13, W=21, stride=32):
    rng = np.random.default_rng(seed + K)
    cls = (rng.uniform(0, 1, (B, A * K, H, W)) ** 4).astype(np.float32)
    if K > 4:
        cls[0, :4] = cls[0, 4:8]                              # equal scores across classes
    reg = (rng.standard_normal((B, 4 * A, H, W)) * 0.5).astype(np.float32)
    info = np.array([[H * stride - 20, W * stride - 40, 1.0], [H * stride, W * stride, 1.6]], np.float32)
    anchors = oracle.gen_anchor(H, W, stride, tuple(4 * 2 ** (i / 3) for i in range(3)), (0.5, 1, 2))
    return cls, reg, info, anchors


@pytest.mark.parametrize("K,thresh,pre,one_hot", RETINA_CASES)
def test_gen_proposal_retina_gpu_operator(K, thresh, pre, one_hot):
    cls, reg, info, anchors = retina_case(K)
    kw = dict(num_anchors=9, rpn_pre_nms_top_n=pre, rpn_min_size=40, thresh=thresh, anchor_mean=(0.0, 0.1, 0.0, -0.1),
              anchor_std=(0.1, 0.1, 0.2, 0.2), output_one_hot=one_hot)
    box, score = ref_cxx.forward("_contrib_GenProposalRetina", dict(kw, feature_stride=32, workspace=256),
                                 [cls, reg, info, anchors], dev="gpu")
    rb, rs = oracle.gen_proposal_retina(cls, reg, info, anchors, **kw)
    assert same(box, rb) and same(score, rs)
    assert (rs != 0).any()


# -------------------------------------------------------------------------------------------------- ProposalMaskTarget
# proposal_mask_target.cc compiled against a stand-in maskApi.h (oracle/shim/coco_api/common/maskApi.h: cocoapi is not
# in the reference tree).  Pins the operator - matching, sampling, the polygon transform into roi coordinates
# (y first, :184-186), the union over segments - not the rasteriser, which is restated on both sides.
MASK_KW = dict(num_classes=81, image_rois=64, fg_thresh=0.5, bg_thresh_hi=0.5, bg_thresh_lo=0.0, proposal_without_gt=False)


@pytest.mark.parametrize("M", [14, 28])
@pytest.mark.parametrize("filter_scales,few_fg", [(False, False), (True, False), (False, True)])
def test_proposal_mask_target_operator(M, filter_scales, few_fg):
    rng = np.random.default_rng(60 + M)
    B, R, G, PL = 2, 200, 8, 400
    rois, gt, polys = synth.mask_scene(rng, B, R, G, PL)
    if few_fg:                                                # fewer foreground rois than mask rows: -1 rows stay (-inl.h:242)
        rois[:, 5:R - 20] = synth.random_rois(rng, B, R - 25, min_side=8, max_side=30)
    vr = np.array([[0, 150], [120, 1e5]], np.float32)
    kw = dict(MASK_KW, filter_scales=filter_scales)
    ref_cxx.set_rand_const(0)
    ins = [rois, gt, polys] + ([vr] if filter_scales else [])
    outs = ref_cxx.forward("ProposalMaskTarget", dict(kw, num_args=len(ins), batch_images=B, mask_size=M), ins)
    assert len(outs) >= 6 and outs[5].shape == (B, 16, M, M)
    o = oracle_under_constant_rand(rois, gt, kw, 0, v2=True, valid_ranges=vr if filter_scales else None, polys=polys,
                                   mask_size=M)
    for i, name in enumerate(("rois", "label", "bbox_target", "bbox_weight", "match_gt_iou", "mask_target")):
        assert same(outs[i], o[i]), name
    assert (o[5] == 1).sum() > 50 and (o[5] == 0).any() and (o[5] == -1).any() == few_fg


def mask_ratio_case(M, few_fg):
    rng = np.random.default_rng(70 + M)
    B, R, G, PL = 2, 200, 8, 400
    rois, gt, polys = synth.mask_scene(rng, B, R, G, PL)
    rois = (np.round(rois * 4) / 4).astype(np.float32) if few_fg else rois   # quarter-pixel corners: int() truncates
    if few_fg:
        rois[:, 5:R - 20] = synth.random_rois(rng, B, R - 25, min_side=8, max_side=30)
    return rois, gt, polys


MASK_RATIO_CASES = [(14, False), (28, True)]


@pytest.mark.parametrize("M,few_fg", MASK_RATIO_CASES)
def test_proposal_mask_target_output_ratio(M, few_fg):
    """Mask Scoring R-CNN form (models/msrcnn/builder.py:219-239): output_iou + output_ratio, 7 outputs.  The ratio
    is counted on integer rasters the size of the roi and of the polygon's extent (proposal_mask_target.cc:20-152),
    and the mask's vertex transform runs in double there (float in the plain operator)."""
    rois, gt, polys = mask_ratio_case(M, few_fg)
    B = rois.shape[0]
    ref_cxx.set_rand_const(0)
    outs = ref_cxx.forward("ProposalMaskTarget", dict(MASK_KW, num_args=3, batch_images=B, mask_size=M, output_iou=True,
                                                      output_ratio=True), [rois, gt, polys])
    assert len(outs) == 7 and outs[6].shape == (B, 16)
    o = oracle_under_constant_rand(rois, gt, MASK_KW, 0, polys=polys, mask_size=M, output_ratio=True)
    for i, name in enumerate(("rois", "label", "bbox_target", "bbox_weight", "match_gt_iou", "mask_target", "mask_ratio")):
        assert same(outs[i], o[i]), name
    r = o[6]
    assert ((r > 0) & (r <= 1)).sum() >= 5 and (r == 0).any() == few_fg and np.unique(r).size > 4
