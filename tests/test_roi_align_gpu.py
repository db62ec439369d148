"""Parity of the CUDA RoIAlign_v2 / fused-FPN kernels with the oracle, through the C ABI.

Bar (BASELINE.json north_star): floats within 1e-4 relative.  The kernels are written to round
exactly like the reference's CPU build, so forward is checked BIT-EXACT (out, argmax_x,
argmax_y, empties); backward (unordered fp32 atomics) within rtol=1e-4."""
import numpy as np
import pytest
import torch

import oracle
from simpledet_b200 import ops, synth

pytestmark = pytest.mark.gpu


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _check_fwd(data, rois, pooled, scale, dev):
    out, ax, ay = ops.roi_align_v2_raw(_t(data, dev), _t(rois, dev), pooled, scale)
    ro, rx, ry = oracle.roi_align_v2_forward(data, rois, pooled, scale)
    o, x, y = out.cpu().numpy(), ax.cpu().numpy(), ay.cpu().numpy()
    assert np.array_equal(o, ro), f"out mismatch at {np.argwhere(o != ro)[:5]}"
    assert np.array_equal(x, rx) and np.array_equal(y, ry)
    out2, _, _ = ops.roi_align_v2_raw(_t(data, dev), _t(rois, dev), pooled, scale, with_argmax=False)
    assert np.array_equal(out2.cpu().numpy(), ro)
    # the inline-preamble path (no workspace) must agree with the pre-kernel path
    o3, x3, y3 = ops.roi_align_v2_raw(_t(data, dev), _t(rois, dev), pooled, scale, use_plan=False)
    assert torch.equal(o3, out) and torch.equal(x3, ax) and torch.equal(y3, ay)
    return ro, rx, ry


def test_config1_bit_exact(cuda):
    data, rois, pooled, scale = synth.config1(0)
    _check_fwd(data, rois, pooled, scale, cuda)


@pytest.mark.parametrize("pooled", [(7, 7), (14, 14), (3, 5), (1, 1), (32, 32)])
@pytest.mark.parametrize("C", [1, 16, 37])
def test_random_shapes(cuda, pooled, C):
    rng = np.random.default_rng(C * 100 + pooled[0])
    data = rng.standard_normal((2, C, 50, 84)).astype(np.float32)
    rois = synth.random_rois(rng, 2, 40, 800, 1333)
    _check_fwd(data, rois, pooled, 1 / 16, cuda)


def test_edge_cases(cuda):
    """Empty / zero rois, rois outside the image, integer-aligned samples, degenerate strides,
    whole-map windows (generic path), NaN roi, inverted roi."""
    rng = np.random.default_rng(7)
    data = rng.standard_normal((1, 8, 25, 42)).astype(np.float32)
    rois = np.array([[
        [0, 0, 0, 0],                 # zeroed roi (how FPN masks a level)
        [-500, -400, -100, -50],      # fully outside (negative)
        [5000, 4000, 6000, 5000],     # fully outside (beyond)
        [0, 0, 1343, 799],            # whole image -> whole-map window
        [96, 96, 96 + 7 * 48, 96 + 7 * 48],   # integer-aligned bins on the stride-32 grid
        [100, 100, 100.2, 100.2],     # tiny: stride < 0.01 -> step clamps to 0.01
        [100, 100, 101.5, 250],       # tiny in x only
        [64, 64, 64.96, 64.96],       # h_stride == 0.01 -> 3 samples per axis possible
        [300, 200, 100, 50],          # inverted (x2 < x1): negative bin size
        [np.nan, 10, 200, 300],       # NaN coordinate
        [1200, 700, 1400, 900],       # straddles the bottom-right border
        [-30, -30, 60, 60],           # straddles the top-left border
    ]], np.float32)
    _check_fwd(data, rois, (7, 7), 1 / 32, cuda)
    _check_fwd(data, rois, (14, 14), 1 / 32, cuda)


def test_ties_first_max_wins(cuda):
    """Constant and piecewise-constant maps make all samples tie; strict `>` keeps the first."""
    data = np.ones((1, 4, 50, 50), np.float32)
    data[:, 1] = 0.0
    data[:, 2, ::2] = 2.0
    data[:, 3] = -1.0
    rois = synth.random_rois(np.random.default_rng(2), 1, 64, 800, 800)
    _check_fwd(data, rois, (7, 7), 1 / 16, cuda)


def test_special_values(cuda):
    data = np.random.default_rng(4).standard_normal((1, 4, 20, 20)).astype(np.float32)
    data[0, 0, 5, 5] = np.inf
    data[0, 1, 6:9, 6:9] = -np.inf
    data[0, 2, 4:12, 4:12] = np.nan
    data[0, 3] = -np.finfo(np.float32).max
    rois = np.array([[[16, 16, 200, 200], [60, 60, 120, 130], [0, 0, 310, 310]]], np.float32)
    out, ax, ay = ops.roi_align_v2_raw(_t(data, cuda), _t(rois, cuda), (7, 7), 1 / 16)
    ro, rx, ry = oracle.roi_align_v2_forward(data, rois, (7, 7), 1 / 16)
    np.testing.assert_array_equal(out.cpu().numpy(), ro)  # NaN-aware equality
    np.testing.assert_array_equal(ax.cpu().numpy(), rx)
    np.testing.assert_array_equal(ay.cpu().numpy(), ry)


def test_batch_index_is_n_div_N(cuda):
    rng = np.random.default_rng(9)
    data = rng.standard_normal((3, 5, 30, 30)).astype(np.float32)
    rois = synth.random_rois(rng, 3, 17, 480, 480)
    _check_fwd(data, rois, (7, 7), 1 / 16, cuda)


@pytest.mark.parametrize("pooled", [(7, 7), (14, 14)])
def test_backward_matches_oracle(cuda, pooled):
    rng = np.random.default_rng(11)
    data = rng.standard_normal((2, 16, 50, 84)).astype(np.float32)
    rois = synth.random_rois(rng, 2, 64, 800, 1333)
    ro, rx, ry = oracle.roi_align_v2_forward(data, rois, pooled, 1 / 16)
    g = rng.standard_normal(ro.shape).astype(np.float32)
    d = _t(data, cuda).requires_grad_(True)
    out = ops.ROIAlign_v2(d, _t(rois, cuda), pooled, 1 / 16)
    assert np.array_equal(out.detach().cpu().numpy(), ro)
    out.backward(_t(g, cuda))
    rg = oracle.roi_align_v2_backward(g, rx, ry, data.shape)
    np.testing.assert_allclose(d.grad.cpu().numpy(), rg, rtol=1e-4, atol=1e-4)


def test_fpn_fused_equals_reference_graph(cuda):
    """fpn_roi_assign + 4 x ROIAlign_v2 + add_n (models/FPN/builder.py:573-605) == fused kernel."""
    rng = np.random.default_rng(13)
    shapes = synth.fpn_shapes(400, 672)
    feats = [rng.standard_normal((2, 8, h, w)).astype(np.float32) for h, w in shapes]
    rois = synth.random_rois(rng, 2, 96, 400, 672, 8, 600)
    rois[0, :4] = [[0, 0, 111, 111], [0, 0, 223, 223], [0, 0, 447, 447], [0, 0, 0, 0]]
    ref, idx = oracle.fpn_roi_align_v2_forward(feats, rois, synth.FPN_STRIDES, (7, 7))
    out, ax, ay, lv = ops.fpn_roi_align_raw([_t(f, cuda) for f in feats], _t(rois, cuda),
                                            synth.FPN_STRIDES, 7)
    assert np.array_equal(lv.cpu().numpy(), idx)
    assert np.array_equal(out.cpu().numpy(), ref)
    # backward: gradient lands only on the assigned level
    fs = [_t(f, cuda).requires_grad_(True) for f in feats]
    o = ops.fpn_roi_align(fs, _t(rois, cuda), synth.FPN_STRIDES, 7)
    g = rng.standard_normal(ref.shape).astype(np.float32)
    o.backward(_t(g, cuda))
    for i, (f, s) in enumerate(zip(feats, synth.FPN_STRIDES)):
        m = (idx == i)[..., None, None, None]
        rg = oracle.roi_align_v2_backward(np.where(m, g, 0).astype(np.float32),
                                          np.where(m, ax.cpu().numpy(), -1).astype(np.float32),
                                          np.where(m, ay.cpu().numpy(), -1).astype(np.float32), f.shape)
        np.testing.assert_allclose(fs[i].grad.cpu().numpy(), rg, rtol=1e-4, atol=1e-4)


def test_headline_shape_properties(cuda):
    """BASELINE size (512 rois x 256 ch x 14x14 on the 800x1333 pyramid): the oracle is too slow
    to run everything here, so check a channel slice bit-exactly plus size-independent
    properties: channel-permutation equivariance and max-of-samples bounds."""
    rng = np.random.default_rng(17)
    shapes = synth.fpn_shapes()
    feats = [torch.randn((1, 256, h, w), device=cuda) for h, w in shapes]
    rois = synth.random_rois(rng, 1, 512)
    out, ax, ay, lv = ops.fpn_roi_align_raw(feats, _t(rois, cuda), synth.FPN_STRIDES, 14)
    sl = slice(100, 104)
    ref, idx = oracle.fpn_roi_align_v2_forward([f[:, sl].cpu().numpy() for f in feats], rois,
                                               synth.FPN_STRIDES, (14, 14))
    assert np.array_equal(lv.cpu().numpy(), idx)
    assert np.array_equal(out[:, :, sl].cpu().numpy(), ref)
    perm = torch.randperm(256, device=cuda)
    out_p = ops.fpn_roi_align_raw([f[:, perm] for f in feats], _t(rois, cuda), synth.FPN_STRIDES,
                                  14, with_argmax=False)[0]
    assert torch.equal(out_p, out[:, :, perm])
    # a bilinear sample is a convex combination: |out| <= max |feat| of the level
    for i, f in enumerate(feats):
        m = (lv[0] == i)
        if m.any():
            assert out[0, m].abs().max() <= f.abs().max() * (1 + 1e-6)
    assert ((ax == -1) == (ay == -1)).all()


@pytest.mark.parametrize("pooled,n", [(7, 512), (14, 128)])
def test_training_forward_full_channels_with_argmax(cuda, pooled, n):
    """The training forward (argmax planes) at mask_train's shapes: B=2, 256 channels on the 800x1333 pyramid,
    512 rois per image at 7x7 and 128 at 14x14.  out, argmax_x and argmax_y bit for bit against the oracle, run once
    per level on the rois assigned to it (equivalent to the literal graph: test_fpn_fused_equals_reference_graph)."""
    rng = np.random.default_rng(19 + pooled)
    rois = synth.random_rois(rng, 2, n)
    feats = [rng.standard_normal((2, 256, h, w)).astype(np.float32) for h, w in synth.fpn_shapes()]
    out, ax, ay, lv = ops.fpn_roi_align_raw([_t(f, cuda) for f in feats], _t(rois, cuda), synth.FPN_STRIDES, pooled)
    idx = oracle.fpn_assign_levels(rois, synth.FPN_STRIDES).reshape(2, n)
    assert np.array_equal(lv.cpu().numpy(), idx)
    assert set(np.unique(idx)) == {0, 1, 2, 3}, "every level must receive rois"
    o, x, y = out.cpu().numpy(), ax.cpu().numpy(), ay.cpu().numpy()
    for b in range(2):
        for i, s in enumerate(synth.FPN_STRIDES):
            m = idx[b] == i
            if not m.any():
                continue
            ro, rx, ry = oracle.roi_align_v2_forward(feats[i][b:b + 1], rois[b:b + 1, m], (pooled, pooled), 1.0 / s)
            assert np.array_equal(o[b, m], ro[0]), f"out differs on image {b}, level {i}"
            assert np.array_equal(x[b, m], rx[0]) and np.array_equal(y[b, m], ry[0]), f"argmax, image {b} level {i}"


def test_error_codes(cuda):
    from simpledet_b200._lib import SdetError

    d = torch.zeros((1, 4, 8, 8), device=cuda)
    r = torch.zeros((1, 2, 4), device=cuda)
    with pytest.raises(SdetError, match="pooled_size"):
        ops.roi_align_v2_raw(d, r, (64, 64), 0.5)
    with pytest.raises(ValueError):
        ops.roi_align_v2_raw(d, torch.zeros((2, 2, 4), device=cuda), (7, 7), 0.5)
    with pytest.raises(TypeError):
        ops.roi_align_v2_raw(d.half(), r, (7, 7), 0.5)
