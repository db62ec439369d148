"""Channels-last RoIAlign_v2 forward (roi_align_cl.cu: NHWC features, warp = 64 channels of one output bin, all
coordinates / weights warp-uniform) against the oracle and the per-roi kernel, through the C ABI; both with the
operator's NCHW contract (features re-laid to NHWC inside the call) and with channels-last features given directly.
BIT-EXACT like every forward path."""
import numpy as np
import pytest
import torch

import oracle
from simpledet_b200 import ops, synth

pytestmark = pytest.mark.gpu

CL = 3


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _single(data, rois, pooled, scale, dev):
    d, r = _t(data, dev), _t(rois, dev)
    out, _, _, used = ops.roi_align_v2_raw(d, r, pooled, scale, with_argmax=False, path=3, return_path=True)
    assert used == CL, f"channels-last path not taken (path_used={used})"
    ref, _, _ = oracle.roi_align_v2_forward(data, rois, pooled, scale)
    o = out.cpu().numpy()
    assert np.array_equal(o, ref), f"channels-last kernel differs from the oracle at {np.argwhere(o != ref)[:5]}"
    # the automatic choice for NCHW features is the planned per-roi kernel (fastest measured): same bits
    out0, _, _, used0 = ops.roi_align_v2_raw(d, r, pooled, scale, with_argmax=False, return_path=True)
    assert used0 == 1 and torch.equal(out0, out)
    # channels-last features handed in directly (single level = a 1-level pyramid with the matching stride)
    stride = int(round(1 / scale))
    if abs(1 / stride - scale) < 1e-12 and stride & (stride - 1) == 0:
        nh, _ = ops.fpn_roi_align_nhwc([d.permute(0, 2, 3, 1).contiguous()], r, (stride,), pooled)
        assert torch.equal(nh, out)


def test_config1_cl(cuda):
    data, rois, pooled, scale = synth.config1(0)
    _single(data, rois, pooled, scale, cuda)


@pytest.mark.parametrize("pooled", [(7, 7), (14, 14), (3, 5), (1, 1), (16, 16)])
@pytest.mark.parametrize("C", [2, 36, 64, 130])
def test_random_shapes_cl(cuda, pooled, C):
    rng = np.random.default_rng(C * 100 + pooled[0])
    data = rng.standard_normal((2, C, 50, 84)).astype(np.float32)
    rois = synth.random_rois(rng, 2, 60, 800, 1333)
    _single(data, rois, pooled, 1 / 16, cuda)


def test_edge_cases_cl(cuda):
    """Zero / outside / whole-map / integer-aligned / sub-0.01-stride (3 samples per axis: general table walk) /
    inverted / NaN / border-straddling rois."""
    rng = np.random.default_rng(7)
    data = rng.standard_normal((1, 8, 25, 42)).astype(np.float32)
    rois = np.array([[
        [0, 0, 0, 0], [-500, -400, -100, -50], [5000, 4000, 6000, 5000], [0, 0, 1343, 799],
        [96, 96, 96 + 7 * 48, 96 + 7 * 48], [100, 100, 100.2, 100.2], [100, 100, 101.5, 250],
        [64, 64, 64.96, 64.96], [300, 200, 100, 50], [np.nan, 10, 200, 300], [1200, 700, 1400, 900],
        [-30, -30, 60, 60], [10, 10, 700, 40], [10, 10, 40, 700],
    ]], np.float32)
    _single(data, rois, (7, 7), 1 / 32, cuda)
    _single(data, rois, (14, 14), 1 / 32, cuda)


def test_ties_cl(cuda):
    data = np.ones((1, 4, 50, 50), np.float32)
    data[:, 1] = 0.0
    data[:, 2, ::2] = 2.0
    data[:, 3] = -1.0
    rois = synth.random_rois(np.random.default_rng(2), 1, 64, 800, 800)
    _single(data, rois, (7, 7), 1 / 16, cuda)


def test_odd_maps_and_three_images_cl(cuda):
    rng = np.random.default_rng(5)
    data = rng.standard_normal((3, 10, 25, 25)).astype(np.float32)   # odd H*W: fine for channels-last
    rois = synth.random_rois(rng, 3, 50, 400, 400)
    _single(data, rois, (7, 7), 1 / 16, cuda)


def _fpn(B, N, C, pooled, dev, seed, check_oracle):
    rng = np.random.default_rng(seed)
    shapes = synth.fpn_shapes()
    feats_np = [rng.standard_normal((B, C, h, w)).astype(np.float32) for h, w in shapes]
    rois_np = synth.random_rois(rng, B, N)
    feats = [_t(f, dev) for f in feats_np]
    rois = _t(rois_np, dev)
    out, _, _, lv, used = ops.fpn_roi_align_raw(feats, rois, synth.FPN_STRIDES, pooled, with_argmax=False, path=3,
                                                return_path=True)
    assert used == CL
    per, _, _, lv1, used1 = ops.fpn_roi_align_raw(feats, rois, synth.FPN_STRIDES, pooled, with_argmax=False, path=1,
                                                  return_path=True)
    assert used1 == 1 and torch.equal(lv, lv1)
    assert torch.equal(out, per), "channels-last kernel differs from the per-roi kernel"
    nh, lv2 = ops.fpn_roi_align_nhwc([f.permute(0, 2, 3, 1).contiguous() for f in feats], rois, synth.FPN_STRIDES, pooled)
    assert torch.equal(nh, out) and torch.equal(lv2, lv)
    if check_oracle:
        ref, rl = oracle.fpn_roi_align_v2_forward(feats_np, rois_np, synth.FPN_STRIDES, (pooled, pooled))
        assert np.array_equal(lv.cpu().numpy(), rl) and np.array_equal(out.cpu().numpy(), ref)


def test_fpn_target_shape_small_c_cl(cuda):
    _fpn(1, 512, 16, 14, cuda, 0, True)


def test_fpn_bench_shape_small_c_cl(cuda):
    _fpn(2, 1000, 8, 7, cuda, 1, True)


def test_fpn_target_shape_full_cl(cuda):
    """The north-star shape, all 256 channels, bit for bit against the oracle's literal 4-level graph."""
    _fpn(1, 512, 256, 14, cuda, 0, True)


def test_fpn_bench_shape_full_cl(cuda):
    """roi_align_cl_kernel<256, 2>, the kernel of the headline metric, at the bench shape: all 256 channels against
    the oracle."""
    _fpn(2, 1000, 256, 7, cuda, 1, True)
