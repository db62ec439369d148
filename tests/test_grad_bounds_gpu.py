"""The backward kernels against a float64 reference with a rounding-error bound (tests/grad_bounds.py), at the shapes
training runs and at the branches where kernels go wrong.

The backward kernels accumulate with unordered float32 atomics, so their result is not reproducible bit for bit; the
bound accepts any summation order and nothing else.  Each reference below recomputes every branch decision of the
kernel in float32, with the same operations (numpy float32 arithmetic rounds to nearest like the kernels, which are
built with -fmad=false), and forms the terms in float64 from those float32 weights.  The number of roundings k of
each term is read off the kernel source and written beside the check."""
import ctypes
import zlib

import numpy as np
import pytest
import torch

from grad_bounds import Accumulator
from simpledet_b200 import _lib, ops, synth
from simpledet_b200._lib import check

pytestmark = pytest.mark.gpu

F32 = np.float32
OLD_RA = (1e-4, 1e-4)      # (rtol, atol) of the older RoIAlign / ROIPooling backward tests
OLD_DCN_DATA = (1e-3, 1e-4)
OLD_DCN_OFF = (1e-3, 1e-3)
OLD_DCN2 = (2e-3, 2e-3)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _np(t):
    torch.cuda.synchronize()
    return t.detach().cpu().numpy()


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


# ---------------------------------------------------------------------------------------------------------------------
# RoIAlign_v2 backward (roi_align.cu: roi_align_v2_bwd_kernel)
# ---------------------------------------------------------------------------------------------------------------------
def _roi_align_ref(ograd, ax, ay, levels, shapes, C):
    """One Accumulator per level.  float32 decisions as in the kernel:
        skip if ax == -1 || ay == -1 (or the roi's level < 0)
        hl = clamp((int)floorf(ay), 0, H-1), hh = clamp((int)ceilf(ay), 0, H-1)  (same for x)
        al = hl == hh ? 0.5 : (ay - (float)hl) / (float)(hh - hl)                 (float32 sub, div)
    terms (float64 from the float32 al, be): d*(1-al)*(1-be), d*(1-al)*be, d*al*(1-be), d*al*be."""
    B, N, _, PH, PW = ograd.shape
    PP = PH * PW
    lv = np.zeros((B, N), np.int32) if levels is None else levels
    valid = (ax != F32(-1)) & (ay != F32(-1))
    accs = []
    for li, (H, W) in enumerate(shapes):
        acc = Accumulator(B * C * H * W)
        sel = np.flatnonzero(valid & (lv == li)[:, :, None, None, None])
        x, y, d = ax.ravel()[sel], ay.ravel()[sel], ograd.ravel()[sel].astype(np.float64)
        nc = sel // PP
        c, n = nc % C, nc // C
        base = ((n // N) * C + c) * H * W
        hl = np.clip(np.floor(y).astype(np.int64), 0, H - 1)
        hh = np.clip(np.ceil(y).astype(np.int64), 0, H - 1)
        wl = np.clip(np.floor(x).astype(np.int64), 0, W - 1)
        wr = np.clip(np.ceil(x).astype(np.int64), 0, W - 1)
        with np.errstate(divide="ignore", invalid="ignore"):
            al = np.where(hl == hh, F32(0.5), (y - hl.astype(F32)) / (hh - hl).astype(F32)).astype(np.float64)
            be = np.where(wl == wr, F32(0.5), (x - wl.astype(F32)) / (wr - wl).astype(F32)).astype(np.float64)
        corners = ((hl, wl, 1 - al, 1 - be), (hl, wr, 1 - al, be), (hh, wl, al, 1 - be), (hh, wr, al, be))
        acc.add(np.concatenate([base + hi * W + wi for hi, wi, _, _ in corners]),
                np.concatenate([d * wy * wx for _, _, wy, wx in corners]))
        accs.append(acc)
    return accs


# k = 3: __fmul_rn(__fmul_rn(d, a0), b0) with a0 = __fsub_rn(1, al) (the al/be branches have k = 2)
K_RA = 3


def _ra_bwd_abi(ograd, ax, ay, H, W, init=None, grad_rois=None):
    B, N, C, PH, PW = ograd.shape
    grad = torch.empty((B, C, H, W), device=ograd.device) if init is None else init.clone()
    check(_lib.lib().sdet_roi_align_v2_backward(_p(ograd), _p(ax), _p(ay), _p(grad), _p(grad_rois), B, N, C, H, W, PH,
                                                PW, 0 if init is None else 1, None))
    return grad


def _fpn_bwd_abi(ograd, ax, ay, levels, shapes, inits=None):
    B, N, C, PH, PW = ograd.shape
    L = len(shapes)
    grads = [torch.empty((B, C, h, w), device=ograd.device) if inits is None else inits[i].clone()
             for i, (h, w) in enumerate(shapes)]
    check(_lib.lib().sdet_fpn_roi_align_v2_backward(
        _p(ograd), _p(ax), _p(ay), _p(levels), (ctypes.c_void_p * L)(*[g.data_ptr() for g in grads]),
        (ctypes.c_int * L)(*[h for h, _ in shapes]), (ctypes.c_int * L)(*[w for _, w in shapes]), L, B, N, C, PH, PW,
        0 if inits is None else 1, None))
    return grads


@pytest.mark.parametrize("pooled,n", [(7, 512), (14, 128)])
def test_fpn_roi_align_backward_mask_train_shapes(cuda, pooled, n):
    """mask_train: B=2, 256 channels on the 800x1333 pyramid, rois on all four levels; through ops.fpn_roi_align with
    a contiguous ograd, with the non-contiguous ograd of out.sum().backward(), and through the ABI in kAddTo mode
    into pre-filled buffers (the initial value is one more term)."""
    rng = np.random.default_rng(100 + pooled)
    shapes = synth.fpn_shapes()
    rois = _t(synth.random_rois(rng, 2, n), cuda)
    feats = [torch.randn((2, 256, h, w), device=cuda, requires_grad=True) for h, w in shapes]
    out, ax, ay, lv = ops.fpn_roi_align_raw(feats, rois, synth.FPN_STRIDES, pooled)
    lv_np = _np(lv)
    assert set(np.unique(lv_np)) == {0, 1, 2, 3}
    ax_np, ay_np = _np(ax), _np(ay)

    g = torch.randn(out.shape, device=cuda)
    o = ops.fpn_roi_align(feats, rois, synth.FPN_STRIDES, pooled)
    o.backward(g)
    accs = _roi_align_ref(_np(g), ax_np, ay_np, lv_np, shapes, 256)
    for i, f in enumerate(feats):
        accs[i].check(_np(f.grad), K_RA, f"fpn RoIAlign bwd {pooled}x{pooled} level {i}", old_tol=OLD_RA)
        f.grad = None

    o = ops.fpn_roi_align(feats, rois, synth.FPN_STRIDES, pooled)
    o.sum().backward()  # ograd: an expanded scalar (stride 0)
    ones = _roi_align_ref(np.ones(out.shape, F32), ax_np, ay_np, lv_np, shapes, 256)
    for i, f in enumerate(feats):
        ones[i].check(_np(f.grad), K_RA, f"fpn RoIAlign bwd {pooled}x{pooled} sum() level {i}", old_tol=OLD_RA)

    inits = [torch.randn((2, 256, h, w), device=cuda) for h, w in shapes]
    grads = _fpn_bwd_abi(g, ax, ay, lv, shapes, inits)
    for i in range(4):
        accs[i].check(_np(grads[i]), K_RA, f"fpn RoIAlign bwd {pooled}x{pooled} kAddTo level {i}",
                      init=_np(inits[i]), old_tol=OLD_RA)


def test_roi_align_backward_same_roi_512_times(cuda):
    """Thousands of atomics per pixel; ograd a non-contiguous view; grad_rois all zero when passed."""
    rng = np.random.default_rng(5)
    data = torch.randn((2, 64, 50, 84), device=cuda, requires_grad=True)
    rois = _t(np.tile(np.array([[[200.3, 150.7, 420.9, 330.1]]], F32), (2, 512, 1)), cuda)
    out = ops.ROIAlign_v2(data, rois, (7, 7), 1 / 16)
    big = torch.randn(out.shape[:-1] + (14,), device=cuda)
    g = big[..., ::2]
    assert not g.is_contiguous()
    out.backward(g)
    _, ax, ay = ops.roi_align_v2_raw(data.detach(), rois, (7, 7), 1 / 16)
    acc = _roi_align_ref(_np(g), _np(ax), _np(ay), None, [(50, 84)], 64)[0]
    st = acc.check(_np(data.grad), K_RA, "RoIAlign bwd same roi x512", old_tol=OLD_RA)
    assert st["max_n"] >= 512
    gr = torch.full((2, 512, 4), float("nan"), device=cuda)
    grad = _ra_bwd_abi(g.contiguous(), ax, ay, 50, 84, grad_rois=gr)
    acc.check(_np(grad), K_RA, "RoIAlign bwd same roi x512 (ABI)", old_tol=OLD_RA)
    assert (_np(gr).view(np.uint32) == 0).all(), "grad_rois must be +0.0 everywhere"


def _special_argmax(rng, shape, H, W):
    """Argmax planes the kernel's branches care about: exact integers (hl == hh: both halves to one pixel), the last
    row / column, (H-1, H) and (-1, 0) (clamped: one pixel), 0, and the -1 sentinel on either plane."""
    ay = rng.uniform(-0.99, H - 0.01, shape).astype(F32)
    ax = rng.uniform(-0.99, W - 0.01, shape).astype(F32)
    r = rng.random(shape)
    ay[r < 0.1] = np.floor(ay[r < 0.1])
    ax[(r > 0.05) & (r < 0.15)] = np.floor(ax[(r > 0.05) & (r < 0.15)])
    ay[(r >= 0.15) & (r < 0.2)] = H - 1
    ax[(r >= 0.18) & (r < 0.23)] = W - 1
    ay[(r >= 0.23) & (r < 0.26)] = F32(H - 0.5)
    ax[(r >= 0.26) & (r < 0.29)] = F32(-0.25)
    ay[(r >= 0.29) & (r < 0.31)] = 0
    ax[(r >= 0.31) & (r < 0.36)] = -1
    ay[(r >= 0.36) & (r < 0.41)] = -1
    return ax, ay


def test_roi_align_backward_branches_single_level(cuda):
    """Synthetic argmax planes through the ABI: every clamp / integer branch, NaN in ograd at the sentinel bins (a read
    of one poisons the result), kAddTo into a pre-filled buffer, grad_rois zeroed."""
    rng = np.random.default_rng(6)
    B, N, C, H, W = 2, 300, 16, 13, 21
    ax, ay = _special_argmax(rng, (B, N, C, 7, 7), H, W)
    g = rng.standard_normal(ax.shape).astype(F32)
    g[(ax == -1) | (ay == -1)] = np.nan
    acc = _roi_align_ref(g, ax, ay, None, [(H, W)], C)[0]
    gd, axd, ayd = _t(g, cuda), _t(ax, cuda), _t(ay, cuda)
    gr = torch.full((B, N, 4), float("nan"), device=cuda)
    acc.check(_np(_ra_bwd_abi(gd, axd, ayd, H, W, grad_rois=gr)), K_RA, "RoIAlign bwd branches", old_tol=OLD_RA)
    assert (_np(gr).view(np.uint32) == 0).all()
    init = torch.randn((B, C, H, W), device=cuda)
    acc.check(_np(_ra_bwd_abi(gd, axd, ayd, H, W, init=init)), K_RA, "RoIAlign bwd branches kAddTo",
              init=_np(init), old_tol=OLD_RA)


def test_fpn_roi_align_backward_branches_and_unused_level(cuda):
    """Fused FPN backward through the ABI: rois with level -1 (NaN ograd: never read) and a level no roi is assigned
    to (its gradient stays exactly +0.0, or exactly its initial value in kAddTo mode)."""
    rng = np.random.default_rng(8)
    B, N, C = 2, 200, 8
    shapes = [(40, 60), (20, 30), (10, 15), (5, 8)]
    lv = rng.choice(np.array([-1, 0, 1, 3], np.int32), (B, N)).astype(np.int32)   # level 2 receives nothing
    ax = np.empty((B, N, C, 7, 7), F32)
    ay = np.empty_like(ax)
    for li, (H, W) in enumerate(shapes):
        x, y = _special_argmax(rng, ax.shape, H, W)
        m = np.broadcast_to((lv == li)[:, :, None, None, None], ax.shape)
        ax[m], ay[m] = x[m], y[m]
    m = np.broadcast_to((lv == -1)[:, :, None, None, None], ax.shape)
    ax[m], ay[m] = 1.5, 2.5
    g = rng.standard_normal(ax.shape).astype(F32)
    g[((ax == -1) | (ay == -1)) | m] = np.nan
    accs = _roi_align_ref(g, ax, ay, lv, shapes, C)
    args = (_t(g, cuda), _t(ax, cuda), _t(ay, cuda), _t(lv, cuda), shapes)
    for i, got in enumerate(_fpn_bwd_abi(*args)):
        accs[i].check(_np(got), K_RA, f"fpn RoIAlign bwd branches level {i}", old_tol=OLD_RA)
    assert (_np(_fpn_bwd_abi(*args)[2]).view(np.uint32) == 0).all()
    inits = [torch.randn((B, C, h, w), device=cuda) for h, w in shapes]
    for i, got in enumerate(_fpn_bwd_abi(*args, inits=inits)):
        accs[i].check(_np(got), K_RA, f"fpn RoIAlign bwd branches kAddTo level {i}", init=_np(inits[i]),
                      old_tol=OLD_RA)


# ---------------------------------------------------------------------------------------------------------------------
# ROIPooling_v1 backward (roi_pool.cu: roi_pool_v1_bwd_kernel)
# ---------------------------------------------------------------------------------------------------------------------
def _roi_pool_ref(ograd, max_idx, rois, B, C, H, W):
    """terms: ograd[r, c, ph, pw] itself at max_idx (k = 0: no arithmetic before the sum), for max_idx >= 0 and a
    batch index (int)rois[r, 0] in [0, B)."""
    R = ograd.shape[0]
    bi = rois[:, 0].astype(np.int64)
    ok = (max_idx >= 0) & ((bi >= 0) & (bi < B))[:, None, None, None]
    sel = np.flatnonzero(ok)
    PP = ograd.shape[2] * ograd.shape[3]
    nc = sel // PP
    c, r = nc % C, nc // C
    acc = Accumulator(B * C * H * W)
    acc.add((bi[r] * C + c) * H * W + max_idx.ravel()[sel].astype(np.int64), ograd.ravel()[sel].astype(np.float64))
    return acc


def _pool_rois(rng, B, n, img_h, img_w):
    r = synth.random_rois(rng, B, n, img_h, img_w).reshape(B * n, 4)
    return np.concatenate([np.repeat(np.arange(B, dtype=F32), n)[:, None], r], 1).astype(F32)


def test_roi_pool_backward_training_shape(cuda):
    """B=2, 512 rois per image, 256 channels, 7x7, through ops.ROIPooling_v1."""
    rng = np.random.default_rng(21)
    data = torch.randn((2, 256, 50, 84), device=cuda, requires_grad=True)
    rois = _t(_pool_rois(rng, 2, 512, 800, 1333), cuda)
    out = ops.ROIPooling_v1(data, rois, (7, 7), 1 / 16)
    g = torch.randn(out.shape, device=cuda)
    out.backward(g)
    _, idx = ops.roi_pooling_v1_raw(data.detach(), rois, (7, 7), 1 / 16)
    acc = _roi_pool_ref(_np(g), _np(idx), _np(rois), 2, 256, 50, 84)
    acc.check(_np(data.grad), 0, "ROIPooling bwd 2x512x256 7x7", old_tol=OLD_RA)


def test_roi_pool_backward_ties_overlap_empty_bins_kaddto(cuda):
    """Constant maps (every bin ties: the first index wins, checked against the oracle), heavily overlapping rois,
    rois partly outside the map (empty bins, max_idx -1, NaN ograd there), kAddTo, grad_rois zeroed."""
    import oracle

    rng = np.random.default_rng(22)
    B, C, H, W = 2, 8, 30, 40
    data = rng.standard_normal((B, C, H, W)).astype(F32)
    data[:, :3] = 1.0
    data[1, 3] = -2.0
    rois = np.concatenate([
        np.tile(np.array([[0, 100, 90, 300, 260], [1, 96, 96, 240, 240]], F32), (40, 1)),   # 80 overlapping rois
        _pool_rois(rng, B, 60, 480, 640),
        np.array([[0, 560, 400, 900, 700], [1, -300, -200, 50, 60], [0, 600, 100, 1000, 200]], F32),  # beyond edges
    ])
    out, idx = ops.roi_pooling_v1_raw(_t(data, cuda), _t(rois, cuda), (7, 7), 1 / 16)
    ro, ri = oracle.roi_pool_v1_forward(data, rois, (7, 7), 1 / 16)
    np.testing.assert_array_equal(_np(out), ro)
    np.testing.assert_array_equal(_np(idx), ri)
    assert (ri == -1).any(), "no empty bin"
    g = rng.standard_normal(ro.shape).astype(F32)
    g[ri == -1] = np.nan
    acc = _roi_pool_ref(g, ri, rois, B, C, H, W)
    R = rois.shape[0]
    for init in (None, torch.randn((B, C, H, W), device=cuda)):
        grad = torch.empty((B, C, H, W), device=cuda) if init is None else init.clone()
        gr = torch.full((R, 5), float("nan"), device=cuda)
        check(_lib.lib().sdet_roi_pooling_v1_backward(_p(_t(g, cuda)), _p(idx), _p(_t(rois, cuda)), _p(grad), _p(gr),
                                                      B, R, C, H, W, 7, 7, 1 / 16, 0 if init is None else 1, None))
        acc.check(_np(grad), 0, "ROIPooling bwd ties/overlap/empty" + ("" if init is None else " kAddTo"),
                  init=None if init is None else _np(init), old_tol=OLD_RA)
        assert (_np(gr).view(np.uint32) == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# DCN v1 deform_col2im_kernel and v2 mdeform_col2im_kernel (dcn.cu), driven with a random grad_col
# ---------------------------------------------------------------------------------------------------------------------
def _out_hw(H, W, kh, kw, pad, stride, dil):
    return ((H + 2 * pad[0] - (dil[0] * (kh - 1) + 1)) // stride[0] + 1,
            (W + 2 * pad[1] - (dil[1] * (kw - 1) + 1)) // stride[1] + 1)


def _dcn_ref(data, offset, mask, gcol, k, pad, stride, dil, dg):
    """-> (Accumulator data, Accumulator offset, Accumulator mask or None).  float32 decisions as in the kernels:
        h = (float)(h_col*stride - pad + i*dil) + offset           (float32 add)
        v1: inside 0 <= h < H;  h_low = floorf(h); h_low >= H-1 -> h_low = h_high = H-1, h = h_low (offset grad 0)
        v2: inside -1 < h < H;  corners outside [0, H-1] read 0 and receive nothing
        lh = h - h_low, hh = 1 - lh                                (float32)
    terms in float64 from those float32 weights."""
    B, C, H, W = data.shape
    kh, kw = k
    T = kh * kw
    Ho, Wo = _out_hw(H, W, kh, kw, pad, stride, dil)
    P = Ho * Wo
    cpg = C // dg
    v2 = mask is not None
    acc_d = Accumulator(B * C * H * W)
    acc_o = np.zeros((3, B, dg, T, 2, P))       # exact, absum, count of the offset gradient
    acc_m = np.zeros((3, B, dg, T, P))
    ti, tj = np.divmod(np.arange(T), kw)
    hb = (np.arange(Ho)[None, :, None] * stride[0] - pad[0] + ti[:, None, None] * dil[0]).repeat(Wo, 2).reshape(T, P)
    wb = (np.arange(Wo)[None, None, :] * stride[1] - pad[1] + tj[:, None, None] * dil[1]).repeat(Ho, 1).reshape(T, P)
    for b in range(B):
        for g in range(dg):
            off = offset[b, g * 2 * T:(g + 1) * 2 * T].reshape(T, 2, P)
            h = hb.astype(F32) + off[:, 0]
            w = wb.astype(F32) + off[:, 1]
            if v2:
                inside = (h > F32(-1)) & (w > F32(-1)) & (h < F32(H)) & (w < F32(W))
            else:
                inside = (h >= F32(0)) & (w >= F32(0)) & (h < F32(H)) & (w < F32(W))
            h = np.where(inside, h, F32(0))
            w = np.where(inside, w, F32(0))
            hl = np.floor(h).astype(np.int64)
            wl = np.floor(w).astype(np.int64)
            if v2:
                hcl = wcl = np.zeros_like(inside)
            else:
                hcl, wcl = hl >= H - 1, wl >= W - 1
                hl = np.where(hcl, H - 1, hl)
                wl = np.where(wcl, W - 1, wl)
                h = np.where(hcl, hl.astype(F32), h)
                w = np.where(wcl, wl.astype(F32), w)
            hh_i = np.where(hcl, hl, hl + 1)
            wh_i = np.where(wcl, wl, wl + 1)
            lh = (h - hl.astype(F32)).astype(np.float64)
            lw = (w - wl.astype(F32)).astype(np.float64)
            hh = (F32(1) - (h - hl.astype(F32))).astype(np.float64)
            hw = (F32(1) - (w - wl.astype(F32))).astype(np.float64)
            corners = [(hl, wl), (hl, wh_i), (hh_i, wl), (hh_i, wh_i)]
            oks = [inside & (hi >= 0) & (hi <= H - 1) & (wi >= 0) & (wi <= W - 1) for hi, wi in corners]
            cs = slice(g * cpg, (g + 1) * cpg)
            im = data[b, cs].reshape(cpg, H * W).astype(np.float64)
            vals = [np.where(ok, im[:, np.clip(hi, 0, H - 1) * W + np.clip(wi, 0, W - 1)], 0.0)
                    for (hi, wi), ok in zip(corners, oks)]                       # (cpg, T, P)
            go = gcol[b, cs.start * T:cs.stop * T].reshape(cpg, T, P).astype(np.float64)
            gm = go * mask[b, g * T:(g + 1) * T].reshape(T, P).astype(np.float64) if v2 else go
            base = (b * C + np.arange(g * cpg, (g + 1) * cpg))[:, None, None] * H * W
            for (hi, wi), ok, wgt in zip(corners, oks, (hh * hw, hh * lw, lh * hw, lh * lw)):
                sel = np.broadcast_to(ok, go.shape)
                acc_d.add((base + hi * W + wi)[sel], (gm * wgt)[sel])
            v1_, v2_, v3_, v4_ = vals
            a1, a2, a3, a4 = (np.abs(v) for v in vals)
            for comp, live, t_, ta in ((0, inside & ~hcl, hw * (v3_ - v1_) + lw * (v4_ - v2_),
                                        hw * (a3 + a1) + lw * (a4 + a2)),
                                       (1, inside & ~wcl, hh * (v2_ - v1_) + lh * (v4_ - v3_),
                                        hh * (a2 + a1) + lh * (a4 + a3))):
                acc_o[0, b, g, :, comp] = np.where(live, (gm * t_).sum(0), 0.0)
                acc_o[1, b, g, :, comp] = np.where(live, (np.abs(gm) * ta).sum(0), 0.0)
                acc_o[2, b, g, :, comp] = np.where(live, cpg, 0)
            if v2:
                s = hh * hw * v1_ + hh * lw * v2_ + lh * hw * v3_ + lh * lw * v4_
                sa = hh * hw * a1 + hh * lw * a2 + lh * hw * a3 + lh * lw * a4
                acc_m[0, b, g] = np.where(inside, (go * s).sum(0), 0.0)
                acc_m[1, b, g] = np.where(inside, (np.abs(go) * sa).sum(0), 0.0)
                acc_m[2, b, g] = np.where(inside, cpg, 0)
    ao = Accumulator(acc_o[0].size)
    ao.add_dense(*acc_o)
    am = None
    if v2:
        am = Accumulator(acc_m[0].size)
        am.add_dense(*acc_m)
    return acc_d, ao, am


# roundings per term (dcn.cu, built with -fmad=false):
#   v1 data   go * hh * hw                                    k = 2
#   v1 offset go * (hw * (v3 - v1) + lw * (v4 - v2))          k = 4  (sub, mul, add, mul)
#   v2 data   (go * m) * hh * hw                              k = 3
#   v2 offset (go * m) * (hw * (v3 - v1) + lw * (v4 - v2))    k = 5
#   v2 mask   go * (hh*hw*v1 + hh*lw*v2 + lh*hw*v3 + lh*lw*v4) k = 6  (2 products, 3 sums, 1 product)
K_V1_DATA, K_V1_OFF, K_V2_DATA, K_V2_OFF, K_V2_MASK = 2, 4, 3, 5, 6


def _run_col2im(data, offset, mask, gcol, k, pad, stride, dil, dg, dev):
    B, C, H, W = data.shape
    d, o, gc = _t(data, dev), _t(offset, dev), _t(gcol, dev)
    gd, go = torch.empty_like(d), torch.empty_like(o)
    geo = (B, C, H, W, k[0], k[1], pad[0], pad[1], stride[0], stride[1], dil[0], dil[1], dg, None)
    if mask is None:
        check(_lib.lib().sdet_deformable_col2im(_p(gc), _p(d), _p(o), _p(gd), _p(go), *geo))
        return _np(gd), _np(go), None
    m = _t(mask, dev)
    gm = torch.empty_like(m)
    check(_lib.lib().sdet_modulated_deformable_col2im(_p(gc), _p(d), _p(o), _p(m), _p(gd), _p(go), _p(gm), *geo))
    return _np(gd), _np(go), _np(gm)


def _edge_offsets(rng, B, dg, k, Ho, Wo, H, W, pad, stride, dil):
    """Offsets that put samples exactly on integers, on 0, -1, H-1 and H, inside [H-1, H) and inside (-1, 0), mixed
    with random positions (same rule on the w axis)."""
    kh, kw = k
    T = kh * kw
    hb = (np.arange(Ho)[:, None] * stride[0] - pad[0]).repeat(Wo, 1).ravel()
    wb = (np.arange(Wo)[None, :] * stride[1] - pad[1]).repeat(Ho, 0).ravel()
    off = np.empty((B, dg, T, 2, Ho * Wo), F32)
    for ax_, base, n, dl, kk in ((0, hb, H, dil[0], np.arange(T) // kw), (1, wb, W, dil[1], np.arange(T) % kw)):
        special = np.array([0, -1, n - 1, n, n - 0.5, n - 0.75, -0.5, -0.125, 1, 2, n // 2, n - 2], F32)
        tgt = rng.uniform(-2, n + 1, (B, dg, T, Ho * Wo)).astype(F32)
        pick = rng.random(tgt.shape) < 0.6
        tgt[pick] = rng.choice(special, int(pick.sum()))
        off[:, :, :, ax_] = (tgt - (base[None, None, None] + kk[None, None, :, None] * dl)).astype(F32)
    return off.reshape(B, dg * 2 * T, Ho, Wo)


DCN_CASES = {
    # name: (B, C, H, W, k, pad, stride, dil, dg, offsets)
    "block_2x256x50x84_dg4": (2, 256, 50, 84, (3, 3), (1, 1), (1, 1), (1, 1), 4, "random"),
    "dg1": (1, 8, 13, 17, (3, 3), (1, 1), (1, 1), (1, 1), 1, "random"),
    "C6_dg3": (2, 6, 13, 17, (3, 3), (1, 1), (1, 1), (1, 1), 3, "random"),
    "stride2_dil2_pad0": (2, 8, 23, 31, (3, 3), (0, 0), (2, 2), (2, 2), 2, "random"),
    "stride2_dil2_pad2": (1, 8, 27, 19, (3, 3), (2, 2), (2, 2), (2, 2), 2, "random"),
    "edges": (2, 8, 11, 14, (3, 3), (1, 1), (1, 1), (1, 1), 2, "edges"),
    "edges_stride2_pad0": (1, 6, 12, 9, (3, 3), (0, 0), (2, 2), (1, 1), 3, "edges"),
    "one_pixel_contention": (1, 4, 30, 40, (3, 3), (1, 1), (1, 1), (1, 1), 1, "one_pixel"),
}


@pytest.mark.parametrize("case", list(DCN_CASES))
@pytest.mark.parametrize("version", ["v1", "v2"])
def test_dcn_col2im_bound(cuda, case, version):
    B, C, H, W, k, pad, stride, dil, dg, kind = DCN_CASES[case]
    rng = np.random.default_rng(zlib.crc32(f"{case}/{version}".encode()))
    Ho, Wo = _out_hw(H, W, *k, pad, stride, dil)
    T = k[0] * k[1]
    assert case != "stride2_dil2_pad0" or (Ho * Wo) % 256 != 0
    data = rng.standard_normal((B, C, H, W)).astype(F32)
    if kind == "random":
        offset = (rng.standard_normal((B, dg * 2 * T, Ho, Wo)) * 2).astype(F32)
    elif kind == "edges":
        offset = _edge_offsets(rng, B, dg, k, Ho, Wo, H, W, pad, stride, dil)
    else:  # every tap of every output pixel samples around (5.25, 7.5)
        offset = _edge_offsets(rng, B, dg, k, Ho, Wo, H, W, pad, stride, dil)
        o = offset.reshape(B, dg, T, 2, Ho * Wo)
        hb = (np.arange(Ho)[:, None] * stride[0] - pad[0]).repeat(Wo, 1).ravel()
        wb = (np.arange(Wo)[None, :] * stride[1] - pad[1]).repeat(Ho, 0).ravel()
        o[:, :, :, 0] = (F32(5.25) - (hb[None] + (np.arange(T) // k[1])[:, None] * dil[0])).astype(F32)
        o[:, :, :, 1] = (F32(7.5) - (wb[None] + (np.arange(T) % k[1])[:, None] * dil[1])).astype(F32)
        offset = o.reshape(B, dg * 2 * T, Ho, Wo)
    mask = rng.uniform(0, 1, (B, dg * T, Ho, Wo)).astype(F32) if version == "v2" else None
    gcol = rng.standard_normal((B, C * T, Ho * Wo)).astype(F32)
    gd, go, gm = _run_col2im(data, offset, mask, gcol, k, pad, stride, dil, dg, cuda)
    ad, ao, am = _dcn_ref(data, offset, mask, gcol, k, pad, stride, dil, dg)
    name = f"DCN{version} col2im {case}"
    if version == "v1":
        ad.check(gd, K_V1_DATA, name + " data", old_tol=OLD_DCN_DATA)
        ao.check(go, K_V1_OFF, name + " offset", old_tol=OLD_DCN_OFF)
        if kind == "edges":
            assert (ao.count == 0).any(), "no clamped sample: the zero offset-gradient rule was not exercised"
    else:
        ad.check(gd, K_V2_DATA, name + " data", old_tol=OLD_DCN2)
        ao.check(go, K_V2_OFF, name + " offset", old_tol=OLD_DCN2)
        am.check(gm, K_V2_MASK, name + " mask", old_tol=OLD_DCN2)
    if kind == "one_pixel":
        assert ad.count.max() >= T * Ho * Wo


def test_dcn_channels_last_data_through_the_operator(cuda):
    """ops.DeformableConvolution with channels-last data (the NHWC im2col and its GEMM layout).  The weight is the
    identity on the (channel, tap) columns, so grad_col == grad_out exactly, whatever the GEMM's precision: gout is
    drawn with 8 significant bits.  data and offset gradients meet the same bound as through the ABI."""
    rng = np.random.default_rng(31)
    B, C, H, W, dg = 2, 16, 20, 24, 2
    T = 9
    data = rng.standard_normal((B, C, H, W)).astype(F32)
    offset = _edge_offsets(rng, B, dg, (3, 3), H, W, H, W, (1, 1), (1, 1), (1, 1))
    weight = np.zeros((C * T, C, 3, 3), F32)
    for c in range(C):
        for t in range(T):
            weight[c * T + t, c, t // 3, t % 3] = 1.0
    gout = rng.standard_normal((B, C * T, H, W)).astype(F32)
    m, e = np.frexp(gout)
    gout = np.ldexp(np.round(m * 256) / 256, e).astype(F32)
    x = _t(data, cuda).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    off = _t(offset, cuda).requires_grad_(True)
    y = ops.DeformableConvolution(x, off, _t(weight, cuda), kernel=(3, 3), pad=(1, 1), num_deformable_group=dg,
                                  no_bias=True)
    y.backward(_t(gout, cuda))
    ad, ao, _ = _dcn_ref(data, offset, None, gout.reshape(B, C * T, H * W), (3, 3), (1, 1), (1, 1), (1, 1), dg)
    ad.check(_np(x.grad).reshape(B, C, H, W), K_V1_DATA, "DCNv1 channels-last op data", old_tol=OLD_DCN_DATA)
    ao.check(_np(off.grad), K_V1_OFF, "DCNv1 channels-last op offset", old_tol=OLD_DCN_OFF)
