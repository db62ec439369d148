"""Pins the oracle against the REFERENCE'S OWN CODE: (a) golden vectors produced by running
operator_py/{bbox_transform,nms}.py and the compiled operator_py/cython/*.pyx
(tests/golden/make_golden.py, committed fixture), (b) random comparisons with the compiled Cython."""
import os
from types import SimpleNamespace

import numpy as np
import pytest

import oracle
from oracle import np_ops
from reference_replay import Reference, same

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_python_ops.npz"))


def test_bbox_overlaps_golden():
    assert np.array_equal(oracle.bbox_overlaps(G["overlaps_boxes"], G["overlaps_query"]), G["overlaps_out"])
    assert np.array_equal(oracle.bbox_selfoverlaps(G["overlaps_boxes"], G["overlaps_query"]), G["selfoverlaps_out"])


def test_greedy_nms_golden():
    assert np.array_equal(oracle.greedy_nms(G["nms_dets"], 0.5), G["greedy_keep_0.5"])
    # operator_py/nms.py `nms` keeps ovr <= thr; with distinct IoUs != thr it equals greedy_nms' set
    assert np.array_equal(np_ops.py_nms(G["nms_dets"], 0.5), G["py_nms_0.5"])
    assert np.array_equal(np_ops.set_nms(G["set_nms_dets"], 0.4), G["set_nms_0.4"])
    for lo, hi in ((0.3, 0.6), (0.5, 0.5)):
        got, want = np_ops.py_weighted_nms(G["nms_dets"], lo, hi), G[f"weighted_nms_{lo}_{hi}"]
        assert got.shape == want.shape and got.dtype == want.dtype and np.array_equal(got, want)


@pytest.mark.parametrize("method", [0, 1, 2])
def test_soft_nms_golden(method):
    bx, idx = oracle.soft_nms(G["nms_dets"], 0.5, 0.3, 0.05, method)
    assert np.array_equal(bx, G[f"soft_boxes_{method}"]) and np.array_equal(idx, G[f"soft_inds_{method}"])


def test_soft_nms_wrapper_defaults_golden():
    # cython_soft_nms_wrapper(thresh): Nt=thresh, sigma=0.5, score_thresh=0.001, linear (nms.py:5-16)
    bx, _ = oracle.soft_nms(G["nms_dets"], 0.5, 0.5, 0.001, 1)
    assert np.array_equal(bx, G["soft_wrapper_linear"])


def test_bbox_transform_golden():
    ex, gt, dl = G["xf_ex"], G["xf_gt"], G["xf_deltas"]
    assert np.array_equal(np_ops.nonlinear_transform(ex, gt), G["nonlinear_transform"])
    pred = np_ops.nonlinear_pred(ex.astype(np.float32), dl)
    assert np.array_equal(pred, G["nonlinear_pred"])
    assert np.array_equal(np_ops.iou_pred(ex.astype(np.float32), dl), G["iou_pred"])
    assert np.array_equal(np_ops.clip_boxes(pred, (400, 500)), G["clip_boxes"])
    assert np.array_equal(np_ops.flip_boxes(ex, 640), G["flip_boxes"])


def test_live_against_compiled_reference():
    """Random comparisons with the compiled Cython; where oracle/_ref is absent, against digests of what it returned
    (tests/reference_replay.py)."""
    mods = oracle.ref_cython()
    ref = Reference(None if mods is None else SimpleNamespace(
        bbox_overlaps_cython=mods["bbox"].bbox_overlaps_cython, greedy_nms=mods["cpu_nms"].greedy_nms,
        soft_nms=mods["cpu_nms"].soft_nms))
    rng = np.random.default_rng(0)
    for _ in range(10):
        b = rng.uniform(0, 500, (300, 4)).astype(np.float32)
        b[:, 2:] += b[:, :2]
        q = rng.uniform(0, 500, (37, 4)).astype(np.float32)
        q[:, 2:] += q[:, :2]
        assert same(ref.bbox_overlaps_cython(b, q), oracle.bbox_overlaps(b, q))
        d = np.concatenate([b, rng.uniform(0, 1, (300, 1)).astype(np.float32)], 1)
        assert same(ref.greedy_nms(d, np.float32(0.5)), oracle.greedy_nms(d, 0.5))
        for m in (0, 1, 2):
            r1 = oracle.soft_nms(d, 0.5, 0.3, 0.001, m)
            r2 = ref.soft_nms(d, np.float32(0.5), np.float32(0.3), np.float32(0.001), np.uint8(m))
            assert same(r2[0], r1[0]) and same(r2[1], r1[1])


def test_box_voting_matches_reference():
    for meth, beta in (("ID", 1.0), ("AVG", 1.0), ("IOU_AVG", 1.0), ("GENERALIZED_AVG", 2.0), ("QUASI_SUM", 0.5),
                       ("TEMP_AVG", 0.7)):
        got = np_ops.box_voting(G["vote_top"], G["nms_dets"], 0.5, meth, beta)
        assert got.dtype == G[f"vote_{meth}"].dtype and np.array_equal(got, G[f"vote_{meth}"]), meth
