"""CPU suite, part 1: pin the oracle against everything the reference's own tests hold for this
path (SURVEY 8c) and against what the literal nms.c returned on the same inputs (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

from multipathnet_b200 import workloads as wl
from conftest import literal_golden, literal_nms_rows

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_iou_known_answer(oracle_built):
    """reference test.lua:40-52 (utiltest.boxoverlap): 5 boxes vs {50,50,150,150} -> {1/7,1/3,1/3,1,1/7} within 5e-3"""
    O = oracle_built
    a = np.array([[0, 0, 100, 100], [0, 50, 100, 150], [50, 0, 150, 100], [50, 50, 150, 150], [100, 100, 200, 200]], np.float32)
    b = np.array([50, 50, 150, 150], np.float32)
    gt = np.array([1 / 7, 1 / 3, 1 / 3, 1, 1 / 7], np.float32)
    mine = np.array([O.overlap(x, b) for x in a], np.float32)
    assert np.max(mine - gt) < 5e-3
    lit = literal_golden("boxoverlap")               # the literal nms.c:boxoverlap
    assert np.array_equal(mine, lit)                  # bit-exact vs the reference's own code


def test_bbox_parametrization_roundtrip(oracle_built):
    """reference test.lua:17-38: convertTo o convertFrom round trip < 1e-8 in fp64"""
    O = oracle_built
    rng = np.random.default_rng(0)
    for _ in range(50):
        A, B = rng.random(2) * 100, rng.random(2) * 100
        bbox = np.array([A[0], A[1], A[0] + rng.integers(1, 41), A[1] + rng.integers(1, 41)])
        tbox = np.array([B[0], B[1], B[0] + rng.integers(1, 41), B[1] + rng.integers(1, 41)])
        y = O.convert_to_f64(bbox, tbox)
        back = O.convert_from_f64(bbox, y)
        assert np.max(np.abs(back - tbox)) < 1e-8


def test_convert_from_fp32_matches_fp64(oracle_built):
    O = oracle_built
    rng = np.random.default_rng(1)
    boxes = wl.random_boxes(64, 600, 800, 1)
    d = (rng.standard_normal((64, 8)) * 0.2).astype(np.float32)
    out = O.convert_from(d, boxes)
    for i in range(64):
        for c in range(2):
            ref = O.convert_from_f64(boxes[i].astype(np.float64), d[i, 4 * c:4 * c + 4].astype(np.float64))
            assert np.max(np.abs(out[i, 4 * c:4 * c + 4] - ref)) < 1e-3


@pytest.mark.parametrize("n,seed", [(1, 0), (2, 1), (17, 2), (64, 3), (65, 4), (400, 5), (1000, 6), (2000, 7)])
def test_nms_restatement_equals_literal_reference(oracle_built, n, seed):
    """orc_nms (index-returning restatement of nms.c:59-108) must reproduce the literal nms.c row for row"""
    O = oracle_built
    sb = wl.nms_sweep_boxes(n, 1, 100 + seed)[0]
    rows = literal_nms_rows(f"cpu_distinct_{n}", sb, 0.3)
    keep = O.nms(sb, 0.3)
    assert np.array_equal(sb[keep], rows)
    # distinct scores => the reference keeps rows in descending-score order (SURVEY A.3)
    assert np.all(np.diff(sb[keep, 4]) < 0)


@pytest.mark.parametrize("seed", range(8))
def test_nms_restatement_ties(oracle_built, seed):
    """tied scores: nms.c's order is an artefact of its swap permutation; the restatement must follow it"""
    O = oracle_built
    sb = wl.nms_sweep_boxes(300, 1, 200 + seed, ties=True)[0]
    assert np.array_equal(sb[O.nms(sb, 0.3)], literal_nms_rows(f"cpu_ties_{seed}", sb, 0.3))


def test_nms_thresholds_and_empty(oracle_built):
    O = oracle_built
    assert len(O.nms(np.zeros((0, 5), np.float32), 0.3)) == 0
    sb = wl.nms_sweep_boxes(200, 1, 9)[0]
    for thr in (0.0, 0.3, 0.5, 0.99, 1.0):
        assert np.array_equal(sb[O.nms(sb, thr)], literal_nms_rows(f"cpu_thr_{thr}", sb, thr))


def test_bbox_vote_restatement_equals_literal(oracle_built):
    O = oracle_built
    sb = wl.nms_sweep_boxes(300, 1, 11)[0]
    rows = literal_nms_rows("cpu_vote", sb, 0.3)
    assert np.array_equal(O.bbox_vote(rows, sb, 0.5), literal_golden("cpu_vote_out"))


def test_foveal_regions(oracle_built):
    """Foveal.lua:36-39: regions x1, x1.5, x2, x4 about the box centre; ContextRegion(s) is the same map in fp32"""
    O = oracle_built
    rois = np.concatenate([np.ones((32, 1), np.float32), wl.random_boxes(32, 600, 800, 3)], 1)
    f = O.foveal(rois).reshape(32, 4, 5)
    assert np.array_equal(f[:, 0], rois)
    for k, s in ((1, 1.5), (2, 2.0), (3, 4.0)):
        w, h = rois[:, 3] - rois[:, 1], rois[:, 4] - rois[:, 2]
        np.testing.assert_allclose(f[:, k, 3] - f[:, k, 1], s * w, rtol=1e-5)
        np.testing.assert_allclose(f[:, k, 4] - f[:, k, 2], s * h, rtol=1e-5)
        np.testing.assert_allclose((f[:, k, 1] + f[:, k, 3]) / 2, (rois[:, 1] + rois[:, 3]) / 2, rtol=1e-5)
        np.testing.assert_allclose(O.context_region(rois, s), f[:, k], rtol=1e-5, atol=1e-3)


def test_roi_pool_chunk_invariance_and_shapes(oracle_built):
    """reference modules/test.lua:60-83: ROIPooling(7,7,1/16) on randn(1,512,38,50) with 40 rois randn*50
    (often negative / inverted => clipped and empty bins): chunked (25) == unchunked exactly"""
    O = oracle_built
    rng = np.random.default_rng(7)
    fm = rng.standard_normal((1, 64, 38, 50)).astype(np.float32)
    rois = (rng.standard_normal((40, 5)) * 50).astype(np.float32)
    rois[:, 0] = 1
    for variant in (1, 2):
        full = O.roi_pool(fm, rois, 7, 7, 1 / 16, variant)
        parts = np.concatenate([O.roi_pool(fm, rois[:25], 7, 7, 1 / 16, variant), O.roi_pool(fm, rois[25:], 7, 7, 1 / 16, variant)])
        assert np.array_equal(full, parts)
        assert full.shape == (40, 64, 7, 7)


def test_roi_pool_semantics(oracle_built):
    """hand-checkable case: 8x8 map with value = h*8+w, ROI covering cells [0..7]^2 at scale 1 (v1)"""
    O = oracle_built
    fm = np.arange(64, dtype=np.float32).reshape(1, 1, 8, 8)
    roi = np.array([[1, 1, 1, 8, 8]], np.float32)       # 1-based px -> cells 0..7 inclusive (v1)
    out, am = O.roi_pool(fm, roi, 2, 2, 1.0, 1, with_argmax=True)
    assert out.reshape(-1).tolist() == [27, 31, 59, 63]
    assert am.reshape(-1).tolist() == [27, 31, 59, 63]
    out2 = O.roi_pool(fm, roi, 2, 2, 1.0, 2)             # v2: end exclusive -> cells 0..6
    assert out2.reshape(-1).tolist() == [27, 30, 51, 54]
    # fully outside the map => all bins empty => zeros, argmax -1
    out3, am3 = O.roi_pool(fm, np.array([[1, 100, 100, 120, 120]], np.float32), 2, 2, 1.0, 2, with_argmax=True)
    assert np.all(out3 == 0) and np.all(am3 == -1)


def test_maxpool_ceil_mode_sizes(oracle_built):
    """SURVEY 8a5: ceil-mode 2x2 pools take 600x800 to 38x50 at conv5 (modules/test.lua:62 uses 38x50)"""
    O = oracle_built
    h, w = 600, 800
    for _ in range(4):
        h, w = O.pool_out(h, 2, 2, 0, 1), O.pool_out(w, 2, 2, 0, 1)
    assert (h, w) == (38, 50)


def test_golden_vectors(oracle_built):
    """committed fixtures (tests/golden/make_golden.py): literal-nms.c outputs + oracle outputs on seeded inputs"""
    O = oracle_built
    g = np.load(os.path.join(GOLD, "nms_golden.npz"))
    for key in [k[:-3] for k in g.files if k.endswith("_sb")]:
        sb, rows, thr = g[key + "_sb"], g[key + "_rows"], float(g[key + "_thr"])
        assert np.array_equal(sb[O.nms(sb, thr)], rows), key
    g = np.load(os.path.join(GOLD, "ops_golden.npz"))
    assert np.array_equal(O.foveal(g["rois"]), g["foveal"])
    assert np.array_equal(O.roi_pool(g["fmap"], g["rois_neg"], 7, 7, 1 / 16, 2), g["roi_v2"])
    assert np.array_equal(O.roi_pool(g["fmap"], g["rois_neg"], 7, 7, 1 / 16, 1), g["roi_v1"])
    np.testing.assert_allclose(O.convert_from(g["deltas"], g["boxes"]), g["decoded"], rtol=1e-6, atol=1e-4)
    assert np.array_equal(O.nms_dense(g["dense_sb"], 0.3), g["dense_pick"])
