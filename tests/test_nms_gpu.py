"""GPU parity: batched NMS / nms_dense / bbox_vote through the C ABI vs the literal reference nms.c (its outputs on the
same seeded inputs, stored by tests/golden/make_golden.py) and its C restatement. Criterion: BIT-EXACT keep indices / rows."""
import os

import numpy as np
import pytest

from multipathnet_b200 import workloads as wl
from oracle import ref as O
from conftest import literal_golden, literal_nms_rows

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _expect_rows(key, sb, thr):
    rows = O.nms(sb, thr)
    assert np.array_equal(sb[rows], literal_nms_rows(key, sb, thr))
    return rows


@pytest.mark.parametrize("n", [1, 2, 31, 63, 64, 65, 127, 128, 129, 400, 1000, 2000, 5000])
def test_nms_distinct_scores_bit_exact(ctx, n):
    sb = wl.nms_sweep_boxes(n, 1, 1000 + n)[0]
    keep = ctx.nms(sb, 0.3)
    assert np.array_equal(keep, _expect_rows(f"gpu_distinct_{n}", sb, 0.3))


@pytest.mark.parametrize("seed", range(6))
def test_nms_tied_scores_follow_reference_permutation(ctx, seed):
    """ties: nms.c's selection order is an artefact of its pointer swaps; the exact-emulation kernel must match"""
    sb = wl.nms_sweep_boxes(300 + 97 * seed, 1, 2000 + seed, ties=True)[0]
    assert np.array_equal(ctx.nms(sb, 0.3), _expect_rows(f"gpu_ties_{seed}", sb, 0.3))


def test_nms_all_equal_scores_and_duplicates(ctx):
    sb = wl.nms_sweep_boxes(257, 1, 5)[0]
    sb[:, 4] = 0.5
    assert np.array_equal(ctx.nms(sb, 0.3), _expect_rows("gpu_all_equal", sb, 0.3))
    dup = np.repeat(wl.nms_sweep_boxes(40, 1, 6)[0], 3, axis=0)       # identical boxes AND scores
    assert np.array_equal(ctx.nms(dup, 0.3), _expect_rows("gpu_duplicates", dup, 0.3))


@pytest.mark.parametrize("thr", [0.0, 0.1, 0.3, 0.5, 0.7, 0.99, 1.0])
def test_nms_thresholds(ctx, thr):
    sb = wl.nms_sweep_boxes(700, 1, 31)[0]
    assert np.array_equal(ctx.nms(sb, thr), _expect_rows(f"gpu_thr_{thr}", sb, thr))


def test_nms_empty_and_degenerate_boxes(ctx):
    assert len(ctx.nms(np.zeros((0, 5), np.float32), 0.3)) == 0
    sb = wl.nms_sweep_boxes(200, 1, 8)[0]
    sb[::7, 2] = sb[::7, 0] - 5            # inverted boxes: w<=0 => overlap 0 (nms.c:40)
    sb[::11, :4] = 0
    assert np.array_equal(ctx.nms(sb, 0.3), _expect_rows("gpu_degenerate", sb, 0.3))


def test_nms_batched_ragged_segments(ctx):
    """one launch set for all classes of an image (Tester_FRCNN.lua:106-117), ragged + empty + tied segments"""
    sizes = [0, 1, 500, 64, 0, 1000, 333, 65]
    segs = []
    for i, n in enumerate(sizes):
        segs.append(wl.nms_sweep_boxes(max(n, 1), 1, 300 + i, ties=(i == 6))[0][:n])
    sb = np.concatenate(segs, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    keeps = ctx.nms_batched(sb, offs, 0.3)
    for i, (s, k) in enumerate(zip(segs, keeps)):
        assert np.array_equal(k, _expect_rows(f"gpu_ragged_{i}", s, 0.3))


def test_nms_80_classes_of_1000(ctx):
    """cfg 5 shape at N=1000: 80 classes in one call"""
    allsb = wl.nms_sweep_boxes(1000, 80, 5 + 1000)
    keeps = ctx.nms_batched(allsb.reshape(-1, 5), np.arange(81) * 1000, 0.3)
    for c in range(80):
        assert np.array_equal(keeps[c], O.nms(allsb[c], 0.3))


def test_nms_large_segment_20k(ctx):
    sb = wl.nms_sweep_boxes(20000, 1, 77)[0]
    assert np.array_equal(ctx.nms(sb, 0.3), O.nms(sb, 0.3))


def test_nms_idempotent_and_sorted(ctx):
    """size-independent properties: NMS(NMS(x)) == NMS(x) rows; kept scores descending for distinct scores"""
    sb = wl.nms_sweep_boxes(3000, 1, 99)[0]
    k1 = ctx.nms(sb, 0.3)
    kept = sb[k1]
    k2 = ctx.nms(kept, 0.3)
    assert np.array_equal(kept[k2], kept)
    assert np.all(np.diff(kept[:, 4]) < 0)


def test_nms_golden_fixtures(ctx):
    g = np.load(os.path.join(GOLD, "nms_golden.npz"))
    for key in [k[:-3] for k in g.files if k.endswith("_sb")]:
        sb, rows, thr = g[key + "_sb"], g[key + "_rows"], float(g[key + "_thr"])
        assert np.array_equal(sb[ctx.nms(sb, thr)], rows), key       # rows produced by the reference's own nms.c


def test_nms_dense(ctx):
    for n, seed in [(1, 0), (64, 1), (300, 2), (1500, 3)]:
        sb = wl.nms_sweep_boxes(n, 1, 400 + seed)[0]
        assert np.array_equal(ctx.nms_dense(sb, 0.3), O.nms_dense(sb, 0.3))
    assert len(ctx.nms_dense(np.zeros((0, 5), np.float32), 0.3)) == 0
    g = np.load(os.path.join(GOLD, "ops_golden.npz"))
    assert np.array_equal(ctx.nms_dense(g["dense_sb"], 0.3), g["dense_pick"])


def test_bbox_vote_bit_exact(ctx):
    sb = wl.nms_sweep_boxes(600, 1, 12)[0]
    rows = sb[ctx.nms(sb, 0.3)]
    got = ctx.bbox_vote(rows, sb, 0.5)
    assert np.array_equal(got, O.bbox_vote(rows, sb, 0.5))
    assert np.array_equal(rows, literal_nms_rows("gpu_vote", sb, 0.3))
    assert np.array_equal(got, literal_golden("gpu_vote_out"))


def test_nms_sweep_50k_single_class(ctx):
    """cfg 5 upper end: 50k boxes in one segment (mask 50k x 782 words = 312 MB)"""
    sb = wl.nms_sweep_boxes(50000, 1, 5 + 50000)[0]
    assert np.array_equal(ctx.nms(sb, 0.3), O.nms(sb, 0.3))


def test_nms_sweep_10k_x_80(ctx):
    allsb = wl.nms_sweep_boxes(10000, 80, 5 + 10000)
    keeps = ctx.nms_batched(allsb.reshape(-1, 5), np.arange(81) * 10000, 0.3)
    for c in (0, 17, 79):
        assert np.array_equal(keeps[c], O.nms(allsb[c], 0.3))


@pytest.mark.parametrize("n,seed", [(1025, 1), (1500, 2), (2048, 3), (3000, 4), (4096, 5), (4097, 6)])
def test_nms_medium_segments_with_ties(ctx, n, seed):
    """1024 < n <= 4096: warp-serial walk with the mask in L2 (2 removed-words per lane); 4097: chunked path"""
    sb = wl.nms_sweep_boxes(n, 1, 3000 + seed, ties=True)[0]
    assert np.array_equal(ctx.nms(sb, 0.3), _expect_rows(f"gpu_medium_ties_{n}", sb, 0.3))
    sb2 = wl.nms_sweep_boxes(n, 1, 3100 + seed)[0]
    assert np.array_equal(ctx.nms(sb2, 0.3), _expect_rows(f"gpu_medium_{n}", sb2, 0.3))


def test_nms_duplicate_rows_many_classes(ctx):
    """identical proposals (same pooled features => same score in EVERY class) are the common source of ties in the
    pipeline: 80 segments that all contain the same tied pairs"""
    base = wl.nms_sweep_boxes(600, 80, 4242)
    for c in range(80):
        base[c, 100:110] = base[c, 200:210]          # 10 exact duplicates (box and score)
        base[c, 300:305, 4] = base[c, 400:405, 4]    # 5 score ties with different boxes
    keeps = ctx.nms_batched(base.reshape(-1, 5), np.arange(81) * 600, 0.3)
    for c in range(0, 80, 7):
        assert np.array_equal(keeps[c], O.nms(base[c], 0.3))
