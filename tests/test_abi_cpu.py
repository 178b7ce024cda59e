"""CPU suite, part 2: the C-ABI library loads and exports exactly what include/mpn_abi.h declares
(no compute without a GPU), and the host-side logic (specs, workloads, ImageDetect geometry)."""
import ctypes
import os
import re

import numpy as np
import pytest

import multipathnet_b200 as mpn
from multipathnet_b200 import _lib, models, workloads as wl
from multipathnet_b200.image_detect import ImageDetect, _image_scale
from multipathnet_b200.modules import ImageTransformer
from conftest import literal_golden, literal_nms_rows, rel_err


def _header_functions():
    src = open(_lib.HEADER_PATH).read()
    body = src[src.index("MPN_CDEF_BEGIN"):src.index("MPN_CDEF_END")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return sorted(set(re.findall(r"\b(mpn_[a-z0-9_]+)\s*\(", body)))


def test_library_exports_every_declared_symbol():
    lib = mpn.load_library()
    declared = _header_functions()
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in mpn_abi.h but not exported"
    assert sorted(_lib.SIGNATURES) == declared, "ctypes signature table out of sync with the header"
    assert b"sm_100a" in lib.mpn_version()


def test_no_gpu_means_loud_failure_not_fallback():
    """without a CUDA device context creation must fail with a message (never a CPU fallback)"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(mpn.MpnError):
        mpn.Context(0)
    with pytest.raises(mpn.MpnError):
        mpn.Context(0, own_stream=True)                       # mpn_ctx_create_stream: the same loud failure
    with pytest.raises(mpn.MpnError):
        mpn.ModelReplicas(0, models.vgg16_fast_rcnn(21, seed=1, width_div=16, fc_dim=64), 2)
    lib = mpn.load_library()
    assert lib.mpn_ctx_stream(None) is None and lib.mpn_ctx_wait_ctx(None, None) < 0
    assert len(lib.mpn_last_error(None)) > 0
    # NULL-handle calls are rejected, not crashes
    assert lib.mpn_ctx_synchronize(None) < 0
    assert lib.mpn_ctx_launch_count(None) == -1
    lib.mpn_ctx_destroy(None); lib.mpn_model_destroy(None)


def test_struct_layout_matches_header():
    assert ctypes.sizeof(_lib.CLayer) == 14 * 4
    assert ctypes.sizeof(_lib.CHead) == 5 * 4
    assert ctypes.sizeof(_lib.CTower) == 4 * (2 + 3 + 3 + 6)
    assert ctypes.sizeof(_lib.CImageTransform) == 4 * (3 + 1 + 3 + 3 + 1)


def test_vgg16_flops_match_survey():
    s = models.vgg16_fast_rcnn(21, seed=None)
    assert abs(models.trunk_flops(s, 600, 800) / 1e9 - 294.0) < 0.1          # SURVEY 8a5
    assert abs(models.head_flops_per_roi(s) / 1e6 - 239.9) < 0.1             # SURVEY 8a12
    s81 = models.vgg16_fast_rcnn(81, seed=None, fc_dim=4096)
    assert abs(models.head_flops_per_roi(s81) / 1e6 - 242.4) < 0.1
    assert s.taps == {"conv3": 9, "conv4": 13, "conv5": 17}


def test_multipathnet_spec_structure():
    s = models.vgg16_multipathnet(81, seed=None)                              # structure only: no 2.4 GB of random weights
    assert [t.region for t in s.towers] == [0, 1, 2, 3, 1]                   # multipathnet.lua:73-113
    assert [len(t.levels) for t in s.towers] == [3, 2, 2, 1, 3]
    assert s.cls_heads[0].col_len == 4 * 4096 and s.bbox_head.col_begin == 4 * 4096
    assert abs(models.head_flops_per_roi(s) / 1e9 - 1.458) < 0.01            # SURVEY 8a12


def test_resnet50_flops_match_survey():
    s = models.resnet50_fast_rcnn(81, seed=None, integral_k=6)
    assert abs(models.trunk_flops(s, 800, 1000) / 1e9 - 104.9) < 1.5          # SURVEY 8a7
    assert abs(models.head_flops_per_roi(s) / 1e9 - 1.62) < 0.02


def test_workloads_are_seeded_and_valid():
    b1, b2 = wl.random_boxes(100, 600, 800, 2), wl.random_boxes(100, 600, 800, 2)
    assert np.array_equal(b1, b2)
    assert np.all(b1[:, 0] >= 1) and np.all(b1[:, 2] <= 800) and np.all(b1[:, 3] <= 600) and np.all(b1[:, 2] > b1[:, 0])
    sm = wl.sharpmask_boxes(500, 600, 800, 3)
    assert np.all(sm[:, 2] > sm[:, 0]) and np.all(sm[:, 3] > sm[:, 1]) and sm.min() >= 1
    sb = wl.nms_sweep_boxes(64, 3, 5)
    assert sb.shape == (3, 64, 5) and len(np.unique(sb[0, :, 4])) == 64
    assert len(np.unique(wl.nms_sweep_boxes(64, 1, 5, ties=True)[0, :, 4])) < 64


def test_transformers():
    im = wl.raw_image(4, 5, 0)
    r = ImageTransformer("ross").forward(im)
    np.testing.assert_allclose(r[0], im[2] * 255 - 102.9801, rtol=1e-6)      # BGR swap, x255, -mean
    i = ImageTransformer("imagenet").forward(im)
    np.testing.assert_allclose(i[1], (im[1] - 0.45624044862054) / 0.22446679341259, rtol=1e-5)


class _FakeModel:
    C = 21
    def detect(self, img, boxes, im_scale, rec):
        self.args = (None if img is None else img.shape, boxes.shape, im_scale, rec)
        return np.zeros((len(boxes), 21), np.float32), np.zeros((len(boxes), 84), np.float32)


def test_image_detect_scaling_rules():
    """ImageDetect.lua:31-41: im_scale = scale/min side, capped so round(im_scale*max side) <= max_size"""
    d = ImageDetect(_FakeModel(), ImageTransformer("ross"), [600], 1000)
    img, s = d.getImages(wl.raw_image(300, 400, 1))
    assert s == 2.0 and img.shape == (3, 600, 800)
    img, s = d.getImages(wl.raw_image(300, 900, 1))
    assert abs(s - 1000 / 900) < 1e-9 and img.shape[2] == 1000
    img, s = d.getImages(wl.raw_image(600, 800, 1))
    assert s == 1.0 and img.shape == (3, 600, 800)
    d.detect(wl.raw_image(600, 800, 1), wl.random_boxes(5, 600, 800, 1))
    assert d.model.args == ((3, 600, 800), (5, 4), 1.0, True)
    with pytest.raises(ValueError):
        ImageDetect(None, ImageTransformer())
    with pytest.raises(ValueError):
        ImageDetect(_FakeModel(), ImageTransformer(), [480, 600])


def test_image_scale_identity_and_constant():
    im = wl.raw_image(7, 9, 3)
    assert np.array_equal(_image_scale(im, 7, 9), im)
    c = np.full((3, 5, 5), 2.5, np.float32)
    assert np.allclose(_image_scale(c, 11, 13), 2.5) and np.allclose(_image_scale(c, 2, 3), 2.5)


def test_cfg1_alexnet_cpu_plumbing(oracle_built):
    """BASELINE configs[0]: AlexNet (CaffeNet) Fast R-CNN, one synthetic 224px image, 64 random boxes, CPU nn path —
    the whole detect + testOne pipeline through the oracle, no GPU (SURVEY 8d cfg 1)."""
    from oracle import graphs as G
    O = oracle_built
    spec = models.alexnet_fast_rcnn(21, seed=1)
    img = wl.transform(wl.raw_image(224, 224, 1), spec.transformer)
    boxes = wl.random_boxes(64, 224, 224, 1, wmax=64, hmax=64)
    scores, bboxes, keeps = G.test_one(spec, img, boxes, 1.0, 224, 224)
    assert scores.shape == (64, 21) and bboxes.shape == (64, 84) and len(keeps) == 20
    np.testing.assert_allclose(scores.sum(1), 1.0, atol=1e-5)
    assert bboxes.min() >= 1 and bboxes[:, 0::2].max() <= 224
    ts = G.trunk_forward(spec, img)
    assert tuple(ts[9].shape) == (1, 256, 13, 13)                 # conv5 of CaffeNet at 224 px
    stored = literal_golden("cfg1_sb")                            # this forward's rows as the golden run computed them
    for j, k in enumerate(keeps, start=1):                        # keep lists = the literal nms.c on the same rows
        sb = np.concatenate([bboxes[:, 4 * j:4 * j + 4], scores[:, j:j + 1]], 1).astype(np.float32)
        assert rel_err(sb[:, :4], stored[j - 1, :, :4]) < 1e-5 and rel_err(sb[:, 4], stored[j - 1, :, 4]) < 1e-4
        assert np.array_equal(k, O.nms(sb, 0.3))
        assert np.array_equal(stored[j - 1][O.nms(stored[j - 1], 0.3)], literal_nms_rows(f"cfg1_class{j}", stored[j - 1], 0.3))
    # the B200 path refuses this configuration loudly (grouped conv + LRN are CPU-plumbing only)
    with pytest.raises(mpn.MpnError):
        mpn.Model.build_desc(spec)


def test_model_desc_builds_without_gpu():
    d, keep = mpn.Model.build_desc(models.vgg16_fast_rcnn(21, width_div=4, fc_dim=256))
    assert d.n_trunk_layers == 17 and d.n_towers == 1 and d.num_classes == 21 and d.bbox_head.cout == 84
    d, keep = mpn.Model.build_desc(models.vgg16_multipathnet(81, width_div=4, fc_dim=256))
    assert d.n_towers == 5 and d.n_tower_layers == 20 and d.towers[4].region == 1 and d.towers[4].n_levels == 3


def _segwalk(lib, sk, unit, units, tiles, S):
    buf = (ctypes.c_int32 * (3 * 4096))()
    n = ctypes.c_int32(0)
    assert lib.mpn_debug_segwalk(int(sk), unit, units, tiles, S, buf, 4096, ctypes.byref(n)) == 0
    return [(buf[3 * i], buf[3 * i + 1], buf[3 * i + 2]) for i in range(n.value)]


@pytest.mark.parametrize("tiles,S,units", [(22, 24, 74), (44, 24, 74), (125, 12, 74), (250, 6, 74), (66, 24, 74), (13, 24, 74),
                                           (74, 9, 74), (75, 9, 74), (3, 100, 74), (500, 3, 148), (7, 5, 2), (148, 6, 148)])
def test_streamk_partition_is_exact_and_deadlock_free(tiles, S, units):
    """The stream-K work walk of the tcgen05 kernels (host view of the same struct the kernels run, no GPU):
    every (tile, step) is owned by exactly one piece; a unit visits at most one continuation piece (a tile begun by the
    previous unit: it only WRITES a partial, first, never waits), then at most one head piece (the tile's finisher, which
    waits only for continuation pieces = first pieces of later units), then whole tiles; the finisher's tile is completed
    by the immediately following units. (The planner only picks stream-K with >= 4 steps per unit, and the launcher
    refuses less: with fewer steps than units some ranges would be empty and a finisher would wait for nobody.)"""
    assert tiles * S >= 4 * units
    lib = mpn.load_library()
    owner = {}
    first_piece = {}
    for u in range(units):
        pieces = _segwalk(lib, 1, u, units, tiles, S)
        kinds = []
        for (t, s0, s1) in pieces:
            assert 0 <= t < tiles and 0 <= s0 < s1 <= S
            for st in range(s0, s1):
                assert (t, st) not in owner, "step covered twice"
                owner[(t, st)] = u
            kinds.append("writer" if s0 > 0 else ("finisher" if s1 < S else "full"))
        # order: [writer] [finisher] full*
        stripped = kinds[:]
        if stripped and stripped[0] == "writer":
            stripped.pop(0)
        if stripped and stripped[0] == "finisher":
            stripped.pop(0)
        assert all(k == "full" for k in stripped), kinds
        first_piece[u] = pieces[0] if pieces else None
    assert len(owner) == tiles * S, "steps missing"
    # every finisher's tile is completed by the FIRST pieces of the following units (what the kernel waits for)
    for u in range(units):
        for (t, s0, s1) in _segwalk(lib, 1, u, units, tiles, S):
            if s0 == 0 and s1 < S:
                nxt, v = s1, u + 1
                while nxt < S:
                    assert v < units and first_piece[v] is not None
                    tt, a, b = first_piece[v]
                    assert (tt, a) == (t, nxt), "continuation is not the next unit's first piece"
                    nxt, v = b, v + 1
    # plain schedule: whole tiles round-robin
    seen = sorted(p for u in range(units) for p in _segwalk(lib, 0, u, units, tiles, S))
    assert seen == [(t, 0, S) for t in range(tiles)]


def test_committed_bench_line_follows_the_contract():
    """The last committed bench line (profiles/) carries every key of the bench.py contract, with sane values."""
    import glob
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = sorted(glob.glob(os.path.join(root, "profiles", "r01*_bench_n1.json")))
    assert files, "no committed bench line"
    d = json.loads(open(files[-1]).read().strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert k in d, k
    assert d["metric"] == "proposals/sec" and d["unit"] == "proposals/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"] and d["warmup"] >= 3
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"]))
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and {"achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.0 < r["frac"] < 1.0
    assert d["gpu_launches"] > 0 and d["value"] > 1e5
    if "cpu_baseline" in d:
        assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("port", "reference")


def _plan(lib, N, Cin, H, W, Cout, k=3, s=1, p=1, per_roi=0, sm=148):
    out = (ctypes.c_int32 * 8)()
    assert lib.mpn_debug_plan(N, Cin, H, W, Cout, k, s, p, per_roi, sm, out) == 0
    return dict(zip(("mode", "cg", "bn", "splitk", "streamk", "tn", "th", "tw"), out))


def test_planner_choices_for_the_default_workload():
    """Host view of conv_tc_plan (no GPU) on a 148-SM device: the configurations the measured launch lists show
    (profiles/r01h_launches.csv) — a regression guard for the cost model."""
    lib = mpn.load_library()
    want = {  # layer: (args, mode, cg, bn, splitk, streamk)
        "conv1_2": ((1, 64, 600, 800, 64), 1, 2, 64, 1, 0), "conv2_1": ((1, 64, 300, 400, 128), 1, 2, 128, 1, 0),
        "conv2_2": ((1, 128, 300, 400, 128), 1, 2, 128, 1, 0), "conv3_1": ((1, 128, 150, 200, 256), 1, 2, 256, 1, 0),
        "conv3_2": ((1, 256, 150, 200, 256), 1, 2, 128, 1, 1), "conv4_1": ((1, 256, 75, 100, 512), 1, 2, 256, 1, 0),
        "conv4_2": ((1, 512, 75, 100, 512), 1, 2, 256, 1, 0), "conv5_1": ((1, 512, 38, 50, 512), 1, 2, 128, 1, 1),
    }
    for name, (args, mode, cg, bn, sk, stk) in want.items():
        pl = _plan(lib, *args)
        assert (pl["mode"], pl["cg"], pl["bn"], pl["splitk"], pl["streamk"]) == (mode, cg, bn, sk, stk), (name, pl)
        assert (pl["tn"], pl["th"], pl["tw"]) == (1, 16, 8)
    heads = {"fc6": ((1000, 25088, 1, 1, 4096), 240, 1), "fc7": ((1000, 4096, 1, 1, 4096), 240, 1),
             "cls": ((1000, 4096, 1, 1, 21), 64, 8), "bbox": ((1000, 4096, 1, 1, 84), 128, 8)}
    for name, (args, bn, sk) in heads.items():
        pl = _plan(lib, *args, k=1, s=1, p=0, per_roi=1)
        assert (pl["mode"], pl["cg"], pl["bn"], pl["splitk"], pl["streamk"], pl["tw"]) == (0, 2, bn, sk, 0, 128), (name, pl)


@pytest.mark.parametrize("Cout,K", [(21, 4096), (84, 4096), (128, 1024), (160, 2048), (512, 2048), (4096, 25088), (4096, 4096)])
def test_planner_keeps_per_roi_rounding_independent_of_row_count(Cout, K):
    """Per-ROI layers: whatever the number of rows, the accumulator grouping (a function of the N tile class) and the
    split-K count are the same, and stream-K is never used — the preconditions of bit-exact chunk invariance."""
    lib = mpn.load_library()
    acc = lambda bn: 1 if bn > 128 else (2 if bn == 128 else 3)
    seen = set()
    for rows in (1, 7, 100, 128, 129, 300, 1000, 2000, 5000, 40000):
        pl = _plan(lib, rows, K, 1, 1, Cout, k=1, s=1, p=0, per_roi=1)
        assert pl["streamk"] == 0
        seen.add((acc(pl["bn"]), pl["splitk"]))
    assert len(seen) == 1, seen


def test_planner_r3_minpix_knob_moves_only_small_maps(monkeypatch):
    """MPN_TC_R3_MINPIX (experiment knob for the 38 x 50 conv5 maps, profiles/r01h_layer_efficiency.md): unset it changes
    nothing; set to 2000 pixels only conv5 leaves the 3x3 A-reuse kernel."""
    lib = mpn.load_library()
    conv5, conv4 = (1, 512, 38, 50, 512), (1, 512, 75, 100, 512)
    monkeypatch.delenv("MPN_TC_R3_MINPIX", raising=False)
    base5, base4 = _plan(lib, *conv5), _plan(lib, *conv4)
    assert base5["mode"] == 1 and base4["mode"] == 1
    monkeypatch.setenv("MPN_TC_R3_MINPIX", "2000")
    k5, k4 = _plan(lib, *conv5), _plan(lib, *conv4)
    assert k5["mode"] == 0 and k5["streamk"] == 0 and k4 == base4
    monkeypatch.setenv("MPN_TC_R3_MINPIX", "0")
    assert _plan(lib, *conv5) == base5
