"""Generates the fixtures under tests/golden/. Needs a checkout of the original facebookresearch/multipathnet
(oracle/Makefile builds its literal nms.c from there): `REF=<checkout> python tests/golden/make_golden.py`.
The NMS goldens are outputs of the REFERENCE's own nms.c; the others are outputs of the C restatement (parity
unpinned, see DESIGN.md), committed so that any later change to the oracle is caught."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "tests"))
from oracle import graphs as G, ref as O  # noqa: E402
from multipathnet_b200 import models, workloads as wl  # noqa: E402
from test_lua_shim_cpu import _methods, _strip_lua  # noqa: E402

REF = os.environ.get("REF")
if not REF or not os.path.exists(os.path.join(REF, "nms.c")):
    sys.exit("set REF to a checkout of facebookresearch/multipathnet")
O.build()
here = os.path.dirname(os.path.abspath(__file__))
d = {}
cases = [("n1", 1, 0.3, False), ("n64", 64, 0.3, False), ("n65", 65, 0.3, False), ("n300", 300, 0.3, False),
         ("n1000", 1000, 0.3, False), ("n1000_t5", 1000, 0.5, False), ("ties200", 200, 0.3, True), ("ties777", 777, 0.3, True)]
for i, (name, n, thr, ties) in enumerate(cases):
    sb = wl.nms_sweep_boxes(n, 1, 500 + i, ties=ties)[0]
    d[name + "_sb"] = sb
    d[name + "_rows"] = O.ref_nms_rows(sb, thr)          # literal reference nms.c
    d[name + "_thr"] = np.float32(thr)
np.savez_compressed(os.path.join(here, "nms_golden.npz"), **d)

rng = np.random.default_rng(42)
rois = np.concatenate([np.ones((48, 1), np.float32), wl.random_boxes(48, 600, 800, 42)], 1)
fmap = rng.standard_normal((1, 16, 38, 50)).astype(np.float32)
rois_neg = (rng.standard_normal((40, 5)) * 50).astype(np.float32)
rois_neg[:, 0] = 1
deltas = (rng.standard_normal((48, 12)) * 0.3).astype(np.float32)
boxes = rois[:, 1:].copy()
dense_sb = wl.nms_sweep_boxes(300, 1, 77)[0]
np.savez_compressed(os.path.join(here, "ops_golden.npz"), rois=rois, foveal=O.foveal(rois), fmap=fmap, rois_neg=rois_neg,
                    roi_v2=O.roi_pool(fmap, rois_neg, 7, 7, 1 / 16, 2), roi_v1=O.roi_pool(fmap, rois_neg, 7, 7, 1 / 16, 1),
                    deltas=deltas, boxes=boxes, decoded=O.convert_from(deltas, boxes), dense_sb=dense_sb,
                    dense_pick=O.nms_dense(dense_sb, 0.3))

# getImages (SURVEY 8f-1): raw image -> transformer -> image.scale, outputs of the two-pass C restatement (parity unpinned)
g = {}
for name, (H0, W0, scale, max_size, kind) in {"grow": (20, 30, 33, 1000, "ross"), "shrink": (40, 56, 17, 1000, "imagenet"),
                                               "capped": (16, 60, 32, 90, "ross"), "same": (24, 32, 24, 1000, "imagenet")}.items():
    im = wl.raw_image(H0, W0, 900 + H0)
    out, s = O.get_images(im, kind, scale, max_size)
    g[name + "_im"], g[name + "_out"], g[name + "_cfg"] = im, out, np.array([scale, max_size, s, kind == "imagenet"], np.float64)
np.savez_compressed(os.path.join(here, "getimages_golden.npz"), **g)

# the literal nms.c on the seeded inputs of the tests that compare with it (conftest.literal_nms_rows): the indices of the
# kept rows and a fingerprint of the input (the inputs themselves are rebuilt by the tests from their seeds)
lit = {}


def literal(key, sb, thr):
    sb = np.ascontiguousarray(sb, np.float32).reshape(-1, 5)
    rows = O.ref_nms_rows(sb, thr)
    first = {}
    for i in range(sb.shape[0] - 1, -1, -1):
        first[sb[i].tobytes()] = i
    lit[key + "_keep"] = np.array([first[r.tobytes()] for r in rows], np.int32)
    lit[key + "_sha1"] = np.array(hashlib.sha1(sb.tobytes()).hexdigest())
    lit[key + "_thr"] = np.float32(thr)
    return rows


# tests/test_oracle_cpu.py
a = np.array([[0, 0, 100, 100], [0, 50, 100, 150], [50, 0, 150, 100], [50, 50, 150, 150], [100, 100, 200, 200]], np.float32)
lit["boxoverlap"] = O.ref_boxoverlap(a, np.array([50, 50, 150, 150], np.float32))
for n, seed in [(1, 0), (2, 1), (17, 2), (64, 3), (65, 4), (400, 5), (1000, 6), (2000, 7)]:
    literal(f"cpu_distinct_{n}", wl.nms_sweep_boxes(n, 1, 100 + seed)[0], 0.3)
for seed in range(8):
    literal(f"cpu_ties_{seed}", wl.nms_sweep_boxes(300, 1, 200 + seed, ties=True)[0], 0.3)
for thr in (0.0, 0.3, 0.5, 0.99, 1.0):
    literal(f"cpu_thr_{thr}", wl.nms_sweep_boxes(200, 1, 9)[0], thr)
sb = wl.nms_sweep_boxes(300, 1, 11)[0]
lit["cpu_vote_out"] = O.ref_bbox_vote(literal("cpu_vote", sb, 0.3), sb, 0.5)
# tests/test_abi_cpu.py::test_cfg1_alexnet_cpu_plumbing: the per-class rows of the CPU forward (torch-CPU sums are not
# bit-reproducible across hosts, so the rows are stored and the test compares its own within a tolerance)
spec = models.alexnet_fast_rcnn(21, seed=1)
scores, bboxes, _ = G.test_one(spec, wl.transform(wl.raw_image(224, 224, 1), spec.transformer),
                               wl.random_boxes(64, 224, 224, 1, wmax=64, hmax=64), 1.0, 224, 224)
lit["cfg1_sb"] = np.stack([np.concatenate([bboxes[:, 4 * j:4 * j + 4], scores[:, j:j + 1]], 1) for j in range(1, 21)]).astype(np.float32)
for j in range(1, 21):
    literal(f"cfg1_class{j}", lit["cfg1_sb"][j - 1], 0.3)
# tests/test_nms_gpu.py
for n in [1, 2, 31, 63, 64, 65, 127, 128, 129, 400, 1000, 2000, 5000]:
    literal(f"gpu_distinct_{n}", wl.nms_sweep_boxes(n, 1, 1000 + n)[0], 0.3)
for seed in range(6):
    literal(f"gpu_ties_{seed}", wl.nms_sweep_boxes(300 + 97 * seed, 1, 2000 + seed, ties=True)[0], 0.3)
sb = wl.nms_sweep_boxes(257, 1, 5)[0]
sb[:, 4] = 0.5
literal("gpu_all_equal", sb, 0.3)
literal("gpu_duplicates", np.repeat(wl.nms_sweep_boxes(40, 1, 6)[0], 3, axis=0), 0.3)
for thr in [0.0, 0.1, 0.3, 0.5, 0.7, 0.99, 1.0]:
    literal(f"gpu_thr_{thr}", wl.nms_sweep_boxes(700, 1, 31)[0], thr)
sb = wl.nms_sweep_boxes(200, 1, 8)[0]
sb[::7, 2] = sb[::7, 0] - 5
sb[::11, :4] = 0
literal("gpu_degenerate", sb, 0.3)
for i, n in enumerate([0, 1, 500, 64, 0, 1000, 333, 65]):
    literal(f"gpu_ragged_{i}", wl.nms_sweep_boxes(max(n, 1), 1, 300 + i, ties=(i == 6))[0][:n], 0.3)
sb = wl.nms_sweep_boxes(600, 1, 12)[0]
lit["gpu_vote_out"] = O.ref_bbox_vote(literal("gpu_vote", sb, 0.3), sb, 0.5)
for n, seed in [(1025, 1), (1500, 2), (2048, 3), (3000, 4), (4096, 5), (4097, 6)]:
    literal(f"gpu_medium_ties_{n}", wl.nms_sweep_boxes(n, 1, 3000 + seed, ties=True)[0], 0.3)
    literal(f"gpu_medium_{n}", wl.nms_sweep_boxes(n, 1, 3100 + seed)[0], 0.3)
np.savez_compressed(os.path.join(here, "nms_literal_golden.npz"), **lit)

# the method table of the reference's fbcoco.ImageDetect (ImageDetect.lua), for tests/test_lua_shim_cpu.py
with open(os.path.join(here, "image_detect_api.json"), "w") as f:
    json.dump(_methods(_strip_lua(open(os.path.join(REF, "ImageDetect.lua")).read())), f, indent=1)
    f.write("\n")
print("golden fixtures written")
