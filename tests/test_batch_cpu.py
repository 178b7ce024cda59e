"""CPU side of batched detection (mpn_model_trunk_batch / mpn_model_detect_nms_batch*): the batch oracle equals the
single-image oracle on the same padded images, the Python wrappers reject a malformed batch before any library call, and
the header block still holds the new prototypes in a form the Lua cdef reader takes."""
import re

import numpy as np
import pytest

import multipathnet_b200 as mpn
from multipathnet_b200 import _lib, models, workloads as wl
from oracle import graphs as G
import _batch_oracle as BO


def _batch(spec, sizes, Rs, H, W, seed):
    ims = [wl.transform(wl.raw_image(h, w, seed + i), spec.transformer) for i, (w, h) in enumerate(sizes)]
    boxes = [wl.random_boxes(r, h, w, seed + 10 + i) for i, ((w, h), r) in enumerate(zip(sizes, Rs))]
    return BO.pad_images(ims, H, W), boxes


@pytest.mark.parametrize("builder", ["vgg", "mpn"])
def test_oracle_batch_equals_single_image_oracle(builder):
    spec = (models.vgg16_fast_rcnn(21, seed=5, width_div=16, fc_dim=64) if builder == "vgg"
            else models.vgg16_multipathnet(21, seed=5, width_div=16, fc_dim=64))
    sizes, Rs, scales = [(96, 64), (72, 80), (100, 56)], [9, 5, 12], [1.0, 1.0, 1.0]
    imgs, boxes = _batch(spec, sizes, Rs, 80, 100, 3)
    got = BO.test_one_batch(spec, imgs, boxes, scales, sizes)
    det = BO.detect_batch(spec, imgs, boxes, scales)
    for i, (w0, h0) in enumerate(sizes):
        s1, b1 = G.detect(spec, imgs[i], boxes[i], scales[i])
        assert np.array_equal(det[i][0], s1) and np.array_equal(det[i][1], b1)
        s, b, k = G.test_one(spec, imgs[i], boxes[i], scales[i], w0, h0)
        assert np.array_equal(got[i][0], s) and np.array_equal(got[i][1], b)
        assert len(k) == len(got[i][2]) and all(np.array_equal(x, y) for x, y in zip(k, got[i][2]))


def test_batch_rois_carry_the_image_index():
    rois = BO.batch_rois([np.ones((2, 4), np.float32) * 11, np.ones((3, 4), np.float32) * 21], [0.5, 2.0])
    assert rois.shape == (5, 5)
    assert rois[:, 0].tolist() == [1, 1, 2, 2, 2]
    assert np.allclose(rois[:2, 1:], 6.0) and np.allclose(rois[2:, 1:], 41.0)


class _NoLib:
    """stands in for the library: any call means validation let a malformed batch through"""
    def __getattr__(self, name):
        raise AssertionError(f"library entry {name} reached with a malformed batch")


def _fake_model(max_rois=16, C=5):
    m = mpn.Model.__new__(mpn.Model)
    m.ctx = type("Ctx", (), {"lib": _NoLib()})()
    m.h, m.C, m.max_rois, m._trunk_n = None, C, max_rois, 1
    return m


@pytest.mark.parametrize("Rs,scales,sizes,msg", [
    ([3, 0], [1, 1], [(8, 8), (8, 8)], "at least one proposal"),
    ([10, 7], [1, 1], [(8, 8), (8, 8)], "max_rois"),
    ([3, 3], [1], [(8, 8), (8, 8)], "im_scales"),
    ([3, 3], [1, 1], [(8, 8)], "sizes"),
])
def test_batch_arguments_rejected_before_any_library_call(Rs, scales, sizes, msg):
    m = _fake_model()
    imgs = np.zeros((len(Rs), 3, 8, 8), np.float32)
    with pytest.raises(ValueError, match=msg):
        m.detect_nms_batch(imgs, [np.ones((r, 4), np.float32) for r in Rs], scales, sizes)
    with pytest.raises(ValueError, match=msg):
        m.detect_nms_batch_dev(0, len(Rs), 8, 8, 0, Rs, scales, sizes, -1.5, 0.3)


def test_batch_size_and_shape_rejected_before_any_library_call():
    m = _fake_model()
    with pytest.raises(ValueError, match="batch size"):
        m.detect_nms_batch_dev(0, 0, 8, 8, 0, [], [], [], -1.5, 0.3)
    with pytest.raises(ValueError, match="batch size"):
        m.detect_nms_batch_dev(0, mpn.MPN_MAX_BATCH + 1, 8, 8, 0, [1] * (mpn.MPN_MAX_BATCH + 1), [1] * (mpn.MPN_MAX_BATCH + 1),
                               [(8, 8)] * (mpn.MPN_MAX_BATCH + 1), -1.5, 0.3)
    with pytest.raises(ValueError, match="N x 3 x H x W"):
        m.trunk_batch(np.zeros((3, 8, 8), np.float32))
    with pytest.raises(ValueError, match="N x 3 x H x W"):
        m.detect_nms_batch(np.zeros((3, 8, 8), np.float32), [np.ones((1, 4))], [1], [(8, 8)])


def test_batch_offsets_are_the_running_sum():
    offs, sc, w0, h0 = _fake_model(max_rois=100)._batch_args(3, [4, 1, 7], [0.5, 1, 2], [(10, 20), (30, 40), (50, 60)])
    assert offs.dtype == np.int64 and offs.tolist() == [0, 4, 5, 12]
    assert sc.tolist() == [0.5, 1, 2] and w0.tolist() == [10, 30, 50] and h0.tolist() == [20, 40, 60]


def test_header_declares_the_batch_entries_for_the_lua_cdef():
    h = open(_lib.HEADER_PATH).read()
    body = re.search(r"MPN_CDEF_BEGIN \*/(.*?)/\* MPN_CDEF_END", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    assert "#" not in body                                          # no preprocessor lines: ffi.cdef takes the block verbatim
    assert re.search(r"enum\s*\{\s*MPN_MAX_BATCH\s*=\s*64\s*\}\s*;", body)
    assert _lib.MPN_MAX_BATCH == 64
    protos = {m.group(1): m.group(2) for m in re.finditer(r"\b(mpn_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", body, re.S)}
    for name, n in [("mpn_model_trunk_batch", 5), ("mpn_model_trunk_batch_dev", 5), ("mpn_model_detect_nms_batch", 16),
                    ("mpn_model_detect_nms_batch_dev", 16)]:
        assert name in protos and len(protos[name].split(",")) == n, name
        assert len(_lib.SIGNATURES[name][1]) == n, name
