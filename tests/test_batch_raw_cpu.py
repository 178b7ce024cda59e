"""CPU side of batched getImages from raw images (mpn_get_images_batch_size / mpn_get_images_batch_u8 /
mpn_model_detect_nms_batch_submit_u8): the size rule per image and the canvas, the per-element code of get_images_kernel
(built for the host from tests/hd_batch_shim.cpp) against the per-image getImages padded on the host, the Python wrappers
rejecting a malformed batch before any library call, and the header block in a form the Lua cdef reader takes."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import multipathnet_b200 as mpn
from multipathnet_b200 import _lib
from multipathnet_b200.image_detect import _get_images_size
import _batch_oracle as BO

HERE = os.path.dirname(os.path.abspath(__file__))


def _sizes(lib, H0, W0, scale, max_size):
    N = len(H0)
    H0a, W0a = np.array(H0, np.int32), np.array(W0, np.int32)
    h, w, s = np.zeros(N, np.int32), np.zeros(N, np.int32), np.zeros(N, np.float64)
    Hc, Wc = C.c_int32(), C.c_int32()
    rc = lib.mpn_get_images_batch_size(N, H0a.ctypes.data_as(_lib._i32p), W0a.ctypes.data_as(_lib._i32p), float(scale), float(max_size),
                                       h.ctypes.data_as(_lib._i32p), w.ctypes.data_as(_lib._i32p),
                                       s.ctypes.data_as(C.POINTER(C.c_double)), C.byref(Hc), C.byref(Wc))
    return rc, h, w, s, Hc.value, Wc.value


@pytest.mark.parametrize("scale,max_size", [(600, 1000), (800, 1000), (60, 100)])
def test_batch_size_is_the_per_image_rule_and_the_canvas_is_the_maximum(scale, max_size):
    lib = mpn.load_library()                                       # host-only entry: no GPU needed
    rng = np.random.default_rng(scale)
    H0 = [480, 427, 512, 375, 500, 100, 1200] + [int(x) for x in rng.integers(20, 1500, 20)]
    W0 = [640, 640, 640, 500, 333, 1234, 1600] + [int(x) for x in rng.integers(20, 1500, 20)]
    rc, h, w, s, H, W = _sizes(lib, H0, W0, scale, max_size)
    assert rc == 0
    for i, (a, b) in enumerate(zip(H0, W0)):
        hi, wi, si = C.c_int32(), C.c_int32(), C.c_double()
        assert lib.mpn_get_images_size(a, b, float(scale), float(max_size), C.byref(hi), C.byref(wi), C.byref(si)) == 0
        assert (int(h[i]), int(w[i]), float(s[i])) == (hi.value, wi.value, si.value) == _get_images_size(a, b, scale, max_size)
    assert (H, W) == (int(h.max()), int(w.max()))


def test_coco_sizes_give_the_600_x_899_canvas():
    rc, h, w, s, H, W = _sizes(mpn.load_library(), [480, 427, 512], [640, 640, 640], 600, 1000)
    assert rc == 0 and list(zip(h, w)) == [(600, 800), (600, 899), (600, 750)] and (H, W) == (600, 899)


def test_batch_size_rejects_bad_counts_and_sizes():
    lib = mpn.load_library()
    assert _sizes(lib, [], [], 600, 1000)[0] != 0
    assert _sizes(lib, [10] * 65, [10] * 65, 600, 1000)[0] != 0
    assert _sizes(lib, [10] * 64, [10] * 64, 600, 1000)[0] == 0
    assert _sizes(lib, [10, 0], [10, 10], 600, 1000)[0] != 0
    assert _sizes(lib, [10, 10], [10, -3], 600, 1000)[0] != 0
    assert _sizes(lib, [10], [10], 0, 1000)[0] != 0


@pytest.fixture(scope="module")
def hd_batch(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hd") / "libhd_batch.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-o", so, os.path.join(HERE, "hd_batch_shim.cpp")],
                   check=True)
    return C.CDLL(so)


def _hd_batch(lib, ims, kind, scale, max_size):
    from oracle import ref as O
    hw = [_get_images_size(im.shape[0], im.shape[1], scale, max_size)[:2] for im in ims]
    H, W = max(h for h, _ in hw), max(w for _, w in hw)
    mean, std, tscale, swap = O.transformer_params(kind)
    m = np.array(mean, np.float32); sd = None if std is None else np.array(std, np.float32)
    raw = np.concatenate([np.ascontiguousarray(im).reshape(-1) for im in ims])
    i32 = lambda a: (C.c_int * len(a))(*[int(x) for x in a])
    out = np.full((len(ims), 3, H, W), np.nan, np.float32)
    rc = lib.hd_get_images_batch_u8(raw.ctypes.data_as(C.c_void_p), len(ims), i32([im.shape[0] for im in ims]), i32([im.shape[1] for im in ims]),
                                    i32([h for h, _ in hw]), i32([w for _, w in hw]), H, W, i32(swap), C.c_float(tscale),
                                    m.ctypes.data_as(C.c_void_p), None if sd is None else sd.ctypes.data_as(C.c_void_p),
                                    out.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return out, hw


# (H0, W0) at scale 60 / max_size 100: grows to 60 x 80, shrinks to 60 x 80, hits the max_size cap (22 x 100), portrait 96 x 60
SIZES = [(48, 64), (150, 200), (20, 90), (80, 50)]


@pytest.mark.parametrize("kind", ["ross", "imagenet"])
@pytest.mark.parametrize("order", [[0, 1, 2, 3], [3, 2, 1, 0], [1], [2, 3]])
def test_batch_element_code_equals_padded_per_image_getimages(oracle_built, hd_batch, kind, order):
    ims = [np.random.default_rng(40 + i).integers(0, 256, (*SIZES[i], 3), dtype=np.uint8) for i in order]
    got, hw = _hd_batch(hd_batch, ims, kind, 60, 100)
    per = [oracle_built.hd_get_images_u8(im, kind, h, w) for im, (h, w) in zip(ims, hw)]
    want = BO.pad_images(per)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))           # bit for bit, the padding +0.0
    if len(ims) == 1:
        assert got.shape[2:] == hw[0]                                            # a batch of one has no padding at all


def test_sizes_cover_grow_shrink_cap_and_portrait():
    hw = [_get_images_size(h, w, 60, 100) for h, w in SIZES]
    assert hw[0][2] > 1 and hw[1][2] < 1                                         # grows, shrinks
    assert hw[2][1] == 100 and hw[2][0] < 60                                     # capped by max_size
    assert hw[3][0] > hw[3][1]                                                   # portrait among landscape


class _NoLib:
    """stands in for the library: any call means validation let a malformed batch through"""
    def __getattr__(self, name):
        raise AssertionError(f"library entry {name} reached with a malformed batch")


def _fake_ctx():
    c = mpn.Context.__new__(mpn.Context)
    c.lib, c.h, c._models = _NoLib(), None, []
    return c


def _fake_model(max_rois=16, C=5, max_h=128, max_w=160):
    m = mpn.Model.__new__(mpn.Model)
    m.ctx = _fake_ctx()
    m.h, m.C, m.max_rois, m.max_h, m.max_w, m._trunk_n = None, C, max_rois, max_h, max_w, 1
    return m


def _u8(h, w):
    return np.zeros((h, w, 3), np.uint8)


BAD_IMAGES = [
    ([], "list of 1..64"),
    ([_u8(8, 8)] * 65, "list of 1..64"),
    (_u8(8, 8), "list of 1..64"),
    ([_u8(8, 8), np.zeros((8, 8, 3), np.float32)], "image 1: expected an H0 x W0 x 3 uint8"),
    ([np.zeros((8, 8), np.uint8)], "image 0: expected an H0 x W0 x 3 uint8"),
    ([np.zeros((8, 8, 4), np.uint8)], "image 0: expected an H0 x W0 x 3 uint8"),
    ([np.zeros((0, 8, 3), np.uint8)], "image 0: expected an H0 x W0 x 3 uint8"),
]


@pytest.mark.parametrize("ims,msg", BAD_IMAGES)
def test_get_images_batch_rejects_malformed_images_before_any_library_call(ims, msg):
    with pytest.raises(ValueError, match=msg):
        _fake_ctx().get_images_batch_u8(ims, "ross", 60, 100)


@pytest.mark.parametrize("ims,msg", BAD_IMAGES)
def test_batch_submit_rejects_malformed_images_before_any_library_call(ims, msg):
    n = len(ims) if isinstance(ims, list) else 1
    with pytest.raises(ValueError, match=msg):
        _fake_model().detect_nms_batch_submit_u8(ims, [np.ones((1, 4), np.float32)] * n, "ross", 60, 100)


@pytest.mark.parametrize("ims,boxes,msg", [
    ([_u8(48, 64), _u8(45, 64)], [np.ones((3, 4))], "2 images need 2 box arrays"),
    ([_u8(48, 64)], [np.ones((3, 4))] * 2, "1 images need 1 box arrays"),
    ([_u8(48, 64)], [np.ones((3, 5))], "R_i x 4"),
    ([_u8(48, 64), _u8(45, 64)], [np.ones((3, 4)), np.ones((0, 4))], "at least one proposal"),
    ([_u8(48, 64), _u8(45, 64)], [np.ones((10, 4)), np.ones((7, 4))], "max_rois"),
    ([_u8(48, 64), _u8(20, 90)], [np.ones((3, 4))] * 2, "larger than the model's max_h x max_w"),
    ([_u8(80, 50)], [np.ones((3, 4))], "larger than the model's max_h x max_w"),
])
def test_batch_submit_rejects_malformed_batches_before_any_library_call(ims, boxes, msg):
    m = _fake_model(max_h=90, max_w=90)                            # 48 x 64 -> 60 x 80 fits; 20 x 90 -> 22 x 100 and 80 x 50 -> 96 x 60 do not
    with pytest.raises(ValueError, match=msg):
        m.detect_nms_batch_submit_u8(ims, [np.asarray(b, np.float32) for b in boxes], "ross", 60, 100)


def test_header_declares_the_raw_batch_entries_for_the_lua_cdef():
    h = open(_lib.HEADER_PATH).read()
    body = re.search(r"MPN_CDEF_BEGIN \*/(.*?)/\* MPN_CDEF_END", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    assert "#" not in body                                          # no preprocessor lines: ffi.cdef takes the block verbatim
    protos = {m.group(1): m.group(2) for m in re.finditer(r"\b(mpn_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", body, re.S)}
    for name, n in [("mpn_get_images_batch_size", 10), ("mpn_get_images_batch_u8", 9), ("mpn_get_images_batch_u8_dev", 9),
                    ("mpn_model_detect_nms_batch_submit_u8", 17)]:
        assert name in protos and len(protos[name].split(",")) == n, name
        assert len(_lib.SIGNATURES[name][1]) == n, name
