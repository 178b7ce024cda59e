"""GPU: raw uint8 images of different sizes through batched getImages and the pipelined batch path
(mpn_get_images_batch_u8(_dev), mpn_model_detect_nms_batch_submit_u8): each image's block of the padded canvas is the
single-image getImages bit for bit and the rest is +0.0; the pipelined raw batch equals mpn_model_detect_nms_batch on that
canvas byte for byte (scores, boxes, keep lists, sink records); a batch of one is mpn_model_detect_nms_submit_u8; batch and
single tickets interleave across changing canvases; at full size the keep lists are nms.c's; bad arguments fail loudly
before anything is enqueued."""
import ctypes as C

import numpy as np
import pytest
import torch

import multipathnet_b200 as mpn
from multipathnet_b200 import _lib, models, workloads as wl
from test_model_gpu import assert_nms_every_class

pytestmark = pytest.mark.gpu

# (H0, W0) at scale 60 / max_size 100: grows to 60 x 80, shrinks to 60 x 80, hits the max_size cap (22 x 100), portrait 96 x 60
SIZES = [(48, 64), (150, 200), (20, 90), (80, 50)]


def _raw(sizes, seed):
    return [np.random.default_rng(seed + i).integers(0, 256, (h, w, 3), dtype=np.uint8) for i, (h, w) in enumerate(sizes)]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _check_canvas(ctx, ims, batch, scales, hw, kind, scale, max_size):
    H, W = batch.shape[2:]
    assert (H, W) == (max(h for h, _ in hw), max(w for _, w in hw))
    for i, im in enumerate(ims):
        one, s = ctx.get_images_u8(im, kind, scale, max_size)
        h, w = hw[i]
        assert one.shape == (3, h, w) and s == scales[i]
        assert np.array_equal(_bits(batch[i, :, :h, :w]), _bits(one)), f"image {i}"
        pad = np.ones((3, H, W), bool)
        pad[:, :h, :w] = False
        assert not _bits(batch[i])[pad].any(), f"image {i}: padding is not +0.0"


@pytest.mark.parametrize("kind", ["ross", "imagenet"])
@pytest.mark.parametrize("order", [[0, 1, 2, 3], [3, 2, 1, 0], [1]])
def test_padded_getimages_host_and_dev(ctx, kind, order):
    ims = [_raw(SIZES, 40)[i] for i in order]
    batch, scales, hw = ctx.get_images_batch_u8(ims, kind, 60, 100)
    _check_canvas(ctx, ims, batch, scales, hw, kind, 60, 100)
    if len(ims) == 1:
        assert batch.shape[2:] == hw[0]                                        # no padding at all
    # _dev: raw bytes and canvas on the device; the canvas starts as NaN, so an element the kernel does not write fails
    raw = torch.from_numpy(np.concatenate([im.reshape(-1) for im in ims])).cuda()
    out = torch.full(batch.shape, float("nan"), dtype=torch.float32, device="cuda")
    H0 = np.array([im.shape[0] for im in ims], np.int32); W0 = np.array([im.shape[1] for im in ims], np.int32)
    tf = _lib.CImageTransform.of(kind)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.mpn_get_images_batch_u8_dev(ctx.h, raw.data_ptr(), len(ims), H0.ctypes.data_as(_lib._i32p), W0.ctypes.data_as(_lib._i32p),
                                                  C.addressof(tf), 60.0, 100.0, out.data_ptr()), "mpn_get_images_batch_u8_dev")
    ctx.synchronize()
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(batch))


def _sink(m, cap):
    rec = torch.zeros((cap, mpn.MPN_REC_FLOATS), dtype=torch.float32, device="cuda")
    m.set_detection_sink(rec, cap, 100)
    return rec


def _same(a, b, what=""):
    (s1, b1, k1), (s2, b2, k2) = a, b
    assert np.array_equal(_bits(s1), _bits(s2)) and np.array_equal(_bits(b1), _bits(b2)), what
    assert len(k1) == len(k2) and all(np.array_equal(x, y) for x, y in zip(k1, k2)), what


def _spec(builder):
    return (models.vgg16_fast_rcnn(21, seed=13, width_div=4, fc_dim=256) if builder == "vgg"
            else models.vgg16_multipathnet(21, seed=13, width_div=4, fc_dim=256))


def _fp32_batch(ctx, m, ims, boxes, kind, scale, max_size, **kw):
    """what a batch user does without the raw path: the canvas from getImages, then mpn_model_detect_nms_batch"""
    canvas, scales, _ = ctx.get_images_batch_u8(ims, kind, scale, max_size)
    return m.detect_nms_batch(canvas, boxes, scales, [(im.shape[1], im.shape[0]) for im in ims], **kw)


# raw sizes at scale 120 / max_size 200: 120 x 160, 120 x 192, 120 x 139 -> canvas 120 x 192
RAW3 = [(96, 128), (80, 128), (110, 128)]


@pytest.mark.parametrize("builder", ["vgg", "mpn"])
def test_raw_batch_submit_equals_the_fp32_batch_path(ctx, builder):
    spec = _spec(builder)
    m = mpn.Model(ctx, spec, max_rois=512, max_h=192, max_w=256)
    try:
        ims = _raw(RAW3, 7)
        gen = wl.sharpmask_boxes if builder == "mpn" else wl.random_boxes
        boxes = [gen(r, h, w, 20 + i) for i, ((h, w), r) in enumerate(zip(RAW3, [90, 41, 130]))]
        rec = _sink(m, 6)
        got = m.detect_nms_wait(m.detect_nms_batch_submit_u8(ims, boxes, spec.transformer, 120, 200, 0.0, 0.3))
        want = _fp32_batch(ctx, m, ims, boxes, spec.transformer, 120, 200, score_thresh=0.0, nms_thr=0.3)
        assert len(got) == len(want) == 3
        for i in range(3):
            _same(got[i], want[i], f"image {i}")
        torch.cuda.synchronize()
        assert m.detection_sink_count() == 6
        for i in range(3):
            assert torch.equal(rec[i], rec[3 + i]), f"record of image {i}"
    finally:
        m.set_detection_sink(None, 0)
        m.close()


def test_batch_of_one_is_the_single_raw_submit(ctx):
    spec = _spec("vgg")
    m = mpn.Model(ctx, spec, max_rois=256, max_h=192, max_w=256)
    try:
        im = _raw([(110, 128)], 3)[0]
        bx = wl.random_boxes(77, 110, 128, 5)
        rec = _sink(m, 2)
        single = m.detect_nms_wait(m.detect_nms_submit_u8(im, bx, "ross", 120, 200))
        batch = m.detect_nms_wait(m.detect_nms_batch_submit_u8([im], [bx], "ross", 120, 200))
        assert len(batch) == 1
        _same(single, batch[0])
        torch.cuda.synchronize()
        assert m.detection_sink_count() == 2 and torch.equal(rec[0], rec[1])
    finally:
        m.set_detection_sink(None, 0)
        m.close()


def test_pipeline_interleaves_batch_and_single_tickets_across_canvases(ctx):
    """two submissions always in flight; batch sizes 1-3, four different canvases, single-image tickets in between: every
    result equals its synchronous counterpart byte for byte and the sink records arrive in submission order"""
    spec = _spec("vgg")
    m = mpn.Model(ctx, spec, max_rois=512, max_h=200, max_w=256)
    kind, scale, max_size = spec.transformer, 120, 200
    jobs = [("batch", [(96, 128), (80, 128)]),             # canvas 120 x 192
            ("single", [(90, 120)]),                       # 120 x 160
            ("batch", [(110, 128), (96, 128), (60, 100)]), # 120 x 200
            ("batch", [(128, 96)]),                        # 160 x 120 (batch of one)
            ("single", [(80, 128)]),
            ("batch", [(100, 100), (128, 96)]),            # 160 x 120
            ("batch", [(96, 128), (110, 128), (80, 128)]), # 120 x 192
            ("single", [(96, 128)])]
    work = []
    for j, (kind_j, sizes) in enumerate(jobs):
        ims = _raw(sizes, 100 + 10 * j)
        boxes = [wl.random_boxes(30 + 17 * i + 5 * j, h, w, 200 + 10 * j + i) for i, (h, w) in enumerate(sizes)]
        work.append((kind_j, ims, boxes))

    def submit(kind_j, ims, boxes):
        if kind_j == "single":
            return m.detect_nms_submit_u8(ims[0], boxes[0], kind, scale, max_size)
        return m.detect_nms_batch_submit_u8(ims, boxes, kind, scale, max_size)

    try:
        n_rec = sum(len(ims) for _, ims, _ in work)
        rec = _sink(m, n_rec)
        tickets, got = [submit(*work[0]), submit(*work[1])], []
        with pytest.raises(mpn.MpnError, match="two submissions are already in flight"):
            submit(*work[2])
        for j in range(2, len(work)):
            got.append(m.detect_nms_wait(tickets[j - 2]))
            tickets.append(submit(*work[j]))
        got += [m.detect_nms_wait(tickets[-2]), m.detect_nms_wait(tickets[-1])]
        torch.cuda.synchronize()
        assert m.detection_sink_count() == n_rec
        rec_pipe = rec.clone()
        # synchronous counterparts, in the same order, into the same sink
        m.set_detection_sink(rec, n_rec, 100)
        for (kind_j, ims, boxes), g in zip(work, got):
            if kind_j == "single" or len(ims) == 1:
                img, s = ctx.get_images_u8(ims[0], kind, scale, max_size)
                want = m.detect_nms(img, boxes[0], s, ims[0].shape[1], ims[0].shape[0])
                _same(g if kind_j == "single" else g[0], want)
            else:
                want = _fp32_batch(ctx, m, ims, boxes, kind, scale, max_size)
                assert len(g) == len(want)
                for a, b in zip(g, want):
                    _same(a, b)
        torch.cuda.synchronize()
        assert torch.equal(rec, rec_pipe), "sink records differ from the synchronous calls or arrived out of order"
    finally:
        m.set_detection_sink(None, 0)
        m.close()


def test_full_size_cfg2_three_coco_sizes(ctx):
    from bench import WORKLOADS
    wk = WORKLOADS["vgg16_frcnn"]
    spec = getattr(models, wk["model"])(wk["C"], seed=1234, **wk["kw"])
    m = mpn.Model(ctx, spec, max_rois=2200, max_h=608, max_w=904)
    try:
        sizes, Rs = [(480, 640), (427, 640), (512, 640)], [1000, 700, 500]
        ims = _raw(sizes, 11)
        boxes = [wl.random_boxes(r, h, w, 60 + i) for i, ((h, w), r) in enumerate(zip(sizes, Rs))]
        got = m.detect_nms_wait(m.detect_nms_batch_submit_u8(ims, boxes, spec.transformer, 600, 1000))
        canvas, scales, hw = ctx.get_images_batch_u8(ims, spec.transformer, 600, 1000)
        assert canvas.shape == (3, 3, 600, 899) and hw == [(600, 800), (600, 899), (600, 750)]
        want = m.detect_nms_batch(canvas, boxes, scales, [(w, h) for h, w in sizes])
        for i in range(3):
            _same(got[i], want[i], f"image {i}")
            assert got[i][0].shape == (Rs[i], wk["C"])
            assert_nms_every_class(*got[i])
    finally:
        m.close()


def test_bad_arguments_fail_before_anything_is_enqueued(ctx):
    spec = _spec("vgg")
    m = mpn.Model(ctx, spec, max_rois=64, max_h=160, max_w=192)
    lib = ctx.lib
    try:
        ims = _raw([(96, 128), (80, 128)], 1)                      # 120 x 160 and 120 x 192 at scale 120 / max_size 200
        boxes = [wl.random_boxes(20, 96, 128, 2), wl.random_boxes(15, 80, 128, 3)]
        before = m.detect_nms_wait(m.detect_nms_batch_submit_u8(ims, boxes, "ross", 120, 200))
        raw = np.concatenate([im.reshape(-1) for im in ims])
        bx = np.ascontiguousarray(np.concatenate(boxes), np.float32)
        Cn = spec.num_classes
        scores = np.empty((64, Cn), np.float32); bboxes = np.empty((64, 4 * Cn), np.float32)
        keep = np.empty((Cn - 1) * 64, np.int32); counts = np.empty((2, Cn - 1), np.int32)

        def call(N=2, H0=(96, 80), W0=(128, 128), swap=(3, 2, 1), offs=(0, 20, 35), scale=120.0, ims_p=raw, boxes_p=bx, ticket=True, tf_p=True):
            h0 = np.array(H0, np.int32); w0 = np.array(W0, np.int32); o = np.array(offs, np.int64)
            tf = _lib.CImageTransform.of("ross"); tf.swap[:] = list(swap)
            t = C.c_int32(-1)
            return lib.mpn_model_detect_nms_batch_submit_u8(
                m.h, _lib._ptr(ims_p), N, h0.ctypes.data_as(_lib._i32p), w0.ctypes.data_as(_lib._i32p), C.addressof(tf) if tf_p else None,
                scale, 200.0, _lib._ptr(boxes_p), o.ctypes.data_as(_lib._i64p), -1.5, 0.3, _lib._ptr(scores), _lib._ptr(bboxes),
                _lib._ptr(keep), _lib._ptr(counts), C.byref(t) if ticket else None)

        cases = [(dict(N=0), "batch size N"), (dict(N=65), "batch size N"),
                 (dict(H0=(96, 0)), "H0, W0 > 0"), (dict(W0=(-1, 128)), "H0, W0 > 0"),
                 (dict(H0=(96, 40)), "larger than max_h x max_w"),          # 40 x 128 -> 62 x 200
                 (dict(scale=200.0), "larger than max_h x max_w"),          # 150 x 200 canvas
                 (dict(offs=(0, 20, 20)), "at least one proposal"), (dict(offs=(0, 40, 70)), "max_rois"),
                 (dict(offs=(1, 20, 35)), "img_offsets\\[0\\]"),
                 (dict(swap=(0, 2, 1)), "swap entries"), (dict(swap=(3, 2, 4)), "swap entries"),
                 (dict(ims_p=None), "missing"), (dict(boxes_p=None), "missing"), (dict(ticket=False), "missing"),
                 (dict(tf_p=False), "missing")]
        n0 = ctx.launch_count
        for kw, msg in cases:
            rc = call(**kw)
            err = lib.mpn_last_error(ctx.h).decode()
            assert rc != 0, kw
            assert __import__("re").search(msg, err), (kw, err)
        assert ctx.launch_count == n0, "a rejected call launched kernels"
        # the getImages entries refuse the same way
        tf = _lib.CImageTransform.of("ross"); tf.swap[:] = [1, 2, 5]
        h0 = np.array([96, 80], np.int32); w0 = np.array([128, 128], np.int32)
        out = np.empty((2, 3, 120, 192), np.float32)
        assert lib.mpn_get_images_batch_u8(ctx.h, _lib._ptr(raw), 2, h0.ctypes.data_as(_lib._i32p), w0.ctypes.data_as(_lib._i32p),
                                           C.addressof(tf), 120.0, 200.0, _lib._ptr(out)) != 0
        assert "swap entries" in lib.mpn_last_error(ctx.h).decode()
        assert lib.mpn_get_images_batch_u8(ctx.h, _lib._ptr(raw), 0, h0.ctypes.data_as(_lib._i32p), w0.ctypes.data_as(_lib._i32p),
                                           C.addressof(_lib.CImageTransform.of("ross")), 120.0, 200.0, _lib._ptr(out)) != 0
        assert "batch size N" in lib.mpn_last_error(ctx.h).decode()
        assert ctx.launch_count == n0
        after = m.detect_nms_wait(m.detect_nms_batch_submit_u8(ims, boxes, "ross", 120, 200))
        for a, b in zip(before, after):
            _same(a, b)
    finally:
        m.close()
