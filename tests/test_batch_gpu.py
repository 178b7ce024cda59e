"""GPU: a batch of N images through the model path (mpn_model_trunk_batch, mpn_model_detect_nms_batch*): the batch of one
is the single-image call byte for byte; with the fp32 check kernels (conv_impl 1, every convolution a per-element sum)
each image's results equal its own single-image call bit for bit; every ROI pooling implementation reads the image the
ROI's batch index names; at full size the product path meets the oracle's 1e-3 contract per image; a batch index
outside [1, N] fails loudly."""
import numpy as np
import pytest
import torch

import multipathnet_b200 as mpn
from multipathnet_b200 import models, workloads as wl
from oracle import ref as O
from conftest import rel_err, record_parity
from test_model_gpu import assert_nms_every_class
from test_roi_product_gpu import check_tower
import _batch_oracle as BO

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _batch(spec, sizes, Rs, H, W, seed, sharp=False):
    """images of the given original (W0, H0) sizes (im_scale 1), zero-padded to H x W, and their own proposals"""
    ims = [wl.transform(wl.raw_image(h, w, seed + i), spec.transformer) for i, (w, h) in enumerate(sizes)]
    gen = wl.sharpmask_boxes if sharp else wl.random_boxes
    boxes = [gen(r, h, w, seed + 10 + i) for i, ((w, h), r) in enumerate(zip(sizes, Rs))]
    return BO.pad_images(ims, H, W), boxes


def _sink(m, cap):
    rec = torch.zeros((cap, mpn.MPN_REC_FLOATS), dtype=torch.float32, device="cuda")
    m.set_detection_sink(rec, cap, 100)
    return rec


def _same(a, b):
    (s1, b1, k1), (s2, b2, k2) = a, b
    assert np.array_equal(s1, s2) and np.array_equal(b1, b2)
    assert len(k1) == len(k2) and all(np.array_equal(x, y) for x, y in zip(k1, k2))


@pytest.mark.parametrize("full", [False, True])
def test_batch_of_one_is_the_single_image_call(ctx, full):
    if full:
        spec, H, W, R = models.vgg16_fast_rcnn(21, seed=1234), 600, 800, 1000
    else:
        spec, H, W, R = models.vgg16_fast_rcnn(21, seed=7, width_div=4, fc_dim=256), 150, 203, 200
    m = mpn.Model(ctx, spec, max_rois=1024, max_h=608, max_w=800)
    try:
        imgs, boxes = _batch(spec, [(W - 7, H - 3)], [R], H, W, 4)
        rec = _sink(m, 2)
        single = m.detect_nms(imgs[0], boxes[0], 1.0, W - 7, H - 3)
        batch = m.detect_nms_batch(imgs, boxes, [1.0], [(W - 7, H - 3)])
        assert len(batch) == 1
        _same(single, batch[0])
        torch.cuda.synchronize()
        assert m.detection_sink_count() == 2 and torch.equal(rec[0], rec[1])
    finally:
        m.set_detection_sink(None, 0)
        m.close()


@pytest.mark.parametrize("builder", ["vgg", "mpn"])
def test_batch_equals_single_calls_with_fp32_check_kernels(ctx, builder):
    """conv_impl 1: every trunk and head convolution is a per-element fp32 sum and the first layer has no split-K, so an
    image's rows cannot depend on the other images; any difference is a batching bug"""
    spec = (models.vgg16_fast_rcnn(21, seed=9, width_div=4, fc_dim=256) if builder == "vgg"
            else models.vgg16_multipathnet(21, seed=9, width_div=4, fc_dim=256))
    m = mpn.Model(ctx, spec, max_rois=512, max_h=256, max_w=320)
    m.set_conv_impl(1)
    sizes, Rs, H, W = [(200, 144), (176, 160), (208, 120)], [70, 33, 101], 160, 208
    try:
        imgs, boxes = _batch(spec, sizes, Rs, H, W, 21, sharp=(builder == "mpn"))
        rec = _sink(m, 6)
        batch = m.detect_nms_batch(imgs, boxes, [1.0] * 3, sizes)
        singles = [m.detect_nms(imgs[i], boxes[i], 1.0, *sizes[i]) for i in range(3)]
        for i in range(3):
            _same(singles[i], batch[i])
        torch.cuda.synchronize()
        assert m.detection_sink_count() == 6
        for i in range(3):
            assert torch.equal(rec[i], rec[3 + i]), f"record of image {i}"
    finally:
        m.set_detection_sink(None, 0)
        m.set_conv_impl(0)
        m.close()


@pytest.mark.parametrize("roi_impl", [0, 1, 2, 3, 4, 5])
def test_every_roi_impl_reads_the_named_image(ctx, roi_impl):
    """ROIs of image 2 of a batch of two: the pooled tensor of every tower equals the oracle's roi_pool of image 2's own
    trunk slots (read back from the device), with the bars of test_roi_product_gpu.py"""
    spec = models.vgg16_multipathnet(21, seed=11, width_div=4, fc_dim=256)
    m = mpn.Model(ctx, spec, max_rois=256, max_h=256, max_w=320)
    ctx.set_option("roi_impl", roi_impl)
    try:
        imgs, boxes = _batch(spec, [(208, 160), (208, 160)], [1, 128], 160, 208, 6, sharp=True)
        rois = O.project_rois(boxes[1], 1.0)
        rois[:, 0] = 2.0
        m.forward(imgs, rois)
        assert m.trunk_slot(spec.taps["conv5"]).shape[0] == 2
        for t in range(len(spec.towers)):
            check_tower(spec, m, rois, t, slice(0, 128))
    finally:
        ctx.set_option("roi_impl", -1)
        m.close()


def _product_parity(ctx, spec, name, sizes, Rs, H, W, seed, sharp, max_rois, fused_slots):
    m = mpn.Model(ctx, spec, max_rois=max_rois, max_h=H, max_w=W)
    try:
        imgs, boxes = _batch(spec, sizes, Rs, H, W, seed, sharp)
        got = m.detect_nms_batch(imgs, boxes, [1.0] * len(sizes), sizes)
        taps = sorted(set(spec.taps.values()))
        batch_slots = {}
        for impl in (0, 2):                                  # conv_impl 2 materialises the slots the conv + pool fusion elides
            m.set_conv_impl(impl)
            m.trunk_batch(imgs)
            for s in taps:
                if impl == 0 and s in fused_slots:
                    continue
                batch_slots[(impl, s)] = m.trunk_slot(s)
            for i in range(len(sizes)):
                m.trunk(imgs[i])
                for s in taps:
                    if (impl, s) in batch_slots:
                        e = rel_err(batch_slots[(impl, s)][i], m.trunk_slot(s)[0])
                        assert e < 1e-4, (name, impl, s, i, e)
        m.set_conv_impl(0)
        ref = BO.test_one_batch(spec, imgs, boxes, [1.0] * len(sizes), sizes)
        for i, ((s, b, k), (rs, rb, _)) in enumerate(zip(got, ref)):
            es, eb = rel_err(s, rs), rel_err(b, rb)
            record_parity(f"batch_{name}_img{i}", scores=es, bboxes=eb)
            assert es < TOL and eb < TOL, (name, i, es, eb)
            assert_nms_every_class(s, b, k)
    finally:
        m.set_conv_impl(0)
        m.close()


def test_batch_full_size_cfg2(ctx):
    """BASELINE configs[1] at B = 2: VGG-16 Fast R-CNN, two images of different sizes padded to 600 x 800"""
    spec = models.vgg16_fast_rcnn(21, seed=1234)
    fused = {spec.taps["conv3"], spec.taps["conv4"]} if "conv3" in spec.taps else set()
    _product_parity(ctx, spec, "cfg2", [(800, 600), (752, 564)], [1000, 700], 600, 800, 31, False, 2048, fused)


def test_batch_full_size_cfg3(ctx):
    """BASELINE configs[2] at B = 2: MultiPathNet (five towers, foveal regions, three pyramid levels)"""
    spec = models.vgg16_multipathnet(81, seed=1234)
    _product_parity(ctx, spec, "cfg3", [(800, 600), (720, 592)], [400, 300], 600, 800, 41, True, 1024, set())


def test_batch_resnet50_integral_head(ctx):
    """cfg 4 style on a small image: ResNet-50 trunk, per-ROI layer4, integral head (mean of softmaxes), B = 2"""
    spec = models.resnet50_fast_rcnn(21, seed=5, integral_k=3)
    _product_parity(ctx, spec, "cfg4_small", [(224, 160), (200, 150)], [48, 30], 160, 224, 51, True, 128, set())


def test_bad_batch_index_fails_loudly(ctx):
    spec = models.vgg16_fast_rcnn(21, seed=7, width_div=4, fc_dim=256)
    m = mpn.Model(ctx, spec, max_rois=256, max_h=256, max_w=320)
    try:
        imgs, boxes = _batch(spec, [(208, 160), (200, 150)], [40, 40], 160, 208, 8)
        rois = O.project_rois(boxes[1], 1.0)
        rois[:, 0] = 2.0
        ref_cls, ref_bbox = m.forward(imgs, rois)
        for bad in (0.0, 3.0):
            r = rois.copy(); r[5, 0] = bad
            with pytest.raises(mpn.MpnError, match="batch index"):
                m.heads(r)
            rd = torch.from_numpy(r).cuda()
            cls = torch.empty((40, spec.num_classes), device="cuda")
            ctx.check(ctx.lib.mpn_model_heads_dev(m.h, rd.data_ptr(), 40, cls.data_ptr(), None), "heads_dev")
            with pytest.raises(mpn.MpnError, match="batch index"):
                ctx.synchronize()
        cls, bbox = m.heads(rois)                                # the model is still usable and exact
        assert np.array_equal(cls, ref_cls) and np.array_equal(bbox, ref_bbox)
    finally:
        m.close()
