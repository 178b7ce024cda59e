"""CPU oracle of the batched detect path (mpn_model_detect_nms_batch*), built on oracle/graphs.py: the reference's
semantics for a padded batch of N images of one size (ImageDetect.lua:44-50 pads with zeros after the transformer):
the trunk over the N x 3 x H x W tensor, inn.ROIPooling by the ROI's 1-based batch index (ImageDetect.lua:66-70), and
per image the decode against its own original boxes and the clamp to its own W0 x H0 (Tester_FRCNN.lua:75-78).

The trunk of an N-image tensor is the per-image trunk stacked (no layer mixes images); it is evaluated image by image so
that the CPU GEMMs see the same shapes as the single-image oracle and the two agree bit for bit. The heads run per image
on that image's ROIs, pooled from the stacked maps by their batch index."""
import numpy as np
import torch

from oracle import graphs as G, ref as O


def pad_images(images_chw, H=None, W=None):
    """N transformed images of different sizes -> one N x 3 x H x W tensor, zero-padded at the bottom / right"""
    H = H or max(im.shape[1] for im in images_chw)
    W = W or max(im.shape[2] for im in images_chw)
    out = np.zeros((len(images_chw), 3, H, W), np.float32)
    for i, im in enumerate(images_chw):
        out[i, :, :im.shape[1], :im.shape[2]] = im
    return out


def batch_rois(boxes_list, im_scales):
    """project_im_rois of every image with its own im_scale, column 0 = the 1-based image index"""
    rois = []
    for i, (b, s) in enumerate(zip(boxes_list, im_scales)):
        r = O.project_rois(b, np.float32(s))
        r[:, 0] = np.float32(i + 1)
        rois.append(r)
    return np.ascontiguousarray(np.concatenate(rois, 0), np.float32)


def trunk_forward(spec, images_nchw):
    """model:get(1):forward on N x 3 x H x W -> {slot: N x C x H x W tensor}"""
    per = [G.trunk_forward(spec, im) for im in np.asarray(images_nchw, np.float32)]
    return {k: torch.cat([p[k] for p in per], 0) for k in per[0]}


def detect_batch(spec, images_nchw, boxes_list, im_scales):
    """ImageDetect:detect for every image of the padded batch -> [(scores R_i x C, bboxes R_i x 4C)]"""
    ts = trunk_forward(spec, images_nchw)
    out = []
    for i, (b, s) in enumerate(zip(boxes_list, im_scales)):
        rois = O.project_rois(b, np.float32(s))
        rois[:, 0] = np.float32(i + 1)
        cls, bbox = G.heads_forward(spec, ts, rois)
        scores = cls if (spec.no_softmax or len(spec.cls_heads) > 1) else O.softmax(cls)
        out.append((scores, O.convert_from(bbox, b)))
    return out


def test_one_batch(spec, images_nchw, boxes_list, im_scales, sizes, score_thresh=-1.5, nms_thr=0.3, nms_fn=None):
    """Tester_FRCNN:testOne for every image of the padded batch -> [(scores, clamped bboxes, [keep rows per class])]"""
    nms_fn = nms_fn or O.nms
    out = []
    for (scores, bboxes), (W0, H0) in zip(detect_batch(spec, images_nchw, boxes_list, im_scales), sizes):
        bboxes = O.clamp_boxes(bboxes, W0, H0)
        keeps = []
        for j in range(1, scores.shape[1]):
            sel = np.nonzero(scores[:, j] > score_thresh)[0]
            sb = np.concatenate([bboxes[sel, 4 * j:4 * j + 4], scores[sel, j:j + 1]], 1).astype(np.float32)
            keeps.append(sel[nms_fn(sb, nms_thr)].astype(np.int32))
        out.append((scores, bboxes, keeps))
    return out
