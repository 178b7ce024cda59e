"""GPU suite, N > 1: the path's one collective on real NCCL (SURVEY 8e). Two processes, one GPU each (skipped on a
1-GPU box): every rank runs ITS images (round-robin, test_runner.lua:91-104) through detect+NMS with the detection sink on,
the library issues ONE ncclAllGather (mpn_dist_all_gather), and the gathered set must equal — bit for bit — what a
single GPU produces for all the images followed by the host keep_top_k (Tester:keepTopKPerImage, :163-168)."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_IMAGES, H, W, R = 5, 150, 203, 200


def _image(spec, i):
    from multipathnet_b200 import workloads as wl
    return wl.transform(wl.raw_image(H, W, 300 + i), spec.transformer), wl.random_boxes(R, H, W, 300 + i)


def _worker(rank, world, q_id, q_out):
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import multipathnet_b200 as mpn
    from multipathnet_b200 import dist as mdist, models
    torch.cuda.set_device(rank)
    ctx = mpn.Context(rank)
    if rank == 0:
        uid = ctx.dist_unique_id()
        for _ in range(world - 1):
            q_id.put(uid)
    else:
        uid = q_id.get(timeout=120)
    ctx.dist_init(uid, rank, world)
    assert ctx.dist_world() == (rank, world)
    spec = models.vgg16_fast_rcnn(21, seed=7, width_div=4, fc_dim=256)
    m = mpn.Model(ctx, spec, max_rois=512, max_h=256, max_w=320)
    mine = mdist.shard_images(N_IMAGES, rank, world)
    per_rank = (N_IMAGES + world - 1) // world
    rec_d = torch.zeros((per_rank, mpn.MPN_REC_FLOATS), dtype=torch.float32, device=f"cuda:{rank}")     # ranks with fewer images pad with empty records
    m.set_detection_sink(rec_d, per_rank, 100)
    for i in mine:
        img, boxes = _image(spec, i)
        m.detect_nms(img, boxes, 1.0, W, H, -1.5, 0.3, want_raw=False)
    g = mdist.gather_records_dev(ctx, rec_d, per_rank)                    # world x per_rank x REC on every rank
    q_out.put((rank, g))
    m.close(); ctx.dist_destroy(); ctx.close()


def test_two_gpu_gather_equals_single_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    import multipathnet_b200 as mpn
    from multipathnet_b200 import dist as mdist, models
    mpc = mp.get_context("spawn")
    q_id, q_out = mpc.Queue(), mpc.Queue()
    ps = [mpc.Process(target=_worker, args=(r, 2, q_id, q_out)) for r in range(2)]
    [p.start() for p in ps]
    res = dict(q_out.get(timeout=600) for _ in ps)
    [p.join(120) for p in ps]
    assert all(p.exitcode == 0 for p in ps)
    assert np.array_equal(res[0], res[1])                                  # every rank ends with the same gathered set
    # single-GPU result for ALL images + host keep_top_k
    ctx = mpn.Context(0)
    spec = models.vgg16_fast_rcnn(21, seed=7, width_div=4, fc_dim=256)
    m = mpn.Model(ctx, spec, max_rois=512, max_h=256, max_w=320)
    for i in range(N_IMAGES):
        img, boxes = _image(spec, i)
        scores, bboxes, keeps = m.detect_nms(img, boxes, 1.0, W, H, -1.5, 0.3)
        tables = [np.concatenate([bboxes[k, 4 * j:4 * j + 4], scores[k, j:j + 1]], 1).astype(np.float32) for j, k in enumerate(keeps, start=1)]
        want = mdist.pack_record(mdist.tables_to_dets(tables))
        r, slot = i % 2, i // 2                                            # image i ran on rank i mod 2 as its (i div 2)-th image
        assert np.array_equal(res[0][r, slot], want), f"image {i}"
        assert int(want[0]) >= 100
    assert np.all(res[0][1, 2] == 0)                                       # rank 1 had two images: its third slot is an empty record
    m.close(); ctx.close()
