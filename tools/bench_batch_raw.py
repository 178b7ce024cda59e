"""Proposals/s of detection from RAW uint8 images of different sizes, one process on one GPU, three arms alternating in rounds:

  A  mpn_model_detect_nms_submit_u8 once per image (two in flight): raw bytes up, getImages + detect + NMS on the device;
  B  mpn_model_detect_nms_batch_submit_u8 with B images per call (two calls in flight): the packed raw bytes up, getImages
     pads the B images into one canvas on the device, batched trunk + heads + NMS;
  C  what a batch user had to do before B existed: mpn_get_images_u8 per image (bytes up, scaled fp32 image down), zero
     padding on the host, then the synchronous mpn_model_detect_nms_batch (the fp32 canvas up).

Images cycle through a fixed list of landscape COCO sizes (scale 600 / max_size 1000, so canvases change from call to call and
the trunk re-plans), R seeded random boxes per image in original coordinates, every host buffer of A and B pinned. After the
timing every arm-B result is checked byte for byte against mpn_model_detect_nms_batch on the mpn_get_images_batch_u8 canvas
(arm A is not compared with B: padding changes the trunk features near a smaller image's right and bottom edges, as in the
reference). Prints one JSON line with the card name, power limit and SM clock read before and after.

    python tools/bench_batch_raw.py [--config vgg16_frcnn|multipathnet] [--batches 2,4] [--images 240] [--rounds 4]
"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

COCO_SIZES = [(480, 640), (427, 640), (512, 640), (375, 500), (424, 640), (333, 500), (480, 640), (426, 640)]   # H0 x W0


def main():
    from bench import WORKLOADS
    from bench_batch import gpu_info
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="vgg16_frcnn", choices=["vgg16_frcnn", "multipathnet"])
    ap.add_argument("--batches", default="2,4")
    ap.add_argument("--images", type=int, default=240, help="images timed per arm (at least 200)")
    ap.add_argument("--rounds", type=int, default=4, help="alternations of the arms")
    ap.add_argument("--warmup", type=int, default=2, help="warm-up passes over the image list per arm")
    ap.add_argument("--R", type=int, default=1000, help="proposals per image")
    args = ap.parse_args()
    args.images = max(args.images, 200)

    import numpy as np
    import torch
    import multipathnet_b200 as mpn
    from multipathnet_b200 import _lib, models, workloads as wl
    from multipathnet_b200.image_detect import _get_images_size

    info_before = gpu_info()
    wk = WORKLOADS[args.config]
    R, Cn = args.R, wk["C"]
    batches = [int(b) for b in args.batches.split(",")]
    Bmax = max(batches)
    scale, max_size = 600.0, 1000.0
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ctx = mpn.Context(0, own_stream=True)
    lib = ctx.lib
    spec = getattr(models, wk["model"])(Cn, seed=1234, **wk["kw"])
    tf = _lib.CImageTransform.of(spec.transformer)
    # one model per arm: each keeps its own plans, as a serving process would run one kind of call
    mA = mpn.Model(ctx, spec, max_rois=R, max_h=608, max_w=904)
    mB = mpn.Model(ctx, spec, max_rois=R * Bmax, max_h=608, max_w=904)
    mC = mpn.Model(ctx, spec, max_rois=R * Bmax, max_h=608, max_w=904)

    n_img = len(COCO_SIZES) * Bmax                  # distinct images; every batch size divides the list
    sizes = [COCO_SIZES[k % len(COCO_SIZES)] for k in range(n_img)]
    raws = [np.random.default_rng(k).integers(0, 256, (h, w, 3), dtype=np.uint8) for k, (h, w) in enumerate(sizes)]
    boxes = [wl.random_boxes(R, h, w, 1000 + k) for k, (h, w) in enumerate(sizes)]
    scaled = [_get_images_size(h, w, scale, max_size) for h, w in sizes]
    raw_pin = [torch.from_numpy(r).pin_memory() for r in raws]
    box_pin = [torch.from_numpy(b).pin_memory() for b in boxes]
    # arm B: the packed bytes, boxes, sizes and offsets of every batch, prepared once (the decoder would write them in place)
    packed = {}
    for B in batches:
        lst = []
        for k0 in range(0, n_img, B):
            ks = range(k0, k0 + B)
            lst.append(dict(ks=list(ks), raw=torch.from_numpy(np.concatenate([raws[k].reshape(-1) for k in ks])).pin_memory(),
                            box=torch.from_numpy(np.concatenate([boxes[k] for k in ks])).pin_memory(),
                            H0=np.array([sizes[k][0] for k in ks], np.int32), W0=np.array([sizes[k][1] for k in ks], np.int32),
                            offs=np.arange(B + 1, dtype=np.int64) * R))
        packed[B] = lst

    def outs(n):
        return [torch.empty(n * R * Cn, dtype=torch.float32).pin_memory(), torch.empty(n * R * 4 * Cn, dtype=torch.float32).pin_memory(),
                torch.empty((Cn - 1) * n * R, dtype=torch.int32).pin_memory(), torch.empty(n * (Cn - 1), dtype=torch.int32).pin_memory()]
    slot_out = [outs(Bmax), outs(Bmax)]

    def pipelined(submit, n_calls, m):
        tickets = []
        for i in range(n_calls):
            if i >= 2:
                ctx.check(lib.mpn_model_detect_nms_wait(m.h, tickets[i - 2]), "wait")
            tickets.append(submit(i, slot_out[i & 1]))
        for t in tickets[-2:]:
            ctx.check(lib.mpn_model_detect_nms_wait(m.h, t), "wait")

    def submit_a(i, o):
        k = i % n_img
        t = C.c_int32(-1)
        ctx.check(lib.mpn_model_detect_nms_submit_u8(mA.h, raw_pin[k].data_ptr(), sizes[k][0], sizes[k][1], C.addressof(tf), scale, max_size,
                                                     box_pin[k].data_ptr(), R, -1.5, 0.3, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(),
                                                     o[3].data_ptr(), C.byref(t)), "detect_nms_submit_u8")
        return t.value

    def submit_b(B):
        def f(i, o):
            p = packed[B][i % len(packed[B])]
            t = C.c_int32(-1)
            ctx.check(lib.mpn_model_detect_nms_batch_submit_u8(
                mB.h, p["raw"].data_ptr(), B, p["H0"].ctypes.data_as(_lib._i32p), p["W0"].ctypes.data_as(_lib._i32p), C.addressof(tf), scale,
                max_size, p["box"].data_ptr(), p["offs"].ctypes.data_as(_lib._i64p), -1.5, 0.3, o[0].data_ptr(), o[1].data_ptr(),
                o[2].data_ptr(), o[3].data_ptr(), C.byref(t)), "detect_nms_batch_submit_u8")
            return t.value
        return f

    host_c = {}

    def arm_c(B, n_calls):
        """per-image getImages to the host, host padding, synchronous fp32 batch call"""
        for i in range(n_calls):
            p = packed[B][i % len(packed[B])]
            hw = [scaled[k][:2] for k in p["ks"]]
            H, W = max(h for h, _ in hw), max(w for _, w in hw)
            canvas = np.zeros((B, 3, H, W), np.float32)
            for j, k in enumerate(p["ks"]):
                h, w = hw[j]
                buf = host_c.setdefault((h, w), torch.empty((3, h, w), dtype=torch.float32).pin_memory())
                ctx.check(lib.mpn_get_images_u8(ctx.h, raw_pin[k].data_ptr(), sizes[k][0], sizes[k][1], C.addressof(tf), h, w, buf.data_ptr()),
                          "get_images_u8")
                canvas[j, :, :h, :w] = buf.numpy()
            sc = np.array([scaled[k][2] for k in p["ks"]], np.float32)
            w0, h0 = p["W0"].astype(np.float32), p["H0"].astype(np.float32)
            o = slot_out[0]
            ctx.check(lib.mpn_model_detect_nms_batch(
                mC.h, canvas.ctypes.data, B, H, W, p["box"].data_ptr(), p["offs"].ctypes.data_as(_lib._i64p), sc.ctypes.data,
                w0.ctypes.data, h0.ctypes.data, -1.5, 0.3, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr()),
                "detect_nms_batch")

    arms = {"A_single_submit_u8": lambda n: pipelined(submit_a, n, mA)}
    for B in batches:
        arms[f"B{B}_batch_submit_u8"] = (lambda B: lambda n: pipelined(submit_b(B), math.ceil(n / B), mB))(B)
        arms[f"C{B}_host_getimages_pad_batch"] = (lambda B: lambda n: arm_c(B, math.ceil(n / B)))(B)
    per_round = math.ceil(args.images / args.rounds / n_img) * n_img         # whole passes over the image list
    for name, fn in arms.items():
        for _ in range(args.warmup):
            fn(n_img)
    ctx.synchronize()
    secs = {k: 0.0 for k in arms}
    t_wall = time.time()
    for _ in range(args.rounds):
        for name, fn in arms.items():
            t0 = time.perf_counter()
            fn(per_round)
            ctx.synchronize()
            secs[name] += time.perf_counter() - t0
    n_timed = per_round * args.rounds
    raw_bytes = sum(3 * h * w for h, w in sizes) / n_img
    box_bytes = R * 16
    canvas_px = {B: sum(max(scaled[k][0] for k in p["ks"]) * max(scaled[k][1] for k in p["ks"]) * B for p in packed[B]) / n_img for B in batches}
    scaled_px = sum(h * w for h, w, _ in scaled) / n_img
    out = {"tool": "tools/bench_batch_raw.py", "workload": wk["name"], "config": args.config, "R_per_image": R,
           "image_sizes_H0xW0": [f"{h}x{w}" for h, w in COCO_SIZES], "scale": scale, "max_size": max_size, "images_per_arm": n_timed,
           "rounds": args.rounds, "gpu_before": info_before, "arms": {}}
    base = secs["A_single_submit_u8"]
    for name in arms:
        a = {"ms_per_image": round(secs[name] * 1e3 / n_timed, 4), "proposals_per_s": round(n_timed * R / secs[name]),
             "over_A": round(base / secs[name], 4)}
        if name.startswith("A"):
            a["h2d_bytes_per_image"] = round(raw_bytes + box_bytes)
        elif name.startswith("B"):
            B = int(name[1:].split("_")[0])
            a["h2d_bytes_per_image"] = round(raw_bytes + box_bytes)
            a["canvas_pixels_over_scaled_pixels"] = round(canvas_px[B] / scaled_px, 4)
        else:
            B = int(name[1:].split("_")[0])
            a["h2d_bytes_per_image"] = round(raw_bytes + 3 * 4 * canvas_px[B] + box_bytes)
            a["d2h_getimages_bytes_per_image"] = round(3 * 4 * scaled_px)
        out["arms"][name] = a
    out["wall_s"] = round(time.time() - t_wall, 1)

    # ---- correctness: every arm-B batch against mpn_model_detect_nms_batch on the mpn_get_images_batch_u8 canvas, byte for byte
    checked, identical = 0, 0
    for B in batches:
        for p in packed[B]:
            ims = [raws[k] for k in p["ks"]]
            bxs = [boxes[k] for k in p["ks"]]
            got = mB.detect_nms_wait(mB.detect_nms_batch_submit_u8(ims, bxs, spec.transformer, scale, max_size))
            canvas, scs, _ = ctx.get_images_batch_u8(ims, spec.transformer, scale, max_size)
            want = mB.detect_nms_batch(canvas, bxs, scs, [(im.shape[1], im.shape[0]) for im in ims])
            for (s1, b1, k1), (s2, b2, k2) in zip(got, want):
                checked += 1
                identical += int(s1.tobytes() == s2.tobytes() and b1.tobytes() == b2.tobytes() and len(k1) == len(k2)
                                 and all(np.array_equal(x, y) for x, y in zip(k1, k2)))
    out["check_B_vs_batch_on_canvas"] = f"{identical}/{checked} images byte-identical"
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))
    mA.close(); mB.close(); mC.close(); ctx.close()
    assert identical == checked, out["check_B_vs_batch_on_canvas"]


if __name__ == "__main__":
    main()
