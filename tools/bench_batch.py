"""Proposals/s of batched detection (mpn_model_detect_nms_batch_dev) against the single-image loop
(mpn_model_detect_nms_dev once per image), device-resident inputs, one model per arm on one stream, CUDA events.

For B in {1, 2, 4} images per call the two arms alternate in one process (rounds of single, batched, single, ...), each
warmed, each timing at least --images images; afterwards every image's batched result is compared with its single-image
result (scores / boxes normwise, keep lists exactly). Prints one JSON line with the card name, power limit and SM clock
read in the same run.

    python tools/bench_batch.py [--config vgg16_frcnn|multipathnet] [--images 240] [--rounds 4]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip().split(", ")
        return dict(zip(("name", "power_limit_w", "sm_mhz", "sm_max_mhz"), out))
    except Exception as e:                                  # the numbers are still printed, flagged as unattributed
        return {"error": str(e)}


def main():
    from bench import WORKLOADS
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="vgg16_frcnn", choices=["vgg16_frcnn", "multipathnet"])
    ap.add_argument("--batches", default="1,2,4")
    ap.add_argument("--images", type=int, default=240, help="images timed per arm and batch size (at least 200)")
    ap.add_argument("--rounds", type=int, default=4, help="alternations of the two arms")
    ap.add_argument("--warmup", type=int, default=3, help="warm-up calls per arm before the timed rounds")
    args = ap.parse_args()
    args.images = max(args.images, 200)

    import numpy as np
    import torch
    import multipathnet_b200 as mpn
    from multipathnet_b200 import models, workloads as wl

    wk = WORKLOADS[args.config]
    H, W, R, C = wk["H"], wk["W"], wk["R"], wk["C"]
    batches = [int(b) for b in args.batches.split(",")]
    Bmax = max(batches)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ctx = mpn.Context(0, own_stream=True)
    stream = torch.cuda.ExternalStream(ctx.stream_handle, device=dev)
    spec = getattr(models, wk["model"])(C, seed=1234, **wk["kw"])
    # one model per arm on the same stream: a model re-plans its trunk (and heads) whenever the image count changes, so
    # alternating the arms on one model would time the re-planning
    m1 = mpn.Model(ctx, spec, max_rois=R, max_h=H + 8, max_w=W)
    mb = mpn.Model(ctx, spec, max_rois=R * Bmax, max_h=H + 8, max_w=W)
    mkbox = wl.random_boxes if wk["boxes"] == "random" else wl.sharpmask_boxes
    imgs_h = np.stack([wl.transform(wl.raw_image(H, W, i), spec.transformer) for i in range(Bmax)])
    boxes_h = [mkbox(R, H, W, i) for i in range(Bmax)]
    imgs_d = torch.from_numpy(imgs_h).to(dev)
    boxes_d = torch.from_numpy(np.concatenate(boxes_h)).to(dev)
    # outputs: the single arm writes image i's results at the same places the batched call does
    sc = torch.empty((Bmax * R, C), dtype=torch.float32, device=dev)
    bb = torch.empty((Bmax * R, 4 * C), dtype=torch.float32, device=dev)
    kp = torch.empty(((C - 1) * Bmax * R,), dtype=torch.int32, device=dev)
    kc = torch.empty((Bmax, C - 1), dtype=torch.int32, device=dev)
    img_bytes = 3 * H * W * 4

    def single(B):
        for i in range(B):
            m1.detect_nms_dev(imgs_d.data_ptr() + i * img_bytes, H, W, boxes_d[i * R:(i + 1) * R], R, 1.0, W, H, -1.5, 0.3,
                             sc[i * R:], bb[i * R:], kp[(C - 1) * i * R:], kc[i])

    def batched(B):
        mb.detect_nms_batch_dev(imgs_d, B, H, W, boxes_d, [R] * B, [1.0] * B, [(W, H)] * B, -1.5, 0.3, sc, bb, kp, kc)

    def results(B):
        torch.cuda.synchronize(dev)
        s, b, k, c = sc[:B * R].cpu().numpy(), bb[:B * R].cpu().numpy(), kp[:(C - 1) * B * R].cpu().numpy(), kc[:B].cpu().numpy()
        return [(s[i * R:(i + 1) * R].copy(), b[i * R:(i + 1) * R].copy(),
                 [k[(C - 1) * i * R + j * R:(C - 1) * i * R + j * R + c[i, j]].copy() for j in range(C - 1)]) for i in range(B)]

    def rel(a, b):
        return float(np.abs(a.astype(np.float64) - b).max() / max(np.abs(b).max(), 1e-30))

    out = {"tool": "tools/bench_batch.py", "workload": wk["name"], "config": args.config, "R_per_image": R, "H": H, "W": W,
           "gpu": gpu_info(), "arms": {}}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t_wall = time.time()
    with torch.cuda.stream(stream):
        for B in batches:
            calls = math.ceil(args.images / (B * args.rounds))          # per round and arm
            for _ in range(args.warmup):
                single(B); batched(B)
            torch.cuda.synchronize(dev)
            ms = {"single": 0.0, "batched": 0.0}
            for _ in range(args.rounds):
                for arm, fn in (("single", single), ("batched", batched)):
                    ev[0].record(stream)
                    for _ in range(calls):
                        fn(B)
                    ev[1].record(stream)
                    ev[1].synchronize()
                    ms[arm] += ev[0].elapsed_time(ev[1])
            ctx.synchronize()
            n_img = calls * args.rounds * B
            single(B); ref = results(B)
            batched(B); got = results(B)
            ctx.synchronize()
            es = max(rel(g[0], r[0]) for g, r in zip(got, ref))
            eb = max(rel(g[1], r[1]) for g, r in zip(got, ref))
            same_keeps = sum(all(np.array_equal(x, y) for x, y in zip(g[2], r[2])) for g, r in zip(got, ref))
            arm = {"images_per_arm": n_img}
            for a in ("single", "batched"):
                arm[f"{a}_ms_per_image"] = round(ms[a] / n_img, 4)
                arm[f"{a}_proposals_per_s"] = round(n_img * R / (ms[a] / 1e3))
            arm["batched_over_single"] = round(ms["single"] / ms["batched"], 4)
            arm["agree"] = {"scores_rel_err_max": es, "bboxes_rel_err_max": eb, "images_with_identical_keep_lists": f"{same_keeps}/{B}"}
            out["arms"][f"B{B}"] = arm
            assert es < 1e-3 and eb < 1e-3, (B, es, eb)
    out["wall_s"] = round(time.time() - t_wall, 1)
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))
    m1.close(); mb.close(); ctx.close()


if __name__ == "__main__":
    main()
