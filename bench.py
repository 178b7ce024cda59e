#!/usr/bin/env python
"""bench.py — proposals/sec of the detection forward hot path on B200.

Workload (BASELINE.json configs[1], the config `metric` is quoted on): VGG-16 Fast R-CNN, one
600x800 image + 1000 random proposals per step, C=21, fp32-faithful (bf16x3 split on tcgen05, fp32
accumulate; fc6 / fc7 two fp16 products). A "step" = ONE image through trunk -> fused ROI pooling -> fc6/fc7/cls/bbox -> BBoxNorm
-> decode + clamp -> softmax -> per-class gather -> batched NMS (20 classes), i.e. everything
ImageDetect:detect + Tester_FRCNN:testOne do per image.

  python bench.py [--gpus N --steps K --warmup W]          our arm (N>1: launched by torchrun, one rank/GPU)
  python bench.py --impl reference [...]                    the reference's CPU path on the host cores

`--replicas K` (default 2): K model replicas per GPU, each on its own mpn_ctx / stream, images dealt round-robin (the
            reference's one-replica-per-donkey-thread runner, test_runner.lua:55-66, with K threads per GPU): the kernels of one
            replica fill the layer-boundary / NMS-chain bubbles of the others. `ms_per_image_p50` stays the latency of ONE image
            on ONE replica.
`value`   : proposals/s with image+proposals already resident in HBM (mpn_model_detect_nms_dev).
`e2e`     : proposals/s through the host-buffer C-ABI (mpn_model_detect_nms_submit/_wait, two images in flight per
            model: pinned host image and boxes copied H2D, scores/boxes/keep lists copied D2H every step, inside the
            timed region); `e2e.sync_value` is the same through one blocking mpn_model_detect_nms call per image.
`roofline`: the tcgen05 conv/GEMM kernels (dominant, tensor-bound): algorithmic FLOPs of the step divided
            by the CUDA-event time of those launches, against MEASURED_PEAKS.json bf16 peak. NOTE the
            engine issues 3 bf16 MMAs per algorithmic MAC (bf16x3 fp32 emulation); `issued_frac` = 3x.
`cpu_baseline`: the CPU oracle port (torch-CPU fp32 dense layers + C restatement + literal nms.c) timed
            on the box's host cores on one image of the same workload (rank 0, N=1 only).
`--dump-outputs DIR`: after the run, rank 0 writes what the last step of the `value` loop returned, as float32 .npy files:
            scores (R x C), bboxes (R x 4C), keep ((C-1) x R proposal rows in NMS emission order, -1 past keep_count),
            keep_count (C-1) and detections (the gathered records of every rank's last image, N x MPN_REC_FLOATS). The inputs
            are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs[1..3] (configs[4], the NMS sweep, is --config nms_sweep). The default, and the line the driver
# records, is configs[1]; the others are extra evidence for SURVEY 8 rows a6/a7/a9/a11/a13.
WORKLOADS = {
    "vgg16_frcnn": dict(H=600, W=800, R=1000, C=21, boxes="random", model="vgg16_fast_rcnn", kw={},
                        name="VGG-16 Fast R-CNN, 600x800 image, 1000 ROIs/image, C=21, detect+NMS (BASELINE configs[1])"),
    "multipathnet": dict(H=600, W=800, R=1000, C=81, boxes="sharpmask", model="vgg16_multipathnet", kw={},
                         name="VGG-16 MultiPathNet 4-foveal + het tower, skip-concat, 600x800, 1000 SharpMask-shaped ROIs, C=81 (BASELINE configs[2])"),
    "resnet50": dict(H=800, W=1000, R=2000, C=81, boxes="sharpmask", model="resnet50_fast_rcnn", kw={"integral_k": 6},
                     name="ResNet-50 Fast R-CNN + integral-loss head (K=6), 800x1000, 2000 ROIs, C=81 (BASELINE configs[3], per-GPU shard)"),
}
H, W, R, C = 600, 800, 1000, 21
WORKLOAD = WORKLOADS["vgg16_frcnn"]["name"]


def traffic_from_profiles(config):
    """DRAM bytes (read + write) per launch of the dominant launch of the dominant kernel family, from the committed
    `ncu --set full` capture (profiles/traffic.json); None when no capture of this config is committed."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")) as f:
            t = json.load(f).get(config)
        return None if t is None else {"dram_bytes_per_launch": t["dram_bytes_per_launch"], "launch": t["dominant_launch"],
                                       "algorithmic_bytes_per_launch": t["algorithmic_bytes_per_launch"], "source": t["source"]}
    except (OSError, ValueError, KeyError):
        return None


def roi_algorithmic_bytes(spec, shapes, R):
    """SURVEY 8d: each pooled feature map once + R*5*4 + sum over towers of the pooled output (fp32-equivalent bytes)."""
    used = {}
    out = 0
    for t in spec.towers:
        ct = 0
        for slot, _ in t.levels:
            used[slot] = shapes[slot]
            ct += shapes[slot][0]
        out += R * ct * t.pooled_h * t.pooled_w * 4
    return sum(c * h * w * 4 for (c, h, w) in used.values()) + R * 5 * 4 + out


def trunk_shapes(spec, H, W):
    from multipathnet_b200.models import _pool_out
    shp = {0: (3, H, W)}
    for L in spec.trunk_layers:
        c, h, w = shp[L.in_slot]
        if L.kind == 1:
            shp[L.out_slot] = (L.cout, (h + 2 * L.pad - L.kh) // L.stride + 1, (w + 2 * L.pad - L.kw) // L.stride + 1)
        else:
            shp[L.out_slot] = (c, _pool_out(h, L.kh, L.stride, L.pad, L.ceil_mode), _pool_out(w, L.kw, L.stride, L.pad, L.ceil_mode))
    return shp


def run_nms_sweep(args, rank, world, local_rank):
    """BASELINE configs[4]: "NMS + BBoxNorm sweep 1k-50k boxes x 80 classes, 1/2/4/8 B200 vs nms.c CPU".
    One unit = ONE image worth of post-network work for N proposals and 80 foreground classes: nn.BBoxNorm + convertFrom +
    clamp of the N x 4*81 deltas, per-class gather, NMS at 0.3 (mpn_post_detect_dev). The 80 classes shard over the ranks
    (strong scaling, no collective: every rank owns whole classes). Beside every N the LITERAL nms.c (oracle/_ref, built from
    /root/reference/nms.c) is timed on the GPU's own decoded boxes for a bounded number of classes — single thread, and one
    thread per class over the host cores — and its keep lists are compared with the GPU's (bit-exact) on the way."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    import numpy as np
    import torch
    import torch.distributed as dist
    import multipathnet_b200 as mpn
    from multipathnet_b200 import workloads as wl
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ctx = mpn.Context(local_rank)
    NC, CC = 80, 81
    c0 = 1 + (NC * rank) // world; c1 = 1 + (NC * (rank + 1)) // world      # this rank's foreground classes [c0, c1)
    ncls = c1 - c0
    mean = np.zeros(4, np.float32); std = np.float32([0.1, 0.1, 0.2, 0.2])
    H0, W0 = 600.0, 800.0
    res = {}
    lit = None
    if rank == 0:
        from oracle import ref as O
        O.build()
        lit = O if O.ref_available() else None
    for N in (1000, 2000, 5000, 10000, 20000, 50000):
        rng = np.random.default_rng(5 + N)                         # same data on every rank: the class range is what differs
        boxes = wl.random_boxes(N, int(H0), int(W0), 5 + N, wmax=0.4 * W0, hmax=0.4 * H0)
        deltas = (rng.standard_normal((N, 4 * CC)) * 0.5).astype(np.float32)
        # distinct scores inside every class (as workloads.nms_sweep_boxes: ties are a parity-test case, not a bench case)
        scores = ((rng.permuted(np.tile(np.arange(N, dtype=np.float64), (CC, 1)), axis=1).T + rng.random((N, CC)) * 0.5) / N).astype(np.float32)
        sc_d, dl_d, bx_d = (torch.from_numpy(x).to(dev) for x in (scores, deltas, boxes))
        bb_d = torch.empty((N, 4 * CC), dtype=torch.float32, device=dev)
        keep = torch.empty((ncls, N), dtype=torch.int32, device=dev)
        cnt = torch.empty((ncls,), dtype=torch.int32, device=dev)

        def call():
            ctx.check(ctx.lib.mpn_post_detect_dev(ctx.h, sc_d.data_ptr(), dl_d.data_ptr(), bx_d.data_ptr(), N, CC, mean.ctypes.data, std.ctypes.data,
                                                  W0, H0, -1.5, 0.3, c0, c1, bb_d.data_ptr(), keep.data_ptr(), cnt.data_ptr()), "mpn_post_detect_dev")
        for _ in range(3):
            call()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10 if N <= 10000 else 3
        e0.record()
        for _ in range(reps):
            call()
        e1.record(); torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                # the image is done when the slowest class range is
        ms = float(t.item())
        row = {"classes_per_rank": ncls, "ms_per_image": ms, "boxes_per_s": NC * N / (ms / 1e3), "kept_mean": float(cnt.float().mean().item())}
        if rank == 0 and lit is not None and not args.no_cpu_baseline:
            bb = bb_d.cpu().numpy(); kp = keep.cpu().numpy(); ct = cnt.cpu().numpy()
            n_cpu = 8 if N <= 5000 else (4 if N <= 20000 else 2)       # bounded CPU sample: classes timed single-threaded
            sbs = [np.ascontiguousarray(np.concatenate([bb[:, 4 * j:4 * j + 4], scores[:, j:j + 1]], 1), np.float32) for j in range(c0, c0 + min(n_cpu, ncls))]
            t0 = time.perf_counter()
            rows = [lit.ref_nms_rows(sb, 0.3) for sb in sbs]
            t_single = (time.perf_counter() - t0) / len(sbs)
            ok = all(np.array_equal(sb[kp[i, :ct[i]]], r) for i, (sb, r) in enumerate(zip(sbs, rows)))
            row["cpu_nms_c"] = {"kind": "reference (literal nms.c)", "classes_timed": len(sbs), "s_per_class_1thread": t_single,
                                "ms_per_image_1thread": 1e3 * t_single * NC, "keeps_equal_gpu": bool(ok)}
            if N <= 10000:                                            # one thread per class over the host cores (ctypes drops the GIL)
                thr = min(os.cpu_count() or 1, NC)
                allsb = [sbs[i % len(sbs)] for i in range(NC)]
                with ThreadPoolExecutor(thr) as ex:
                    list(ex.map(lambda sb: lit.ref_nms_rows(sb, 0.3), allsb[:thr]))        # warm the pool
                    t0 = time.perf_counter()
                    list(ex.map(lambda sb: lit.ref_nms_rows(sb, 0.3), allsb))
                    row["cpu_nms_c"].update({"threads": thr, "ms_per_image_thread_per_class": 1e3 * (time.perf_counter() - t0)})
            row["speedup_vs_nms_c_1thread"] = row["cpu_nms_c"]["ms_per_image_1thread"] / ms
        res[N] = row
    if rank == 0:
        print(json.dumps({"metric": "NMS + BBoxNorm boxes/sec (80-class sweep)", "value": res[10000]["boxes_per_s"], "unit": "boxes/s", "n_gpus": world,
                          "higher_is_better": True, "scaling": "strong (the 80 classes shard over the ranks, no collective)", "dtype": "fp32", "data": "synthetic",
                          "config": {"workload": "BBoxNorm + decode + clamp + per-class gather + NMS, N boxes x 80 classes, thr 0.3 (BASELINE configs[4])"},
                          "host_cpus": os.cpu_count(), "sweep": res}))
    if world > 1:
        dist.destroy_process_group()


def bench_config(world, replicas=2):
    """`config` of the JSON line: ONE dict for both arms (ours / --impl reference) so the driver's same-config check holds;
    arm-specific facts (CPU thread count, ...) live in other keys of the line."""
    return {"workload": WORKLOAD,
            "replicas_per_gpu": f"GPU arm: {replicas} model replica(s) per GPU, each on its own stream, images dealt round-robin (test_runner.lua:55-66 with {replicas} donkey thread(s) per GPU); CPU arm: n/a",
            "parallelism": (f"images sharded over {world} rank(s), one NCCL all-gather of the packed top-100 detection records at the end"
                            if world > 1 else "single GPU"),
            "l2": "GPU arm: inputs larger than L2, each step streams 0.55 GB of weights + ~1 GB of activations (L2 = 126 MB); CPU arm: n/a",
            "nms_thr": 0.3, "score_thresh": -1.5, "roi_variant": 2, "top_k_per_image": 100}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            self.proc.kill(); out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pick_cpu_threads(torch):
    """The CPU legs should be the host at its best, and oneDNN / MKL on a many-core box are not fastest with every
    logical CPU on this batch-1 workload (128 threads were 2x slower than 8 on another host): time a proxy of the two
    dominant layers (conv3_2, fc6) at a few thread counts and keep the fastest. Returns (threads, {threads: seconds})."""
    import torch.nn.functional as F
    n = os.cpu_count() or 1
    cands = sorted({max(min(n, 4), n >> s) for s in range(6)}, reverse=True)       # nproc, /2, /4, ... /32 (never below 4)
    x, w = torch.randn(1, 256, 150, 200), torch.randn(256, 256, 3, 3)
    a, b = torch.randn(1000, 25088), torch.randn(4096, 25088)
    tried = {}
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            F.conv2d(x, w, padding=1); F.linear(a[:64], b)                 # primitive creation / first touch
            t0 = time.perf_counter()
            F.conv2d(x, w, padding=1); F.linear(a, b)
            tried[c] = round(time.perf_counter() - t0, 3)
    best = min(tried, key=tried.get)
    torch.set_num_threads(best)
    return best, tried


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores. Torch-7 cannot run
    here, so the nn graph is the oracle port (PyTorch-CPU fp32 + C restatement) and NMS is the LITERAL nms.c."""
    if rank != 0:
        return
    import numpy as np
    import torch
    from multipathnet_b200 import models, workloads as wl
    from oracle import graphs as G, ref as O
    O.build()
    cores, tried = pick_cpu_threads(torch)
    spec = models.vgg16_fast_rcnn(C, seed=1234)
    use_lit = O.ref_available()

    def nms_fn(sb, thr):          # literal reference nms.c when its build travelled, timing-equivalent restatement otherwise
        if use_lit:
            return np.arange(len(O.ref_nms_rows(sb, thr)))
        return O.nms(sb, thr)

    def step(i):
        img = wl.transform(wl.raw_image(H, W, 100 + i), spec.transformer)
        boxes = wl.random_boxes(R, H, W, 100 + i)
        t0 = time.perf_counter()
        G.test_one(spec, img, boxes, 1.0, W, H, -1.5, 0.3, nms_fn=nms_fn)
        return time.perf_counter() - t0

    # one full image costs about a second on the host cores: one warm-up image whatever --warmup says, then --steps images
    t_first = step(0) if args.warmup > 0 else None
    ts = [step(1 + i) for i in range(args.steps)]
    total = sum(ts)
    val = R * len(ts) / total
    line = {"impl": "reference", "metric": "proposals/sec", "value": val, "unit": "proposals/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "steps_timed": len(ts), "warmup_run": 1 if t_first is not None else 0,
            "ms_per_step": 1e3 * total / len(ts), "ms_per_image_p50": 1e3 * statistics.median(ts),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": bench_config(args.gpus, args.replicas),
            "host": {"arm": "CPU only", "threads": cores, "logical_cpus": os.cpu_count(), "thread_count_proxy_s": tried},
            "cpu_baseline": {"value": val, "unit": "proposals/s", "cores": cores,
                             "kind": "port", "sample": f"{len(ts)} full images (1000 ROIs each); dense layers PyTorch-CPU fp32, "
                                                       f"ROI/decode C restatement, NMS {'literal nms.c' if use_lit else 'nms.c restatement'}"},
            "e2e": {"value": val, "unit": "proposals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 3 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 5; 1 with --impl reference)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--replicas", type=int, default=2, help="model replicas per GPU, each on its own mpn_ctx / stream (images dealt round-robin)")
    ap.add_argument("--config", default="vgg16_frcnn", choices=list(WORKLOADS) + ["nms_sweep"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "nms_sweep"):
        ap.error("--dump-outputs writes the outputs of the GPU arm's detection workloads")
    if args.steps is None:
        args.steps = 3 if args.impl == "reference" else 200       # the CPU arm's defaults are sized for a run of a few minutes
    if args.warmup is None:
        args.warmup = 1 if args.impl == "reference" else 5
    global H, W, R, C, WORKLOAD
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    if args.config == "nms_sweep":
        return run_nms_sweep(args, rank, world, local_rank)
    wk = WORKLOADS[args.config]
    H, W, R, C, WORKLOAD = wk["H"], wk["W"], wk["R"], wk["C"], wk["name"]

    import numpy as np
    import torch
    import torch.distributed as dist
    import multipathnet_b200 as mpn
    from multipathnet_b200 import models, workloads as wl, dist as mdist

    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    # K model replicas on this GPU, each on its own mpn_ctx / non-blocking stream (multipathnet_b200/replicas.py): the kernels of
    # one replica fill the layer-boundary and NMS-chain bubbles of the others. Images are dealt round-robin.
    K = max(1, args.replicas)
    spec = getattr(models, wk["model"])(C, seed=1234, **wk["kw"])
    reps = mpn.ModelReplicas(local_rank, spec, K, max_rois=max(R, 1024), max_h=H + 8, max_w=W)
    ctx, model = reps.ctxs[0], reps.models[0]          # replica 0: p50 loop, blocking-call leg, profiling pass, the collective
    streams = [torch.cuda.ExternalStream(c.stream_handle, device=dev) for c in reps.ctxs]
    stream = streams[0]

    # ---- synthetic inputs: a small rotating set of distinct images/proposals per rank (seeded by rank)
    NIMG = 4
    imgs_h = [wl.transform(wl.raw_image(H, W, 1000 * rank + i), spec.transformer) for i in range(NIMG)]
    mkbox = wl.random_boxes if wk["boxes"] == "random" else wl.sharpmask_boxes
    boxes_h = [mkbox(R, H, W, 1000 * rank + i) for i in range(NIMG)]
    imgs_d = [torch.from_numpy(x).to(dev) for x in imgs_h]
    boxes_d = [torch.from_numpy(x).to(dev) for x in boxes_h]
    outs_d = [(torch.empty((R, C), dtype=torch.float32, device=dev), torch.empty((R, 4 * C), dtype=torch.float32, device=dev),
               torch.empty((C - 1, R), dtype=torch.int32, device=dev), torch.empty((C - 1,), dtype=torch.int32, device=dev)) for _ in range(K)]

    def step_dev(i):
        k = i % NIMG
        reps.models[i % K].detect_nms_dev(imgs_d[k], H, W, boxes_d[k], R, 1.0, W, H, -1.5, 0.3, *outs_d[i % K])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- the path's ONE collective, issued by the library (mpn_dist_*, csrc/dist.cu): every detect+NMS pass also packs the
    # image's record (keep_top_k 100 + fixed-size layout, csrc/post.cu) into its replica's slice of `records_d`; after the last
    # image replica 0's stream waits for the others (mpn_ctx_wait_ctx) and ONE ncclAllGather ships K x PER x MPN_REC_FLOATS
    # floats per rank (image i = record [i mod K, i div K]). At N = 1 the same calls run (the gather degenerates to a copy).
    REC = mpn.MPN_REC_FLOATS
    PER = (max(args.steps, args.warmup, 3) + K - 1) // K
    records_d = torch.zeros((K, PER, REC), dtype=torch.float32, device=dev)
    gathered_d = torch.zeros((world, K, PER, REC), dtype=torch.float32, device=dev)
    gathered_h = torch.empty((world, K, PER, REC), dtype=torch.float32).pin_memory()
    if world > 1:
        idt = torch.zeros(mpn.MPN_DIST_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(ctx.dist_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        ctx.dist_init(bytes(idt.cpu().numpy().tobytes()), rank, world)

    def sinks_on():
        for k, m in enumerate(reps.models):
            m.set_detection_sink(records_d[k], PER, 100)      # (re)sets the record count of the replica

    def sinks_off():
        for m in reps.models:
            m.set_detection_sink(None, 0, 100)

    def gather_dev():
        reps.join()
        ctx.dist_all_gather_dev(records_d, K * PER * REC, gathered_d)

    # warm-up: the exact sequence of the timed region (steps with the sinks on, then the join + the collective: the first NCCL
    # call on a communicator sets up its channels — tens of ms that are not part of a steady-state run)
    barrier()
    sinks_on()
    for i in range(max(args.warmup, 2 * K)):
        step_dev(i)
    gather_dev()
    barrier()

    # ---- timed region 1: device-resident throughput (`value`)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    sinks_on()
    launches0 = reps.launch_count
    barrier()
    ev0, ev_loop, end_ev = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    ev0.record(stream)                                               # every replica stream is idle here
    for i in range(args.steps):
        step_dev(i)
    reps.join()
    ev_loop.record(stream)                                           # this rank's K steps are done on every replica
    ctx.dist_all_gather_dev(records_d, K * PER * REC, gathered_d)    # THE collective of the path, inside the timed region
    end_ev.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev0.elapsed_time(end_ev)
    collective_ms = ev_loop.elapsed_time(end_ev)                     # the all-gather incl. the wait for the slowest rank
    launches = reps.launch_count - launches0
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    loop_ms = ev0.elapsed_time(ev_loop)                               # this rank's K steps alone, before the collective
    per_rank_ms = [loop_ms / args.steps]
    if world > 1:
        tl_ = torch.tensor([loop_ms], dtype=torch.float64, device=dev)
        allt = [torch.empty_like(tl_) for _ in range(world)]
        dist.all_gather(allt, tl_)
        # diagnostics: each rank's own loop time (the job total also contains the wait for the slowest GPU in the
        # one all-gather: GPUs of one box differ by several % under the power cap)
        per_rank_ms = [float(x.item()) / args.steps for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * R * args.steps / (total_ms_max / 1e3)
    # what was gathered: every rank's records, real detections (count field = rows kept by keep_top_k, <= MPN_MAX_DET)
    g = gathered_d.cpu().numpy()
    det_counts = np.array([[g[r, i % K, i // K, 0] for i in range(args.steps)] for r in range(world)])
    assert np.array_equal(g[rank], records_d.cpu().numpy()), "gathered records differ from this rank's own"
    assert det_counts.min() >= 1 and det_counts.max() <= mpn.MPN_MAX_DET, "gathered detection records are empty or overflowed"
    dump = None
    if args.dump_outputs and rank == 0:             # the last step's buffers, before the loops below overwrite them
        last = args.steps - 1
        sc, bb, kp, ct = (x.cpu().numpy() for x in outs_d[last % K])
        dump = {"scores": sc, "bboxes": bb, "keep": np.where(np.arange(R) < ct[:, None], kp, -1), "keep_count": ct,
                "detections": g[:, last % K, last // K]}

    # ---- p50 latency of ONE image on ONE replica over --steps images (SURVEY 8d)
    sinks_off()
    P50_STEPS, P50_WARM = args.steps, 20

    def step_one(i):
        k = i % NIMG
        model.detect_nms_dev(imgs_d[k], H, W, boxes_d[k], R, 1.0, W, H, -1.5, 0.3, *outs_d[0])

    for i in range(P50_WARM):
        step_one(i)
    evp = [torch.cuda.Event(enable_timing=True) for _ in range(P50_STEPS + 1)]
    evp[0].record(stream)
    for i in range(P50_STEPS):
        step_one(i)
        evp[i + 1].record(stream)
    torch.cuda.synchronize(dev)
    per_step = [evp[i].elapsed_time(evp[i + 1]) for i in range(P50_STEPS)]

    # ---- timed region 2: end to end through the host-buffer C-ABI call (`e2e`)
    pin_img = [torch.from_numpy(x).pin_memory() for x in imgs_h]
    pin_box = [torch.from_numpy(x).pin_memory() for x in boxes_h]
    sc_h = torch.empty((R, C), dtype=torch.float32).pin_memory()
    bb_h = torch.empty((R, 4 * C), dtype=torch.float32).pin_memory()
    kp_h = torch.empty((C - 1, R), dtype=torch.int32).pin_memory()
    ct_h = torch.empty((C - 1,), dtype=torch.int32).pin_memory()
    lib = ctx.lib

    def step_e2e(i):
        k = i % NIMG
        ctx.check(lib.mpn_model_detect_nms(model.h, pin_img[k].data_ptr(), H, W, pin_box[k].data_ptr(), R, 1.0, float(W), float(H),
                                           -1.5, 0.3, sc_h.data_ptr(), bb_h.data_ptr(), kp_h.data_ptr(), ct_h.data_ptr()), "detect_nms")

    for i in range(3):
        step_e2e(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(i)
    torch.cuda.synchronize(dev)
    e2e_sync_s = time.perf_counter() - t0

    # pipelined public API (two images in flight per replica, like the reference's one image per donkey thread): every step
    # still copies its own inputs host->device and its own results device->host inside the timed region
    outs = [[(torch.empty((R, C), dtype=torch.float32).pin_memory(), torch.empty((R, 4 * C), dtype=torch.float32).pin_memory(),
              torch.empty((C - 1, R), dtype=torch.int32).pin_memory(), torch.empty((C - 1,), dtype=torch.int32).pin_memory()) for _ in range(2)]
            for _ in range(K)]
    import ctypes as _C
    from collections import deque

    def run_pipelined(n, submit_fn):
        """deal image i to replica i mod K; at most two submissions in flight per replica (the API's limit)"""
        pend = [deque() for _ in range(K)]
        for i in range(n):
            rk = i % K
            if len(pend[rk]) == 2:
                reps.ctxs[rk].check(lib.mpn_model_detect_nms_wait(reps.models[rk].h, pend[rk].popleft()), "detect_nms_wait")
            pend[rk].append(submit_fn(i, rk, outs[rk][(i // K) & 1]))
        for rk in range(K):
            while pend[rk]:
                reps.ctxs[rk].check(lib.mpn_model_detect_nms_wait(reps.models[rk].h, pend[rk].popleft()), "detect_nms_wait")

    def submit(i, rk, o):
        k = i % NIMG
        t = _C.c_int32(-1)
        reps.ctxs[rk].check(lib.mpn_model_detect_nms_submit(reps.models[rk].h, pin_img[k].data_ptr(), H, W, pin_box[k].data_ptr(), R, 1.0, float(W), float(H),
                                                            -1.5, 0.3, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), _C.byref(t)),
                            "detect_nms_submit")
        return t.value

    def gather_host():       # the join + the collective + the gathered records to (pinned) host memory, synchronous
        reps.join()
        ctx.check(lib.mpn_dist_all_gather(ctx.h, records_d.data_ptr(), K * PER * REC, gathered_h.data_ptr()), "mpn_dist_all_gather")

    sinks_on()
    run_pipelined(max(3, 2 * K), submit)
    gather_host()
    barrier()
    sinks_on()
    t0 = time.perf_counter()
    run_pipelined(args.steps, submit)
    gather_host()
    e2e_s = time.perf_counter() - t0
    sinks_off()
    t = torch.tensor([e2e_s, e2e_sync_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * R * args.steps / float(t[0].item())
    e2e_sync_value = world * R * args.steps / float(t[1].item())
    # ---- same pipeline fed with the RAW decoder bytes (SURVEY 8f-1): a 480 x 640 x 3 uint8 image per step, getImages (transformer +
    # im_scale rule + image.scale to 600 x 800) on the device in front of the trunk; boxes in original-image coordinates
    e2e_raw = None
    if args.config == "vgg16_frcnn":
        H0r, W0r = (H * 4) // 5, (W * 4) // 5                      # 480 x 640 -> scale 600 / max 1000 gives exactly H x W
        rng = np.random.default_rng(77 + rank)
        raw_pin = [torch.from_numpy(rng.integers(0, 256, (H0r, W0r, 3), dtype=np.uint8)).pin_memory() for _ in range(NIMG)]
        rbox_pin = [torch.from_numpy(wl.random_boxes(R, H0r, W0r, 2000 * rank + i)).pin_memory() for i in range(NIMG)]
        from multipathnet_b200._lib import CImageTransform
        tfm = CImageTransform.of(spec.transformer)

        def submit_raw(i, rk, o):
            k = i % NIMG
            t = _C.c_int32(-1)
            reps.ctxs[rk].check(lib.mpn_model_detect_nms_submit_u8(reps.models[rk].h, raw_pin[k].data_ptr(), H0r, W0r, _C.addressof(tfm), 600.0, 1000.0,
                                                                   rbox_pin[k].data_ptr(), R, -1.5, 0.3, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(),
                                                                   o[3].data_ptr(), _C.byref(t)), "detect_nms_submit_u8")
            return t.value

        run_pipelined(max(3, 2 * K), submit_raw)
        barrier()
        t0 = time.perf_counter()
        run_pipelined(args.steps, submit_raw)
        raw_s = time.perf_counter() - t0
        tr = torch.tensor([raw_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tr, op=dist.ReduceOp.MAX)
        e2e_raw = {"value": world * R * args.steps / float(tr.item()), "unit": "proposals/s", "h2d_bytes_per_step": H0r * W0r * 3 + R * 4 * 4,
                   "api": "mpn_model_detect_nms_submit_u8 / _wait: raw 480x640x3 uint8 image in, getImages on the device (get_images_kernel)"}
    h2d = 3 * H * W * 4 + R * 4 * 4
    d2h = R * C * 4 + R * 4 * C * 4 + (C - 1) * R * 4 + (C - 1) * 4 + world * REC * 4      # + this image's share of the gathered records

    # ---- per-kernel-category CUDA-event timing of the same steps (roofline numerators)
    # (ONE replica, in order: the events between the launches serialise them, so the categories describe the kernels themselves)
    torch.cuda.synchronize(dev)
    ctx.profile_begin()
    for i in range(args.steps):
        step_one(i)
    prof = ctx.profile_end()
    L0 = spec.trunk_layers[0]
    first_flops = 2.0 * L0.cin * L0.cout * L0.kh * L0.kw * ((H + 2 * L0.pad - L0.kh) // L0.stride + 1) * ((W + 2 * L0.pad - L0.kw) // L0.stride + 1)
    tflop_step = (models.trunk_flops(spec, H, W) - first_flops + models.head_flops_per_roi(spec) * R) / 1e12   # tcgen05 layers only
    tc_ms_step = prof["conv_gemm_tc"][0] / args.steps
    peak_tf, hbm_gbs, peak_src = load_peaks()
    achieved = tflop_step / (tc_ms_step / 1e3) if tc_ms_step > 0 else 0.0
    n_tc = prof["conv_gemm_tc"][1] // args.steps
    # issued MMA work: three bf16 products per algorithmic MAC, two fp16 products in the "w16" Linears (fc6 / fc7 of single-tower graphs)
    w16_on = os.environ.get("MPN_FC_W16", "") != "0"
    tflop_w16 = (models.w16_flops_per_roi(spec) * R / 1e12) if w16_on else 0.0
    issued = (3.0 * (tflop_step - tflop_w16) + 2.0 * tflop_w16) / (tc_ms_step / 1e3) if tc_ms_step > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "conv3x3_tc_kernel / conv_gemm_tc_kernel<BN> (tcgen05 implicit-GEMM, %d launches/step)" % n_tc,
                "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf if peak_tf else None,
                "issued_frac": issued / peak_tf if peak_tf else None, "issued_tflops": issued,
                "products_per_mac": {"three_bf16": tflop_step - tflop_w16, "two_fp16_w16": tflop_w16, "unit": "algorithmic TFLOP/step"},
                "peak_source": peak_src,
                "traffic": (traffic_from_profiles(args.config) or {}).get("dram_bytes_per_launch"),   # bytes, or None
                "traffic_detail": traffic_from_profiles(args.config),
                "algorithmic_tflop_per_step": tflop_step, "kernel_ms_per_step": tc_ms_step,
                "by_category_ms_per_step": {k: v[0] / args.steps for k, v in prof.items()}}
    # ROI pooling (HBM-bound secondary kernel): algorithmic bytes = feature map once + rois + pooled output (SURVEY 8d)
    roi_bytes = roi_algorithmic_bytes(spec, trunk_shapes(spec, H, W), R)
    roi_ms = prof["roi_pool"][0] / args.steps
    roofline["roi_pool"] = {"bound": "hbm", "achieved": roi_bytes / (roi_ms / 1e3) / 1e9 if roi_ms > 0 else None, "peak": hbm_gbs,
                            "unit": "GB/s", "frac": (roi_bytes / (roi_ms / 1e3) / 1e9 / hbm_gbs) if roi_ms > 0 and hbm_gbs else None,
                            "algorithmic_bytes": roi_bytes}

    line = {"metric": "proposals/sec", "value": value, "unit": "proposals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "ms_per_image_p50": statistics.median(per_step), "p50_steps": P50_STEPS,
            "p50_note": "latency of one image on one replica (in-order loop); ms_per_step = wall / images with %d replica(s) overlapped" % K,
            "replicas_per_gpu": K,
            "per_rank_loop_ms_per_step": per_rank_ms,
            "collective": {"api": "mpn_dist_all_gather_dev (ncclAllGather issued by libmpn_b200.so on the ctx stream)" if world > 1 else "world of 1: device copy",
                           "ms": collective_ms, "bytes_per_rank": K * PER * REC * 4, "in_timed_region": True, "in_e2e_region": True,
                           "detections_per_image_mean": float(det_counts.mean())},
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32 (tcgen05 split emulation, fp32 accumulate: 3 bf16 products per MAC" + (", 2 fp16 products in fc6/fc7)" if tflop_w16 > 0 else ")"), "data": "synthetic",
            "config": bench_config(world, K),
            "e2e": {"value": e2e_value, "unit": "proposals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "mpn_model_detect_nms_submit / _wait (pinned host buffers, 2 images in flight per replica) + mpn_ctx_wait_ctx + mpn_dist_all_gather (records to host) at the end",
                    "sync_value": e2e_sync_value, "sync_api": "mpn_model_detect_nms (host buffers, one blocking call per image)"},
            "e2e_raw": e2e_raw,
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline}

    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.config == "vgg16_frcnn":
        # bounded CPU sample: ONE full image (1000 ROIs) through the oracle port on all host cores
        from oracle import graphs as G, ref as O
        O.build()
        cores, tried = pick_cpu_threads(torch)
        use_lit = O.ref_available()
        nms_fn = (lambda sb, thr: np.arange(len(O.ref_nms_rows(sb, thr)))) if use_lit else None
        t0 = time.perf_counter()
        G.test_one(spec, imgs_h[0], boxes_h[0], 1.0, W, H, -1.5, 0.3, nms_fn=nms_fn)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": R / dt, "unit": "proposals/s", "cores": cores, "kind": "port",
                                "logical_cpus": os.cpu_count(), "thread_count_proxy_s": tried,
                                "sample": f"1 full image (1000 ROIs), {dt:.1f} s; dense layers PyTorch-CPU fp32, ROI/decode C restatement, "
                                          f"NMS {'literal nms.c' if use_lit else 'nms.c restatement'}"}
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, np.float32))
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        ctx.dist_destroy()
        dist.destroy_process_group()
    reps.close()


if __name__ == "__main__":
    main()
