#!/usr/bin/env python
"""bench.py -- images/sec of the full ColorHandPose3DNetwork.inference pipeline on synthetic 320x320 batches.

  python bench.py --gpus N --steps K --warmup W            # our sm_100a path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement of the TF1 reference (oracle)

One JSON line on stdout (rank 0).  A "step" is one pass of the full pipeline (HandSegNet -> mask/crop ->
PoseNet2D -> PosePrior/Viewpoint lifting -> x8 up-sampling -> key-point arg-max) over one batch of
`--batch` synthetic images PER GPU (weak scaling; BASELINE config 4 shards 32 images per GPU).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GFLOP_PER_IMAGE = 142.258408192          # conv + FC FLOPs of the full pipeline (SURVEY.md 8a.1 / arch.conv_flops_per_image)
METRIC = "images/sec full pipeline 320x320"

# BASELINE.json configs -> defaults (explicit flags win).  stage: "full" = inference(), "2d" = inference2d(), "posenet" =
# inference_pose2d + x8 up-sampling + detect_keypoints on 256x256 crops (eval2d_gt_cropped.py:45-50,78).
CONFIGS = {
    1: dict(batch=1, stage="full", precision="bf16x3", cuda_graph=1, height=320, width=320,
            name="config 1: run.py shape, single 320x320 image, full pipeline (CUDA-graph replay)"),
    2: dict(batch=32, stage="posenet", precision="bf16x3", cuda_graph=0, height=256, width=256,
            name="config 2: PoseNet-only (eval2d_gt_cropped path), 32 crops of 256x256 per GPU"),
    3: dict(batch=64, stage="2d", precision="bf16x3", cuda_graph=0, height=320, width=320,
            name="config 3: HandSegNet+PoseNet (eval2d path, inference2d), 64 images of 320x320 per GPU"),
    4: dict(batch=32, stage="full", precision="bf16x3", cuda_graph=0, height=320, width=320,
            name="config 4 shard: full ColorHandPose3DNetwork.inference incl. PosePrior lifting, 32 images per GPU (256 on 8 GPUs)"),
    5: dict(batch=64, stage="full", precision="fp16", cuda_graph=0, height=320, width=320,
            name="config 5 shard: fp16 single-pass tensor-core conv path (tolerance 1e-2), 64 images per GPU (512 on 8 GPUs)"),
}


def stage_gflop_per_image(stage, H, W):
    """conv + FC GFLOP per image of the measured stage (arch.py layer tables)."""
    from hand3d_b200 import arch
    def net(layers, h, w):
        tot = 0
        for name, k, s, cin, cout, _ in layers:
            if k == 0:
                tot += 2 * cin * cout; continue
            h, w = -(-h // s), -(-w // s)
            tot += 2 * h * w * k * k * cin * cout
            if name in arch.HANDSEGNET_POOL_AFTER and layers is not arch.POSEPRIOR and layers is not arch.VIEWPOINT:
                h, w = h // 2, w // 2
        return tot
    if stage == "posenet":
        return net(arch.POSENET2D, H, W) / 1e9
    seg, pose = net(arch.HANDSEGNET, H, W), net(arch.POSENET2D, 256, 256)
    if stage == "2d":
        return (seg + pose) / 1e9
    return (seg + pose + net(arch.POSEPRIOR, 32, 32) + net(arch.VIEWPOINT, 32, 32)) / 1e9


def measured_traffic(precision="bf16x3"):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/*_summary.json), or None."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    if os.path.isdir(pdir):
        for fn in sorted(os.listdir(pdir)):
            if fn.endswith("_summary.json") and (("f8c" in fn) == (precision == "fp16_f8c")):
                try:
                    d = json.load(open(os.path.join(pdir, fn)))
                    if "tc_conv" in d:
                        best = (fn, d["tc_conv"])
                except Exception:
                    pass
    return best


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {"tflops_burst": float(d["bf16_tflops"]), "tflops_sustained": float(d["bf16_tflops_sustained"]),
                    "hbm_gbs": float(d["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
        except Exception:
            pass
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            names = {getattr(N, k): k for k in dir(N) if k.startswith("nvmlClocksEventReason") or k.startswith("nvmlClocksThrottleReason")}
            while not self.stop_flag:
                self.sm.append(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM))
                try:
                    mask = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if isinstance(bit, int) and bit and (mask & bit) == bit and bin(bit).count("1") == 1:
                        self.reasons.add(nm.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
                time.sleep(0.002)
        except Exception as e:  # NVML unavailable: report that instead of clocks
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        r = sorted(x for x in self.reasons if x not in ("GpuIdle", "None", "ApplicationsClocksSetting"))
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": r, "samples": len(self.sm)}


def oracle_stage(stage):
    """The oracle's restatement of the measured stage as f(images, hand_side, weights)."""
    from oracle import hand3d_oracle as O
    from oracle import tf1_ops as T
    if stage == "full":
        return lambda img, hs, wd: O.inference(img, hs, wd, literal_mask=False)
    if stage == "2d":
        return lambda img, hs, wd: O.inference2d(img, wd, literal_mask=False)

    def posenet(img, hs, wd):     # eval2d_gt_cropped.py:45-50,78
        sm = T.resize_bilinear_tf1(O.inference_pose2d(img, wd)[-1], img.shape[1], img.shape[2])
        return [O.detect_keypoints(m) for m in sm]
    return posenet


def cpu_reference_throughput(n_images, H, W, seconds_cap=40.0, stage="full"):
    """Times the oracle (CPU restatement of the TF1 graph; the reference itself needs TensorFlow 1.3, which cannot be
    installed here) on the host cores.  Thread-count candidates are swept in ASCENDING order (16, 32, 64, all cores: the
    oracle's convolutions stop scaling long before 128 threads and the largest counts are the slowest), each one is timed on
    one batched oracle.inference() after a one-image warm-up, at least two candidates are always measured and the best
    throughput is kept; the cap only stops the sweep early.  The mask grower runs in its fast boolean form (bit-identical to
    the literal 32 x dilation2d sequence, tests/test_oracle_kat.py), which is the generous choice for the CPU side.
    Returns (images/s, threads used, sample description)."""
    import torch
    from hand3d_b200 import weights as Wt
    from oracle import hand3d_oracle as O
    cores = os.cpu_count() or 1
    wd = Wt.synthetic_weights(0)
    img = Wt.synthetic_images(n_images, H, W, seed=100)
    hs = Wt.synthetic_hand_side(n_images, seed=2)
    run = oracle_stage(stage)
    best, best_thr, t_start = 0.0, cores, time.perf_counter()
    cands = sorted({min(cores, 16), min(cores, 32), min(cores, 64), cores})
    tried = []
    for thr in cands:
        torch.set_num_threads(thr)
        run(img[:1], hs[:1], wd)                                              # warm-up for this thread count
        t0 = time.perf_counter()
        run(img, hs, wd)
        v = n_images / (time.perf_counter() - t0)
        tried.append((thr, round(v, 3)))
        if v > best:
            best, best_thr = v, thr
        if len(tried) >= 2 and time.perf_counter() - t_start > seconds_cap:
            break
    torch.set_num_threads(cores)
    return best, best_thr, "one batched oracle inference() of [%d,%d,%d,3] per thread count, ascending sweep %s (threads, images/s), best kept (%d threads of %d cores)" % (
        n_images, H, W, tried, best_thr, cores)


def metric_name(args):
    return METRIC if (args.stage == "full" and args.height == 320 and args.width == 320) else "images/sec %s %dx%d" % (args.stage, args.height, args.width)


def workload_name(args):
    what = {"full": "full ColorHandPose3DNetwork.inference (HandSegNet+PoseNet2D+PosePrior/Viewpoint, %dx%d input, 256x256 crop)" % (args.height, args.width),
            "2d": "ColorHandPose3DNetwork.inference2d (HandSegNet+PoseNet2D, %dx%d input, 256x256 crop)" % (args.height, args.width),
            "posenet": "ColorHandPose3DNetwork.inference_pose2d + x8 up-sampling + detect_keypoints on %dx%d crops" % (args.height, args.width)}[args.stage]
    cfg = CONFIGS.get(args.config, {}).get("name", "custom")
    return "%s, %d images per GPU per step (BASELINE %s)" % (what, args.batch, cfg)


def run_reference(args):
    """Reference arm: the CPU restatement of the TF1 graph (oracle/) on the host cores -- the unmodified reference cannot run
    (TensorFlow 1.3 is not installable offline, and the repo ships no weights).  Warm-up = ascending thread-count sweep; each
    timed step = one batched oracle call of the same stage, sized so that the whole run stays within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from hand3d_b200 import weights as Wt
    v0, thr, sample = cpu_reference_throughput(min(args.ref_images, 4), args.height, args.width, seconds_cap=60.0, stage=args.stage)
    torch.set_num_threads(thr)
    n = int(max(1, min(args.ref_images, round(150.0 * v0 / max(1, args.steps)))))      # ~150 s of timed CPU work in total
    wd = Wt.synthetic_weights(0)
    img = Wt.synthetic_images(n, args.height, args.width, seed=100)
    hs = Wt.synthetic_hand_side(n, seed=2)
    run = oracle_stage(args.stage)
    for _ in range(max(0, args.warmup - 1)):
        run(img, hs, wd)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run(img, hs, wd)
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    line = {
        "impl": "reference", "metric": metric_name(args), "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args) + "; CPU restatement of the TF1 reference (oracle/), TensorFlow 1.3 is not installable",
                   "images_per_step": n, "threads": thr, "stage": args.stage},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": thr, "kind": "port",
                         "sample": "%d steps x one batched oracle call of %d images, %d torch threads (best of the warm-up sweep: %s)" % (
                             args.steps, n, thr, sample)},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa(index):
    """Best effort: pin this rank's host threads to the CPUs NVML reports as local to its GPU BEFORE the pinned staging buffers
    are allocated (first-touch places them on that NUMA node), so that eight ranks do not pull their inputs across sockets."""
    try:
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = N.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


RHD_RECORD_BYTES, RHD_IMAGE_OFF = 410520, 878     # data/BinaryDbReader.py:103-208 (header 876 B + 2 B pad, then 320x320x3 u8)
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, result):
    """Writes the arrays of one step's result dict as <out_dir>/<name>.npy in float32 (the int32 key-point indices are exact
    in float32), so that two builds run with the same arguments can be compared output for output.  Above DUMP_LIMIT_BYTES
    every array keeps the same seeded sample of images, whose indices go to sample_rows.npy."""
    arrays = {k: v.detach().cpu().numpy().astype(np.float32) for k, v in result.items() if v is not None}
    B = next(iter(arrays.values())).shape[0]
    per_row = sum(a.nbytes for a in arrays.values()) // B
    if B * per_row > DUMP_LIMIT_BYTES:
        n = (DUMP_LIMIT_BYTES - (1 << 20)) // (per_row + 8)          # 1 MB left for the index file's and the headers' slack
        rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from hand3d_b200 import runtime, weights as Wt
    from hand3d_b200.distributed import P2PGather, gather_records

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device -- hand3d_b200 has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = bind_to_gpu_numa(local_rank) if world > 1 else 0
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, H, W, stage = args.batch, args.height, args.width, args.stage
    full = stage == "full"

    ctx = runtime.Context(local_rank, precision=args.precision)
    ctx.load_weights(Wt.synthetic_weights(0))
    ctx.ensure_workspace(B, H, W)
    # synthetic inputs: NBUF different batches per rank (rotated every step so that inputs > L2 never repeat back to back)
    NBUF = 4
    host_imgs = [torch.from_numpy(Wt.synthetic_images(B, H, W, seed=1000 + 17 * rank + i)).pin_memory() for i in range(NBUF)]
    host_hs = [torch.from_numpy(Wt.synthetic_hand_side(B, seed=2000 + 17 * rank + i)).pin_memory() for i in range(NBUF)]
    dev_imgs = [t.to(dev) for t in host_imgs]
    dev_hs = [t.to(dev) for t in host_hs]

    # multi-GPU result exchange (full pipeline): fused pack + peer-memory all-gather kernel (NCCL all_gather with --gather nccl)
    p2p = None
    if world > 1 and full and args.gather == "p2p":
        p2p = P2PGather(ctx, max_batch=B)

    def exchange(r):
        if not full:
            return r["keypoints_uv"]
        if p2p is not None:
            return p2p.gather(r["keypoint_coord3d"], r["keypoints_uv"], r["center"], r["scale_crop"])
        rec = ctx.pack_records(r["keypoint_coord3d"], r["keypoints_uv"], r["center"], r["scale_crop"])
        return gather_records(rec) if world > 1 else rec

    def run_stage(img, hs, outputs="keypoints"):
        if stage == "posenet":
            return ctx.pose2d(img, outputs=outputs)
        return ctx.pipeline(img, hs if full else None, full, outputs=outputs)

    # one CUDA graph per input buffer (the forward pass is sync-free with fixed pointers: ~80 launches replay as one)
    graphs = None
    if args.cuda_graph:
        if stage == "posenet":
            raise SystemExit("--cuda-graph is wired for the pipeline stages")
        graphs = []
        for k in range(NBUF):
            c0 = ctx.launch_count
            replay, res = ctx.capture_pipeline(dev_imgs[k], dev_hs[k] if full else None, full, outputs="keypoints")
            graphs.append((replay, res, (ctx.launch_count - c0) // 2))   # warm-up + capture each issue the step once
    graph_launches = [0]

    def step_device(i):
        if graphs is not None:
            replay, r, nl = graphs[i % NBUF]
            replay()
            graph_launches[0] += nl
        else:
            r = run_stage(dev_imgs[i % NBUF], dev_hs[i % NBUF])
        exchange(r)
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up
    for i in range(args.warmup):
        step_device(i)
    barrier()

    # ---- the exchange kernel against NCCL, outside the timed region: bit-identical records at every N (multimem at N = 8)
    gather_verified = None
    if p2p is not None:
        r = run_stage(dev_imgs[0], dev_hs[0])
        got = p2p.gather(r["keypoint_coord3d"], r["keypoints_uv"], r["center"], r["scale_crop"]).clone()
        want = gather_records(ctx.pack_records(r["keypoint_coord3d"], r["keypoints_uv"], r["center"], r["scale_crop"]))
        torch.cuda.synchronize()
        ok = torch.tensor([int(torch.equal(got.view(torch.int32), want.view(torch.int32)))], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        gather_verified = bool(ok.item())
        if not gather_verified:
            raise RuntimeError("bench.py: records gathered by h3d_gather_records_p2p differ from NCCL all_gather")
        barrier()

    # ---- timed region (device-resident inputs)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count + graph_launches[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        last = step_device(i)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = ctx.launch_count + graph_launches[0] - l0
    sampler.stop_flag = True
    sampler.join(timeout=2.0)
    value = world * B * args.steps / (ms / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)      # before any later replay overwrites the graph's result buffers

    # ---- sustained: the same loop for several seconds (power / thermal steady state), reported beside the K-step value
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1000.0 / max(ms / args.steps, 1e-3)))
        s2 = ClockSampler(local_rank); s2.start()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        g0.record()
        for i in range(n_sus):
            step_device(i)
        g1.record()
        barrier()
        ms_sus = max_over_ranks(g0.elapsed_time(g1))
        s2.stop_flag = True; s2.join(timeout=2.0)
        sustained = {"value": world * B * n_sus / (ms_sus / 1000.0), "unit": "images/s", "steps": n_sus, "seconds": ms_sus / 1000.0,
                     "ms_per_step": ms_sus / n_sus, "sm_mhz": s2.summary().get("sm_mhz")}

    # ---- end to end through the public API: every step copies its inputs from pinned host memory and reads its result back.
    # Input forms: "records" = the dataset's uint8 records (data/BinaryDbReader.py:103-208, 410 520 B per 320x320 sample) decoded on
    # the device by h3d_decode_records (image = u8 / 255 - 0.5 as the reader computes it): the form eval2d.py / eval_full.py feed;
    # "f32" = the fp32 NHWC image run.py builds on the host.  Double-buffered: the copy of step i+1 runs on a copy stream while
    # step i computes; results leave on a second copy stream.
    use_records = args.e2e_input == "records" and stage != "posenet" and H == 320 and W == 320
    if use_records:
        host_recs = []
        for i in range(NBUF):
            rec = torch.zeros((B, RHD_RECORD_BYTES), dtype=torch.uint8)
            u8 = torch.clamp(torch.round((host_imgs[i] + 0.5) * 255.0), 0, 255).to(torch.uint8)       # the same synthetic images, quantised
            rec[:, RHD_IMAGE_OFF:RHD_IMAGE_OFF + H * W * 3] = u8.reshape(B, -1)
            host_recs.append(rec.pin_memory())
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    if use_records:
        stage_in = [torch.empty((B, RHD_RECORD_BYTES), dtype=torch.uint8, device=dev) for _ in range(2)]
    else:
        stage_in = [torch.empty((B, H, W, 3), dtype=torch.float32, device=dev) for _ in range(2)]
    stage_hs = [torch.empty((B, 2), dtype=torch.float32, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    host_out = [None, None]
    d2h_done = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        k = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k])            # the compute stream is done reading this staging buffer
            stage_in[k].copy_((host_recs if use_records else host_imgs)[i % NBUF], non_blocking=True)
            stage_hs[k].copy_(host_hs[i % NBUF], non_blocking=True)
            ready[k].record(copy_stream)

    def result_tensors(r, all_outputs):
        if not all_outputs:
            return [exchange(r)]
        keys = {"full": ["hand_scoremap", "image_crop", "scale_crop", "center", "keypoints_scoremap", "keypoint_coord3d"],   # run.py:61-64
                "2d": ["keypoints_scoremap", "image_crop", "scale_crop", "center"],                                          # eval2d.py:58
                "posenet": ["keypoints_scoremap"]}[stage]                                                                   # eval2d_gt_cropped.py:45-50
        return [r[k] for k in keys]

    def run_e2e(n, all_outputs):
        cur = torch.cuda.current_stream()
        for k in range(2):
            consumed[k].record(cur)
        prefetch(0)
        d2h_bytes = 0
        for i in range(n):
            k = i & 1
            if i + 1 < n:
                prefetch(i + 1)
            if host_out[k] is not None:
                d2h_done[k].synchronize()                  # the results of step i-2 have landed on the host (a consumer reads them here)
            cur.wait_event(ready[k])
            img = ctx.decode_records(stage_in[k], "rhd", want_aux=False)["image"] if use_records else stage_in[k]
            r = run_stage(img, stage_hs[k], outputs="all" if all_outputs else "keypoints")
            outs = result_tensors(r, all_outputs)
            consumed[k].record(cur)
            done = torch.cuda.Event()
            done.record(cur)
            if host_out[k] is None:
                host_out[k] = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done)
                for h, o in zip(host_out[k], outs):
                    h.copy_(o, non_blocking=True)          # device -> host read of the step's result
                    try:
                        o.record_stream(d2h_stream)        # the caching allocator must not recycle `o` under the copy
                    except Exception:
                        pass                               # views of the symmetric gather buffer are not allocator-owned
                d2h_done[k].record(d2h_stream)
            d2h_bytes = sum(o.numel() * o.element_size() for o in outs)
        return d2h_bytes

    def time_e2e(all_outputs):
        host_out[0] = host_out[1] = None
        run_e2e(max(2, args.warmup // 2), all_outputs)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        f0.record()
        nbytes = run_e2e(args.steps, all_outputs)
        d2h_stream.synchronize()
        f1.record()
        barrier()
        return world * B * args.steps / (max_over_ranks(f0.elapsed_time(f1)) / 1000.0), nbytes

    e2e_value, d2h = time_e2e(False)
    h2d = (B * RHD_RECORD_BYTES if use_records else B * H * W * 3 * 4) + B * 2 * 4
    e2e_all = None
    if args.e2e_all_outputs:
        v_all, d2h_all = time_e2e(True)
        e2e_all = {"value": v_all, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_all,
                   "outputs": "every tensor the reference's sess.run fetches for this stage (run.py:61-64 / eval2d.py:58 / eval2d_gt_cropped.py:45-50)"}
    ctx.check_errors()

    # ---- per-kernel-class timing (CUDA events around every launch; separate pass so it does not perturb `value`)
    gflop_img = stage_gflop_per_image(stage, H, W)
    prof_steps = min(3, args.steps)
    ctx.profile_begin()
    for i in range(prof_steps):
        run_stage(dev_imgs[i % NBUF], dev_hs[i % NBUF])
    prof = ctx.profile_end()
    peaks = measured_peaks()
    roof = None
    dominant = "tc_conv" if prof["tc_conv"]["launches"] else "direct_conv"
    d = prof[dominant]
    if d["ms"] > 0:
        achieved = d["flops"] / (d["ms"] * 1e-3) / 1e12
        peak = peaks["tflops_sustained"] if dominant == "tc_conv" else 75.0
        tr = measured_traffic(args.precision) if (dominant == "tc_conv" and args.precision in ("bf16x3", "fp16_f8c") and full and B == 32) else None
        passes = 3 if args.precision in ("bf16x3", "fp16x3") else (2 if args.precision == "fp16_f8c" else 1)
        roof = {"bound": "tensor", "kernel": "conv_tc2_kernel / conv_tc_kernel / conv_c64x2_kernel / conv_c64_kernel / conv_c1f_kernel (tcgen05 implicit GEMM: every conv layer - conv1_1 fused into conv1_2 - and the FC stacks)" if dominant == "tc_conv" else "conv_direct_kernel (fp32 FFMA)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": tr[1]["dram_bytes_per_launch"] if tr else None,
                "traffic_source": ("ncu dram__bytes_read+write per launch, B=32, profiles/%s" % tr[0]) if tr else None,
                "achieved_per_launch": {"gflop": d["flops"] / max(1, d["launches"]) / 1e9, "us": 1e3 * d["ms"] / max(1, d["launches"])},
                "peak_source": peaks["source"] + (", bf16 sustained" if dominant == "tc_conv" else ", nominal fp32 FFMA"),
                "launches_per_step": d["launches"] // prof_steps, "ms_per_step": d["ms"] / prof_steps,
                "mma_passes": passes,
                # fp32 parity costs `passes` tensor-core passes per algorithmic FLOP: the executed rate is what the tensor pipe sees
                "executed": {"value": achieved * passes, "unit": "TFLOP/s", "frac": achieved * passes / peak} if dominant == "tc_conv" else None,
                "share_of_step": (d["ms"] / prof_steps) / (ms / args.steps),
                "by_class_ms_per_step": {k: v["ms"] / prof_steps for k, v in prof.items()}}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample = cpu_reference_throughput(min(args.cpu_images, max(1, B)), H, W, seconds_cap=25.0, stage=stage)
            cpu = {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample}
        line = {
            "metric": metric_name(args), "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16x3": "bf16 hi/lo split x3 MMA passes, fp32 accumulate (fp32 parity, 1e-3)",
                      "fp16x3": "fp16 hi/lo split x3 MMA passes, fp32 accumulate (fp32 parity, 1e-3)",
                      "fp16_f8c": "fp16 main pass + two fp8 (e4m3) correction passes, fp32 accumulate (fp32 parity, 1e-3)",
                      "fp16": "fp16 (1e-2 path)", "bf16": "bf16", "fp32_ffma": "f32"}[args.precision],
            "data": "synthetic",
            "config": {"workload": workload_name(args), "baseline_config": args.config, "stage": stage,
                       "global_batch": world * B, "precision": args.precision, "parallelism": "dp%d" % world, "cuda_graph": bool(args.cuda_graph),
                       "l2": "inputs rotate over %d distinct batches per rank (%.0f MB > L2); activations per step %.1f GB" % (
                           NBUF, NBUF * B * H * W * 12 / 1e6, B * 0.312),
                       "e2e_input": "uint8 RHD records + on-device decode (h3d_decode_records)" if use_records else "fp32 NHWC images",
                       "numa_bound_cpus": numa_cpus,
                       "collective": ("none (single GPU)" if world == 1 else "none (per-rank results)" if not full else
                                      "fused pack + all-gather of 432 B/image records over NVLink peer memory (h3d_gather_records_p2p, %s), verified bit-identical to NCCL all_gather before the timed region" % (
                                          "multimem store" if (p2p is not None and p2p.mc) else "peer stores")
                                      if p2p is not None else "NCCL all_gather of 432 B/image records")},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "e2e_all_outputs": e2e_all,
            "sustained": sustained,
            "gather_verified": gather_verified,
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": roof,
            "cpu_baseline": cpu,
            "gflop_per_image": gflop_img,
            "tflops_algorithmic": value * gflop_img / 1e3,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS), help="BASELINE.json config (1-5); sets the defaults of --batch / --stage / --precision / --cuda-graph / --height / --width")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step")
    ap.add_argument("--stage", default=None, choices=["full", "2d", "posenet"])
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--precision", default=os.environ.get("H3D_PRECISION"), choices=["bf16x3", "fp16x3", "fp16", "bf16", "fp32_ffma", "fp16_f8c"])
    ap.add_argument("--cpu-images", type=int, default=8, help="bounded CPU-baseline sample (images per oracle call)")
    ap.add_argument("--ref-images", type=int, default=8, help="--impl reference: images per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default=os.environ.get("H3D_GATHER", "p2p"), choices=["p2p", "nccl"], help="multi-GPU result exchange")
    ap.add_argument("--cuda-graph", type=int, default=None, help="replay the step from a CUDA graph")
    ap.add_argument("--sustain-seconds", type=float, default=3.0, help="extra sustained loop after the timed K steps (0 = off)")
    ap.add_argument("--e2e-input", default="records", choices=["records", "f32"], help="what the end-to-end loop copies host -> device")
    ap.add_argument("--e2e-all-outputs", type=int, default=1, help="also time the end-to-end loop with every reference output read back")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = CONFIGS[args.config]
    for k in ("batch", "stage", "height", "width", "precision", "cuda_graph"):
        if getattr(args, k) is None:
            setattr(args, k, cfg[k] if k != "cuda_graph" else int(os.environ.get("H3D_CUDA_GRAPH", cfg[k])))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
