#!/usr/bin/env python
"""bench.py -- images/sec of the end-to-end VGG16 Faster R-CNN forward path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision bf16x3|bf16] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config #2): synthetic 600x1000 image (uniform(0,255) - BGR means), random-init weights
(heads N(0,0.01), He-normal trunk), test-mode ProposalLayer (6000 -> NMS 0.7 -> 300), 21 classes.
One step = one image through the whole graph (trunk, RPN, ProposalLayer, RoI pool, fc6/fc7, heads,
softmax/decode/clip and the caller's per-class NMS of forward.py:48-57) on each GPU; images shard one per GPU with
no collective ("scaling": "weak").

Prints ONE JSON line (rank 0).  `value`   : device-timed (CUDA events) images/s, inputs resident in HBM, 4 images in
                                            flight per GPU (`detail.one_image_in_flight` = the batch-1 latency view).
                                `e2e`     : the same metric through the REFERENCE's interface, per image inside the timed
                                            region: models.faster_rcnn.FasterRCNN.__call__ on a HOST float32
                                            (1,3,600,1000) array (7.2 MB H2D) + the caller's 20 models.cpu_nms.cpu_nms
                                            calls on host arrays, 8 caller threads; the one-thread number, the
                                            standalone-NMS numbers and the build's streaming API are reported beside it.
                                `roofline`: the conv/GEMM tensor-core kernel, timed live per launch (frac vs the burst
                                            peak), a second run of the lanes (vs the sustained peak), DRAM traffic and
                                            per-kernel HBM fractions from the committed ncu pass of this binary.
                                `cpu_baseline`: the CPU oracle pipeline on this box's host cores (rank 0, N=1).
Every timed leg of the B200 arm runs --steps images.  `--dump-outputs DIR` writes what the last timed image computed
(see dump_outputs); the inputs are seeded, so two builds can be compared output for output.
`--impl reference` times the reference-equivalent CPU pipeline instead (torch-CPU fp32 dense ops standing in for
Chainer-NumPy -- Chainer is not installable offline -- plus the reference's own compiled cpu_nms.pyx when
oracle/_ref holds it, else the C restatement).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# More hardware work queues than the default 8: the B200 arm keeps 4 lane streams, a copy stream and, in the reference-interface
# leg, a graph stream + a host-NMS stream per caller thread; with 8 queues unrelated streams alias onto one queue and a 30 us NMS
# kernel can sit behind another thread's 1.4 ms graph (must be set before the CUDA context exists).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "chainer-faster-rcnn_b200"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

H_IMG, W_IMG = 600, 1000
CONV_STACK_GFLOP = 379.17       # trunk 367.74 + RPN 3x3 11.30 + RPN 1x1 0.13 (SURVEY.md 8d)
WHOLE_GFLOP = 451.15


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1421.6), d.get("hbm_gbs", 6571.9), "measured"
    return 1590.0, 6650.0, "fallback"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------- CPU (reference-equivalent) arm
def cpu_pipeline_once(orc, params, x, info, ref_nms=None, raw=None):
    """One image through the reference-equivalent CPU path.  Returns (seconds, nms_seconds).
    raw: optional uint8 (h0,w0,3) BGR image -- then forward.py's img_preprocessing (34-45) is part of the timed work
    and replaces `x`, like the B200 arm's e2e."""
    t0 = time.perf_counter()
    if raw is not None:
        x = orc.img_preprocessing(raw)[0][None]
    if ref_nms is not None:
        saved = orc.cpu_nms
        tn = [0.0]

        def timed_nms(dets, thr):
            s = time.perf_counter()
            k = [int(v) for v in ref_nms.cpu_nms(np.ascontiguousarray(dets, dtype=np.float32), thr)]
            tn[0] += time.perf_counter() - s
            return k
        orc.cpu_nms = timed_nms
    else:
        tn = [0.0]
        saved = orc.cpu_nms

        def timed_nms2(dets, thr):
            s = time.perf_counter()
            k = saved(dets, thr)
            tn[0] += time.perf_counter() - s
            return k
        orc.cpu_nms = timed_nms2
    try:
        cls_prob, pred_boxes, _ = orc.faster_rcnn_forward(x, params, info)
        orc.detect(cls_prob, pred_boxes, 0.3, 0.8)          # forward.py:48-57
    finally:
        orc.cpu_nms = saved
    return time.perf_counter() - t0, tn[0]


def pick_cpu_threads(torch):
    """Give the CPU arm its best case: time one mid-trunk 3x3 convolution at a few intra-op thread counts and keep the
    fastest (all hardware threads is often NOT the fastest for torch-CPU on a many-core host)."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16) if 1 <= c <= cores}, reverse=True)
    x = torch.randn(1, 256, 150, 250)
    w = torch.randn(256, 256, 3, 3)
    best, best_t = cores, None
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.conv2d(x, w, padding=1)
        t = None
        for _ in range(5):
            t0 = time.perf_counter()
            torch.nn.functional.conv2d(x, w, padding=1)
            dt = time.perf_counter() - t0
            t = dt if t is None else min(t, dt)
        if best_t is None or t < 0.9 * best_t:          # fewer threads only when clearly (>10%) faster
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def run_reference_arm(args, rank):
    if rank != 0:
        return
    import torch
    import frcnn_oracle as orc
    import build_ref
    cores = pick_cpu_threads(torch)
    ref_nms = build_ref.load()
    params = orc.make_params(seed=1234)
    x = None
    raw = np.random.default_rng(7).integers(0, 256, (375, 625, 3), dtype=np.uint8)     # resizes to 600x1000
    info = np.array([[H_IMG, W_IMG]], np.int32)
    warm = max(args.warmup, 3)               # the same warm-up count as the B200 arm
    for _ in range(warm):
        t_probe, _ = cpu_pipeline_once(orc, params, x, info, ref_nms, raw=raw)
    steps = args.steps
    if t_probe * steps > 240.0:                 # keep the whole run within a few minutes
        steps = max(1, int(240.0 / t_probe))
    ts, tn = [], []
    for _ in range(steps):
        a, b = cpu_pipeline_once(orc, params, x, info, ref_nms, raw=raw)
        ts.append(a)
        tn.append(b)
    total = sum(ts)
    val = steps / total
    kind = "reference" if ref_nms is not None else "port"
    line = {
        "impl": "reference", "metric": "images/sec end-to-end VGG16 Faster R-CNN forward @600x1000",
        "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * total / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(),
        "detail": {"device": "host CPU", "requested_steps": args.steps},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": "%d whole image(s): raw uint8 375x625 -> preprocessing -> 600x1000 forward -> per-class "
                                   "NMS; dense ops torch-CPU fp32 (Chainer not installable offline), NMS = %s; NMS share %.1f%%" %
                                   (steps, "reference cpu_nms.pyx (oracle/_ref)" if ref_nms is not None else "C port",
                                    100.0 * sum(tn) / total)},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- B200 arm
def hbm_fractions(tj, table, peak_hbm):
    """Per-kernel HBM fractions (VERDICT r01 item 3): DRAM bytes of each launch from the ncu pass of this binary
    (profiles/r02_conv_stack_dram.json) over the launch's LIVE CUDA-event time where bench.py times it (the GEMM launches:
    same order as `table`), else over its duration under ncu (cold caches, serialised)."""
    out = {}
    gl = tj.get("gemm_launches") or []
    if len(gl) == len(table):
        for name, idx in (("conv1_1", 0), ("conv1_2", 1), ("fc6", len(table) - 3), ("fc7", len(table) - 2)):
            mb, ms = gl[idx]["dram_mb"], table[idx][1]
            out[name] = {"dram_mb_ncu": mb, "ms_live": round(ms, 4), "gbs": round(mb / ms, 1),
                         "frac_of_hbm_peak": round(mb / ms / peak_hbm, 3)}
    for name, sub in (("pack_image_c8", "pack_image_c8_kernel"), ("roi_pool", "roi_pool")):
        for key, e in (tj.get("per_kernel") or {}).items():
            if sub in key:
                out[name] = {"kernel": key.replace("void ", "").replace("frcnn::", ""), "dram_mb_ncu": e["dram_mb"], "us_under_ncu": e["us"],
                             "gbs": round(e["dram_mb"] / e["us"] * 1e3, 1),
                             "frac_of_hbm_peak": round(e["dram_mb"] / e["us"] * 1e3 / peak_hbm, 3)}
                break
    return out


def conv_layer_table(plan, torch, reps=3, spin=True):
    """Per-launch device time of the tensor-core kernel over one forward: eager re-run with CUDA events around each
    frcnn_conv2d / frcnn_linear call (same stream, same buffers).  Returns [(name, ms, gflop)].  (frcnn_linear = the
    split-K GEMM + its small reduction kernel, timed together.)"""
    from frcnn_b200 import ops
    rows = []
    orig_conv, orig_lin = ops.conv2d, ops.linear

    def bracket(fn, gflop, name):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # a ~40 us spin kernel first: while the GPU spins, the host enqueues e0 + the launch + e1, so the interval
        # between the events is the kernel's execution alone (no host launch latency inside it, even on a slow host)
        if spin:
            torch.cuda._sleep(80000)
        e0.record()
        r = fn()
        e1.record()
        rows.append([(e0, e1), gflop, name])
        return r

    def timed_conv(x, w_hi, w_lo, bias, ksize, relu, **kw):
        Hh, Ww, Cin = x.hi.shape
        taps, Cout, _ = w_hi.shape
        k_true = 27 if (Cin == 32 and taps == 1 and Hh > 1) else taps * Cin     # conv1_1 = im2col GEMM, 27 real K
        return bracket(lambda: orig_conv(x, w_hi, w_lo, bias, ksize, relu, **kw), 2.0 * Hh * Ww * Cout * k_true / 1e9,
                       "%dx%dx%d->%d k%d" % (Hh, Ww, Cin, Cout, ksize))

    def timed_lin(x, w_hi, w_lo, bias, relu, **kw):
        _, R, K = x.hi.shape
        Cout = w_hi.shape[1]
        return bracket(lambda: orig_lin(x, w_hi, w_lo, bias, relu, **kw), 2.0 * R * Cout * K / 1e9,
                       "linear %dx%d->%d" % (R, K, Cout))
    orig_c8 = ops.conv3x3_c8

    def timed_c8(x_c8, H, W, w_hi, w_lo, bias, relu=True, out=None):
        Cout = w_hi.shape[1]
        return bracket(lambda: orig_c8(x_c8, H, W, w_hi, w_lo, bias, relu, out=out), 2.0 * H * W * Cout * 27 / 1e9,
                       "%dx%dx3->%d k3 (compact image, K=3x32)" % (H, W, Cout))
    ops.conv2d, ops.linear, ops.conv3x3_c8 = timed_conv, timed_lin, timed_c8
    acc = {}
    try:
        for _ in range(reps):
            rows.clear()
            plan._run()
            torch.cuda.synchronize()
            for i, (ev, gf, name) in enumerate(rows):
                acc.setdefault(i, [name, gf, []])[2].append(ev[0].elapsed_time(ev[1]))
    finally:
        ops.conv2d, ops.linear, ops.conv3x3_c8 = orig_conv, orig_lin, orig_c8
    return [(v[0], min(v[2]), v[1]) for _, v in sorted(acc.items())]


WORKLOAD = ("VGG16 Faster R-CNN forward + the caller's per-class NMS (forward.py:48-57: thresh 0.3, conf 0.8), synthetic "
            "600x1000, 300 proposals (config #2), one image per GPU")


def bench_config():
    """The SAME `config` object in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "image": [H_IMG, W_IMG], "proposals": 300, "num_classes": 21,
            "l2": "no L2 flush needed: the per-step working set (activations + weights, ~1.5 GB) exceeds the 126 MB L2 and 4 "
                  "input images are rotated"}


def host_link_probe(torch, nbytes=7200000, reps=20):
    """Bare pinned-memory H2D / D2H bandwidth of this box (CUDA events on the copying stream), so that an e2e number
    limited by the host link can be told from one limited by the code."""
    h = torch.empty((nbytes,), dtype=torch.uint8).pin_memory()
    d = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
    out = {}
    for name, (dst, src) in (("h2d", (d, h)), ("d2h", (h, d))):
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        out[name + "_gbs_median"] = nbytes / ts[len(ts) // 2] / 1e6
        out[name + "_gbs_worst"] = nbytes / ts[-1] / 1e6
    out["bytes"] = nbytes
    return out


def build_reference_api_model(params):
    """models.faster_rcnn.FasterRCNN (the drop-in mirror of the reference class) filled with `params`."""
    from frcnn_b200 import dropin
    dropin.install()
    from models.faster_rcnn import FasterRCNN
    from models.vgg16 import VGG16Prev
    model = FasterRCNN(trunk_class=VGG16Prev)
    model.rcnn_train = False
    model.rpn_train = False
    named = dict(model.namedparams())
    for k, v in params.items():
        named["/" + k].data[...] = v
    model._params_changed()
    return model


def reference_api_image(model, x_var, info_var, nms, np_):
    """One image through the REFERENCE's interface, exactly what forward.py does per image (:88-99, :48-57):
    model(x, img_info) with a HOST float32 image, then the caller's per-class loop of 20 cpu_nms calls on host arrays."""
    cls_score, bbox_pred = model(x_var, info_var)
    prob = cls_score.data
    n_det = 0
    for cls_id in range(1, 21):
        _cls = prob[:, cls_id][:, np_.newaxis]
        _bbx = bbox_pred[:, cls_id * 4: (cls_id + 1) * 4]
        dets = np_.hstack((_bbx, _cls))
        keep = nms(dets, 0.3)
        dets = dets[keep, :]
        n_det += int((dets[:, -1] >= 0.8).sum())
    return prob.shape[0], n_det


def dump_outputs(out_dir, plan):
    """Writes what the caller of the timed path receives for the image `plan` ran last: the proposals (rois, scores), the
    class probabilities (prob), the decoded boxes (boxes) and the per-class NMS result (keep_idx per class with entries
    past keep_count set to -1, keep_count, conf_count) as out_dir/<name>.npy.  Integers are stored as float64 (exact)."""
    os.makedirs(out_dir, exist_ok=True)
    r = plan.unpack_result(plan.result.cpu().numpy())
    r["count"] = np.array([r["count"]])
    r["keep_idx"] = np.where(np.arange(r["keep_idx"].shape[1]) < r["keep_count"][:, None], r["keep_idx"], -1)
    for name, a in r.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def run_b200_arm(args, rank, local_rank, world):
    import torch
    import frcnn_oracle as orc              # synthetic weights / image generators + cpu_baseline only
    from frcnn_b200 import shard
    from frcnn_b200.engine import Engine, LanePool, StreamRunner

    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    anchors = orc.generate_anchors(ratios=(0.5, 1, 2), scales=(8, 16, 32))
    params = orc.make_params(seed=1234)
    if args.smem_reserve_kb:
        from frcnn_b200 import ops as _o
        _o.set_conv_smem_reserve(1024 * args.smem_reserve_kb)
    # the whole north_star path: the caller's per-class NMS (forward.py:48-57, thresholds of :75-76) runs inside the graph
    eng = Engine(params, precision=args.precision, anchors=anchors, use_graph=True, with_detect=True,
                 det_nms_thresh=0.3, det_conf=0.8)
    plan = eng.plan(H_IMG, W_IMG)
    n_img = 4                                # rotate distinct images: no step sees the previous step's input
    imgs_np = [orc.make_image(H_IMG, W_IMG, seed=shard.image_seed(rank, i)) for i in range(n_img)]       # (1,3,H,W) float32
    from frcnn_b200 import ops as _ops
    imgs_host = []
    for a in imgs_np:                        # pinned by the library (cudaHostAlloc), see frcnn_host_alloc
        blk = _ops.PinnedBlock(a[0].shape, np.float32)
        blk.np[...] = a[0]
        imgs_host.append(blk)
    imgs_dev = [torch.from_numpy(a[0]).cuda() for a in imgs_np]
    warm = max(args.warmup, 3)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-timed value: inputs resident in HBM
    pool = LanePool(plan, lanes=args.in_flight)      # args.in_flight independent images in flight (one stream + graph each)
    # clocks / throttle reasons are sampled (nvidia-smi, every 100 ms) from the warm-up through the timed region, the
    # one-image-in-flight repeat of it and the sustained run: the GPU is under the same load throughout
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    pool.fork()
    for i in range(warm):
        pool.submit(i, imgs_dev[i % n_img])
    pool.join()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    pool.fork()
    for i in range(args.steps):
        last = pool.submit(i, imgs_dev[i % n_img])   # every step = one whole image through the whole path
    pool.join()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)        # before the legs below reuse the lanes' buffers
    R_last = int(plan.prop.count.item())
    n_conf_last = int(plan.det[2].sum().item())
    # tie-free-ness of the run (SURVEY 8d): distinct fg scores among the anchors of the last image
    fg = torch.softmax(plan.rpn_out[:, :18], dim=1)[:, 9:18].reshape(-1)
    unique_fg = int(torch.unique(fg).numel())
    # the same K steps with ONE image in flight (no overlap between images): reported beside the headline
    barrier()
    e0.record()
    for i in range(args.steps):
        plan.forward(imgs_dev[i % n_img])
    e1.record()
    barrier()
    ms_single = e0.elapsed_time(e1)
    # the lanes once more after the legs above: the number to hold against bf16_tflops_sustained (a long --steps makes it
    # a sustained run; every timed leg runs --steps images)
    n_sus = args.steps
    barrier()
    e0.record()
    pool.fork()
    for i in range(n_sus):
        pool.submit(i, imgs_dev[i % n_img])
    pool.join()
    e1.record()
    barrier()
    ms_sus = shard.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    clocks = sampler.stop() if rank == 0 else None
    # per-launch times of the tensor-core kernel, taken right here: same thermal / power state as the timed region above
    table = conv_layer_table(plan, torch) if rank == 0 else None
    ms_max = shard.max_over_ranks(ms, device="cuda")          # slowest rank decides
    value = world * args.steps / (ms_max / 1e3)
    # seeds 0-4 (SURVEY 8d): one image in flight, --steps images per seed, this rank
    seed_rates = {}
    if rank == 0:
        for sd in range(5):
            xi = torch.from_numpy(orc.make_image(H_IMG, W_IMG, seed=sd)[0]).cuda()
            plan.forward(xi)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                plan.forward(xi)
            e1.record()
            torch.cuda.synchronize()
            seed_rates[str(sd)] = {"images_per_s": args.steps * 1e3 / e0.elapsed_time(e1), "proposals": int(plan.prop.count.item())}
    barrier()

    # The e2e legs run Python per image.  A full (generation-2) garbage collection in a process that has imported torch walks
    # ~1M objects and takes 70-80 ms (measured: the "periodic stall" of round 1 and the 81 ms outliers of
    # profiles/r02_host_api_profile.txt); a serving process moves its start-up objects out of the collector's way once.
    import gc
    gc.collect()
    gc.freeze()

    # ---------------- e2e (1): the public streaming call -- host image in, host result out, every step
    runner = StreamRunner(pool)
    seq = [imgs_host[i % n_img] for i in range(args.steps)]
    runner.run(seq[: min(4, len(seq))])                      # warm-up
    barrier()
    t0 = time.perf_counter()
    counts = runner.run(seq)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    assert len(counts) == args.steps and all(c > 0 for c in counts)
    e2e_f32_val = world * args.steps / shard.max_over_ranks(t_e2e, device="cuda")
    # same streaming call fed with RAW uint8 375x625 BGR images: mean-subtract + OpenCV-compatible bilinear resize to
    # 600x1000 run on the device (forward.py:34-45 moved onto the GPU)
    rng8 = np.random.default_rng(7 + rank)
    raw = []
    for _ in range(n_img):
        blk = _ops.PinnedBlock((375, 625, 3), np.uint8)
        blk.np[...] = rng8.integers(0, 256, (375, 625, 3), dtype=np.uint8)
        raw.append(blk)
    runner8 = StreamRunner(pool, src_hw=(375, 625))
    seq8 = [raw[i % n_img] for i in range(args.steps)]
    runner8.run(seq8[: min(4, len(seq8))])
    barrier()
    t0 = time.perf_counter()
    runner8.run(seq8)
    torch.cuda.synchronize()
    e2e8_val = world * args.steps / shard.max_over_ranks(time.perf_counter() - t0, device="cuda")

    # ---------------- e2e (2): the REFERENCE's interface -- models.faster_rcnn.FasterRCNN.__call__ fed a host float32
    # (1,3,600,1000) chainer.Variable + img_info, then the caller's 20 models.cpu_nms.cpu_nms calls (forward.py:88-99,48-57)
    import threading

    def cgroup_cpu():
        out = {}
        for name in ("cpu.max", "cpu.stat"):
            try:
                with open("/sys/fs/cgroup/" + name) as f:
                    out[name] = f.read().split()
            except OSError:
                pass
        st = out.get("cpu.stat", [])
        d = {st[i]: int(st[i + 1]) for i in range(0, len(st) - 1, 2) if st[i + 1].isdigit()}
        return {"cpu_max": " ".join(out.get("cpu.max", [])) or None, "nr_throttled": d.get("nr_throttled"),
                "throttled_usec": d.get("throttled_usec")}
    cg0 = cgroup_cpu()
    model = build_reference_api_model(params)
    model.precision = args.precision
    from chainer import Variable
    from models.cpu_nms import cpu_nms as ref_nms
    info_var = Variable(np.array([[H_IMG, W_IMG]], dtype=np.int32))
    x_vars = [Variable(a) for a in imgs_np]
    for i in range(3):
        reference_api_image(model, x_vars[i % n_img], info_var, ref_nms, np)
    barrier()
    from frcnn_b200 import engine as _engine_mod
    _engine_mod.HOST_PROFILE = []
    per_image = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        ta = time.perf_counter()
        r_api = reference_api_image(model, x_vars[i % n_img], info_var, ref_nms, np)
        per_image.append(1e3 * (time.perf_counter() - ta))
    t_api = time.perf_counter() - t0
    phases = np.array(_engine_mod.HOST_PROFILE)
    _engine_mod.HOST_PROFILE = None
    per_image = np.array(per_image)
    api_phases = {"upload_pageable_to_device_ms_median": float(np.median(phases[:, 1])),
                  "graph_replay_enqueue_ms_median": float(np.median(phases[:, 2])), "d2h_and_wait_ms_median": float(np.median(phases[:, 3])),
                  "forward_host_ms_mean": float(phases.sum(1).mean()), "forward_host_ms_max": float(phases.sum(1).max()),
                  "per_image_ms_median": float(np.median(per_image)), "per_image_ms_mean": float(per_image.mean()),
                  "per_image_ms_p90": float(np.percentile(per_image, 90)), "per_image_ms_max": float(per_image.max())}
    api_serial = world * args.steps / shard.max_over_ranks(t_api, device="cuda")
    # the same serial loop with the in-graph hand-off of the per-class NMS switched off: every cpu_nms call is its own kernel
    # launch + host round trip (models/cpu_nms.py)
    import models.cpu_nms as _caller_nms
    _caller_nms.HANDOFF = False
    reference_api_image(model, x_vars[0], info_var, ref_nms, np)
    t0 = time.perf_counter()
    for i in range(args.steps):
        reference_api_image(model, x_vars[i % n_img], info_var, ref_nms, np)
    api_serial_standalone = world * args.steps / shard.max_over_ranks(time.perf_counter() - t0, device="cuda")
    _caller_nms.HANDOFF = True
    # the model call alone (no caller NMS), serial: where the time of the serial number goes
    t0 = time.perf_counter()
    for i in range(args.steps):
        model(x_vars[i % n_img], info_var)
    api_model_only_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    # T caller threads, each running the same serial per-image code on its own images (a thread-per-request server):
    # the drop-in keeps a plan per calling thread, so the threads' graphs overlap on the GPU
    T = max(1, args.api_threads)
    # every caller thread (and every rank's main thread) spins on a core while it waits for the GPU: stay inside the
    # container's CPU quota (the GPU boxes: cpu.max = 16 CPUs) when several ranks share it
    try:
        q = cg0["cpu_max"].split() if cg0["cpu_max"] else []
        cpus = int(q[0]) // int(q[1]) if len(q) == 2 and q[0] != "max" else (os.cpu_count() or 8)
    except (ValueError, ZeroDivisionError):
        cpus = os.cpu_count() or 8
    T = max(2, min(T, cpus // world - 1)) if world > 1 else T
    # every image makes ~45 short library calls that release the GIL; with CPython's default 5 ms switch interval a thread
    # coming back from such a call can wait that long for the GIL while another one runs bytecode -- a server that drives
    # the model from several threads lowers the interval (the caller's setting, restored below)
    import sys as _sys
    old_switch = _sys.getswitchinterval()
    _sys.setswitchinterval(1e-4)
    per = [(args.steps + T - 1 - k) // T for k in range(T)]          # --steps images over the T threads (e2e.images_timed)

    def threads_leg():
        errs = []
        thread_secs = [0.0] * T

        def worker(k, n_local, sync):
            try:
                torch.cuda.set_device(local_rank)
                if args.smem_reserve_kb:
                    _ops.set_conv_smem_reserve(1024 * args.smem_reserve_kb)
                for i in range(2):
                    reference_api_image(model, x_vars[(k + i) % n_img], info_var, ref_nms, np)     # per-thread plan + graph
                sync.wait()
                tw = time.perf_counter()
                for i in range(n_local):
                    reference_api_image(model, x_vars[(k + i) % n_img], info_var, ref_nms, np)
                thread_secs[k] = time.perf_counter() - tw
            except Exception as exc:          # noqa: BLE001
                errs.append(repr(exc))
                try:
                    sync.abort()
                except Exception:             # noqa: BLE001
                    pass
        sync = threading.Barrier(T + 1)
        ths = [threading.Thread(target=worker, args=(k, per[k], sync)) for k in range(T)]
        for t in ths:
            t.start()
        try:
            sync.wait()
        except threading.BrokenBarrierError:
            pass
        t0 = time.perf_counter()
        for t in ths:
            t.join()
        t_thr = time.perf_counter() - t0
        if errs:
            raise RuntimeError("reference-API worker failed: %s" % errs[0])
        # the rate of the threads' own timed loops (first start to last finish is what t_thr adds: thread start-up and teardown)
        t_loop = max(thread_secs) if all(v > 0 for v in thread_secs) else t_thr
        return world * sum(per) / shard.max_over_ranks(t_loop, device="cuda"), t_thr, thread_secs

    nms_stats0 = dict(_caller_nms.stats)
    api_threads, t_thr, thread_secs = threads_leg()
    nms_stats1 = dict(_caller_nms.stats)
    _caller_nms.HANDOFF = False
    api_threads_standalone, _, thread_secs_standalone = threads_leg()
    _caller_nms.HANDOFF = True
    _sys.setswitchinterval(old_switch)
    link = host_link_probe(torch) if rank == 0 else None
    cg1 = cgroup_cpu()
    cgroup = {"cpu_max": cg1["cpu_max"],
              "throttled_periods_during_api_legs": None if cg1["nr_throttled"] is None or cg0["nr_throttled"] is None
              else cg1["nr_throttled"] - cg0["nr_throttled"],
              "throttled_ms_during_api_legs": None if cg1["throttled_usec"] is None or cg0["throttled_usec"] is None
              else (cg1["throttled_usec"] - cg0["throttled_usec"]) / 1e3}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the tensor-core kernel (live, CUDA events, rank 0)
    pk = {}
    if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
    peak_burst = pk.get("bf16_tflops", 1590.0)
    peak_sus = pk.get("bf16_tflops_sustained", 1421.6)
    peak_hbm = pk.get("hbm_gbs", 6571.9)
    peak_src = "MEASURED_PEAKS.json" if pk else "fallback (B200_PROFILING.md)"
    conv_rows = [r for r in table if " k3" in r[0] or "->64 k1" in r[0]]   # trunk + RPN convs (3x3 incl. conv1_1, the twin 1x1)
    conv_ms = sum(r[1] for r in conv_rows)
    all_ms = sum(r[1] for r in table)
    exec_mult = 3.0 if args.precision == "bf16x3" else 1.0
    traffic, traffic_src, hbm_frac = None, None, None
    tpath = os.path.join(ROOT, "profiles", "r02_conv_stack_dram.json")
    if args.precision == "bf16x3" and os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_src = tj["conv_stack_dram_bytes_per_step"], tj["source"]
        hbm_frac = hbm_fractions(tj, table, peak_hbm)
    achieved = CONV_STACK_GFLOP / conv_ms          # GFLOP/ms == TFLOP/s (algorithmic flops)
    sus_ips = n_sus / (ms_sus / 1e3)               # per rank set: all ranks ran n_sus images in ms_sus
    roofline = {
        "bound": "tensor", "kernel": "conv_gemm_kernel (tcgen05 implicit-GEMM; %d GEMM launches/step)" % len(table),
        # isolated per-launch timings (a spin kernel ahead of every launch, clocks near max) -> the BURST peak applies
        "achieved": achieved, "peak": peak_burst, "unit": "TFLOP/s", "frac": achieved / peak_burst,
        "peak_source": "%s bf16_tflops (burst: every launch timed alone between CUDA events)" % peak_src,
        "algorithmic_gflop_per_step": CONV_STACK_GFLOP, "conv_stack_ms": conv_ms, "all_gemm_ms": all_ms,
        "executed_mma_flop_multiplier": exec_mult, "executed_tflops": achieved * exec_mult,
        "executed_frac_of_burst": achieved * exec_mult / peak_burst,
        # the whole step over a long run against the SUSTAINED peak: images/s x conv-stack GFLOP
        "sustained": {"images": n_sus, "images_per_s_per_gpu": sus_ips, "ms_per_image": ms_sus / n_sus,
                      "achieved": sus_ips * CONV_STACK_GFLOP / 1e3, "peak": peak_sus, "unit": "TFLOP/s",
                      "frac": sus_ips * CONV_STACK_GFLOP / 1e3 / peak_sus,
                      "executed_frac": sus_ips * CONV_STACK_GFLOP * exec_mult / 1e3 / peak_sus,
                      "note": "whole forward steps (3 images in flight), conv-stack flops only in the numerator; "
                              "peak = bf16_tflops_sustained"},
        "traffic": traffic,     # DRAM read+write bytes of the conv-stack launches of one step (ncu pass of this binary)
        "traffic_source": traffic_src,
        # every conv-stack activation written once + read once (hi+lo planes, 4 B/elem), the im2col input read
        # once, weights (17.1 M params, hi+lo) read once: 1.02 GB (DESIGN.md 4)
        "algorithmic_bytes_per_step": 1.02e9 if args.precision == "bf16x3" else 0.51e9,
        "hbm_peak_gbs": peak_hbm,
        "hbm_fractions": hbm_frac,   # per-kernel DRAM GB/s over the HBM peak for the kernels that move the most bytes
        "layers": [{"shape": n, "ms": round(m, 4), "tflops_algorithmic": round(g / m, 1)} for n, m, g in table],
    }

    # ---------------- CPU baseline (rank 0, N == 1 only): the oracle pipeline on this box's cores
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        import build_ref
        cores = pick_cpu_threads(torch)
        ref_nms_c = build_ref.load()
        raw0 = np.random.default_rng(7).integers(0, 256, (375, 625, 3), dtype=np.uint8)
        info = np.array([[H_IMG, W_IMG]], np.int32)
        cpu_pipeline_once(orc, params, None, info, ref_nms_c, raw=raw0)          # warm-up
        tt, tn = cpu_pipeline_once(orc, params, None, info, ref_nms_c, raw=raw0)
        cpu_baseline = {"value": 1.0 / tt, "unit": "images/s", "cores": cores,
                        "kind": "reference" if ref_nms_c is not None else "port",
                        "sample": "1 whole image (raw 375x625 -> 600x1000) after 1 warm-up (%.2f s, NMS %.2f s); dense ops torch-CPU fp32 "
                                  "stand-in for Chainer, NMS = %s" %
                                  (tt, tn, "reference cpu_nms.pyx" if ref_nms_c is not None else "C port of cpu_nms.pyx")}

    d2h_api = 4 * plan.result_words()
    line = {
        "metric": "images/sec end-to-end VGG16 Faster R-CNN forward @600x1000",
        "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16x3 (bf16 hi/lo split operands, 3 tcgen05 MMAs per product, fp32 accumulate)"
                 if args.precision == "bf16x3" else "bf16 (fp32 accumulate)",
        "data": "synthetic",
        "config": bench_config(),
        "detail": {"precision": args.precision, "proposals_last_step": R_last, "detections_conf_0.8_last_step": n_conf_last,
                   "unique_fg_scores_last_step": [unique_fg, int(fg.numel())],
                   "images_in_flight_per_gpu": len(pool),
                   "one_image_in_flight": {"images_per_s_this_rank": args.steps / (ms_single / 1e3),
                                           "ms_per_image": ms_single / args.steps},
                   "seeds_one_image_in_flight": seed_rates,
                   "cuda_graph": True, "programmatic_dependent_launch": os.environ.get("FRCNN_PDL", "0") == "1",
                   "launches_per_image": plan.n_launches,
                   "frac_of_conv_roofline_burst": (value / world) * CONV_STACK_GFLOP / 1e3 / peak_burst},
        "clocks": clocks,
        # headline e2e = the REFERENCE's interface: FasterRCNN.__call__ with a host float32 (1,3,600,1000) Variable and
        # img_info, then the caller's 20 cpu_nms calls on host arrays -- per image, inside the timed region: the upload of
        # the 7.2 MB image, the graph (which, as the model's default caller_nms_thresh = 0.3 says, also runs forward.py's
        # per-class NMS), ONE download of (prob, boxes, proposals, keep lists), and the 20 cpu_nms calls, each of which
        # checks its rows bit for bit against the downloaded block and hands the device-computed keep list over
        # (models/cpu_nms.py).  `*_standalone_nms` = the same with that hand-off switched off: 20 kernel launches + host
        # round trips per image.
        "e2e": {"value": api_threads, "unit": "images/s", "h2d_bytes_per_step": 4 * 3 * H_IMG * W_IMG,
                "d2h_bytes_per_step": d2h_api,
                "mode": "models.faster_rcnn.FasterRCNN.__call__(Variable float32 (1,3,600,1000) HOST, img_info) + 20 x "
                        "models.cpu_nms.cpu_nms(dets, 0.3) per image (forward.py:88-99,48-57), %d caller threads; per-class NMS "
                        "computed in the image's graph (frcnn_detect), handed to cpu_nms after a bit-exact input check" % T,
                "cpu_nms_calls": {"handed_over_from_graph": nms_stats1["handoff"] - nms_stats0["handoff"],
                                  "standalone_kernel": nms_stats1["standalone"] - nms_stats0["standalone"]},
                "reference_api_threads_standalone_nms": {"value": api_threads_standalone, "unit": "images/s",
                                                         "h2d_bytes_per_step": 4 * 3 * H_IMG * W_IMG + 20 * 300 * 5 * 4,
                                                         "d2h_bytes_per_step": d2h_api + 20 * 300 * 4,
                                                         "thread_seconds": [round(v, 4) for v in thread_secs_standalone]},
                "reference_api_one_thread_standalone_nms": {"value": api_serial_standalone, "unit": "images/s"},
                "reference_api_one_thread": {"value": api_serial, "unit": "images/s", "ms_per_image": 1e3 / (api_serial / world),
                                             "model_call_only_ms": api_model_only_ms, "last": list(r_api), "phases": api_phases},
                "reference_api_threads": T, "images_timed": int(sum(per)), "reference_api_wall_incl_thread_start_stop_s": round(t_thr, 4), "reference_api_thread_seconds": [round(v, 4) for v in thread_secs],
                "stream_runner_raw_uint8": {"value": e2e8_val, "unit": "images/s", "h2d_bytes_per_step": runner8.h2d_bytes,
                                            "d2h_bytes_per_step": runner8.d2h_bytes,
                                            "note": "the build's own streaming API (engine.StreamRunner): pinned RAW uint8 375x625 "
                                                    "image H2D + device preprocessing (forward.py:34-45) + graph incl. per-class "
                                                    "NMS + one D2H of (prob, boxes, proposals, keep lists), ring of %d slots" % runner8.depth},
                "stream_runner_float32": {"value": e2e_f32_val, "unit": "images/s", "h2d_bytes_per_step": runner.h2d_bytes,
                                          "d2h_bytes_per_step": runner.d2h_bytes},
                "host_link": link, "host_cgroup_cpu": cgroup},
        "gpu_launches": plan.n_launches * args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_train_arm(args, rank, local_rank, world):
    """Secondary workload (BASELINE config #5, a "next" row): one train_rpn.py step per image -- forward, AnchorTargetLayer,
    RPN losses, backward through 15 convs, gradient all-reduce over the ranks, WeightDecay + MomentumSGD.  Not the headline."""
    import torch
    import frcnn_oracle as orc
    from frcnn_b200 import shard
    from frcnn_b200.train_engine import RpnTrainer
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    anchors = orc.generate_anchors(ratios=(0.5, 1, 2), scales=(8, 16, 32))
    params = orc.make_params(seed=1234)
    tr = RpnTrainer(params, H_IMG, W_IMG, anchors, precision=args.precision, subsample="device")
    tr.set_grad_exchange(args.grad_dtype, overlap=not args.no_overlap)
    imgs = [torch.from_numpy(orc.make_image(H_IMG, W_IMG, seed=shard.image_seed(rank, i))[0]).cuda() for i in range(4)]
    gt = torch.tensor([[100, 120, 400, 380, 3], [500, 200, 900, 560, 7], [50, 50, 200, 180, 1], [600, 30, 780, 150, 5]],
                      dtype=torch.float32).cuda()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    for i in range(max(args.warmup, 3)):
        tr.step(imgs[i % 4], gt)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        tr.step(imgs[i % 4], gt)
    e1.record()
    barrier()
    ms = shard.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    clocks = sampler.stop() if rank == 0 else None
    losses = [float(v) for v in tr.last_losses.cpu().numpy()]
    # exposed gradient exchange: per step, the time between "backward enqueued work done" (compute stream) and "all-reduce
    # done" (communication stream), CUDA events, 8 extra steps with a sync after each; max over ranks of the median
    exposed = []
    for i in range(8):
        tr.step(imgs[i % 4], gt)
        torch.cuda.synchronize()
        exposed.append(tr.last_exposed_exchange_ms())
    exposed_ms = shard.max_over_ranks(sorted(exposed)[len(exposed) // 2], device="cuda") if world > 1 else 0.0
    if rank == 0:
        cpu_baseline = None
        if not args.no_cpu_baseline and world == 1:
            cores = pick_cpu_threads(torch)
            x = orc.make_image(H_IMG, W_IMG, seed=0)
            info = np.array([[H_IMG, W_IMG]], np.int32)
            t0 = time.perf_counter()
            r = orc.anchor_target_layer(38, 63, gt.cpu().numpy()[None], info, choice=lambda a, n: np.asarray(a)[:n])
            orc.rpn_train_step(params, x, r["labels"], r["targets"], r["inds_inside"], dtype="float32")
            tt = time.perf_counter() - t0
            cpu_baseline = {"value": 1.0 / tt, "unit": "images/s", "cores": cores, "kind": "port",
                            "sample": "1 step, 600x1000: AnchorTargetLayer restatement + torch-CPU fp32 autograd standing in for "
                                      "Chainer's backward (%.1f s)" % tt}
        print(json.dumps({
            "metric": "images/sec through the train_rpn.py step (forward + AnchorTargetLayer + RPN loss + backward + MomentumSGD) @600x1000",
            "value": world * args.steps / (ms / 1e3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": "train_rpn.py step, VGG16 trunk + RPN trainable, one 600x1000 image per GPU per step, "
                                   "all-reduce(SUM) of the gradient bucket (config #5; secondary workload)",
                       "gradient_exchange": {"dtype": args.grad_dtype, "bucket_bytes": int(tr.g_flat.numel()) * (2 if args.grad_dtype == "bf16" else 4),
                                             "buckets": "deep layers (conv4_1..heads) reduced on a side stream during the rest of "
                                                        "backward; shallow layers after it" if not args.no_overlap else "one all-reduce after backward",
                                             "exposed_ms_median_max_over_ranks": exposed_ms},
                       "last_losses_cls_bbox_acc_total": losses},
            "clocks": clocks, "cpu_baseline": cpu_baseline}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_train_rcnn_arm(args, rank, local_rank, world):
    """Secondary workload: one train_rcnn.py step per image (frozen RPN -> ProposalTargetLayer -> RoI pool -> fc6/fc7 with
    dropout -> losses -> backward through head, RoI pool and trunk -> MomentumSGD), device-side sampling disabled: the
    reference-faithful NumPy sampling (one small D2H per step) is what is timed.  Not the headline."""
    import torch
    import frcnn_oracle as orc
    from frcnn_b200 import shard
    from frcnn_b200.train_engine import RcnnTrainer
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    anchors = orc.generate_anchors(ratios=(0.5, 1, 2), scales=(8, 16, 32))
    params = orc.make_params(seed=1234)
    tr = RcnnTrainer(params, H_IMG, W_IMG, anchors, precision=args.precision, lr=1e-5)
    imgs = [torch.from_numpy(orc.make_image(H_IMG, W_IMG, seed=shard.image_seed(rank, i))[0]).cuda() for i in range(4)]
    gt = torch.tensor([[100, 120, 400, 380, 3], [500, 200, 900, 560, 7], [50, 50, 200, 180, 1], [600, 30, 780, 150, 5]],
                      dtype=torch.float32).cuda()
    np.random.seed(1234 + rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    for i in range(max(args.warmup, 3)):
        tr.step(imgs[i % 4], gt)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        tr.step(imgs[i % 4], gt)
    e1.record()
    barrier()
    ms = shard.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        print(json.dumps({
            "metric": "images/sec through the train_rcnn.py step @600x1000 (300 proposals, 128 RoIs per image)",
            "value": world * args.steps / (ms / 1e3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": "train_rcnn.py step, trunk + fc6/fc7/cls_score/bbox_pred trainable, one 600x1000 image per GPU "
                                   "per step (secondary workload)", "kept_rois_last_step": int(tr.keep.numel()),
                       "last_losses_cls_bbox_acc_total": [float(v) for v in tr.last_losses.cpu().numpy()]},
            "clocks": clocks}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_resnet_arm(args, rank, local_rank, world):
    """Secondary workload (BASELINE config #4, a "next" row): ResNet-101 trunk Faster R-CNN forward, 800x1333, 1000 proposals,
    one image per GPU.  Device-timed with inputs resident in HBM, args.in_flight images in flight.  Not the headline."""
    import torch
    import frcnn_oracle as orc
    from frcnn_b200 import shard
    from frcnn_b200.engine import LanePool
    from frcnn_b200.resnet_engine import ResNetEngine
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    H, W = 800, 1333
    anchors = orc.generate_anchors(ratios=(0.5, 1, 2), scales=(8, 16, 32))
    params = orc.make_resnet_params(101, seed=4321)
    eng = ResNetEngine(params, 101, precision=args.precision, anchors=anchors, use_graph=True, post_n=1000)
    plan = eng.plan(H, W)
    imgs = [torch.from_numpy(orc.make_image(H, W, seed=shard.image_seed(rank, i))[0]).cuda() for i in range(4)]
    pool = LanePool(plan, lanes=args.in_flight)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    pool.fork()
    for i in range(max(args.warmup, 3)):
        pool.submit(i, imgs[i % 4])
    pool.join()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    pool.fork()
    for i in range(args.steps):
        pool.submit(i, imgs[i % 4])
    pool.join()
    e1.record()
    barrier()
    ms = shard.max_over_ranks(e0.elapsed_time(e1), device="cuda")
    clocks = sampler.stop() if rank == 0 else None
    R_last = int(plan.prop.count.item())
    barrier()
    e0.record()
    for i in range(args.steps):
        plan.forward(imgs[i % 4])
    e1.record()
    barrier()
    ms1 = e0.elapsed_time(e1)
    if rank == 0:
        print(json.dumps({
            "metric": "images/sec end-to-end ResNet-101 Faster R-CNN forward @800x1333, 1000 proposals",
            "value": world * args.steps / (ms / 1e3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": "ResNet-101 trunk Faster R-CNN forward, synthetic 800x1333, 1000 proposals, one image per GPU "
                                   "(config #4; secondary workload)", "images_in_flight_per_gpu": len(pool),
                       "proposals_last_step": R_last, "one_image_in_flight_ms": ms1 / args.steps,
                       "launches_per_image": plan.n_launches},
            "clocks": clocks}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--in-flight", type=int, default=4, help="independent images in flight per GPU (streams/graphs)")
    ap.add_argument("--grad-dtype", default="bf16", choices=["bf16", "fp32"],
                    help="train_rpn workload: dtype of the all-reduced gradient bucket (BASELINE config #5 says bf16)")
    ap.add_argument("--no-overlap", action="store_true", help="train_rpn workload: one all-reduce after backward instead of bucket overlap")
    ap.add_argument("--smem-reserve-kb", type=int, default=0,
                    help="shared memory per SM the conv kernels leave to other streams' small kernels (tuning experiment)")
    ap.add_argument("--api-threads", type=int, default=8, help="caller threads of the reference-interface e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="forward workload: write the results of the last timed image as DIR/<name>.npy (rank 0)")
    ap.add_argument("--workload", default="forward", choices=["forward", "train_rpn", "train_rcnn", "resnet101"],
                    help="forward = the headline metric (default); train_rpn / resnet101 = secondary workloads (configs #5 / #4)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.workload == "train_rpn":
        run_train_arm(args, rank, local_rank, world)
        return
    if args.workload == "resnet101":
        run_resnet_arm(args, rank, local_rank, world)
        return
    if args.workload == "train_rcnn":
        run_train_rcnn_arm(args, rank, local_rank, world)
        return
    run_b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
