#!/usr/bin/env python
"""bench.py -- candidate-window scoring throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the whole post-MSER detection chain (K1 expand/filter, K2 crop+resize, K5 histogram + fold
x2, K3 masks, K4 score, detection records) over one batch of synthetic 1360x800 BGR frames with 200 MSER-like
candidates per frame (BASELINE.json configs[2]; SURVEY.md section 8(d)).  Frames are sharded by image: every rank owns
its own batch (weak scaling), no collective on the hot path, one small gather of detection records at the end.

Prints ONE JSON line (rank 0).  `value` = raw candidate windows/s, inputs resident in HBM; `e2e` = the same metric
through the public host-buffer API (pinned host frames, H2D + D2H inside the timed region); `roofline` = the dominant
kernel (largest stage time) against the measured HBM peak, `roofline_stages` = the same figure for every stage; `cpu_baseline` = the reference pipeline (oracle/ref_port.py: cv2 + the
reference's Python loops) on the host cores over a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, NBOX, D = 800, 1360, 200, 25
UNIQUE_FRAMES = 32
METRIC = "candidate windows/sec (1360x800 frames, ~200 MSER candidates/frame, detection scoring)"


def bench_config(world):
    """`config` of the JSON line: identical keys and values for both arms (the per-arm batch size is reported beside it)."""
    return {"workload": "synthetic 1360x800 BGR frames, 200 MSER-like candidates/frame, detection-only scoring (BASELINE configs[2])",
            "boxes_per_frame": NBOX, "window": D, "frame_bytes": H * W * 3, "parallelism": "frames sharded by image, dp%d" % world,
            "l2": "inputs larger than L2: every step reads its own batch of distinct resident frames (3.26 MB each, >= 100 MB per step), "
                  "so no step finds its frames in the 126 MB L2"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """Per-kernel DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture, divided by the
    aspect-passing windows of that capture) recorded under profiles/; scaled by the run's window count in the report."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def templates():
    g = np.load(os.path.join(ROOT, "tests", "golden", "det_templates.npz"))
    return g["red6"], g["blue6"]


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML every 10 ms DURING the timed region (B200_PROFILING.md recipe;
    an nvidia-smi subprocess takes longer to start than the timed region lasts)."""

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.t, self.h = index, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # torch device index -> NVML index through the PCI bus id (CUDA_VISIBLE_DEVICES may remap)
            import torch
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            if bus is not None:
                for k in range(pynvml.nvmlDeviceGetCount()):
                    hk = pynvml.nvmlDeviceGetHandleByIndex(k)
                    if pynvml.nvmlDeviceGetPciInfo(hk).bus == bus:
                        self.h = hk
                        break
        except Exception:
            self.h = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h),
                                     nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.h is None:
            return
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        reasons = sorted(k for k, bit in names.items() if any(r & bit for _, r, _ in self.samples))
        sm = [c for c, _, _ in self.samples]
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = None
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "power_w_max": max((p for _, _, p in self.samples), default=None), "reasons": reasons}


def algorithmic_bytes(boxes, offsets, counts, hist_entries=0, row_words=7, enlarge=1.30, D=D, Hf=H, Wf=W, recognize=False):
    """SURVEY.md section 8(d) per-unit figures x the units one launch processes (independent of the implementation).
    K2: in 3*min(w_c,2D)*min(h_c,2D) + out 3*D*D per aspect-passing window; k5_hist: 3*D*D + 16 per window; k5_pairs:
    the sparse histograms + moments + energies read once, bit rows written; k5_fold: in 3*D*D+16 per input window, out
    3*D*D+16 per survivor; K3: 3*D*D in, bit-packed masks out (160 B); K4: 160 B in, 8 out; K6: 3*D*D in, D*D out;
    K7: D*D in, 324 f32 out; K8: 324 f32 in, 6 f64 logits + label out."""
    b = boxes.astype(np.int64)
    w, h = b[:, 2].astype(np.float64), b[:, 3].astype(np.float64)
    pm1 = enlarge - 1
    ratio = w / np.maximum(h, 1e-300)
    ok = (0.8 < ratio) & (ratio < 1.20)
    x1 = np.maximum(b[:, 0] - w * pm1 * 0.5, 0).astype(np.int64); y1 = np.maximum(b[:, 1] - h * pm1 * 0.5, 0).astype(np.int64)
    x2 = (b[:, 0] + b[:, 2] + w * pm1 * 0.5).astype(np.int64); y2 = (b[:, 1] + b[:, 3] + h * pm1 * 0.5).astype(np.int64)
    cw = np.minimum(x2, Wf) - np.minimum(x1, Wf); ch = np.minimum(y2, Hf) - np.minimum(y1, Hf)
    k2_in = (3 * np.minimum(cw, 2 * D) * np.minimum(ch, 2 * D))[ok].sum()
    npass, nsurv = int(ok.sum()), int(counts[2])
    px = D * D
    alg = {
        "k1_expand_filter": int(len(b) * 33),
        "k2_crop_resize": int(k2_in + npass * 3 * px),
        "k5_hist": int(npass * (3 * px + 16)),
        # every window's sparse histogram (4 B per non-zero bin) + moments (48 B) + group energies (100 B) read once,
        # two bit rows written per window
        "k5_pairs": int(4 * hist_entries + npass * (48 + 100 + 8 * row_words)),
        "k5_fold": int(npass * (3 * px + 16) + nsurv * (3 * px + 16)),
        "detections": int(counts[3] * 32),
    }
    if recognize:
        alg.update({"k6_gray": int(nsurv * 4 * px), "k7_hog": int(nsurv * (px + 324 * 4)), "k8_lda": int(nsurv * (324 * 4 + 49))})
    else:
        # inside the chain K3 hands K4 bit-packed masks (2 x 20 words per window); the byte masks of SURVEY's 2*D*D figure are
        # written only by the tsd_color_masks entry point (TSD_KEEP_MASKS=1 restores them in the chain)
        alg.update({"k3_masks": int(nsurv * (3 * px + 8 * ((px + 31) // 32))), "k4_score": int(nsurv * (8 * ((px + 31) // 32) + 8))})
    return alg, npass


# ---------------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """--impl reference: the reference's CPU pipeline (oracle/ref_port.py) on all host cores, same config/metric.
    Rank 0 alone runs; the other ranks exit 0."""
    if rank != 0:
        return
    import multiprocessing as mp
    import tsd_b200
    from oracle import ref_port
    cores = os.cpu_count() or 1
    red6, blue6 = templates()
    fpc = max(1, args.cpu_frames_per_core)
    F = cores * fpc
    frames = tsd_b200.synth.make_frames(min(F, UNIQUE_FRAMES))
    frames = frames[np.arange(F) % len(frames)]
    boxes, off = tsd_b200.synth.make_boxes(F, NBOX)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=ref_port._worker_init, initargs=(red6, blue6)) as pool:
        for _ in range(args.warmup):
            ref_port.run_parallel(pool, frames[:cores], boxes[:off[cores]], off[:cores + 1], cores)
        t0 = time.perf_counter()
        ndet = 0
        for _ in range(args.steps):
            ndet += ref_port.run_parallel(pool, frames, boxes, off, cores)
        dt = time.perf_counter() - t0
    value = F * NBOX * args.steps / dt
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "windows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "frames_per_sec": F * args.steps / dt,
        "config": bench_config(args.gpus), "frames_per_step": F,
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": cores, "kind": "port",
                         "sample": "%d frames x %d candidates per step (%d per core), oracle/ref_port.py = reference pipeline with cv2 + its Python loops" % (F, NBOX, fpc)},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "detections": ndet,
    }
    print(json.dumps(out))


def cpu_baseline_sample(args):
    """Bounded sample of the same workload on the host cores (rank 0, N=1): ~64 frames."""
    import multiprocessing as mp
    import tsd_b200
    from oracle import ref_port
    cores = os.cpu_count() or 1
    red6, blue6 = templates()
    F = max(cores, 64 // cores * cores)
    frames = tsd_b200.synth.make_frames(min(F, UNIQUE_FRAMES))
    frames = frames[np.arange(F) % len(frames)]
    boxes, off = tsd_b200.synth.make_boxes(F, NBOX)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=ref_port._worker_init, initargs=(red6, blue6)) as pool:
        ref_port.run_parallel(pool, frames[:cores], boxes[:off[cores]], off[:cores + 1], cores)      # warm the workers
        t0 = time.perf_counter()
        ref_port.run_parallel(pool, frames, boxes, off, cores)
        dt = time.perf_counter() - t0
    return {"value": F * NBOX / dt, "unit": "windows/s", "cores": cores, "kind": "port", "frames_per_sec": F / dt, "seconds": dt,
            "sample": "%d frames x %d candidates, one worker per host core, oracle/ref_port.py (reference pipeline: cv2 + its Python loops)" % (F, NBOX)}


# ---------------------------------------------------------------------------------------------------------------------
def _time_steps(torch, stream, ctx, fn, steps=10, warm=3):
    for _ in range(warm):
        fn()
    ctx.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    ctx.synchronize()
    return e0.elapsed_time(e1) / steps


def _staged(torch, ctx, stream, fn, steps):
    """Per-stage device times (ms per step) of `steps` enqueues with the library's stage events on (serialised batches)."""
    ctx.set_profiling(True)
    for _ in range(steps):
        fn()
    ctx.synchronize()
    st = {k: v / steps for k, v in ctx.stage_times()}
    ctx.set_profiling(False)
    return st


def recognize_run(torch, tsd_b200, dev, local_rank, rank, world, dist, peak):
    """BASELINE configs[3]: the detect + recognise chain (K1 K2 K5 K5 K6 K7 K8, x1.15 / 32x32, HOG + 6 LDA in f64) on 1024
    synthetic frames PER RANK with the LDA weights the reference fitted (tests/golden/rec_golden.npz).  Runs on every rank: the
    value is the whole job's windows/s over the slowest rank's device time, so the 2/4/8-GPU lines carry detect+recognise."""
    F = 1024
    uniq = tsd_b200.synth.make_frames(16, seed=tsd_b200.synth.FRAME_SEED + 500 + rank)
    boxes, off = tsd_b200.synth.make_boxes(F, NBOX, seed=tsd_b200.synth.BOX_SEED + 500 + rank, enlarge=1.15, D=32)
    d_frames = torch.from_numpy(uniq).to(dev)[torch.arange(F, device=dev) % 16].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    r = np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz"))
    with tsd_b200.Context(device=local_rank, flavour="rec") as rc:
        rc.set_lda(r["lda_W"], r["lda_b"])
        st = torch.cuda.ExternalStream(rc.stream, device=dev)

        def step():
            rc.enqueue_frames(d_frames.data_ptr(), F, H, W, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), mode=tsd_b200.RUN_RECOGNIZE,
                              max_boxes_per_frame=NBOX)
        for _ in range(3):
            step()
        rc.synchronize()
        if dist is not None:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(10):
            step()
        rc.flush()
        e1.record(st)
        rc.synchronize()
        ms = e0.elapsed_time(e1) / 10
        stages = _staged(torch, rc, st, step, 5)
        _, cnt = rc.fetch_detections(int(off[-1]))
        nnz = rc.stat_hist_entries()
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    alg, _ = algorithmic_bytes(boxes, off, cnt, nnz, (NBOX + 31) // 32, enlarge=1.15, D=32, recognize=True)
    rec_only = {k: stages.get(k) for k in ("k6_gray", "k7_hog", "k8_lda") if stages.get(k)}
    dom = max(rec_only, key=rec_only.get) if rec_only else None
    out = {"windows_per_s": world * F * NBOX / (ms * 1e-3), "frames_per_s": world * F / (ms * 1e-3), "ms_per_step": ms, "frames_per_gpu": F, "n_gpus": world,
           "stage_counts": [int(v) for v in cnt], "stages_ms_per_step": stages,
           "stages_alg_gbs": {k: alg.get(k, 0) / (v * 1e-3) / 1e9 for k, v in stages.items() if v > 0 and alg.get(k)},
           "config": "synthetic 1360x800, 200 candidates/frame, x1.15 / 32x32, HOG + 6 LDA (f64) (BASELINE configs[3])"}
    if dom:
        ach = alg[dom] / (rec_only[dom] * 1e-3) / 1e9
        out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                           "algorithmic_bytes_per_launch": alg[dom], "kernel_ms_per_launch": rec_only[dom], "traffic": None,
                           "note": "dominant kernel of the recognition branch (K6/K7/K8); the K1/K2/K5 stages are shared with detection"}
    return out


def sweep_4k(torch, tsd_b200, dev, local_rank, peak):
    """BASELINE configs[4]: candidate-window sweep at 4K frames (3840x2160), 50 .. 2000 candidates per frame, device-resident
    detection chain.  Frames: 8 distinct synthetic 4K frames tiled to the batch; candidates: 16 distinct per-frame lists tiled."""
    H4, W4, U, UB = 2160, 3840, 8, 16
    red6, blue6 = templates()
    uniq = tsd_b200.synth.make_frames(U, H4, W4, seed=tsd_b200.synth.FRAME_SEED + 900)
    d_uniq = torch.from_numpy(uniq).to(dev)
    rows = []
    with tsd_b200.Context(device=local_rank, flavour="det") as ctx:
        ctx.set_templates(red6, blue6)
        st = torch.cuda.ExternalStream(ctx.stream, device=dev)
        for N in (50, 200, 500, 1000, 2000):
            F = 256
            d_frames = d_uniq[torch.arange(F, device=dev) % U].contiguous()       # 256 resident 4K frames = 6.4 GB
            bu, _ = tsd_b200.synth.make_boxes(UB, N, H4, W4, seed=tsd_b200.synth.BOX_SEED + 900 + N)
            boxes = np.ascontiguousarray(bu.reshape(UB, N, 4)[np.arange(F) % UB].reshape(-1, 4))
            off = (np.arange(F + 1) * N).astype(np.int32)
            d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)

            def step():
                ctx.enqueue_frames(d_frames.data_ptr(), F, H4, W4, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), max_boxes_per_frame=N)
            for _ in range(3):
                step()
            ctx.synchronize()
            steps = 10 if N <= 500 else 5
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(steps):
                step()
            ctx.flush()
            e1.record(st)
            ctx.synchronize()
            ms = e0.elapsed_time(e1) / steps
            stages = _staged(torch, ctx, st, step, 3)
            _, cnt = ctx.fetch_detections(int(off[-1]))
            nnz = ctx.stat_hist_entries()
            alg, _ = algorithmic_bytes(boxes, off, cnt, nnz, (min(N, 1024) + 31) // 32, Hf=H4, Wf=W4)
            tot = sum(alg.values())
            rows.append({"candidates_per_frame": N, "frames": F, "windows_per_s": F * N / (ms * 1e-3), "frames_per_s": F / (ms * 1e-3), "ms_per_step": ms,
                         "stage_counts": [int(v) for v in cnt], "stages_ms_per_step": stages,
                         "chain_alg_gbs": tot / (ms * 1e-3) / 1e9, "chain_frac_of_peak": tot / (ms * 1e-3) / 1e9 / peak})
            del d_frames
    return {"config": "synthetic 3840x2160 BGR frames, 256 resident frames (6.4 GB), detection chain, device-resident (BASELINE configs[4])", "rows": rows}


def real_mser_run(torch, tsd_b200, dev, ctx_det, stream_det):
    """The detection chain on REAL frames with REAL cv2.MSER boxes (SURVEY 8(d)): the three stored test frames and the boxes the
    reference's MSER produced for them, tiled to 1024 frames."""
    import cv2
    F = 1024
    g = np.load(os.path.join(ROOT, "tests", "golden", "det_frames.npz"))
    names = ["00604", "00639", "00719"]
    imgs = np.stack([cv2.imread(os.path.join(ROOT, "tests", "golden", "det_frame_%s.png" % k)) for k in names])
    bl = [g[k + "_boxes"].astype(np.int32) for k in names]
    boxes = np.concatenate([bl[f % 3] for f in range(F)])
    off = np.concatenate([[0], np.cumsum([len(bl[f % 3]) for f in range(F)])]).astype(np.int32)
    d_frames = torch.from_numpy(imgs).to(dev)[torch.arange(F, device=dev) % 3].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    mb = int(max(len(b) for b in bl))
    l0 = ctx_det.launch_count
    ms = _time_steps(torch, stream_det, ctx_det, lambda: ctx_det.enqueue_frames(d_frames.data_ptr(), F, H, W, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]),
                                                                                max_boxes_per_frame=mb))
    launches = (ctx_det.launch_count - l0) / 13.0            # 3 warm + 10 timed steps
    _, cnt = ctx_det.fetch_detections(int(off[-1]))
    return {"windows_per_s": int(off[-1]) / (ms * 1e-3), "frames_per_s": F / (ms * 1e-3), "ms_per_step": ms, "frames": F, "launches_per_step": launches,
            "boxes_per_frame_mean": float(off[-1]) / F, "stage_counts": [int(v) for v in cnt],
            "config": "3 real GTSDB test frames + the boxes cv2.MSER(7,200,2000,0.15) gives for them, tiled to 1024 frames"}


def dump_outputs(out_dir, det, counts):
    """--dump-outputs: what a caller of the timed path receives for its last step (Context.fetch_detections), as float64 .npy files,
    so that two builds can be compared output for output on the same seeded inputs.  detections.npy [n,7] = frame, x1, y1, x2, y2,
    id, hundredths in record order; stage_counts.npy [4] = raw, aspect-passing, survivors, detections.  Records beyond 60 MB are
    cut to a fixed seeded sample (kept in record order), so a dump stays under 64 MB.  With --gpus N > 1 only rank 0 calls this, so
    the dump holds rank 0's records (its own frames), not the other ranks'."""
    os.makedirs(out_dir, exist_ok=True)
    cols = ("frame", "x1", "y1", "x2", "y2", "id", "hundredths")
    rec = np.stack([det[c] for c in cols], 1).astype(np.float64)
    cap = (60 << 20) // (8 * len(cols))
    if len(rec) > cap:
        rec = rec[np.sort(np.random.default_rng(0).choice(len(rec), cap, replace=False))]
    np.save(os.path.join(out_dir, "detections.npy"), rec)
    np.save(os.path.join(out_dir, "stage_counts.npy"), counts.astype(np.float64))


def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and so the first-touch placement of its page-locked host frames) to the CPUs of the NUMA node
    the GPU hangs off: the e2e leg reads host memory from the GPU, a remote node costs PCIe/UPI bandwidth.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.replace(",", "").isdigit() else local_rank
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        return None
    return None


def run_b200(args, rank, world, local_rank):
    # The CPU baseline forks worker processes: run it BEFORE this process touches CUDA (rank 0, N=1 only)
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline_sample(args)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    import torch
    import tsd_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    red6, blue6 = templates()
    F = args.frames
    uniq = tsd_b200.synth.make_frames(UNIQUE_FRAMES, seed=tsd_b200.synth.FRAME_SEED + rank)
    boxes, off = tsd_b200.synth.make_boxes(F, NBOX, seed=tsd_b200.synth.BOX_SEED + rank)
    d_uniq = torch.from_numpy(uniq).to(dev)
    d_frames = d_uniq[torch.arange(F, device=dev) % UNIQUE_FRAMES].contiguous()     # F distinct resident frames (3.26 MB each)
    del d_uniq
    d_boxes = torch.from_numpy(boxes).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    nb = int(off[-1])

    ctx = tsd_b200.Context(device=local_rank, flavour="det")
    ctx.set_templates(red6, blue6)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def step():
        ctx.enqueue_frames(d_frames.data_ptr(), F, H, W, d_boxes.data_ptr(), d_off.data_ptr(), nb, max_boxes_per_frame=NBOX)

    for _ in range(max(args.warmup, 3)):
        step()
    ctx.synchronize()
    det, counts = ctx.fetch_detections(nb)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    # ---- timed region: EXACTLY K steps, CUDA events on the launching stream ----------------------------------------
    # (a step splits its frames into chunks that alternate between two streams, so the latency-bound fold of one chunk
    #  overlaps the throughput-bound kernels of the next; the per-kernel times for the roofline come from a second pass
    #  of K steps, right after, with the chunks serialised and CUDA events between the stages)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank)
    l0 = ctx.launch_count
    barrier()
    sampler.start()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ctx.flush()                                              # (overlap mode defers the last batch's join: the stream waits for it here)
    ev1.record(stream)
    ctx.synchronize()
    barrier()
    n_timed = len(sampler.samples)
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *ctx.fetch_detections(nb))
    ctx.set_profiling(True)                                  # second pass: same K steps, serialised, per-stage CUDA events
    evp0, evp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evp0.record(stream)
    for _ in range(args.steps):
        step()
    evp1.record(stream)
    ctx.synchronize()
    stage_ms = dict(ctx.stage_times())
    ms_serial = evp0.elapsed_time(evp1)
    ctx.set_profiling(False)
    # NVML answers in ~10-30 ms, so a short timed region yields few samples: keep sampling over an UNTIMED window of
    # the same steps (>= 0.5 s of the same load) and report both counts
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 0.5:
        for _ in range(4):
            step()
        ctx.synchronize()
    clocks = sampler.stop()
    clocks["samples_in_timed_region"] = n_timed
    clocks["note"] = "NVML, 10 ms period; samples span the timed region plus 0.5 s of the same steps run untimed right after it"
    det, counts = ctx.fetch_detections(nb)
    hist_entries = ctx.stat_hist_entries()
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        from tsd_b200 import sharding
        allrec = sharding.gather_detections(det, rank * F, dist, device=dev)      # the one small NCCL gather, for the report
        ndet_total = len(allrec)
    else:
        ndet_total = len(det)
    value = world * F * NBOX * args.steps / (ms * 1e-3)

    # ---- e2e: public host-buffer API, host frames, H2D + D2H inside the timed region ----------------------------------------
    Fe = min(args.e2e_frames, F) if not args.no_e2e else 1
    h_frames = torch.empty((Fe, H, W, 3), dtype=torch.uint8).pin_memory()
    for f0 in range(0, Fe, 256):
        h_frames[f0:min(f0 + 256, Fe)].copy_(d_frames[f0:min(f0 + 256, Fe)])
    hf = h_frames.numpy()
    hb, ho = boxes[:off[Fe]], off[:Fe + 1]

    def e2e_leg(frames_np, steps):
        for _ in range(2):
            ctx.detect_frames(frames_np, hb, ho)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            edet, ecounts = ctx.detect_frames(frames_np, hb, ho)
        ctx.synchronize()
        dt = (time.perf_counter() - t0) / steps
        if dist is not None:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt, edet, ecounts
    ctx.stat_staged_bytes(reset=True)
    e_dt, edet, ecounts = e2e_leg(hf, args.e2e_steps)
    staged = ctx.stat_staged_bytes(reset=True) // (args.e2e_steps + 2)          # (2 warm-up calls inside e2e_leg): bytes per call, counted on the device
    alg_e, _ = algorithmic_bytes(hb, ho, ecounts)
    roi_bytes = int(alg_e["k2_crop_resize"] - int(ecounts[1]) * 3 * D * D)      # source bytes of the candidate ROIs (section 8(d) formula)
    e2e = {"value": world * Fe * NBOX / e_dt, "unit": "windows/s", "h2d_bytes_per_step": int(staged + hb.nbytes + ho.nbytes),
           "d2h_bytes_per_step": int(len(edet) * 32 + 16), "frames_per_step": Fe, "ms_per_step": e_dt * 1e3,
           "frames_per_sec": world * Fe / e_dt, "host_input_bytes_per_step": int(hf.nbytes + hb.nbytes + ho.nbytes),
           "roi_bytes_algorithmic": roi_bytes, "h2d_gbs": (staged + hb.nbytes + ho.nbytes) / e_dt / 1e9,
           "api": "Context.detect_frames (tsd_detect_frames, TSD_MEM_HOST) on PAGE-LOCKED host frames: every 32-byte sector the candidate ROIs "
                  "touch is copied over PCIe once per batch into a device mirror (stage_mark + stage_copy kernels), then the chain runs on the "
                  "mirror; h2d_bytes_per_step = those bytes (counted by the copy kernel) + boxes; detection records D2H"}
    if not args.no_e2e and world == 1:
        # the same call on PAGEABLE frames (what cv2.imread returns): whole frames are copied in double-buffered chunks
        pg = np.array(hf[:min(Fe, 256)], copy=True)
        hb_s, ho_s = hb, ho
        hb, ho = boxes[:off[len(pg)]], off[:len(pg) + 1]
        p_dt, pdet, _ = e2e_leg(pg, 3)
        e2e["pageable"] = {"value": len(pg) * NBOX / p_dt, "unit": "windows/s", "frames_per_step": len(pg), "ms_per_step": p_dt * 1e3,
                           "h2d_bytes_per_step": int(pg.nbytes + hb.nbytes + ho.nbytes), "d2h_bytes_per_step": int(len(pdet) * 32 + 16),
                           "api": "same call, pageable numpy frames: 32-frame chunks copied whole (cudaMemcpyAsync from pageable memory), chain of chunk k under the copy of chunk k+1"}
        hb, ho = hb_s, ho_s

    peak, peak_src = load_peaks()
    secondary = None
    if not args.no_secondary:
        secondary = {}
        try:                                                 # every rank (collective timing inside); never breaks the bench line
            secondary["recognize_chain"] = recognize_run(torch, tsd_b200, dev, local_rank, rank, world, dist, peak)
        except Exception as e:
            secondary["recognize_chain"] = {"error": str(e)[:300]}
            if dist is not None:
                raise
        if rank == 0:
            try:
                secondary["real_mser_frames"] = real_mser_run(torch, tsd_b200, dev, ctx, stream)
            except Exception as e:
                secondary["real_mser_frames"] = {"error": str(e)[:300]}
            if world == 1 and not args.no_sweep:
                del d_frames                                 # the sweep needs 6.4 GB of its own
                try:
                    secondary["sweep_4k"] = sweep_4k(torch, tsd_b200, dev, local_rank, peak)
                except Exception as e:
                    secondary["sweep_4k"] = {"error": str(e)[:300]}
    if rank == 0:
        alg, npass = algorithmic_bytes(boxes, off, counts, hist_entries, (NBOX + 31) // 32)
        traffic = load_traffic()
        per_stage = {k: v / args.steps for k, v in stage_ms.items()}
        dom = max(per_stage, key=per_stage.get) if per_stage else "k2_crop_resize"
        achieved = alg.get(dom, 0) / (per_stage.get(dom, 1e9) * 1e-3) / 1e9
        fused_bytes = sum(alg.values())
        out = {
            "metric": METRIC, "value": value, "unit": "windows/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "frames_per_sec": world * F * args.steps / (ms * 1e-3),
            "config": bench_config(world), "frames_per_step": F * world, "frames_per_gpu": F,
            "resident": "%d frames (%.1f GB) per GPU, ROI bytes touched per step %.0f MB" % (F, F * H * W * 3 / 1e9, alg["k2_crop_resize"] / 1e6),
            "stage_counts": {"raw": int(counts[0]), "aspect_passing": int(counts[1]), "survivors": int(counts[2]), "detections": int(counts[3])},
            "detections_all_ranks": int(ndet_total),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic.get(dom, {}).get("dram_bytes_per_window", 0) * npass or None,
                         "traffic_source": traffic.get(dom, {}).get("source"), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg.get(dom, 0),
                         "kernel_ms_per_launch": per_stage.get(dom)},
            # the same figure for every stage (the fold is latency-bound and mostly hidden under the next batch's kernels; K2 is the
            # heaviest mover of bytes and the kernel the round-1 review named)
            "roofline_stages": {k: {"achieved": alg.get(k, 0) / (v * 1e-3) / 1e9, "frac": alg.get(k, 0) / (v * 1e-3) / 1e9 / peak, "ms": v,
                                    "algorithmic_bytes_per_launch": alg.get(k, 0),
                                    "traffic": traffic.get(k, {}).get("dram_bytes_per_window", 0) * npass or None}
                                for k, v in per_stage.items() if v > 0},
            "stages_ms_per_step": per_stage, "ms_per_step_serialised": ms_serial / args.steps,
            "stages_alg_gbs": {k: alg.get(k, 0) / (v * 1e-3) / 1e9 for k, v in per_stage.items() if v > 0},
            "chain": {"algorithmic_bytes_per_step": fused_bytes, "gbs": fused_bytes / (ms / args.steps * 1e-3) / 1e9,
                      "frac_of_peak": fused_bytes / (ms / args.steps * 1e-3) / 1e9 / peak},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "numa_node_rank0": numa_node,
        }
        if cpu_base is not None:
            out["cpu_baseline"] = cpu_base
        if secondary is not None:
            out["secondary"] = secondary
        print(json.dumps(out))
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=4096, help="resident frames per GPU per step")
    ap.add_argument("--e2e-frames", type=int, default=1024)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-frames-per-core", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary (recognition chain, real-MSER frames) measurements")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 4K candidate sweep (BASELINE configs[4]) of the secondary measurements")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (used for the ncu launch list of the device-resident step)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the detection records and stage counts of the last timed step (rank 0) "
                                                         "to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29400 + os.getpid() % 500), os.path.abspath(__file__)] + sys.argv[1:]
        os.environ["WORLD_SIZE_LAUNCHED"] = "1"
        raise SystemExit(subprocess.call(cmd))
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
