"""One batch of frames of different sizes against the same frames as size-grouped uniform calls.

Device-resident: 4096 frames, 1024 each of 640x480, 1360x800, 1920x1080 and 2560x1440 (about 22 GB, larger than L2 by far),
200 synth.make_boxes candidates per frame at each frame's size, RUN_DETECT.  One step is either ONE tsd_enqueue_frames_ragged
call over a table that interleaves the four sizes, or FOUR tsd_enqueue_frames calls, one per size group (the same frames, each
group contiguous).  The two alternate in one process; each step is timed with CUDA events on the context's stream (enqueue,
tsd_flush, synchronise) and the tool reports windows/s (aspect-passing windows of the step over its time), median and spread.
Both give the same records per frame (checked).

Host: HOST_PER_SIZE pageable numpy frames of each size through Context.detect_frames, as one mixed list (packed into the
context's page-locked buffer, staged route) against np.stack per size group (four pageable uniform calls); host clock around
each call, which synchronises.

Writes one JSON file (--out, default profiles/ragged_step_b200.json) with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SIZES = ((480, 640), (800, 1360), (1080, 1920), (1440, 2560))     # (H, W)
PER_SIZE, NBOX, DISTINCT, HOST_PER_SIZE = 1024, 200, 8, 64


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not measured"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not measured"
    return info


def stats(v):
    v = np.asarray(v, np.float64)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "spread_pct": float((v.max() - v.min()) / np.median(v) * 100), "n": len(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ragged_step_b200.json"))
    a = ap.parse_args()
    import torch
    import tsd_b200
    from tsd_b200 import synth
    dev = torch.device("cuda", 0)
    red6, blue6 = (np.load(os.path.join(ROOT, "tests", "golden", "det_templates.npz"))[k] for k in ("red6", "blue6"))
    ctx = tsd_b200.Context(0, "det")
    ctx.set_templates(red6, blue6)
    # device frames: one contiguous group per size (DISTINCT synthetic frames repeated), boxes per group
    groups = []
    big = torch.empty(sum(PER_SIZE * H * W * 3 for H, W in SIZES), dtype=torch.uint8, device=dev)     # one buffer behind the table
    o = 0
    for g, (H, W) in enumerate(SIZES):
        src = torch.from_numpy(synth.make_frames(DISTINCT, H, W, seed=100 + g)).to(dev)
        d = big[o:o + PER_SIZE * H * W * 3].view(PER_SIZE, H, W, 3)
        o += PER_SIZE * H * W * 3
        for k in range(0, PER_SIZE, DISTINCT):
            d[k:k + DISTINCT].copy_(src[:min(DISTINCT, PER_SIZE - k)])
        boxes, off = synth.make_boxes(PER_SIZE, NBOX, H, W, seed=200 + g)
        groups.append(dict(H=H, W=W, d=d, boxes=boxes, off=off, d_boxes=torch.from_numpy(boxes).to(dev), d_off=torch.from_numpy(off).to(dev)))
    # the ragged batch: table entry i = frame i // 4 of group i % 4 (the sizes interleaved), one buffer of all four groups
    base = big.data_ptr()
    n = PER_SIZE * len(SIZES)
    table = np.zeros(n, tsd_b200.FRAME_DESC_DTYPE)
    rboxes = np.empty((n * NBOX, 4), np.int32)
    for i in range(n):
        gr, k = groups[i % 4], i // 4
        fb = gr["H"] * gr["W"] * 3
        table[i] = (gr["d"].data_ptr() - base + k * fb, gr["W"] * 3, gr["H"], gr["W"])
        rboxes[i * NBOX:(i + 1) * NBOX] = gr["boxes"][k * NBOX:(k + 1) * NBOX]
    assert table["offset"].min() >= 0
    roff = (np.arange(n + 1) * NBOX).astype(np.int32)
    d_rb, d_ro = torch.from_numpy(rboxes).to(dev), torch.from_numpy(roff).to(dev)
    s = torch.cuda.ExternalStream(ctx.stream)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step(kind):
        torch.cuda.synchronize()
        ev0.record(s)
        if kind == "ragged":
            ctx.enqueue_frames_ragged(base, table, d_rb.data_ptr(), d_ro.data_ptr(), len(rboxes), max_boxes_per_frame=NBOX)
        else:
            for gr in groups:
                ctx.enqueue_frames(gr["d"].data_ptr(), PER_SIZE, gr["H"], gr["W"], gr["d_boxes"].data_ptr(), gr["d_off"].data_ptr(),
                                   len(gr["boxes"]), max_boxes_per_frame=NBOX)
        ctx.flush()
        ev1.record(s)
        ev1.synchronize()
        return ev0.elapsed_time(ev1)

    def records(kind):
        """-> (records as (group, frame in group, x1, y1, x2, y2, id, hundredths) sorted, aspect-passing windows)."""
        out, wins = [], 0
        if kind == "ragged":
            step(kind)
            det, counts = ctx.fetch_detections(len(rboxes))
            out = [(int(d["frame"]) % 4, int(d["frame"]) // 4) + tuple(int(d[k]) for k in ("x1", "y1", "x2", "y2", "id", "hundredths")) for d in det]
            wins = int(counts[1])
        else:
            for g, gr in enumerate(groups):
                ctx.enqueue_frames(gr["d"].data_ptr(), PER_SIZE, gr["H"], gr["W"], gr["d_boxes"].data_ptr(), gr["d_off"].data_ptr(),
                                   len(gr["boxes"]), max_boxes_per_frame=NBOX)
                det, counts = ctx.fetch_detections(len(gr["boxes"]))
                out += [(g, int(d["frame"])) + tuple(int(d[k]) for k in ("x1", "y1", "x2", "y2", "id", "hundredths")) for d in det]
                wins += int(counts[1])
        return sorted(out), wins

    rr, wins = records("ragged")
    gg, wins_g = records("grouped")
    assert rr == gg and wins == wins_g, "ragged and grouped records differ"
    for _ in range(a.warmup):
        step("ragged"); step("grouped")
    t = {"ragged": [], "grouped": []}
    for _ in range(a.reps):
        for kind in ("ragged", "grouped"):
            t[kind].append(step(kind))
    dev_res = {k: dict(ms=stats(v), windows_per_s=stats([wins / (x / 1e3) for x in v])) for k, v in t.items()}
    dev_res["windows_per_step"] = wins
    dev_res["records_per_step"] = len(rr)
    dev_res["ragged_over_grouped_median"] = dev_res["ragged"]["ms"]["median"] / dev_res["grouped"]["ms"]["median"]
    # host: pageable numpy frames
    hf = [synth.make_frames(HOST_PER_SIZE, H, W, seed=300 + g) for g, (H, W) in enumerate(SIZES)]
    hb = [synth.make_boxes(HOST_PER_SIZE, NBOX, H, W, seed=400 + g) for g, (H, W) in enumerate(SIZES)]
    mixed = [hf[i % 4][i // 4] for i in range(HOST_PER_SIZE * 4)]
    mboxes = np.concatenate([hb[i % 4][0][(i // 4) * NBOX:(i // 4 + 1) * NBOX] for i in range(HOST_PER_SIZE * 4)])
    moff = (np.arange(HOST_PER_SIZE * 4 + 1) * NBOX).astype(np.int32)

    def host(kind):
        t0 = time.perf_counter()
        if kind == "ragged":
            det, _ = ctx.detect_frames(mixed, mboxes, moff)
            nrec = len(det)
        else:
            nrec = 0
            for g in range(4):
                frames = np.stack([mixed[i] for i in range(g, len(mixed), 4)])
                det, _ = ctx.detect_frames(frames, hb[g][0], hb[g][1])
                nrec += len(det)
        return time.perf_counter() - t0, nrec

    ht = {"ragged": [], "grouped": []}
    nrec = {}
    for i in range(a.warmup + max(3, a.reps // 3)):
        for kind in ("ragged", "grouped"):
            dt, nrec[kind] = host(kind)
            if i >= a.warmup:
                ht[kind].append(dt * 1e3)
    assert nrec["ragged"] == nrec["grouped"]
    host_res = {k: dict(ms=stats(v), frames_per_s=stats([len(mixed) / (x / 1e3) for x in v])) for k, v in ht.items()}
    host_res["frames"] = len(mixed)
    res = {"gpu": gpu_info(torch), "workload": dict(sizes_hw=SIZES, frames_per_size=PER_SIZE, boxes_per_frame=NBOX, host_frames_per_size=HOST_PER_SIZE),
           "device_resident": dev_res, "host_pageable": host_res}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    ctx.close()


if __name__ == "__main__":
    main()
