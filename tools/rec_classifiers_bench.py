"""Step times of the recognition chain for the four classifiers (HOG / GRAY descriptors x LDA / KNN), and tsd_knn_predict alone on
both sides of its training-set split.

The chain runs bench.py's recognize_run inputs: 1 024 synthetic 1360x800 frames x 200 candidates (16 unique frames), x1.15, 32x32.
The reference's own LDA biases and KNN training sets label nothing on these frames, so the LDA modes use the reference's weights with
biases at the 0.85 quantile of each classifier's logits, and the KNN modes the reference's reducer with 14 574 training rows sampled
around the survivors' Z (labels 0..6): records are then written, as on real data.  Each mode: warm-up, then device events over
--steps enqueues (batches overlapped, CUDA graphs on), then per-stage times from tsd_set_profiling over 5 serialised steps.

tsd_knn_predict (public API only, device pointers) is timed on 36 871 queries -- the survivors of the recorded recognition step
(profiles/r02_bench_v5.json) -- and on 300 queries, with the reference's 324-feature model (14 574 training rows, k = 4).  The
first needs no split; the second is below one 128-query CTA per SM and splits the training set.  --old-lib names another build of
libtsd_b200.so: the leg then runs in child processes that alternate between the two libraries (TSD_LIB), so both are measured on one
card, and their labels are compared.

    python tools/rec_classifiers_bench.py --out result.json [--old-lib path/to/libtsd_b200.so] [--steps 10] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
F, NBOX, H, W = 1024, 200, 800, 1360
KNN_SIZES = (36871, 300)


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not measured"
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = "not measured"
    return info


def knn_leg(reps=20):
    """Child process: median device time of tsd_knn_predict (MEM_DEVICE) at each KNN_SIZES, and a digest of the labels."""
    import hashlib
    import torch
    import tsd_b200
    from tsd_b200 import _capi as A
    r = np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz"))
    dev = torch.device("cuda", 0)
    out = {}
    with tsd_b200.Context(0, "rec") as c:
        c.set_knn(r["knn_xbar"], r["knn_scalings"], r["knn_Ztrain"], r["knn_ytrain"], 4)
        st = torch.cuda.ExternalStream(c.stream, device=dev)
        for n in KNN_SIZES:
            X = torch.from_numpy(np.ascontiguousarray(np.resize(r["hog"], (n, 324)))).to(dev)
            lab = torch.zeros(n, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()

            def call():
                A.check(c._L.tsd_knn_predict(c._h, A.ptr(X.data_ptr()), n, None, A.ptr(lab.data_ptr()), A.MEM_DEVICE))
            for _ in range(3):
                call()
            c.synchronize()
            ts = []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                call()
                e1.record(st)
                c.synchronize()
                ts.append(e0.elapsed_time(e1))
            out[str(n)] = {"ms_median": float(np.median(ts)), "ms_min": float(np.min(ts)),
                           "labels_sha1": hashlib.sha1(lab.cpu().numpy().tobytes()).hexdigest()}
    print(json.dumps(out))


def chain_modes(torch, tsd_b200, steps, warmup):
    from tsd_b200 import synth
    dev = torch.device("cuda", 0)
    uniq = synth.make_frames(16, seed=synth.FRAME_SEED + 500)
    boxes, off = synth.make_boxes(F, NBOX, seed=synth.BOX_SEED + 500, enlarge=1.15, D=32)
    d_frames = torch.from_numpy(uniq).to(dev)[torch.arange(F, device=dev) % 16].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    r = np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz"))
    rg = np.load(os.path.join(ROOT, "tests", "golden", "rec_gray_golden.npz"))
    res = {}
    with tsd_b200.Context(0, "rec") as c:
        # the survivors' descriptors of the 16 unique frames (stage entry points), for the biases and the sampled training sets
        wins, coords, woff = c.windows(uniq, boxes[:off[16]], off[:17])
        w1, c1, o1 = c.dedup(wins, coords, woff, False, 0.85)
        w2, _, _ = c.dedup(w1, c1, o1, True, 0.95)
        gray = c.bgr2gray(w2)
        desc = {"HOG": (c.hog(gray).astype(np.float64), r), "GRAY": (gray.reshape(-1, 1024).astype(np.float64), rg)}
        rng = np.random.default_rng(7)
        st = torch.cuda.ExternalStream(c.stream, device=dev)
        for dname, (X, g) in desc.items():
            for cname in ("LDA", "KNN"):
                mode = tsd_b200.RUN_RECOGNIZE | (tsd_b200.REC_GRAY if dname == "GRAY" else 0) | (tsd_b200.REC_KNN if cname == "KNN" else 0)
                if cname == "LDA":
                    c.set_lda(g["lda_W"], -np.quantile(X @ g["lda_W"], 0.85, axis=0))
                else:
                    Zq = (X - g["knn_xbar"]) @ g["knn_scalings"]
                    Zt = Zq[rng.integers(0, len(Zq), 14574)] + 0.3 * rng.standard_normal((14574, 6))
                    c.set_knn(g["knn_xbar"], g["knn_scalings"], Zt, rng.integers(0, 7, 14574), 4)

                def step():
                    c.enqueue_frames(d_frames.data_ptr(), F, H, W, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), mode=mode,
                                     max_boxes_per_frame=NBOX)
                for _ in range(warmup):
                    step()
                c.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                for _ in range(steps):
                    step()
                c.flush()
                e1.record(st)
                c.synchronize()
                ms = e0.elapsed_time(e1) / steps
                det, cnt = c.fetch_detections(int(off[-1]))
                c.set_profiling(True)
                for _ in range(5):
                    step()
                c.synchronize()
                stages = {k: v / 5 for k, v in c.stage_times()}
                c.set_profiling(False)
                res["%s+%s" % (dname, cname)] = {"ms_per_step": ms, "steps": steps, "stage_counts": [int(v) for v in cnt],
                                                  "distinct_labels": sorted(set(int(d["id"]) for d in det)), "stages_ms_per_step": stages}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=False)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--old-lib", default=None)
    ap.add_argument("--alternations", type=int, default=3)
    ap.add_argument("--knn-leg", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.knn_leg:
        return knn_leg()
    import torch
    import tsd_b200
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    out = {"gpu": gpu_info(torch), "workload": "1024 synthetic 1360x800 frames x 200 candidates, x1.15, 32x32 (bench.py recognize_run)"}
    out["chain"] = chain_modes(torch, tsd_b200, a.steps, a.warmup)
    libs = {"this": tsd_b200._capi.LIB_PATH}
    if a.old_lib:
        libs["old"] = os.path.abspath(a.old_lib)
    runs = {k: [] for k in libs}
    for _ in range(a.alternations):
        for name, path in libs.items():
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--knn-leg"], env=dict(os.environ, TSD_LIB=path),
                               capture_output=True, text=True, check=True)
            runs[name].append(json.loads(p.stdout.strip().splitlines()[-1]))
    out["knn_predict"] = {name: {str(n): {"ms_median_per_run": [r[str(n)]["ms_median"] for r in rs], "labels_sha1": rs[0][str(n)]["labels_sha1"]}
                                 for n in KNN_SIZES} for name, rs in runs.items()}
    out["knn_predict"]["model"] = "reference HOG model: 324 features, 14 574 training rows, k = 4; queries = rec_golden HOG rows repeated"
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
