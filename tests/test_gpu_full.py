"""GPU (-m gpu): the known-answer tests BASELINE.json's north_star names, through the C ABI.

  * the reference's resultado.txt for ALL 150 frames of test_alumnos_jpg (DET/source.py:659,708-745), byte for byte;
  * K2 and the whole chain on 24 real frames decoded from their JPEG bytes;
  * the GRAY descriptor classifiers (REC/source.py:517-521, REC/constants.py:10-12) with 1024 features;
  * the large seeded fuzz regimes (device-resident chain vs the oracle, record by record);
  * the exact-f64 fallback of the pair classification (cv2.compareHist within 2e-6 of a threshold) is taken and agrees.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _lines(files, det):
    """resultado.txt lines (DET/source.py:501-508) from detection records."""
    return ["%s;%d;%d;%d;%d;%d;%s" % (files[int(d["frame"])], d["x1"], d["y1"], d["x2"], d["y2"], d["id"], str(int(d["hundredths"]) / 100))
            for d in det]


def test_full_dataset_kat(ctx_det, det_full150, resultado150):
    """All 150 frames: K1 on the 18 540 MSER boxes, K5 (both passes) on the reference's 3 581 post-resize windows, K3 + K4 on the
    742 survivors -> the 192 lines of the reference's resultado.txt, byte for byte, in order."""
    g = det_full150
    files = [str(f) for f in g["files"]]
    coords, valid = ctx_det.expand_boxes(g["boxes"])
    assert np.array_equal(valid, g["valid"]) and np.array_equal(coords[valid], g["coords"])
    w1, c1, o1 = ctx_det.dedup(g["windows"], g["coords"], g["offsets"], False, 0.85)
    assert np.array_equal(o1, g["p1_offsets"]) and np.array_equal(c1, g["p1_coords"])
    w2, c2, o2 = ctx_det.dedup(w1, c1, o1, True, 0.95)
    assert np.array_equal(o2, g["surv_offsets"]) and np.array_equal(c2, g["surv_coords"]) and np.array_equal(w2, g["surv_windows"])
    r = ctx_det.score_windows(w2)
    frame_of = np.repeat(np.arange(len(files)), np.diff(o2))
    lines = ["%s;%d;%d;%d;%d;%d;%s" % (files[frame_of[i]], c2[i][0], c2[i][1], c2[i][2], c2[i][3], r["id"][i], str(int(r["hundredths"][i]) / 100))
             for i in range(len(c2)) if r["emit"][i]]
    assert len(lines) == 192 and lines == resultado150
    assert np.array_equal(np.bincount(frame_of[r["emit"]], minlength=len(files)), np.diff(g["det_offsets"]))


def test_real_frames_whole_chain(ctx_det, det_full150, jpeg24, resultado150):
    """24 real frames (the ones with the most windows / detections: 1 488 windows, 89 detections) from their JPEG bytes through
    K1+K2 (windows equal the reference's cv2.resize output) and through the whole chain in ONE batch, pageable and page-locked
    (K2 reading host memory in place): exactly those frames' lines of resultado.txt."""
    g = det_full150
    idx = jpeg24["index"]
    frames = jpeg24["frames"]
    boxes = np.concatenate([g["boxes"][g["box_offsets"][f]:g["box_offsets"][f + 1]] for f in idx])
    off = np.concatenate([[0], np.cumsum([g["box_offsets"][f + 1] - g["box_offsets"][f] for f in idx])]).astype(np.int32)
    wins, coords, woff = ctx_det.windows(frames, boxes, off)
    exp_w = np.concatenate([g["windows"][g["offsets"][f]:g["offsets"][f + 1]] for f in idx])
    exp_c = np.concatenate([g["coords"][g["offsets"][f]:g["offsets"][f + 1]] for f in idx])
    assert np.array_equal(coords, exp_c) and np.array_equal(wins, exp_w)
    expect = [ln for ln in resultado150 if ln.split(";")[0] in set(jpeg24["files"])]
    det, counts = ctx_det.detect_frames(frames, boxes, off)
    assert _lines(jpeg24["files"], det) == expect
    assert counts.tolist() == [int(off[-1]), len(exp_c), int(sum(g["surv_offsets"][f + 1] - g["surv_offsets"][f] for f in idx)), len(expect)]
    pinned = np.ascontiguousarray(frames.copy())
    ctx_det.pin(pinned)
    try:
        det2, counts2 = ctx_det.detect_frames(pinned, boxes, off)
    finally:
        ctx_det.unpin(pinned)
    assert np.array_equal(det, det2) and np.array_equal(counts, counts2)


def test_gray_descriptor_classifiers(tsd, rec_golden, rec_gray_golden):
    """GRAY_LDA_LDABAYES and GRAY_LDA_KNN: 1024 raw grey pixels per window (REC/source.py:520-521) through K8 / K8b with
    nfeat = 1024 -> sklearn's logits (relative 1e-9), LDA-transformed coordinates and labels on the reference's 1 623 held-out
    windows; the mirror's computeDescriptors gives the same feature vector as the reference's image.ravel()."""
    g = rec_gray_golden
    gray = rec_golden["gray"]
    X = np.stack([tsd.source_rec.computeDescriptors(im, (None, "GRAY")) for im in gray[:50]])
    assert X.dtype == np.uint8 and np.array_equal(X, gray[:50].reshape(50, 1024))
    X = gray.reshape(-1, 1024).astype(np.float32)
    with tsd.Context(device=0, flavour="rec") as c:
        c.set_lda(g["lda_W"], g["lda_b"])
        lg, lab = c.lda_predict(X)
        assert np.max(np.abs(lg - g["logits"]) / np.maximum(1.0, np.abs(g["logits"]))) < 1e-9
        assert np.array_equal(lab, g["pred_lda"])
        c.set_knn(g["knn_xbar"], g["knn_scalings"], g["knn_Ztrain"], g["knn_ytrain"], 4)
        Z, lk = c.knn_predict(X)
        assert np.max(np.abs(Z - g["knn_Zq"]) / np.maximum(1.0, np.abs(g["knn_Zq"]))) < 1e-9
        assert np.array_equal(lk, g["pred_knn"])
        with pytest.raises(tsd.TsdError):                                 # the chain's HOG branch refuses 1024-feature weights
            c.detect_frames(np.zeros((1, 64, 64, 3), np.uint8), np.array([[1, 1, 20, 20]], np.int32), np.array([0, 1], np.int32), mode=tsd.RUN_RECOGNIZE)


FUZZ = [  # (mode, frames, candidates/frame, seed): ~45 s of oracle time in total
    ("det", 1024, 200, 21),        # the bench regime (~81 windows/frame: 6-block Gram)
    ("det", 1024, 30, 33),         # ~12 windows/frame: 1-block Gram, the regime of real MSER boxes
    ("det", 512, 100, 32),         # ~40 windows: 3 blocks
    ("det", 192, 270, 31),         # ~109 windows: 10 blocks
    ("det", 192, 310, 34),         # ~126 windows: frames on both sides of the 128-window limit
    ("det", 24, 900, 35),          # ~360 windows: frames far above it
    ("rec", 256, 200, 23),         # recognition flavour (x1.15, 32x32, HOG + LDA labels)
]


@pytest.mark.parametrize("mode,F,N,seed", FUZZ)
def test_chain_fuzz_vs_oracle(tsd, oracle, templates, rec_golden, mode, F, N, seed):
    """Device-resident asynchronous chain against the oracle, record by record, on seeded synthetic batches large enough to hit the
    rare paths (merges of merged items, twins, pruning against rewritten histograms, counts above 255)."""
    import torch
    U = 32
    uniq = tsd.synth.make_frames(U, seed=tsd.synth.FRAME_SEED + seed)
    boxes, off = tsd.synth.make_boxes(F, N, seed=tsd.synth.BOX_SEED + 100 + seed)
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(uniq).to(dev)[torch.arange(F, device=dev) % U].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    bad = []
    if mode == "det":
        red6, blue6 = templates
        with tsd.Context(0, "det") as ctx:
            ctx.set_templates(red6, blue6)
            ctx.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), max_boxes_per_frame=N)
            det, counts = ctx.fetch_detections(int(off[-1]))
        got = {}
        for d in det:
            got.setdefault(int(d["frame"]), []).append((int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])))
        tot = np.zeros(4, np.int64)
        for f in range(F):
            o = oracle.detect_frame(uniq[f % U], boxes[off[f]:off[f + 1]], red6, blue6)
            tot += o["stage_counts"]
            exp = [tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
            if got.get(f, []) != exp:
                bad.append(f)
        assert not bad and counts.tolist() == tot.tolist()
    else:
        r = rec_golden
        with tsd.Context(0, "rec") as ctx:
            ctx.set_lda(r["lda_W"], r["lda_b"])
            ctx.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), mode=tsd.RUN_RECOGNIZE,
                               max_boxes_per_frame=N)
            det, counts = ctx.fetch_detections(int(off[-1]))
        got = {}
        for d in det:
            got.setdefault(int(d["frame"]), []).append((int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"])))
        nsurv = 0
        for f in range(F):
            c, v = oracle.expand_boxes(boxes[off[f]:off[f + 1]], 1.15)
            c = c[v]
            wins = np.stack([oracle.crop_resize(uniq[f % U], cc, 32) for cc in c]) if len(c) else np.zeros((0, 32, 32, 3), np.uint8)
            w1, c1 = oracle.dedup(wins, c, False, 0.85)
            w2, c2 = oracle.dedup(w1, c1, True, 0.95)
            nsurv += len(c2)
            exp = []
            if len(c2):
                hog = np.stack([oracle.hog32(oracle.bgr2gray(w)) for w in w2])
                _, lab = oracle.lda_predict(hog, r["lda_W"], r["lda_b"], 0.5)
                exp = [tuple(int(x) for x in cc) + (int(l),) for cc, l in zip(c2, lab) if l != 0]
            if got.get(f, []) != exp:
                bad.append(f)
        assert not bad and int(counts[2]) == nsurv


def test_slot_layout_independent_of_row_words(tsd, oracle, templates):
    """Overlap mode: a batch with wide pair-class bit rows (600 candidates/frame) enqueued back to back with a batch of narrow
    rows (40 candidates/frame), and the reverse, without a host synchronisation in between.  The slot base of the bit matrix must
    not depend on the batch's own row width (round-1 advisor finding: the second batch overwrote rows the first batch's fold was
    still reading)."""
    import torch
    red6, blue6 = templates
    dev = torch.device("cuda", 0)
    batches = []
    for k, (F, N) in enumerate(((48, 600), (64, 40))):
        frames = tsd.synth.make_frames(8, seed=tsd.synth.FRAME_SEED + 60 + k)
        boxes, off = tsd.synth.make_boxes(F, N, seed=tsd.synth.BOX_SEED + 60 + k)
        exp = []
        for f in range(F):
            o = oracle.detect_frame(frames[f % 8], boxes[off[f]:off[f + 1]], red6, blue6)
            exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
        d_frames = torch.from_numpy(frames).to(dev)[torch.arange(F, device=dev) % 8].contiguous()
        batches.append((d_frames, torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev), F, int(off[-1]), N, exp))
    rec = lambda det: [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)

        def enqueue(b):
            ctx.enqueue_frames(b[0].data_ptr(), b[3], 800, 1360, b[1].data_ptr(), b[2].data_ptr(), b[4], max_boxes_per_frame=b[5])
        enqueue(batches[0]); enqueue(batches[1]); enqueue(batches[0])       # the slot layout grows to its final size (a growth synchronises)
        ctx.synchronize()
        for first, second in ((0, 1), (1, 0), (0, 1), (1, 0)):
            enqueue(batches[first]); enqueue(batches[second])
            prev, _ = ctx.fetch_detections(batches[first][4], previous=True)
            last, _ = ctx.fetch_detections(batches[second][4])
            assert rec(prev) == batches[first][6] and rec(last) == batches[second][6], (first, second)


def test_state_setters_join_the_running_batch(tsd, oracle, templates):
    """tsd_set_templates right after an asynchronous enqueue (overlap mode: the batch still runs on an internal stream) must not
    change that batch's scores (round-1 advisor finding)."""
    import torch
    red6, blue6 = templates
    dev = torch.device("cuda", 0)
    F = 64
    frames = tsd.synth.make_frames(8, seed=tsd.synth.FRAME_SEED + 70)
    boxes, off = tsd.synth.make_boxes(F, 200, seed=tsd.synth.BOX_SEED + 70)
    d_frames = torch.from_numpy(frames).to(dev)[torch.arange(F, device=dev) % 8].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    exp = []
    for f in range(F):
        o = oracle.detect_frame(frames[f % 8], boxes[off[f]:off[f + 1]], red6, blue6)
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)
        for _ in range(3):
            ctx.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), max_boxes_per_frame=200)
            ctx.set_templates(np.zeros_like(red6), np.zeros_like(blue6))     # would zero every score if it overtook the batch
            det, _ = ctx.fetch_detections(int(off[-1]))
            got = [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]
            assert got == exp
            ctx.set_templates(red6, blue6)


def test_exact_f64_fallback_is_taken(tsd, oracle, monkeypatch):
    """A pair whose cv2.compareHist value sits 1e-9 (relative) beside the tolerance -- or beside tolerance * 0.8823 -- cannot be
    decided from the integer dot product (its float32-product model is only good to ~1e-7): the kernels must take the exact float64
    path (counter > 0) and reach the reference's decision -- sim > tol deletes, tol*0.8823 <= sim <= tol merges
    (DET/source.py:203-217).  1e-9 is far inside the 2e-6 band that triggers the fallback and far outside the 5e-15 by which two
    float64 summation orders can differ (SURVEY 8c), so the expected decision does not depend on the order.  Both producers of the
    pair classes are covered: the tensor-core Gram kernel (default) and the CUDA-core pair kernel (TSD_GRAM=0)."""
    rng = np.random.default_rng(44)
    base = rng.integers(0, 256, (5, 5, 3)).repeat(5, 0).repeat(5, 1).astype(np.int16)
    wins = [np.clip(base + rng.integers(-25, 26, base.shape), 0, 255).astype(np.uint8) for _ in range(6)]
    wins += [rng.integers(0, 256, (25, 25, 3), dtype=np.uint8) for _ in range(3)]
    wins = np.stack(wins)
    coords = np.array([(40 * i, 30 * i, 40 * i + 50, 30 * i + 50) for i in range(len(wins))], np.int32)
    off = np.array([0, len(wins)], np.int32)
    hists = [oracle.hist_normalized(w) for w in wins]
    sims = sorted({oracle.hist_correl(hists[i], hists[j]) for i in range(6) for j in range(i)})
    assert len(sims) >= 10 and 0.2 < sims[0] and sims[-1] < 0.999
    for gram in ("1", "0"):
        monkeypatch.setenv("TSD_GRAM", gram)
        with tsd.Context(0, "det") as ctx:
            ctx.stat_unsure_pairs(reset=True)
            for s in sims[::3]:
                for tol in (s * (1 - 1e-9), s * (1 + 1e-9), s / 0.8823 * (1 - 1e-9), s / 0.8823 * (1 + 1e-9)):
                    if not 0.0 < tol < 1.0:
                        continue
                    gw, gc, go = ctx.dedup(wins, coords, off, False, float(tol))
                    ow, oc = oracle.dedup(wins, coords, False, float(tol))
                    assert go[1] == len(oc) and np.array_equal(gc, oc) and np.array_equal(gw, ow), (gram, tol)
            assert ctx.stat_unsure_pairs() > 0, "the exact-f64 path was never taken (TSD_GRAM=%s)" % gram


def test_k2_tma_variant_bit_identical(tsd, oracle, templates, det_full150, jpeg24, resultado150, monkeypatch):
    """TSD_K2=tma: the resize kernel whose ROI is staged in shared memory by the Tensor Memory Accelerator (cp.async.bulk.tensor behind
    an mbarrier, tsd_k2_tma.cuh) must give exactly the default kernel's windows: the whole chain on synthetic frames (crops of every
    size class: staged ones of 64 / 128 / 192 / 256-byte boxes, the direct-gather fallback for wide crops, copy and 2x2-AREA paths,
    ROIs clipped at the right / bottom frame edge where the TMA zero-fills) against the oracle, at 1360x800 and at 4K, and on the 24
    real frames against the reference's resultado.txt lines."""
    red6, blue6 = templates
    monkeypatch.setenv("TSD_K2", "tma")
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)
        for (H, W, F, N, seed) in ((800, 1360, 48, 200, 81), (2160, 3840, 2, 700, 82)):
            frames = tsd.synth.make_frames(F, H, W, seed=tsd.synth.FRAME_SEED + seed)
            boxes, off = tsd.synth.make_boxes(F, N, H, W, seed=tsd.synth.BOX_SEED + seed)
            det, counts = ctx.detect_frames(frames, boxes, off)
            exp, tot = [], np.zeros(4, np.int64)
            for f in range(F):
                o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
                tot += o["stage_counts"]
                exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
            got = [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]
            assert counts.tolist() == tot.tolist() and got == exp, (H, W)
        g = det_full150
        idx = jpeg24["index"]
        boxes = np.concatenate([g["boxes"][g["box_offsets"][f]:g["box_offsets"][f + 1]] for f in idx])
        off = np.concatenate([[0], np.cumsum([g["box_offsets"][f + 1] - g["box_offsets"][f] for f in idx])]).astype(np.int32)
        det, _ = ctx.detect_frames(jpeg24["frames"], boxes, off)
        assert _lines(jpeg24["files"], det) == [ln for ln in resultado150 if ln.split(";")[0] in set(jpeg24["files"])]
    # recognition flavour (32x32 windows): survivors' labels through the chain equal the default kernel's
    r = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "rec_golden.npz"))
    frames = tsd.synth.make_frames(16, seed=tsd.synth.FRAME_SEED + 83)
    boxes, off = tsd.synth.make_boxes(16, 200, seed=tsd.synth.BOX_SEED + 83, enlarge=1.15, D=32)
    res = []
    for k2 in ("tma", "v2"):
        monkeypatch.setenv("TSD_K2", k2)
        with tsd.Context(0, "rec") as ctx:
            ctx.set_lda(r["lda_W"], r["lda_b"])
            res.append(ctx.detect_frames(frames, boxes, off, mode=tsd.RUN_RECOGNIZE))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])


def test_timeline_and_stagger_switch(tsd, oracle, templates, monkeypatch):
    """tsd_set_profiling(ctx, 2) + tsd_timeline: the batches keep overlapping (two slots), every stage boundary comes back in
    enqueue order with non-decreasing times inside a batch; and the records of back-to-back batches do not depend on whether the
    front halves of consecutive batches are staggered (TSD_STAGGER) or how many fold CTAs may share an SM (TSD_FOLD_PER_SM)."""
    import torch
    red6, blue6 = templates
    dev = torch.device("cuda", 0)
    F, N = 24, 200
    frames = tsd.synth.make_frames(8, seed=tsd.synth.FRAME_SEED + 90)
    boxes, off = tsd.synth.make_boxes(F, N, seed=tsd.synth.BOX_SEED + 90)
    exp = []
    for f in range(F):
        o = oracle.detect_frame(frames[f % 8], boxes[off[f]:off[f + 1]], red6, blue6)
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    d_frames = torch.from_numpy(frames).to(dev)[torch.arange(F, device=dev) % 8].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    rec = lambda det: [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]
    for stagger, cap in (("1", "2"), ("0", "0"), ("1", "1")):
        monkeypatch.setenv("TSD_STAGGER", stagger)
        monkeypatch.setenv("TSD_FOLD_PER_SM", cap)
        with tsd.Context(0, "det") as ctx:
            ctx.set_templates(red6, blue6)
            one = lambda: ctx.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), max_boxes_per_frame=N)
            for _ in range(4):                               # one key per slot: eager, eager, captured, captured (CUDA graphs holding
                one()                                        # the stagger's event record as an external event node)
            assert ctx.stat_graphs() == (2, 0)
            prev, _ = ctx.fetch_detections(int(off[-1]), previous=True)
            last, _ = ctx.fetch_detections(int(off[-1]))
            assert rec(prev) == exp and rec(last) == exp, (stagger, cap)
            ctx.set_profiling(2)
            for _ in range(3):
                one()
            tl = ctx.timeline()
            ctx.set_profiling(False)
            det, _ = ctx.fetch_detections(int(off[-1]))
            assert rec(det) == exp
            starts = [i for i, (name, _) in enumerate(tl) if name == "start"]
            assert len(starts) == 3 and tl[0][1] == 0.0
            for a, b in zip(starts, starts[1:] + [len(tl)]):
                names = [n for n, _ in tl[a:b]]
                times = [t for _, t in tl[a:b]]
                assert names[:4] == ["start", "k1_expand_filter", "k2_crop_resize", "k5_hist"] and names[-1] == "detections"
                assert all(t1 >= t0 for t0, t1 in zip(times, times[1:]))
