"""The GRAY and k-NN recognition modes (TSD_REC_GRAY, TSD_REC_KNN) on every frame layout, host route, size limit, call sequence
and profiling mode of the chain, against the oracle composition: expand_boxes -> crop_resize -> both dedup passes -> bgr2gray ->
(hog32) -> lda_predict / knn_predict.  Records (frame, x1, y1, x2, y2, label, 0) must be equal; the layout, det_cap, split and
past-4 GiB cases compare the four stage counts too.

  layouts    every layout of test_gpu_layouts through every route (device pointers, pageable chunks, page-locked staged whole
             and in chunks, page-locked read by K2 over PCIe, TSD_STAGE=0, TSD_ZEROCOPY=0), GRAY + LDA, HOG + KNN and GRAY + KNN;
             staged routes move exactly the bytes of the stage_mark model.  det_cap below the record count: TSD_E_NOMEM with
             the count and the stage counts filled in, on two routes per mode.
  split      K8b's training-set split is decided from the batch's window bound, not from its survivors: batches whose bound
             splits with many or no survivors, a bound past the split line with few survivors, bounds just above a multiple
             of 128 with 0, 1 and 128 k + 1 survivors, and the bounds on both sides of the line.  Device pointers (two
             overlapped slots, both splitting) and page-locked staged frames.
  large      GRAY + LDA and GRAY + KNN on 2^22 + 4 099 survivors a batch, two overlapped batches: the grey windows of a batch
             pass 2^31 and 2^32 bytes, and the second slot's start past 4 GiB.  Item i must equal pattern i mod 4 099.
  sequences  GRAY / KNN batches alternating with HOG + LDA and detection batches on one D = 32 context, with overlap, stagger
             and CUDA graphs each on and off; every batch checked; each mode's graph captured then replayed, a model change
             between replays runs the new model eagerly first.
  config     GRAY + LDA at proba_tol 0.2 and 0.8; tsd_set_profiling(1) and (2) per mode: records unchanged, tsd_stage_times
             names as the header lists them, tsd_timeline non-decreasing within every batch.
  knn_k      tsd_create refuses knn_k outside 1..8; Context.set_knn without k uses the config's knn_k.

test_rec_mode_cases_reach_their_regimes checks on the CPU that every case is in the regime it names.
"""
import functools
import inspect
import os
import re

import numpy as np
import pytest

from test_gpu_large import P, dev, distinct_first, is_prime, room, small_frames, square_boxes, tile_records, win_stride, ent_stride
from test_gpu_layouts import F as LF, LAYOUTS, ROUTES, canvas_for, clipped, expand, frames_of, staged_bytes, stages, boxes_for, windows_of
from test_gpu_rec_classifiers import KNN_THREADS, KNN_TILE, SM_B200, knn_robust, run_mode, survivors as chain_survivors
from test_gpu_recognition import chain_inputs, decision_margin
from test_gpu_sequences import gap_bias

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ("gray_lda", "hog_knn", "gray_knn")
ALL_MODES = ("hog_lda",) + MODES
E_NOMEM = -4
SPLIT_LINE = SM_B200 * KNN_THREADS                       # a window bound below this splits the training set (knn_splits)
SPLIT_H, SPLIT_W, SPLIT_POOL, SPLIT_CANDIDATES, SPLIT_DUP = 48, 64, 513, 1800, 64
SPLIT_K = 4
SPLIT_NTRAIN = 14574
# (name, window bound nb, survivors): below / above the line, bounds just above a multiple of 128, the line itself
SPLIT_CASES = (("split", 300, 300), ("bound_past_line_few_survivors", 300 * SPLIT_DUP, 300), ("edge_0", 1281, 0), ("edge_1", 1281, 1),
               ("edge_128k1", 1281, 128 * SPLIT_K + 1), ("below_line", SPLIT_LINE - 128, 128 * SPLIT_K + 1),
               ("above_line", SPLIT_LINE + 1, 128 * SPLIT_K + 1))
LG_N = (1 << 22) + P                                     # survivors a batch in the large case
LG_H = LG_W = 8
LG_BOX = (1, 1, 6, 6)
LG_NTRAIN = 2000
STAGES_REC = {"hog_lda": ["k6_gray", "k7_hog", "k8_lda"], "gray_lda": ["k6_gray", "k8_lda"],
              "hog_knn": ["k6_gray", "k7_hog", "k8_knn"], "gray_knn": ["k6_gray", "k8_knn"]}
SEQ_ENV = {"overlap_stagger_graph": {}, "overlap_graph": {"TSD_STAGGER": "0"}, "serial_graph": {"TSD_OVERLAP": "0"},
           "overlap_stagger": {"TSD_GRAPH": "0"}, "serial": {"TSD_OVERLAP": "0", "TSD_GRAPH": "0"}}
# (X, Y, model change after the first 6 batches): blocks of X Y X Y X Y (X Y X Y X Y)
SEQ_BLOCKS = (("gray_lda", "det", False), ("hog_knn", "hog_lda", True), ("gray_knn", "det", True), ("gray_knn", "gray_lda", False),
              ("hog_knn", "det", False))
SEQ_F = 8
DETCAP_ROUTES = ("device", "staged_chunks")


def _src(name):
    return open(os.path.join(ROOT, "opencv-traffic-sign-detector_b200", "csrc", name)).read()


def cdiv(a, b):
    return -(-a // b)


def knn_splits(n_max, ntrain, sm=SM_B200):
    """tsd_capi.cu knn_splits restated -> (nsplit, rows per split)."""
    qb, nt = cdiv(n_max, KNN_THREADS), cdiv(ntrain, KNN_TILE)
    ns = 1 if qb >= sm else min(nt, cdiv(2 * sm, max(qb, 1)))
    tiles = cdiv(nt, ns)
    return cdiv(nt, tiles), tiles * KNN_TILE


@functools.lru_cache(None)
def _oracle():
    from oracle import oracle as O
    O.build()
    return O


@functools.lru_cache(None)
def goldens():
    return (np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz")),
            np.load(os.path.join(ROOT, "tests", "golden", "rec_gray_golden.npz")))


def oracle_survivors(O, frame, boxes):
    """(coords, grey windows [m,32,32], HOG [m,324]) of one frame's survivors (x1.15, 32 x 32, both dedup passes)."""
    c, v = O.expand_boxes(boxes, 1.15)
    c = c[v]
    w = np.stack([O.crop_resize(frame, cc, 32) for cc in c]) if len(c) else np.zeros((0, 32, 32, 3), np.uint8)
    w1, c1 = O.dedup(w, c, False, 0.85)
    w2, c2 = O.dedup(w1, c1, True, 0.95)
    g = np.stack([O.bgr2gray(x) for x in w2]) if len(c2) else np.zeros((0, 32, 32), np.uint8)
    h = np.stack([O.hog32(x) for x in g]) if len(c2) else np.zeros((0, 324), np.float32)
    return c2, g, h


def feats(sv, gray):
    """Descriptors of a list of oracle_survivors results."""
    parts = [s[1].reshape(-1, 1024).astype(np.float32) if gray else s[2] for s in sv]
    return np.concatenate(parts) if parts else np.zeros((0, 1024 if gray else 324), np.float32)


# ---- models ------------------------------------------------------------------------------------------------------------
def lda_model(X, gray):
    """The real 324- or 1 024-feature LDA weights, biases in gaps of the logits of X (their own biases label nothing here)."""
    g = goldens()[1 if gray else 0]
    return dict(W=g["lda_W"], b=gap_bias(X, g["lda_W"]))


def knn_model(X, gray, seed, k=4, ntrain=SPLIT_NTRAIN, per_row=False, noise=0.01):
    """The real reducer with a training set sampled around the Z of X (each row a query's Z plus Gaussian noise).  Labels 0..6
    per query (rows of one query agree) or, per_row, per row: then a query's k nearest rows disagree, and losing any of them
    (a split's partial list, say) changes the vote of many queries."""
    real = goldens()[1 if gray else 0]
    rng = np.random.default_rng(seed)
    Zq = (X.astype(np.float64) - real["knn_xbar"]) @ real["knn_scalings"]
    _, inv = np.unique(np.round(Zq, 6), axis=0, return_inverse=True)
    qlab = rng.integers(0, 7, inv.max() + 1)[inv.ravel()].astype(np.int32)
    src = rng.integers(0, len(Zq), ntrain)
    yt = rng.integers(0, 7, ntrain).astype(np.int32) if per_row else qlab[src]
    return dict(xbar=real["knn_xbar"], S=real["knn_scalings"], Zt=Zq[src] + noise * rng.standard_normal((ntrain, 6)), yt=yt, k=k)


def predict(model, X, tol=0.5):
    O = _oracle()
    if not len(X):
        return np.zeros(0, np.int32)
    if "W" in model:
        return O.lda_predict(X, model["W"], model["b"], tol)[1]
    return O.knn_predict(X, model["xbar"], model["S"], model["Zt"], model["yt"], model["k"])[1]


def set_model(ctx, model):
    if "W" in model:
        ctx.set_lda(model["W"], model["b"])
    else:
        ctx.set_knn(model["xbar"], model["S"], model["Zt"], model["yt"], model["k"])


def lda_margin(z, X, W, tol, rel):
    """Per window: the distance of the logits from every change of the decision at tol (the sign of each z, logit(tol) when tol >
    0.5, the gap between the two largest z above the threshold) in units of the largest logit change descriptors within rel
    relative (+ rel absolute) can cause."""
    t = np.log(tol / (1 - tol)) if tol > 0.5 else 0.0
    guard = ((rel * np.abs(X.astype(np.float64)) + rel) @ np.abs(W)).max(1) + 1e-300
    d = np.abs(z).min(1)
    if t:
        d = np.minimum(d, np.abs(z - t).min(1))
    zs = np.sort(np.where(z > t, z, -np.inf), 1)
    two = np.isfinite(zs[:, -2])
    gap = np.full(len(z), np.inf)
    gap[two] = zs[two, -1] - zs[two, -2]
    return np.minimum(d, gap) / (2 * guard)


def robust(model, X, gray, tol=0.5):
    """The oracle's labels of X cannot change under the chain's descriptor error: grey bytes are exact (only the f64 summation
    order differs, < 1e-12 relative), K7's HOG within 1e-5 relative + 1e-7 of hog32."""
    O = _oracle()
    if not len(X):
        return True
    if "W" in model:
        z, _ = O.lda_predict(X, model["W"], model["b"], tol)
        if gray:
            return lda_margin(z, X, model["W"], tol, 1e-12).min() > 1
        return (decision_margin(z, X, model["W"]).min() > 1) if tol == 0.5 else lda_margin(z, X, model["W"], tol, 1e-5).min() > 1
    lab = predict(model, X)
    return knn_robust(model, X, lab, *((1e-12, 1e-12) if gray else (1e-5, 1e-7)))


# ---- layouts --------------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def layout_survivors():
    """{layout: [oracle_survivors of frame f]} for the recognition flavour (K1 drops crops that clip to nothing)."""
    O = _oracle()
    out = {}
    for name in LAYOUTS:
        boxes, off = boxes_for(name, 32)
        fr = frames_of(name)
        H, W = LAYOUTS[name][:2]
        keep = np.array([(c := expand(b, 1.15)) is None or min(clipped(c, H, W)[2:]) > 0 for b in boxes], bool)
        out[name] = [oracle_survivors(O, fr[f], boxes[off[f]:off[f + 1]][keep[off[f]:off[f + 1]]]) for f in range(LF)]
    return out


@functools.lru_cache(None)
def layout_models():
    sv = [s for v in layout_survivors().values() for s in v]
    H, G = feats(sv, False), feats(sv, True)
    return {"gray_lda": lda_model(G, True), "hog_knn": knn_model(H, False, 31), "gray_knn": knn_model(G, True, 32)}


@functools.lru_cache(None)
def layout_expected(mode):
    """{layout: (records, stage counts)} of one mode."""
    model = layout_models()[mode]
    gray = mode.startswith("gray")
    out = {}
    for name, per in layout_survivors().items():
        rec, nsurv = [], 0
        for f, s in enumerate(per):
            lab = predict(model, feats([s], gray))
            rec += [(f,) + tuple(int(v) for v in q) + (int(l), 0) for q, l in zip(s[0], lab) if l != 0]
            nsurv += len(s[0])
        boxes, _ = boxes_for(name, 32)
        out[name] = (rec, [len(boxes), len(windows_of(name, 32)[0]), nsurv, len(rec)])
    return out


def detcap_layout(mode):
    """The first layout whose records under this mode are at least 2, in at least 2 frames."""
    for name, (rec, _) in layout_expected(mode).items():
        if len(rec) >= 2 and len({r[0] for r in rec}) >= 2:
            return name
    return None


# ---- split regime -----------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def split_candidates():
    """SPLIT_CANDIDATES frames of 64 x 48 with one square box each, each frame's single survivor, and the two k-NN models (row
    labelled, trained around every candidate's Z)."""
    O = _oracle()
    frames = small_frames(SPLIT_CANDIDATES, SPLIT_H, SPLIT_W, 600)
    boxes = square_boxes(SPLIT_CANDIDATES, SPLIT_H, SPLIT_W, 6, 30, 601)
    sv = [oracle_survivors(O, frames[f], boxes[f:f + 1]) for f in range(SPLIT_CANDIDATES)]
    models = {"hog_knn": knn_model(feats(sv, False), False, 41, k=SPLIT_K, per_row=True),
              "gray_knn": knn_model(feats(sv, True), True, 42, k=SPLIT_K, per_row=True)}
    return frames, boxes, sv, models


@functools.lru_cache(None)
def split_pool():
    """The first SPLIT_POOL candidates whose label neither model's descriptor error can change -> (frames, boxes, survivors)."""
    frames, boxes, sv, models = split_candidates()
    keep = [f for f in range(SPLIT_CANDIDATES) if len(sv[f][0]) == 1 and
            all(robust(m, feats([sv[f]], mode.startswith("gray")), mode.startswith("gray")) for mode, m in models.items())][:SPLIT_POOL]
    return np.ascontiguousarray(frames[keep]), np.ascontiguousarray(boxes[keep]), [sv[f] for f in keep]


@functools.lru_cache(None)
def split_case(name):
    """-> (frames [nf,48,64,3], boxes [nb,4], offsets [nf+1], survivors per frame).  Frame f < survivors holds pool box f (64 times
    in the bound-past-line case, where the first dedup pass merges the copies); the rest of the bound is boxes of aspect 2,
    which K1 drops, spread over the frames."""
    _, nb, ns = dict((c[0], c) for c in SPLIT_CASES)[name]
    frames, pool, psv = split_pool()
    nf = max(ns, 1) if name != "edge_0" else 10
    per = [[tuple(pool[f])] * (SPLIT_DUP if name.startswith("bound_past") else 1) if f < ns else [] for f in range(nf)]
    rng = np.random.default_rng(nb + ns)
    for i in range(nb - sum(len(p) for p in per)):
        s = int(rng.integers(3, 12))
        per[i % nf].append((int(rng.integers(0, SPLIT_W - 2 * s)), int(rng.integers(0, SPLIT_H - s)), 2 * s, s))
    for p in per:
        rng.shuffle(p)
    boxes = np.array([b for p in per for b in p], np.int32).reshape(-1, 4)
    off = np.concatenate([[0], np.cumsum([len(p) for p in per])]).astype(np.int32)
    return np.ascontiguousarray(frames[:nf]), boxes, off, [psv[f] if f < ns else None for f in range(nf)]


def split_models():
    return split_candidates()[3]


@functools.lru_cache(None)
def split_warmup():
    """A batch at least as large as every split case in frames, boxes and boxes per frame (the sticky slot sizes), so that no case
    regrows the two scratch slots -- a regrowth waits for both and ends the previous batch's fetch_previous."""
    cases = [split_case(c[0]) for c in SPLIT_CASES]
    nf = max(len(c[0]) for c in cases)
    nb = max(len(c[1]) for c in cases)
    mb = max(int(np.diff(c[2]).max()) for c in cases)
    frames = split_pool()[0][:nf]
    per = [mb] + [0] * (nf - 1)
    for i in range(nb - mb):
        per[1 + i % (nf - 1)] += 1
    boxes = np.tile(np.array([[0, 0, 8, 4]], np.int32), (nb, 1))
    return np.ascontiguousarray(frames), boxes, np.concatenate([[0], np.cumsum(per)]).astype(np.int32)


def split_expected(name, mode):
    frames, boxes, off, sv = split_case(name)
    model = split_models()[mode]
    gray = mode.startswith("gray")
    rec, nwin, nsurv = [], 0, 0
    for f, s in enumerate(sv):
        if s is None:
            continue
        nwin += int(off[f + 1] - off[f]) if name.startswith("bound_past") else 1
        nsurv += len(s[0])
        lab = predict(model, feats([s], gray))
        rec += [(f,) + tuple(int(v) for v in q) + (int(l), 0) for q, l in zip(s[0], lab) if l != 0]
    return rec, [len(boxes), nwin, nsurv, len(rec)]


# ---- past 4 GiB -------------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def large_patterns(batch):
    """P frames of 8 x 8 noise whose single box gives pairwise different grey windows -> (frames, per-pattern survivors)."""
    O = _oracle()
    rng = np.random.default_rng(7000 + batch)
    cand = rng.integers(0, 256, (2 * P, LG_H, LG_W, 3), dtype=np.uint8)
    box = np.array([LG_BOX], np.int32)
    sv = [oracle_survivors(O, f, box) for f in cand]
    keep = distinct_first(np.stack([s[1][0] for s in sv]), P)
    return np.ascontiguousarray(cand[keep]), [sv[i] for i in keep]


@functools.lru_cache(None)
def large_models():
    G = np.concatenate([feats(large_patterns(bt)[1], True) for bt in (0, 1)])
    return {"gray_lda": lda_model(G, True), "gray_knn": knn_model(G, True, 51, ntrain=LG_NTRAIN)}


def large_buffers():
    """Byte offsets the large case reaches: a batch's grey windows, and the second slot's start (slot_cap windows)."""
    slot_cap = (((LG_N + 3) & ~3) + 63) & ~63
    return {"grey of one batch": LG_N * 1024, "second slot's grey start": slot_cap * 1024,
            "second slot's windows start": slot_cap * win_stride(1024), "second slot's entries start": slot_cap * ent_stride(1024) * 4}


def large_device_gb():
    """Device memory the two-slot chain of the large case allocates: per window slot, windows + entries + grey + the rest of the
    per-window scratch (< 600 B), twice, plus both batches' frames and boxes."""
    per_win = win_stride(1024) + ent_stride(1024) * 4 + 1024 + 600
    return (2 * LG_N * per_win + 2 * LG_N * (LG_H * LG_W * 3 + 16)) / 1e9


# ---- CPU: every case is in its regime ------------------------------------------------------------------------------------
def test_rec_mode_cases_reach_their_regimes(oracle):
    capi, kern = _src("tsd_capi.cu"), _src("tsd_kernels.cuh")
    assert int(re.search(r"kKnnTile = (\d+);", kern).group(1)) == KNN_TILE
    assert int(re.search(r"kKnnThreads = (\d+);", kern).group(1)) == KNN_THREADS
    for line in ("const int qblocks = cdiv(n_max, kKnnThreads), ntiles = cdiv(c->knn_ntrain, kKnnTile);",
                 "int nsplit = qblocks >= c->sm_count ? 1 : std::min(ntiles, cdiv(2 * c->sm_count, std::max(qblocks, 1)));",
                 "const int tiles = cdiv(ntiles, nsplit);", "return cdiv(ntiles, tiles);"):
        assert line in capi, line                                              # knn_splits above restates these
    assert "TRY(hog ? dev_knn(c, hog, d_nsurv, nb, Z, pd, pi, id) : dev_knn(c, gray, d_nsurv, nb, Z, pd, pi, id));" in capi
    # stage names: the header's list and the chain's marks
    h = open(os.path.join(ROOT, "include", "tsd_b200.h")).read()
    assert "k6_gray, k7_hog (absent with TSD_REC_GRAY), then k8_lda" in h and "with TSD_REC_KNN, k8_knn" in h
    for s in ("k6_gray", "k7_hog", "k8_lda", "k8_knn"):
        assert 'mark(c, "%s");' % s in capi, s
    # layouts: every route reached, labels of every mode varied and robust, det_cap layouts exist, staged layouts stage bytes
    assert set(ROUTES) == {"device", "pageable", "staged", "staged_chunks", "gather", "zerocopy_off"}
    rows = {stages(n, r) for n in LAYOUTS for r in ROUTES}
    assert rows == {True, False}
    assert sum(staged_bytes(n, 32)[0] > 0 for n in LAYOUTS if stages(n, "staged")) >= 5
    sv = [s for v in layout_survivors().values() for s in v]
    for mode in MODES:
        gray = mode.startswith("gray")
        X = feats(sv, gray)
        lab = predict(layout_models()[mode], X)
        assert len(set(lab[lab != 0].tolist())) >= 3, mode
        assert robust(layout_models()[mode], X, gray), mode
        assert detcap_layout(mode) is not None, mode
        assert sum(len(r) for r, _ in layout_expected(mode).values()) > 20, mode
    # split regime: each case has the bound and survivors it names, and is on its side of the line
    psv = split_pool()[2]
    assert len(psv) == SPLIT_POOL and all(len(s[0]) == 1 for s in psv)
    assert len(distinct_first(np.stack([s[1][0] for s in psv]), SPLIT_POOL)) == SPLIT_POOL
    for name, nb, ns in SPLIT_CASES:
        frames, boxes, off, _ = split_case(name)
        assert len(boxes) == nb == off[-1], name
        rec, counts = split_expected(name, "gray_knn")
        assert counts[2] == ns, (name, counts)
        nsplit, _ = knn_splits(nb, SPLIT_NTRAIN)
        want_split = name in ("split", "edge_0", "edge_1", "edge_128k1", "below_line")
        assert (nsplit > 1) == want_split, (name, nsplit)
        assert (ns < SPLIT_LINE) and (nb >= SPLIT_LINE) == (not want_split)
        if name.startswith("edge"):
            assert nb % 128 == 1
        assert frames.shape[1:] == (SPLIT_H, SPLIT_W, 3) and (3 * SPLIT_W) % 16 == 0          # the staged route stages them
    assert knn_splits(SPLIT_LINE - 128, SPLIT_NTRAIN)[0] >= 2 and knn_splits(SPLIT_LINE, SPLIT_NTRAIN)[0] == 1
    assert {ns for _, _, ns in SPLIT_CASES} >= {0, 1, 128 * SPLIT_K + 1}
    wf, wb, wo = split_warmup()
    assert len(wo) == len(wf) + 1 and wo[-1] == len(wb) and np.all(np.diff(wo) >= 0)
    for name, nb, _ in SPLIT_CASES:
        frames, boxes, off, _ = split_case(name)
        assert len(wf) >= len(frames) and len(wb) >= nb and np.diff(wo).max() >= np.diff(off).max(), name
    assert not oracle.expand_boxes(wb, 1.15)[1].any()                         # the warm-up's boxes all fail the aspect test
    for mode, m in split_models().items():
        gray = mode.startswith("gray")
        X = feats(psv, gray)
        assert robust(m, X, gray), mode
        # the last split's rows hold some query's k nearest: a merge without its list changes labels
        ns, rps = knn_splits(1281, SPLIT_NTRAIN)
        cut = (ns - 1) * rps
        full = predict(m, X)
        part = _oracle().knn_predict(X, m["xbar"], m["S"], m["Zt"][:cut], m["yt"][:cut], m["k"])[1]
        assert np.sum(full != part) > 10, mode
    # past 4 GiB: sizes, patterns, models
    assert is_prime(P) and P % 2 == 1
    for what, nbytes in large_buffers().items():
        assert nbytes > 1 << 32, what
    assert LG_N * 1024 > (1 << 32) > (1 << 31) and (LG_N - P) * 1024 == 1 << 32
    assert ((1 << 31) // 1024) % P and ((1 << 32) // 1024) % P                 # a wrap lands on another pattern
    for bt in (0, 1):
        fr, psv2 = large_patterns(bt)
        assert all(len(s[0]) == 1 for s in psv2) and len(fr) == P
    G = np.concatenate([feats(large_patterns(bt)[1], True) for bt in (0, 1)])
    for mode, m in large_models().items():
        lab = predict(m, G)
        assert len(set(lab.tolist())) >= 4, mode
        assert robust(m, G, True), mode
    assert 60 < large_device_gb() < 90
    # sequences: the chain survivors of test_gpu_rec_classifiers under both k of each k-NN model and both LDA sizes
    csv = chain_survivors()
    for mode, m in seq_models().items():
        gray = mode[0].startswith("gray")
        X = np.concatenate([s[1].reshape(-1, 1024).astype(np.float32) if gray else s[2] for s in csv])
        assert robust(m, X, gray), mode
        assert len(set(predict(m, X).tolist())) >= 3, mode
    assert seq_models()[("hog_knn", 1)]["k"] != seq_models()[("hog_knn", 0)]["k"]
    assert len(seq_models()[("gray_knn", 1)]["Zt"]) != len(seq_models()[("gray_knn", 0)]["Zt"])
    # config: proba_tol 0.2 and 0.8 decide away from their thresholds and 0.8 removes records
    G = np.concatenate([s[1].reshape(-1, 1024).astype(np.float32) for s in csv])
    m = seq_models()[("gray_lda", 0)]
    for tol in (0.2, 0.8):
        assert robust(m, G, True, tol), tol
    assert np.sum(predict(m, G, 0.8) != 0) < np.sum(predict(m, G, 0.2) != 0)
    # knn_k: the header, the engine and tsd_create agree
    assert "tsd_create: TSD_E_INVALID otherwise" in h and "the k-NN kernels use" in h
    assert 'if (c->cfg.knn_k < 1 || c->cfg.knn_k > kKnnMaxK)' in capi
    import tsd_b200
    assert inspect.signature(tsd_b200.Context.set_knn).parameters["k"].default is None


@functools.lru_cache(None)
def seq_models():
    """(mode, generation) -> model on the chain survivors of test_gpu_rec_classifiers; generation 1 of a k-NN mode has another k
    and another training-set size."""
    csv = chain_survivors()
    H = np.concatenate([s[2] for s in csv])
    G = np.concatenate([s[1].reshape(-1, 1024).astype(np.float32) for s in csv])
    return {("hog_lda", 0): lda_model(H, False), ("gray_lda", 0): lda_model(G, True),
            ("hog_knn", 0): knn_model(H, False, 61), ("hog_knn", 1): knn_model(H, False, 62, k=7, ntrain=20001),
            ("gray_knn", 0): knn_model(G, True, 63), ("gray_knn", 1): knn_model(G, True, 64, k=1, ntrain=3001)}


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------
def _A():
    import tsd_b200
    return tsd_b200._capi


@pytest.fixture
def make_ctx(tsd, monkeypatch):
    """Contexts created under an environment (read at tsd_create); all closed at the end of the test."""
    made = []

    def mk(flavour="rec", env=None, config=None):
        for k in ("TSD_STAGE", "TSD_STAGE_CHUNK", "TSD_CHUNK_FRAMES", "TSD_ZEROCOPY", "TSD_OVERLAP", "TSD_STAGGER", "TSD_GRAPH"):
            monkeypatch.delenv(k, raising=False)
        for k, v in (env or {}).items():
            monkeypatch.setenv(k, v)
        c = tsd.Context(0, flavour, config=config)
        made.append(c)
        return c
    yield mk
    for c in made:
        c.close()


def recs(det):
    return [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]


def det_call(ctx, mode, p, lay, nframes, boxes, off, cap):
    import ctypes as C
    A = _A()
    H, W, rs, fs = lay[:4]
    det = np.zeros(max(cap, 1), A.DET_DTYPE); nd = C.c_int32(-1); counts = np.full(4, -1, np.int32)
    rc = ctx._L.tsd_detect_frames(ctx._h, mode, A.ptr(p), nframes, H, W, rs, fs, A.ptr(boxes), A.ptr(off), A.ptr(det), cap, C.byref(nd),
                                  A.ptr(counts), A.MEM_HOST)
    return rc, det[:max(nd.value, 0)], nd.value, counts.tolist()


def enqueue(ctx, mode, d_frames, nframes, H, W, rs, fs, d_boxes, d_off, nb, maxb=0):
    A = _A()
    A.check(ctx._L.tsd_enqueue_frames(ctx._h, mode, A.ptr(d_frames), nframes, H, W, rs, fs, A.ptr(d_boxes), A.ptr(d_off), nb, maxb))


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- GPU: layouts and host routes ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("mode", MODES)
def test_rec_modes_layouts(tsd, make_ctx, mode, route):
    """Every layout through one route: records and stage counts equal the oracle's; staged layouts first run twice on other
    pixels (both slots' mirrors hold stale bytes), then stage exactly the stage_mark model's bytes; other routes stage none."""
    import torch
    A = _A()
    mem, env = ROUTES[route]
    ctx = make_ctx("rec", env)
    set_model(ctx, layout_models()[mode])
    rm = run_mode(tsd, mode)
    exp_all = layout_expected(mode)
    bad = []
    for name in LAYOUTS:
        boxes, off = boxes_for(name, 32)
        exp, ecounts = exp_all[name]
        canvas, _, lay = canvas_for(name)
        H, W, rs, fs, base = lay
        if mem == "device":
            d_canvas = dev(canvas)
            d_boxes, d_off = dev(boxes), dev(off)
            enqueue(ctx, rm, d_canvas.data_ptr() + base, LF, H, W, rs, fs, d_boxes.data_ptr(), d_off.data_ptr(), len(boxes))
            det, counts = ctx.fetch_detections(len(boxes))
            got, gcounts = recs(det), counts.tolist()
            del d_canvas
        elif mem == "pageable":
            rc, det, _, gcounts = det_call(ctx, rm, canvas.ctypes.data + base, lay, LF, boxes, off, len(boxes))
            A.check(rc)
            got = recs(det)
        else:
            ctx.pin(canvas)
            try:
                real = canvas.copy()
                if stages(name, route):
                    canvas[:] = 255 - real
                    for _ in range(2):
                        A.check(det_call(ctx, rm, canvas.ctypes.data + base, lay, LF, boxes, off, len(boxes))[0])
                    canvas[:] = real
                ctx.stat_staged_bytes(reset=True)
                rc, det, _, gcounts = det_call(ctx, rm, canvas.ctypes.data + base, lay, LF, boxes, off, len(boxes))
                A.check(rc)
                staged = ctx.stat_staged_bytes(reset=True)
            finally:
                ctx.unpin(canvas)
            got = recs(det)
            want = staged_bytes(name, 32)[0] if stages(name, route) else 0
            if staged != want:
                bad.append((name, "staged bytes", staged, want))
        if got != exp or gcounts != list(ecounts):
            bad.append((name, "records", len(got), len(exp), gcounts, list(ecounts)))
    torch.cuda.synchronize()
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("route", DETCAP_ROUTES)
@pytest.mark.parametrize("mode", MODES)
def test_rec_modes_det_cap(tsd, make_ctx, mode, route):
    """det_cap = 0 and n - 1: TSD_E_NOMEM with *ndet = n and the stage counts filled in; det_cap = n: the oracle's records; the
    context keeps working afterwards."""
    import ctypes as C
    A = _A()
    mem, env = ROUTES[route]
    ctx = make_ctx("rec", env)
    set_model(ctx, layout_models()[mode])
    rm = run_mode(tsd, mode)
    name = detcap_layout(mode)
    boxes, off = boxes_for(name, 32)
    exp, ecounts = layout_expected(mode)[name]
    n = len(exp)
    canvas, _, lay = canvas_for(name)
    H, W, rs, fs, base = lay
    if mem == "device":
        d_canvas, d_boxes, d_off = dev(canvas), dev(boxes), dev(off)
        for cap in (0, n - 1, n, n):
            enqueue(ctx, rm, d_canvas.data_ptr() + base, LF, H, W, rs, fs, d_boxes.data_ptr(), d_off.data_ptr(), len(boxes))
            det = np.zeros(max(cap, 1), A.DET_DTYPE); nd = C.c_int32(-1); counts = np.full(4, -1, np.int32)
            rc = ctx._L.tsd_fetch_detections(ctx._h, A.ptr(det), cap, C.byref(nd), A.ptr(counts))
            assert nd.value == n and counts.tolist() == list(ecounts), (cap, nd.value, counts.tolist())
            assert rc == (E_NOMEM if cap < n else 0), cap
            if cap == n:
                assert recs(det[:n]) == exp
        return
    ctx.pin(canvas)
    try:
        for cap in (0, n - 1, n, n):
            rc, det, nd, counts = det_call(ctx, rm, canvas.ctypes.data + base, lay, LF, boxes, off, cap)
            assert nd == n and counts == list(ecounts), (cap, nd, counts)
            assert rc == (E_NOMEM if cap < n else 0), (cap, rc)
            if cap == n:
                assert recs(det) == exp
    finally:
        ctx.unpin(canvas)


# ---- GPU: the split regime ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("route", ("device", "staged"))
@pytest.mark.parametrize("mode", ("hog_knn", "gray_knn"))
def test_knn_split_regime_through_the_chain(tsd, make_ctx, mode, route):
    """The SPLIT_CASES batches in a row.  device: overlapped, each batch read with fetch_previous while the next runs, so two
    splitting batches hold both slots' partial lists at once; staged: page-locked frames staged whole by tsd_detect_frames."""
    if sm_count() != SM_B200:
        pytest.skip("the cases are placed around the split line of a %d-SM device" % SM_B200)
    A = _A()
    mem, env = ROUTES[route]
    ctx = make_ctx("rec", env)
    set_model(ctx, split_models()[mode])
    rm = run_mode(tsd, mode)
    bad, keep, pending = [], [], None
    if mem == "device":
        wf, wb, wo = split_warmup()
        keep.append((dev(wf), dev(wb), dev(wo)))
        enqueue(ctx, rm, keep[0][0].data_ptr(), len(wf), SPLIT_H, SPLIT_W, SPLIT_W * 3, SPLIT_H * SPLIT_W * 3, keep[0][1].data_ptr(),
                keep[0][2].data_ptr(), len(wb), int(np.diff(wo).max()))
        assert ctx.fetch_detections(len(wb))[1].tolist()[1:] == [0, 0, 0]
    for name, nb, _ in SPLIT_CASES:
        frames, boxes, off, _ = split_case(name)
        exp = split_expected(name, mode)
        nf = len(frames)
        lay = (SPLIT_H, SPLIT_W, SPLIT_W * 3, SPLIT_H * SPLIT_W * 3)
        if mem == "device":
            d = (dev(frames), dev(boxes), dev(off))
            keep.append(d)
            enqueue(ctx, rm, d[0].data_ptr(), nf, *lay, d[1].data_ptr(), d[2].data_ptr(), nb, int(np.diff(off).max()))
            if pending is not None:
                det, counts = ctx.fetch_detections(pending[1][1][0], previous=True)
                if (recs(det), counts.tolist()) != pending[1]:
                    bad.append((pending[0], len(recs(det)), len(pending[1][0]), counts.tolist(), pending[1][1]))
            pending = (name, exp)
        else:
            host = np.ascontiguousarray(frames)
            ctx.pin(host)
            try:
                rc, det, _, counts = det_call(ctx, rm, host.ctypes.data, lay, nf, boxes, off, nb)
            finally:
                ctx.unpin(host)
            A.check(rc)
            if (recs(det), counts) != exp:
                bad.append((name, len(recs(det)), len(exp[0]), counts, exp[1]))
    if pending is not None:
        det, counts = ctx.fetch_detections(pending[1][1][0])
        if (recs(det), counts.tolist()) != pending[1]:
            bad.append((pending[0], len(recs(det)), len(pending[1][0]), counts.tolist(), pending[1][1]))
    assert not bad, bad


# ---- GPU: past 4 GiB ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("gray_lda", "gray_knn"))
def test_gray_chain_past_4gib(tsd, make_ctx, mode):
    """Two overlapped tsd_enqueue_frames batches of 2^22 + 4 099 frames of 8 x 8, one box each: every box survives, a batch's grey
    windows span 4.3 GB and the second slot's start 4.3 GB into b_gray.  Batch 1 read with fetch_previous, batch 2 with
    fetch_detections."""
    import torch
    room(large_device_gb() + 4.0, host_gb=1.5)
    model = large_models()[mode]
    ctx = make_ctx("rec")
    set_model(ctx, model)
    rm = run_mode(tsd, mode)
    exp, keep = [], []
    lay = (LG_H, LG_W, LG_W * 3, LG_H * LG_W * 3)
    d_box = dev(np.array([LG_BOX], np.int32)).repeat(LG_N, 1).contiguous()
    d_off = torch.arange(0, LG_N + 1, dtype=torch.int32, device="cuda")
    for bt in (0, 1):
        frames, sv = large_patterns(bt)
        lab = predict(model, feats(sv, True))
        per = [np.array([list(s[0][0]) + [int(l), 0]] if l else [], np.int64).reshape(-1, 6) for s, l in zip(sv, lab)]
        nz = np.asarray(lab) != 0
        exp.append((tile_records(per, LG_N), [LG_N, LG_N, LG_N, int(nz.sum() * (LG_N // P) + nz[:LG_N % P].sum())]))
        d_fr = dev(frames).repeat(-(-LG_N // P), 1, 1, 1)[:LG_N]
        keep.append(d_fr)
        enqueue(ctx, rm, d_fr.data_ptr(), LG_N, *lay, d_box.data_ptr(), d_off.data_ptr(), LG_N, 1)
    got = [ctx.fetch_detections(LG_N, previous=True), ctx.fetch_detections(LG_N)]
    del keep
    for bt in (0, 1):
        det, counts = got[bt]
        erec, ecounts = exp[bt]
        assert counts.tolist() == ecounts, (bt, counts.tolist(), ecounts)
        g = np.stack([det[k] for k in ("frame", "x1", "y1", "x2", "y2", "id", "hundredths")], 1).astype(np.int64)
        if not np.array_equal(g, erec):
            i = np.flatnonzero(np.any(g != erec, 1))[:10] if g.shape == erec.shape else []
            raise AssertionError((bt, g.shape, erec.shape, [(int(j), g[j].tolist(), erec[j].tolist()) for j in i]))


# ---- GPU: sequences ---------------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def det32_expected():
    """Per unique frame of chain_inputs: the oracle's detection records at D = 32, x1.15 (a detection batch on the rec context)."""
    import tsd_b200
    from test_gpu_large import det32_templates
    O = _oracle()
    uniq, per, _, _ = chain_inputs(tsd_b200)
    r6, b6 = det32_templates()
    out = []
    for u in range(len(uniq)):
        o = O.detect_frame(uniq[u], per[u], r6, b6, percentage=1.15, D=32)
        out.append([tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])])
    return out


def seq_expected(kind, model, ids):
    """Records of a batch whose frame f is unique frame ids[f]."""
    if kind == "det":
        d = det32_expected()
        return [(f,) + r for f, u in enumerate(ids) for r in d[u]]
    csv = chain_survivors()
    gray = kind.startswith("gray")
    rec = []
    for f, u in enumerate(ids):
        c2, g, h = csv[u]
        if len(c2):
            lab = predict(model, g.reshape(-1, 1024).astype(np.float32) if gray else h)
            rec += [(f,) + tuple(int(v) for v in q) + (int(l), 0) for q, l in zip(c2, lab) if l != 0]
    return rec


@pytest.mark.gpu
@pytest.mark.parametrize("env", list(SEQ_ENV))
def test_rec_modes_in_sequence(tsd, make_ctx, env):
    """Blocks X Y X Y X Y of two modes (a GRAY or k-NN mode X, and detection or another recognition mode Y) on one D = 32 context,
    each block after its models are set; two blocks change the k-NN model (another k and training-set size) after their sixth
    batch.  Every batch read back (fetch_previous while the next one runs when overlapped).  With graphs each mode's batches run
    eager, captured, replayed -- and the first batch after a model change runs eagerly again."""
    import torch
    from test_gpu_large import det32_templates
    A = _A()
    ctx = make_ctx("rec", SEQ_ENV[env])
    graphs = "TSD_GRAPH" not in SEQ_ENV[env]
    overlap = "TSD_OVERLAP" not in SEQ_ENV[env]
    ctx.set_templates(*det32_templates())
    uniq, per, _, _ = chain_inputs(tsd)
    U = len(uniq)
    bufs = [(torch.empty((SEQ_F, 800, 1360, 3), dtype=torch.uint8, device="cuda"), torch.empty((SEQ_F * 200, 4), dtype=torch.int32, device="cuda"))
            for _ in range(3)]
    d_off = torch.arange(0, SEQ_F * 200 + 1, 200, dtype=torch.int32, device="cuda")
    M = seq_models()

    def mode_of(kind):
        return A.RUN_DETECT if kind == "det" else run_mode(tsd, kind)

    def models_for(x, y, gen):
        out = {}
        for kind in (x, y):
            if kind != "det":
                out[kind] = M.get((kind, gen), M[(kind, 0)])
        return out

    # warm-up: every mode once, so that no scratch buffer grows (a growth starts a new graph generation) inside the blocks
    for kind in ("hog_lda", "hog_knn", "det", "gray_lda", "gray_knn"):
        if kind != "det":
            set_model(ctx, M[(kind, 0)])
        fr, bx = bufs[2]
        fr.copy_(torch.from_numpy(uniq[:SEQ_F])); bx.copy_(torch.from_numpy(np.concatenate(per[:SEQ_F])))
        torch.cuda.synchronize()
        enqueue(ctx, mode_of(kind), fr.data_ptr(), SEQ_F, 800, 1360, 4080, 4080 * 800, bx.data_ptr(), d_off.data_ptr(), SEQ_F * 200, 200)
        ctx.fetch_detections(SEQ_F * 200)
    bad, events, pending, i = [], [], None, 0
    for x, y, change in SEQ_BLOCKS:
        for gen in ((0, 1) if change else (0,)):
            cur = models_for(x, y, gen)
            if pending is not None:                          # (a model change waits for the device anyway)
                if recs(ctx.fetch_detections(SEQ_F * 200)[0]) != pending[1]:
                    bad.append(pending[0])
                pending = None
            for kind, m in cur.items():
                set_model(ctx, m)
            for j in range(6):
                kind = (x, y)[j % 2]
                ids = [(3 * i + 5 * f) % U for f in range(SEQ_F)]
                i += 1
                fr, bx = bufs[j % 2]
                fr.copy_(torch.from_numpy(uniq[ids])); bx.copy_(torch.from_numpy(np.concatenate([per[u] for u in ids])))
                torch.cuda.synchronize()
                c0, r0 = ctx.stat_graphs()
                enqueue(ctx, mode_of(kind), fr.data_ptr(), SEQ_F, 800, 1360, 4080, 4080 * 800, bx.data_ptr(), d_off.data_ptr(), SEQ_F * 200, 200)
                c1, r1 = ctx.stat_graphs()
                events.append(((x, y, gen), kind, j // 2, (c1 - c0, r1 - r0)))
                rec = seq_expected(kind, cur.get(kind), ids)
                if pending is not None and recs(ctx.fetch_detections(SEQ_F * 200, previous=True)[0]) != pending[1]:
                    bad.append(pending[0])
                pending = ((x, y, gen, j, kind), rec)
                if not overlap:
                    if recs(ctx.fetch_detections(SEQ_F * 200)[0]) != rec:
                        bad.append(pending[0])
                    pending = None
    if pending is not None:
        det, counts = ctx.fetch_detections(SEQ_F * 200)
        if recs(det) != pending[1]:
            bad.append(pending[0])
    assert not bad, bad
    # eager, captured, replayed for each mode of each block and model generation; nothing without graphs
    want = [(0, 0), (1, 0), (0, 1)] if graphs else [(0, 0)] * 3
    wrong = [e for e in events if e[3] != want[e[2]]]
    assert not wrong, wrong[:12]


# ---- GPU: config and profiling ---------------------------------------------------------------------------------------------------
def _chain_device_batch(tsd, F):
    uniq, per, boxes, off = chain_inputs(tsd)
    import torch
    d_frames = dev(uniq)[torch.arange(F, device="cuda") % len(uniq)].contiguous()
    return d_frames, dev(boxes[:off[F]]), dev(off[:F + 1]), int(off[F])


@pytest.mark.gpu
@pytest.mark.parametrize("tol", (0.2, 0.8))
def test_gray_lda_proba_tol(tsd, make_ctx, tol):
    """GRAY + LDA with proba_tol 0.2 and 0.8 in the config: the oracle's decision at that tolerance."""
    cfg = tsd.default_config("rec")
    cfg.proba_tol = tol
    ctx = make_ctx("rec", config=cfg)
    m = seq_models()[("gray_lda", 0)]
    set_model(ctx, m)
    F = 64
    d_frames, d_boxes, d_off, nb = _chain_device_batch(tsd, F)
    enqueue(ctx, run_mode(tsd, "gray_lda"), d_frames.data_ptr(), F, 800, 1360, 4080, 4080 * 800, d_boxes.data_ptr(), d_off.data_ptr(), nb, 200)
    det, _ = ctx.fetch_detections(nb)
    csv = chain_survivors()
    exp = []
    for f in range(F):
        c2, g, _ = csv[f % len(csv)]
        if len(c2):
            lab = predict(m, g.reshape(-1, 1024).astype(np.float32), tol)
            exp += [(f,) + tuple(int(v) for v in q) + (int(l), 0) for q, l in zip(c2, lab) if l != 0]
    assert recs(det) == exp


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ALL_MODES)
def test_rec_modes_profiling(tsd, make_ctx, mode):
    """tsd_set_profiling(1): two batches, records unchanged, tsd_stage_times names = the front half, then the header's stages of
    this mode, then "detections".  tsd_set_profiling(2): two overlapped batches, records unchanged, tsd_timeline non-decreasing
    from every batch's "start" to its "detections"."""
    ctx = make_ctx("rec")
    m = seq_models()[(mode, 0)]
    set_model(ctx, m)
    F = 16
    d_frames, d_boxes, d_off, nb = _chain_device_batch(tsd, F)
    exp = seq_expected(mode, m, [f % 32 for f in range(F)])
    rm = run_mode(tsd, mode)
    args = (d_frames.data_ptr(), F, 800, 1360, 4080, 4080 * 800, d_boxes.data_ptr(), d_off.data_ptr(), nb, 200)
    enqueue(ctx, rm, *args)
    assert recs(ctx.fetch_detections(nb)[0]) == exp
    ctx.set_profiling(1)
    for _ in range(2):
        enqueue(ctx, rm, *args)
        assert recs(ctx.fetch_detections(nb)[0]) == exp
    names = [n for n, _ in ctx.stage_times()]
    k = names.index("k5_fold")
    assert names[:2] == ["k1_expand_filter", "k2_crop_resize"] and "k5_hist" in names[:k]
    assert names[k + 1:] == STAGES_REC[mode] + ["detections"], names
    ctx.set_profiling(2)
    enqueue(ctx, rm, *args)
    enqueue(ctx, rm, *args)
    assert recs(ctx.fetch_detections(nb, previous=True)[0]) == exp
    assert recs(ctx.fetch_detections(nb)[0]) == exp
    tl = ctx.timeline()
    starts = [j for j, (n, _) in enumerate(tl) if n == "start"]
    assert len(starts) == 2 and starts[0] == 0
    for a, b in zip(starts, starts[1:] + [len(tl)]):
        seg = tl[a:b]
        assert [n for n, _ in seg][-1] == "detections" and STAGES_REC[mode] == [n for n, _ in seg if n in ("k6_gray", "k7_hog", "k8_lda", "k8_knn")]
        t = [v for _, v in seg]
        assert all(u <= v for u, v in zip(t, t[1:])), seg
    ctx.set_profiling(0)


# ---- GPU: knn_k ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_knn_k_config(tsd, oracle, make_ctx):
    """tsd_create refuses knn_k 0 and 9; a context created with knn_k = 1 (or 8) gets that k from Context.set_knn without k, and
    an explicit k still wins."""
    from test_gpu_rec_classifiers import knn_lattice_sweep
    for k in (0, 9, -1):
        cfg = tsd.default_config("rec")
        cfg.knn_k = k
        with pytest.raises(tsd.TsdError, match="knn_k"):
            make_ctx("rec", config=cfg)
    X, xbar, S, Zt, yt = knn_lattice_sweep(3 * KNN_TILE + 5, 17, nq=500)
    olab = {k: oracle.knn_predict(X, xbar, S, Zt, yt, k)[1] for k in (1, 4, 8)}
    assert np.sum(olab[1] != olab[4]) > 10 and np.sum(olab[8] != olab[4]) > 10
    for k in (1, 8):
        cfg = tsd.default_config("rec")
        cfg.knn_k = k
        ctx = make_ctx("rec", config=cfg)
        ctx.set_knn(xbar, S, Zt, yt)
        assert np.array_equal(ctx.knn_predict(X)[1], olab[k]), k
        ctx.set_knn(xbar, S, Zt, yt, 4)
        assert np.array_equal(ctx.knn_predict(X)[1], olab[4]), k
    ctx = make_ctx("rec")
    ctx.set_knn(xbar, S, Zt, yt)
    assert np.array_equal(ctx.knn_predict(X)[1], olab[4])
