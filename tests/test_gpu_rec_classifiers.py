"""The recognition chain for all four classifiers of the reference (REC/constants.py:10-12): HOG or GRAY descriptors, each with
LDABAYES or KNN, selected by OR-ing TSD_REC_GRAY / TSD_REC_KNN into TSD_RUN_RECOGNIZE, and the tiled k-NN kernels that both the
chain and tsd_knn_predict run.

  modes      1 024 frames x 200 candidates (32 unique frames) through tsd_enqueue_frames and through tsd_detect_frames on page-locked
             host frames, every mode against the oracle composition per frame: windows + both dedup passes -> bgr2gray -> (hog32)
             -> lda_predict / knn_predict.  The real 324- and 1 024-feature LDA weights with gap_bias biases (their own biases label
             nothing on synthetic frames), the real reducers with a training set sampled around the queries' Z (the real training
             sets label nothing or almost nothing).  The chain's k-NN labels also equal tsd_knn_predict on the same descriptors.
  k-NN sweep ntrain = 1, k - 1, tile - 1, tile, tile + 1, many tiles plus a remainder, 14 574 and 200 003; query counts 0, 1, below
             the split threshold and above one CTA; k = 1..8.  Integer lattices, so that exact distance ties straddle every tile
             boundary and therefore every split boundary; labels must follow (distance, index).  Through tsd_knn_predict and the
             chain (GRAY + KNN with a reducer that picks six pixels, so Z is exact and ties are exact too).
  sequences  the four modes in rotation on one overlapped context with CUDA graphs, models replaced mid-sequence.
  refusals   every mode / state refusal before any device work.
  drop-in    source_rec.recognizeBatch on the three stored real frames against the per-frame composition of the drop-in functions.

test_rec_classifier_inputs_reach_their_regimes checks on the CPU that each case is in the regime it names.
"""
import functools
import os
import re
import types

import numpy as np
import pytest

from test_gpu_recognition import chain_inputs
from test_gpu_sequences import gap_bias

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KNN_TILE, KNN_THREADS, SM_B200 = 256, 128, 148          # kKnnTile, kKnnThreads (tsd_kernels.cuh), SMs of a B200
SPLIT_BELOW = KNN_THREADS * SM_B200                      # fewer queries than this: the training set is split across CTAs
MODES = ("hog_lda", "hog_knn", "gray_lda", "gray_knn")
SWEEP_NTRAIN = lambda k: sorted({1, max(k - 1, 1), KNN_TILE - 1, KNN_TILE, KNN_TILE + 1, 9 * KNN_TILE + 77, 14574, 200003})
SWEEP_QUERIES = (0, 1, 300, 20000)


def run_mode(tsd, name):
    m = tsd.RUN_RECOGNIZE
    if name.startswith("gray"):
        m |= tsd.REC_GRAY
    if name.endswith("knn"):
        m |= tsd.REC_KNN
    return m


# ---- inputs -----------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def survivors(seed=41):
    """Per unique frame of chain_inputs(): (coords, grey windows [m,32,32], oracle HOG [m,324])."""
    import tsd_b200 as tsd
    from oracle import oracle as O
    uniq, per, _, _ = chain_inputs(tsd, seed=seed)
    out = []
    for f, bx in zip(uniq, per):
        c, v = O.expand_boxes(bx, 1.15)
        c = c[v]
        w = np.stack([O.crop_resize(f, cc, 32) for cc in c]) if len(c) else np.zeros((0, 32, 32, 3), np.uint8)
        w1, c1 = O.dedup(w, c, False, 0.85)
        w2, c2 = O.dedup(w1, c1, True, 0.95)
        g = np.stack([O.bgr2gray(x) for x in w2]) if len(c2) else np.zeros((0, 32, 32), np.uint8)
        h = np.stack([O.hog32(x) for x in g]) if len(c2) else np.zeros((0, 324), np.float32)
        out.append((c2, g, h))
    return out


def features(sv, gray):
    return np.concatenate([s[1].reshape(-1, 1024).astype(np.float32) if gray else s[2] for s in sv])


def sampled_knn(real, X, seed, k=4):
    """The real reducer with a training set sampled around the queries' Z: 14 574 rows, each a query's Z plus small Gaussian noise,
    labelled 0..6 by the query it comes from (queries with the same Z share a label)."""
    rng = np.random.default_rng(seed)
    Zq = (X.astype(np.float64) - real["knn_xbar"]) @ real["knn_scalings"]
    _, inv = np.unique(np.round(Zq, 6), axis=0, return_inverse=True)
    qlab = rng.integers(0, 7, inv.max() + 1)[inv.ravel()].astype(np.int32)
    src = rng.integers(0, len(Zq), 14574)
    return dict(xbar=real["knn_xbar"], S=real["knn_scalings"], Zt=Zq[src] + 0.01 * rng.standard_normal((14574, 6)), yt=qlab[src], k=k)


@functools.lru_cache(None)
def models():
    """{mode: model dict} for the four modes on survivors()."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz"))
    gg = np.load(os.path.join(ROOT, "tests", "golden", "rec_gray_golden.npz"))
    sv = survivors()
    H, G = features(sv, False), features(sv, True)
    return {"hog_lda": dict(W=g["lda_W"], b=gap_bias(H, g["lda_W"])),
            "gray_lda": dict(W=gg["lda_W"], b=gap_bias(G, gg["lda_W"])),
            "hog_knn": sampled_knn(g, H, 5),
            "gray_knn": sampled_knn(gg, G, 6)}


def predict(oracle, model, X):
    if "W" in model:
        return oracle.lda_predict(X, model["W"], model["b"], 0.5)[1]
    return oracle.knn_predict(X, model["xbar"], model["S"], model["Zt"], model["yt"], model["k"])[1]


def set_model(ctx, model):
    if "W" in model:
        ctx.set_lda(model["W"], model["b"])
    else:
        ctx.set_knn(model["xbar"], model["S"], model["Zt"], model["yt"], model["k"])


def expected_records(oracle, sv, frame_ids, model, gray):
    """Records (frame, x1, y1, x2, y2, label) of a batch whose frame f is unique frame frame_ids[f]."""
    out = []
    labs = {u: predict(oracle, model, features([sv[u]], gray)) if len(sv[u][0]) else [] for u in set(frame_ids)}
    for f, u in enumerate(frame_ids):
        out += [(f,) + tuple(int(v) for v in c) + (int(l),) for c, l in zip(sv[u][0], labs[u]) if l != 0]
    return out


def records(det):
    return [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"])) for d in det]


def knn_lattice_sweep(ntrain, seed, nq=max(SWEEP_QUERIES)):
    """Integer queries and training rows in {0,1,2}^6 (Z = X exactly), the rows around every tile boundary duplicated under
    different labels: rows t*TILE - 2 .. t*TILE + 1 are copies of one point."""
    rng = np.random.default_rng(seed)
    Zt = rng.integers(0, 3, (ntrain, 6)).astype(np.float64)
    for t in range(1, (ntrain - 1) // KNN_TILE + 1):
        b = t * KNN_TILE
        Zt[max(b - 2, 0):min(b + 2, ntrain)] = Zt[b - 1]
    yt = rng.integers(0, 16, ntrain).astype(np.int32)
    X = rng.integers(0, 3, (nq, 6)).astype(np.float32)
    return X, np.zeros(6), np.eye(6), Zt, yt


def pixel_reducer(seed):
    """A 1 024-feature reducer that picks six grey pixels: Z of a window is six of its bytes, exactly."""
    rng = np.random.default_rng(seed)
    S = np.zeros((1024, 6))
    S[rng.choice(1024, 6, replace=False), np.arange(6)] = 1.0
    return np.zeros(1024), S


def chain_lattice(ntrain, seed):
    """Training rows for the chain sweep: Z values of the survivors under pixel_reducer (so queries tie with rows exactly),
    duplicated around every tile boundary under different labels."""
    xbar, S = pixel_reducer(seed)
    G = features(survivors(), True)
    rng = np.random.default_rng(seed)
    Zt = (G.astype(np.float64) @ S)[rng.integers(0, len(G), ntrain)]
    for t in range(1, (ntrain - 1) // KNN_TILE + 1):
        b = t * KNN_TILE
        Zt[max(b - 2, 0):min(b + 2, ntrain)] = Zt[b - 1]
    return xbar, S, Zt, rng.integers(0, 16, ntrain).astype(np.int32)


def knn_robust(m, X, lab, rel=1e-5, eps=1e-7):
    """Every query's label stays the same whichever rows within reach of the k-th distance (for descriptors moved by up to
    rel * |x| + eps each) fill the k places."""
    import itertools
    Z = (X.astype(np.float64) - m["xbar"]) @ m["S"]
    dz = np.sqrt((((rel * np.abs(X.astype(np.float64)) + eps) @ np.abs(m["S"])) ** 2).sum(1))
    k = m["k"]
    for i in range(len(Z)):
        d = ((Z[i] - m["Zt"]) ** 2).sum(1)
        o = np.argsort(d, kind="stable")
        dk = d[o[k - 1]]
        g = 2 * (2 * np.sqrt(dk) * dz[i] + dz[i] ** 2)
        sure = [t for t in o[:k] if d[t] < dk - g]
        maybe = [t for t in o[:k + 8] if abs(d[t] - dk) <= g]
        for pick in itertools.combinations(maybe, k - len(sure)):
            v = np.bincount(m["yt"][list(sure) + list(pick)], minlength=16)
            if int(np.argmax(v)) != int(lab[i]):
                return False
    return True


# ---- CPU --------------------------------------------------------------------------------------------------------------
def test_rec_constants_match_the_header(tsd):
    h = open(os.path.join(ROOT, "include", "tsd_b200.h")).read()
    d = dict((k, int(v)) for k, v in re.findall(r"#define (TSD_(?:RUN|REC)_\w+) (\d+)", h))
    assert d == {"TSD_RUN_DETECT": tsd.RUN_DETECT, "TSD_RUN_RECOGNIZE": tsd.RUN_RECOGNIZE, "TSD_REC_GRAY": tsd.REC_GRAY,
                 "TSD_REC_KNN": tsd.REC_KNN}
    k = open(os.path.join(ROOT, "opencv-traffic-sign-detector_b200", "csrc", "tsd_kernels.cuh")).read()
    assert int(re.search(r"kKnnTile = (\d+);", k).group(1)) == KNN_TILE
    assert int(re.search(r"kKnnThreads = (\d+);", k).group(1)) == KNN_THREADS


def test_rec_classifier_inputs_reach_their_regimes(oracle, tsd):
    sv = survivors()
    M = models()
    # every mode emits records of at least 3 distinct labels, and none of them is within reach of a different decision
    for name in MODES:
        gray = name.startswith("gray")
        X = features(sv, gray)
        lab = predict(oracle, M[name], X)
        assert len(set(lab[lab != 0].tolist())) >= 3, name
        if name == "hog_knn":      # K7's descriptors differ from hog32 by <= 1e-5 relative + 1e-7: no label can follow from that
            assert knn_robust(M[name], X, lab)
        if name == "hog_lda":
            z, _ = oracle.lda_predict(X, M[name]["W"], M[name]["b"], 0.5)
            guard = ((1e-5 * np.abs(X.astype(np.float64)) + 1e-7) @ np.abs(M[name]["W"])).max(1)
            zs = np.sort(np.where(z > 0, z, -np.inf), 1)
            with np.errstate(invalid="ignore"):
                gap = np.where(np.isfinite(zs[:, -2]), zs[:, -1] - zs[:, -2], np.inf)
            assert np.all(np.minimum(np.abs(z).min(1), gap) > 2 * guard)
    # the sweep's training-set sizes and query counts
    for k in range(1, 9):
        nt = SWEEP_NTRAIN(k)
        assert {1, KNN_TILE - 1, KNN_TILE, KNN_TILE + 1, 14574}.issubset(nt) and (k == 1 or k - 1 in nt) and max(nt) >= 200000
        assert any(n > 2 * KNN_TILE and n % KNN_TILE for n in nt)
    assert 0 in SWEEP_QUERIES and 1 in SWEEP_QUERIES
    assert any(KNN_THREADS < q < SPLIT_BELOW for q in SWEEP_QUERIES) and any(q >= SPLIT_BELOW for q in SWEEP_QUERIES)
    assert 8 * 200 < SPLIT_BELOW <= 1024 * 200                     # the chain sweep's 8-frame batch splits, the 1 024-frame one does not
    # lattice ties straddle tile (and so split) boundaries: a query's k nearest include a tie across a boundary that a flipped
    # index rule resolves differently
    X, xbar, S, Zt, yt = knn_lattice_sweep(9 * KNN_TILE + 77, 3, nq=300)
    assert np.array_equal(Zt[KNN_TILE - 1], Zt[KNN_TILE]) and yt[KNN_TILE - 1] != yt[KNN_TILE]
    flips = 0
    for k in (1, 4, 8):
        _, olab = oracle.knn_predict(X, xbar, S, Zt, yt, k)
        _, rlab = oracle.knn_predict(X, xbar, S, Zt[::-1].copy(), yt[::-1].copy(), k)
        flips += int(np.sum(olab != rlab))
    assert flips > 0
    # the chain's lattice: Z is exact (six bytes) and queries sit at exactly the same distance from several rows
    xbar, S, Zt, yt = chain_lattice(14574, 7)
    G = features(sv, True)
    Zq, _ = oracle.knn_predict(G, xbar, S, Zt, yt, 1)
    assert np.array_equal(Zq, G.astype(np.float64) @ S)
    d = ((Zq[:200, None, :] - Zt[None]) ** 2).sum(-1)
    assert np.all((d == d.min(1, keepdims=True)).sum(1) >= 2)


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _device_batch(tsd, U, F):
    import torch
    uniq, per, boxes, off = chain_inputs(tsd)
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(uniq).to(dev)[torch.arange(F, device=dev) % U].contiguous()
    return uniq, per, boxes[:off[F]], off[:F + 1], d_frames, torch.from_numpy(boxes[:off[F]]).to(dev), torch.from_numpy(off[:F + 1]).to(dev)


@pytest.mark.gpu
@pytest.mark.parametrize("name", MODES)
def test_four_modes_match_the_oracle(tsd, oracle, name):
    F = 1024
    uniq, per, boxes, off, d_frames, d_boxes, d_off = _device_batch(tsd, 32, F)
    sv = survivors()
    model = models()[name]
    gray = name.startswith("gray")
    exp = expected_records(oracle, sv, [f % 32 for f in range(F)], model, gray)
    mode = run_mode(tsd, name)
    with tsd.Context(0, "rec") as c:
        set_model(c, model)
        c.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), mode=mode,
                         max_boxes_per_frame=200)
        det, counts = c.fetch_detections(int(off[-1]))
        assert records(det) == exp and int(counts[3]) == len(exp), (name, counts.tolist(), len(exp))
        host = np.ascontiguousarray(uniq[np.arange(F) % 32])
        c.pin(host)
        try:
            det2, counts2 = c.detect_frames(host, boxes, off, mode=mode)
        finally:
            c.unpin(host)
        assert records(det2) == exp and np.array_equal(counts, counts2)
        if name.endswith("knn"):      # the chain's labels = tsd_knn_predict on the same descriptors (K6 / K7 of the GPU)
            lab = {}
            for u in range(32):
                if len(sv[u][0]):
                    X = sv[u][1].reshape(-1, 1024).astype(np.float32) if gray else c.hog(sv[u][1])
                    lab[u] = c.knn_predict(X, want_Z=False)[1]
            mine = [(f,) + tuple(int(v) for v in q) + (int(l),) for f in range(F) if f % 32 in lab
                    for q, l in zip(sv[f % 32][0], lab[f % 32]) if l != 0]
            assert mine == exp


@pytest.mark.gpu
def test_knn_sweep_entry_point(tsd, oracle):
    """tsd_knn_predict at every training-set size and query count of the sweep, k = 1..8, lattice ties across tile boundaries."""
    bad = []
    with tsd.Context(0, "rec") as c:
        for k in range(1, 9):
            for ntrain in SWEEP_NTRAIN(k):
                X, xbar, S, Zt, yt = knn_lattice_sweep(ntrain, 100 * k + ntrain % 97)
                c.set_knn(xbar, S, Zt, yt, k)
                for nq in (q for q in SWEEP_QUERIES if q * ntrain <= 4e8):     # (oracle time; the chain sweep takes 200 003 rows on 1 024 frames)
                    Z, lab = c.knn_predict(X[:nq])
                    oZ, olab = oracle.knn_predict(X[:nq], xbar, S, Zt, yt, k) if nq else (np.zeros((0, 6)), np.zeros(0, np.int32))
                    if not (np.array_equal(Z, oZ) and np.array_equal(lab, olab)):
                        bad.append((k, ntrain, nq, int(np.sum(lab != olab))))
    assert not bad, bad[:10]


@pytest.mark.gpu
@pytest.mark.parametrize("F", (8, 1024))
def test_knn_sweep_through_the_chain(tsd, oracle, F):
    """GRAY + KNN in the chain with a pixel-picking reducer (exact Z, exact ties), every sweep size, k = 1..8.  8 frames: n_max =
    1 600 candidates, so the training set is split; 1 024 frames: 204 800, one CTA range per query block."""
    uniq, per, boxes, off, d_frames, d_boxes, d_off = _device_batch(tsd, 32, F)
    sv = survivors()
    bad = []
    with tsd.Context(0, "rec") as c:
        for k in range(1, 9):
            for ntrain in SWEEP_NTRAIN(k):
                xbar, S, Zt, yt = chain_lattice(ntrain, 10 * k + 1)
                model = dict(xbar=xbar, S=S, Zt=Zt, yt=yt, k=k)
                set_model(c, model)
                c.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]),
                                 mode=run_mode(tsd, "gray_knn"), max_boxes_per_frame=200)
                det, _ = c.fetch_detections(int(off[-1]))
                if records(det) != expected_records(oracle, sv, [f % 32 for f in range(F)], model, True):
                    bad.append((k, ntrain))
    assert not bad, bad


@pytest.mark.gpu
def test_four_modes_in_sequence(tsd, oracle):
    """One overlapped context with graphs: blocks of HOG (HL HK x 3) and GRAY (GL GK x 3) batches, models replaced between blocks and
    once inside one (another k), every batch read back through tsd_fetch_previous while the next one runs."""
    import torch
    F, U = 8, 32
    uniq, per, _, _ = chain_inputs(tsd)
    sv = survivors()
    M = models()
    dev = torch.device("cuda", 0)
    bufs = [(torch.empty((F, 800, 1360, 3), dtype=torch.uint8, device=dev), torch.empty((F * 200, 4), dtype=torch.int32, device=dev))
            for _ in range(2)]
    d_off = torch.arange(0, F * 200 + 1, 200, dtype=torch.int32, device=dev)
    plan = []
    for rep in range(3):
        for block in (("hog_lda", "hog_knn"), ("gray_lda", "gray_knn")):
            for j in range(6):
                plan.append((block[j % 2], j == 0, rep == 1 and j == 3))
    counts = {m: 0 for m in MODES}
    pending = None
    with tsd.Context(0, "rec") as c:
        for i, (name, new_block, change_k) in enumerate(plan):
            if new_block or change_k:
                if pending is not None:
                    det, _ = c.fetch_detections(F * 200)
                    assert records(det) == pending, i
                    pending = None
                gray = name.startswith("gray")
                lda, knn = (("gray_lda", "gray_knn") if gray else ("hog_lda", "hog_knn"))
                set_model(c, M[lda])
                km = dict(M[knn])
                if change_k:
                    km["k"] = 7
                set_model(c, km)
                cur = {"lda": M[lda], "knn": km}
            ids = [(3 * i + 5 * f) % U for f in range(F)]
            fr, bx = bufs[i % 2]
            fr.copy_(torch.from_numpy(uniq[ids]))
            bx.copy_(torch.from_numpy(np.concatenate([per[u] for u in ids])))
            torch.cuda.synchronize()
            c.enqueue_frames(fr.data_ptr(), F, 800, 1360, bx.data_ptr(), d_off.data_ptr(), F * 200, mode=run_mode(tsd, name),
                             max_boxes_per_frame=200)
            exp = expected_records(oracle, sv, ids, cur["knn" if name.endswith("knn") else "lda"], name.startswith("gray"))
            if pending is not None:
                det, _ = c.fetch_detections(F * 200, previous=True)
                assert records(det) == pending, i
            pending = exp
            counts[name] += 1
        det, _ = c.fetch_detections(F * 200)
        assert records(det) == pending
        cap, rep = c.stat_graphs()
    assert min(counts.values()) >= 5 and cap > 0 and rep > 0, (counts, cap, rep)


@pytest.mark.gpu
def test_refusals_before_device_work(tsd):
    import tsd_b200._capi as A
    uniq, per, boxes, off = chain_inputs(tsd)
    frames, boxes, off = uniq[:2], boxes[:400], off[:3]
    g = np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz"))
    gg = np.load(os.path.join(ROOT, "tests", "golden", "rec_gray_golden.npz"))
    det = np.empty(400, A.DET_DTYPE)

    def call(ctx, mode):
        nd, cnt = A.C.c_int32(), np.zeros(4, np.int32)
        before = ctx.launch_count
        rc = ctx._L.tsd_detect_frames(ctx._h, mode, A.ptr(frames), 2, 800, 1360, 1360 * 3, 800 * 1360 * 3, A.ptr(boxes), A.ptr(off),
                                      A.ptr(det), 400, A.C.byref(nd), A.ptr(cnt), A.MEM_HOST)
        assert ctx.launch_count == before
        return rc, ctx._L.tsd_last_error().decode()

    R, GR, KN = tsd.RUN_RECOGNIZE, tsd.REC_GRAY, tsd.REC_KNN
    with tsd.Context(0, "rec") as c:
        for m in (tsd.RUN_DETECT | GR, tsd.RUN_DETECT | KN, R | 16, R | 1, 0, 16 | GR):
            assert call(c, m)[0] == -1, m
        for m, what in ((R, "324-feature LDA"), (R | GR, "1024-feature LDA"), (R | KN, "324-feature KNN"), (R | GR | KN, "1024-feature KNN")):
            rc, msg = call(c, m)
            assert rc == -3 and what in msg, (m, msg)
        c.set_lda(g["lda_W"], g["lda_b"])
        c.set_knn(g["knn_xbar"], g["knn_scalings"], g["knn_Ztrain"], g["knn_ytrain"], 4)
        assert call(c, R | GR)[0] == -3 and call(c, R | GR | KN)[0] == -3
        c.set_lda(gg["lda_W"], gg["lda_b"])
        assert call(c, R)[0] == -3 and call(c, R | GR | KN)[0] == -3
        for m in (R | KN, R | GR):                               # and the context works afterwards
            before = c.launch_count
            det2, counts = c.detect_frames(frames, boxes, off, mode=m)
            assert c.launch_count > before and int(counts[0]) == 400
    with tsd.Context(0, "det") as c:                             # D = 25
        c.set_lda(gg["lda_W"], gg["lda_b"])
        rc, msg = call(c, R | GR)
        assert rc == -3 and "D=32" in msg


@pytest.mark.gpu
def test_recognize_batch_like_the_drop_in_functions(tsd, rec_golden, rec_gray_golden, rec_frames, frames3):
    """source_rec.recognizeBatch for the four classifier strings on the three stored real frames = per frame
    MSERTrafficSignDetector -> windowsToGray -> calculateDescriptors -> predictProbability, with the stored MSER boxes."""
    R = tsd.source_rec
    names = sorted(frames3)
    frames = np.stack([frames3[k] for k in names])
    bl = [rec_frames[k + "_boxes"] for k in names]
    boxes = np.concatenate(bl)
    off = np.concatenate([[0], np.cumsum([len(b) for b in bl])]).astype(np.int32)
    files = [k + ".jpg" for k in names]

    def classifiers(g, kind):
        if kind == "LDABAYES":
            return [types.SimpleNamespace(coef_=g["lda_W"][:, c][None, :], intercept_=np.array([g["lda_b"][c]])) for c in range(6)], None
        knn = types.SimpleNamespace(_fit_X=g["knn_Ztrain"], classes_=np.arange(7), _y=g["knn_ytrain"].astype(np.int64), n_neighbors=4)
        return knn, (types.SimpleNamespace(xbar_=g["knn_xbar"], scalings_=g["knn_scalings"]),)

    for desc, g in (("HOG", rec_golden), ("GRAY", rec_gray_golden)):
        for kind in ("LDABAYES", "KNN"):
            clf, reducer = classifiers(g, kind)
            got, counts = R.recognizeBatch(frames, boxes, off, files, (clf, kind), reducer, (None, desc))
            exp = []
            for f, k in enumerate(names):
                mser = types.SimpleNamespace(detectRegions=lambda img, b=bl[f]: (None, b))
                dets = R.windowsToGray(R.MSERTrafficSignDetector(frames3[k], mser, files[f]))
                descs = R.calculateDescriptors({0: dets}, (None, desc))[0]
                pred, _ = R.predictProbability((clf, kind), reducer, descs, 0.5)
                exp += [(files[f],) + d[1] + (int(p),) for d, p in zip(dets, pred) if int(p) != 0]
                if desc == "HOG" and kind == "LDABAYES":
                    assert [int(p) for p in pred] == rec_frames[k + "_pred_lda"].tolist()
            assert got == exp, (desc, kind)
            assert int(counts[0]) == len(boxes) and int(counts[3]) == len(exp)
