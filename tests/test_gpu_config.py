"""Every window size and every tsd_config field against the oracle.

tsd_create takes a whole tsd_config, and the kernels dispatch on several of its values.  Per window size D = 2 .. 32
(npx = D * D, ws = 3 npx rounded up to 16 bytes, NW = ceil(npx / 32) mask words):

  K2    k2_crop_resize_v2<3, D> at D = 25 / 32, the generic kernel at every other D
  K5    k5_hist / launch_folds <640> for npx <= 640 (D <= 25), <1024> above
  K3    k3_masks_v3 (flag tables built in create_impl) for ws <= 2048 (D <= 26), the generic kernel (HsvBounds) above
  K4    k4_score_bits<20> / <32> at NW = 20 / 32 (D = 25, 29 .. 32), k4_score_kernel on the byte masks at every other D

  window sizes  per D: tsd_windows, tsd_hist, both tsd_dedup passes, tsd_color_masks, tsd_score_masks (with scores) and tsd_score;
                the chain on host pointers (score_tol_hundredths = -1: every survivor is a record), on device pointers, with
                TSD_KEEP_MASKS=1 and with TSD_GRAM=0.  Seeded random templates, one of them degenerate (at most 1 % of the
                pixels set) and one all set.
  HSV bounds    an empty band, a band of everything, hue bounds above 179, single values, identical red bands, a blue band
                overlapping a red one: tsd_color_masks over all 2^24 colours, and the chain at D = 25 / 32 on windows made of
                colours whose H, S or V is one below, on and one above each bound.
  aspect        (0.75, 1.25), (0.5, 2), (0, 1e300), (1, 1) and each bound moved one ulp either way, boxes whose w / h is exactly
                on the bounds, h = 0 and w = 0, enlarge 1.0 / 1.07 / 1.5 / 2.0: tsd_expand_boxes, tsd_windows, counts[1].
  dedup         hist_tol x coord_tol x merge_factor on 4K frames with corner pairs 200 .. 2000 px apart: the chain, and tsd_dedup
                with explicit tolerances (two of them exactly on a pair's similarity and on merge_factor * tol).  A tolerance
                whose lowest acting similarity is not above sqrt(f(65535)) must be refused (pairs beyond the 65 536-entry
                table take no action); so must such a tol in tsd_match_detections.
  thresholds    score_tol_hundredths -1, 0, 54, 55, 56, 99, 100 with windows scoring exactly on each; proba_tol 0.2 / 0.8 in
                RUN_RECOGNIZE against oracle.lda_predict.
  refusals      window 0, 1, 33; tsd_score_masks / tsd_score at another D; the chain before tsd_set_templates.

All comparisons are bit for bit (records, stage counts, windows, histograms, masks, scores).  test_config_inputs_are_in_their_regimes
checks on the CPU that every D is listed and every kernel branch is reached, that the HSV windows hold colours on both sides
of every bound, that the far-corner pairs act in the oracle exactly where tsd_create must refuse, and that each threshold case
has a winner exactly on it.
"""
import functools
import math
import types

import numpy as np
import pytest

from test_gpu_recognition import decision_margin, oracle_rec_frame, spread_lda

E_INVALID, E_STATE = -1, -3
DS = tuple(range(2, 33))


# ---- configuration ------------------------------------------------------------------------------------------------
def ns(flavour="det", **over):
    """A tsd_config as a namespace (the defaults of tsd_config_default, then `over`)."""
    from oracle import oracle as O
    d = dict(O.DEFAULTS, enlarge=1.15 if flavour == "rec" else 1.30, window=32 if flavour == "rec" else 25,
             score_tol_hundredths=55, proba_tol=0.5, knn_k=4)
    d.update(over)
    return types.SimpleNamespace(**d)


def to_ctypes(tsd, cfg):
    c = tsd.default_config()
    for k in ("enlarge", "aspect_lo", "aspect_hi", "hist_tol", "coord_tol", "merge_factor", "proba_tol"):
        setattr(c, k, float(getattr(cfg, k)))
    for k in ("window", "score_tol_hundredths", "knn_k"):
        setattr(c, k, int(getattr(cfg, k)))
    for b in range(2):
        for ch in range(3):
            c.red_lo[b][ch] = cfg.red_lo[b][ch]
            c.red_hi[b][ch] = cfg.red_hi[b][ch]
    for ch in range(3):
        c.blue_lo[ch] = cfg.blue_lo[ch]
        c.blue_hi[ch] = cfg.blue_hi[ch]
    return c


def branches(D):
    npx = D * D
    ws, nw = (3 * npx + 15) & ~15, (npx + 31) >> 5
    return dict(k2="v2" if D in (25, 32) else "generic", k5="640" if npx <= 640 else "1024",
                k3="v3" if ws <= 2048 else "generic", k4="bits%d" % nw if nw in (20, 32) else "bytes")


def sim_limit(oracle):
    return math.sqrt(oracle.eucl_similarity_d2(65535))


def refused(oracle, tol, mf=1.0):
    """Whether a corner tolerance must be refused: its lowest acting similarity is not above the default table's reach."""
    return sim_limit(oracle) >= tol * mf


def records(det):
    return [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]


def oracle_chain(oracle, frames, boxes, off, red6, blue6, cfg):
    rec, counts = [], np.zeros(4, np.int64)
    for f in range(len(frames)):
        o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6, percentage=cfg.enlarge, D=cfg.window,
                                tol_hundredths=cfg.score_tol_hundredths, cfg=cfg)
        rec += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
        counts += o["stage_counts"]
    return rec, counts.tolist()


def oracle_windows(oracle, frames, boxes, off, enlarge, D, cfg=None):
    """K1 + K2 restated: the non-empty aspect-passing crops -> (windows, coords, offsets)."""
    H, W = frames.shape[1:3]
    wins, co, wo = [], [], [0]
    for f in range(len(frames)):
        c, v = oracle.expand_boxes(boxes[off[f]:off[f + 1]], enlarge, cfg=cfg)
        for cc, ok in zip(c, v):
            if ok and min(cc[2], W) > min(cc[0], W) and min(cc[3], H) > min(cc[1], H):
                wins.append(oracle.crop_resize(frames[f], cc, D)); co.append(cc)
        wo.append(len(co))
    wins = np.stack(wins) if wins else np.zeros((0, D, D, 3), np.uint8)
    return wins, np.array(co, np.int32).reshape(-1, 4), np.array(wo, np.int32)


def oracle_dedup(oracle, wins, coords, off, by_coords, tol, mf=0.8823):
    ow, oc, oo = [], [], [0]
    for f in range(len(off) - 1):
        w, c = oracle.dedup(wins[off[f]:off[f + 1]], coords[off[f]:off[f + 1]], by_coords, tol, mf)
        ow.append(w); oc.append(c); oo.append(oo[-1] + len(c))
    D = wins.shape[1]
    return (np.concatenate(ow) if ow else np.zeros((0, D, D, 3), np.uint8)), np.concatenate(oc).reshape(-1, 4), np.array(oo, np.int32)


def oracle_scores(oracle, red, blue, red6, blue6, tol):
    n = len(red)
    sc = np.zeros((n, 2, 6), np.int32)
    ids, hs, em = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, bool)
    for i in range(n):
        for k in range(6):
            sc[i, 0, k] = oracle.score_hundredths(red[i], red6[k])[0]
            sc[i, 1, k] = oracle.score_hundredths(blue[i], blue6[k])[0]
        kr, kb = int(np.argmax(sc[i, 0])), int(np.argmax(sc[i, 1]))          # first maximum (DET:249-259)
        ids[i], hs[i] = (kr + 1, sc[i, 0, kr]) if sc[i, 0, kr] > sc[i, 1, kb] else (kb + 1, sc[i, 1, kb])
        em[i] = hs[i] > tol
    return sc, ids, hs, em


# ---- inputs ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def templates_for(D):
    """-> (red6, blue6) uint8 [6, D * D]: one degenerate template (at most 1 % set), one all set, four random densities."""
    rng = np.random.default_rng(1000 + D)
    npx = D * D
    out = []
    for colour in range(2):
        t = np.zeros((6, npx), np.uint8)
        t[0, rng.permutation(npx)[:npx // 100]] = 255
        t[1] = 255
        for k in range(2, 6):
            t[k] = np.where(rng.random(npx) < rng.uniform(0.1, 0.8), 255, 0)
        out.append(t[rng.permutation(6)] if colour else t)
    return out[0], out[1]


@functools.lru_cache(maxsize=None)
def sweep_inputs(D):
    """3 frames 240 x 320 of coloured rectangles, 60 boxes each (30 % jittered copies)."""
    import tsd_b200
    frames = tsd_b200.synth.make_frames(3, 240, 320, seed=500 + D, nrect=24)
    boxes, off = tsd_b200.synth.make_boxes(3, 60, 240, 320, seed=600 + D, D=D)
    return frames, boxes, off


# HSV bound cases: overrides of the red / blue bounds.  Bands are [red band 0, red band 1, blue] x (H, S, V).
HSV_CASES = {
    "empty_band": dict(red_lo=((0, 50, 10), (170, 50, 10)), red_hi=((10, 255, 255), (160, 255, 255)),
                       blue_lo=(90, 200, 10), blue_hi=(128, 100, 255)),
    "everything": dict(blue_lo=(0, 0, 0), blue_hi=(255, 255, 255)),
    "hue_above_179": dict(red_lo=((0, 50, 10), (175, 50, 10)), red_hi=((10, 255, 255), (250, 255, 255)),
                          blue_lo=(180, 0, 0), blue_hi=(255, 255, 255)),
    "single_values": dict(red_lo=((5, 200, 200), (170, 128, 77)), red_hi=((5, 200, 200), (170, 128, 77)),
                          blue_lo=(100, 150, 220), blue_hi=(100, 150, 220)),
    "identical_red": dict(red_lo=((0, 50, 10), (0, 50, 10)), red_hi=((10, 255, 255), (10, 255, 255))),
    "blue_overlaps_red": dict(blue_lo=(5, 30, 10), blue_hi=(100, 255, 255)),
}
CH_MAX = (179, 255, 255)                              # largest H, S, V 8-bit HSV reaches


def bands(cfg):
    return [(cfg.red_lo[0], cfg.red_hi[0]), (cfg.red_lo[1], cfg.red_hi[1]), (cfg.blue_lo, cfg.blue_hi)]


@functools.lru_cache(maxsize=None)
def all_colours():
    b, g, r = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    return np.stack([b, g, r], -1).reshape(-1, 3)


@functools.lru_cache(maxsize=None)
def all_hsv():
    from oracle import oracle as O
    return O.bgr2hsv(all_colours()).astype(np.int16)


@functools.lru_cache(maxsize=None)
def boundary_palette(case):
    """BGR colours whose H, S or V is bound - 1, bound or bound + 1 of some band, the other two channels inside that band where
    the band allows (so the bound decides).  -> uint8 [m, 3]."""
    cfg = ns(**HSV_CASES[case])
    hsv = all_hsv()
    rng = np.random.default_rng(sum(map(ord, case)))
    pick = []
    for lo, hi in bands(cfg):
        for ch in range(3):
            others = np.ones(len(hsv), bool)
            for o in range(3):
                if o != ch and lo[o] <= hi[o]:
                    others &= (hsv[:, o] >= lo[o]) & (hsv[:, o] <= hi[o])
            for bound in (lo[ch], hi[ch]):
                for t in (bound - 1, bound, bound + 1):
                    if 0 <= t <= CH_MAX[ch]:
                        idx = np.flatnonzero(others & (hsv[:, ch] == t))
                        if len(idx) == 0:
                            idx = np.flatnonzero(hsv[:, ch] == t)
                        pick += list(rng.choice(idx, min(3, len(idx)), replace=False))
    return all_colours()[np.unique(pick)]


@functools.lru_cache(maxsize=None)
def palette_frames(case, D):
    """2 frames of a grid of D x D windows, each filled with a random handful of palette colours; boxes exactly on the windows
    (enlarge 1.0: the chain's windows are exact copies)."""
    pal = boundary_palette(case)
    rng = np.random.default_rng([D, len(pal)])
    G = 7
    frames = np.full((2, G * D + 3, G * D + 5, 3), 128, np.uint8)
    boxes = []
    for f in range(2):
        for gy in range(G):
            for gx in range(G):
                cols = pal[rng.choice(len(pal), 6)]
                frames[f, gy * D:(gy + 1) * D, gx * D:(gx + 1) * D] = cols[rng.integers(0, 6, (D, D))]
                boxes.append((gx * D, gy * D, D, D))
    off = np.array([0, G * G, 2 * G * G], np.int32)
    return frames, np.array(boxes, np.int32), off


# aspect bounds, each also with one bound moved one ulp down / up
ASPECTS = ((0.75, 1.25), (0.5, 2.0), (0.0, 1e300), (1.0, 1.0))
ENLARGES = (1.0, 1.07, 1.5, 2.0)


def aspect_variants():
    out = []
    for lo, hi in ASPECTS:
        out += [(lo, hi), (np.nextafter(lo, -np.inf), hi), (np.nextafter(lo, np.inf), hi), (lo, np.nextafter(hi, -np.inf)),
                (lo, np.nextafter(hi, np.inf))]
    return [(float(a), float(b)) for a, b in out]


@functools.lru_cache(maxsize=None)
def aspect_inputs():
    """One 400 x 400 frame, boxes with w / h exactly 0.75, 1.25, 0.5, 2, 1, in between, outside, h = 0 and w = 0."""
    import tsd_b200
    frame = tsd_b200.synth.make_frames(1, 400, 400, seed=77, nrect=12)
    wh = [(3, 4), (30, 40), (75, 100), (5, 4), (50, 40), (1, 2), (20, 40), (2, 1), (80, 40), (33, 33), (1, 1), (41, 40),
          (39, 40), (29, 40), (51, 40), (19, 40), (81, 40), (7, 0), (0, 7), (0, 0), (100, 1), (1, 100)]
    rng = np.random.default_rng(3)
    boxes = [(int(rng.integers(0, 250)), int(rng.integers(0, 250)), w, h) for w, h in wh for _ in range(2)]
    return frame, np.array(boxes, np.int32), np.array([0, len(boxes)], np.int32)


# dedup tolerances on 4K frames
HIST_TOLS = (0.3, 0.6, 0.99)
COORD_TOLS = (0.3, 0.45, 0.6, 0.99)
MERGE_FACTORS = (0.5, 0.8823, 1.0)


@functools.lru_cache(maxsize=None)
def dedup_inputs():
    """2 frames 2160 x 3840: random boxes, jittered copies, and far-corner pairs -- a red square A = (x, y, s, s) and a box
    B = (x, y, s + d, s + d) over blue with the same top-left corner, d = 145 .. 1414 (bottom-right corners 205 .. 2000 px
    apart).  enlarge 1.0 keeps the corners as given."""
    import tsd_b200
    H, W = 2160, 3840
    frames = tsd_b200.synth.make_frames(2, H, W, seed=91, nrect=40)
    rng = np.random.default_rng(92)
    boxes, off, far = [], [0], []
    for f in range(2):
        bx = []
        for i, d in enumerate((145, 160, 182, 200, 230, 260, 300, 350, 420, 520, 700, 1000, 1414)):
            s = 30 + 4 * i
            x, y = 40 + 280 * i if f == 0 else 3700 - 280 * i - d - s, 60 + 60 * i
            x = max(0, x)
            frames[f, y:y + s + d, x:x + s + d] = (200, 60, 20)                 # blue (BGR)
            frames[f, y:y + s, x:x + s] = (20, 20, 220)                         # red
            bx += [(x, y, s, s), (x, y, s + d, s + d)]
            far.append((f, (x, y, x + s, y + s), (x, y, x + s + d, y + s + d)))
        for _ in range(60):
            s = int(rng.integers(12, 120)); x = int(rng.integers(0, W - s)); y = int(rng.integers(0, H - s))
            bx.append((x, y, s, s + int(rng.integers(-2, 3))))
            for _ in range(int(rng.integers(0, 3))):
                j = rng.integers(-4, 5, 4)
                bx.append((x + int(j[0]), max(0, y + int(j[1])), s + int(j[2]), s + int(j[3])))
        order = rng.permutation(len(bx))
        boxes += [bx[k] for k in order]
        off.append(len(boxes))
    return frames, np.array(boxes, np.int32), np.array(off, np.int32), far


def exact_tols(oracle):
    """-> (t_hi, t_lo): a near pair of dedup_inputs whose similarity s satisfies s == t_hi and t_lo * 0.8823 == s exactly."""
    frames, boxes, off, _ = dedup_inputs()
    wins, co, wo = oracle_windows(oracle, frames, boxes, off, 1.0, 25)
    for f in range(2):
        c = co[wo[f]:wo[f + 1]]
        for i in range(len(c)):
            for j in range(i):
                s = oracle.coord_similarity(c[i], c[j])
                if not 0.6 < s < 0.8:
                    continue
                t = s / 0.8823
                for _ in range(40):
                    if t * 0.8823 == s:
                        return s, t
                    t = float(np.nextafter(t, np.inf if t * 0.8823 < s else -np.inf))
    return None


# score thresholds: red template k = pixels [start_k, start_k + T_k), blue templates empty; a window's mask = the first tp
# pixels of one template, the rest grey.  2 tp / (tp + T) = 0.54, 0.55, 0.56, 0.99, 1.00, 0.53 and an empty mask (0).
THRESH_T = (73, 29, 36, 101, 20, 50)
THRESH_WINDOWS = ((0, 27), (1, 11), (2, 14), (3, 99), (4, 20), (5, 18), (0, 0))
THRESH_TOLS = (-1, 0, 54, 55, 56, 99, 100)


def thresh_templates():
    red6 = np.zeros((6, 625), np.uint8)
    starts = np.concatenate([[0], np.cumsum(THRESH_T)[:-1]])
    for k, (s, t) in enumerate(zip(starts, THRESH_T)):
        red6[k, s:s + t] = 255
    return red6, np.zeros((6, 625), np.uint8), starts


def thresh_inputs():
    """One 25 x 25 window per 40 x 40 frame (no duplicate removal between them), box exactly on it."""
    _, _, starts = thresh_templates()
    frames = np.full((len(THRESH_WINDOWS), 40, 40, 3), 128, np.uint8)
    for f, (k, tp) in enumerate(THRESH_WINDOWS):
        win = np.full((625, 3), 128, np.uint8)
        win[starts[k]:starts[k] + tp] = (0, 0, 255)
        frames[f, 5:30, 7:32] = win.reshape(25, 25, 3)
    boxes = np.array([(7, 5, 25, 25)] * len(THRESH_WINDOWS), np.int32)
    return frames, boxes, np.arange(len(THRESH_WINDOWS) + 1, dtype=np.int32)


PROBA_TOLS = (0.2, 0.8)
REC_SEED = 32


@functools.lru_cache(maxsize=None)
def rec_inputs(oracle):
    """-> frames, boxes, offsets, W, b, [(survivor coords, hog)] per frame (x1.15, 32 x 32, default dedup tolerances)."""
    import tsd_b200
    frames = tsd_b200.synth.make_frames(4, 300, 400, seed=REC_SEED)
    boxes, off = tsd_b200.synth.make_boxes(4, 50, 300, 400, seed=REC_SEED + 1, enlarge=1.15, D=32)
    surv = [oracle_rec_frame(oracle, frames[f], boxes[off[f]:off[f + 1]]) for f in range(4)]
    W, b = spread_lda(np.concatenate([h for _, h in surv]), REC_SEED)
    return frames, boxes, off, W, b, surv


def rec_margin(z, hog, W, tol):
    """decision_margin plus the distance of every logit from +-logit(tol) (where a label changes when tol > 0.5)."""
    guard = ((1e-5 * np.abs(hog.astype(np.float64)) + 1e-7) @ np.abs(W)).max(1)
    m = decision_margin(z, hog, W)
    if tol > 0.5:
        lt = math.log(tol / (1 - tol))
        m = np.minimum(m, np.minimum(np.abs(z - lt), np.abs(z + lt)).min(1) / (2 * guard))
    return m


# ---- CPU: every case is in its regime -------------------------------------------------------------------------------
def test_config_inputs_are_in_their_regimes(oracle):
    # every window size, every branch
    assert DS == tuple(range(2, 33))
    seen = {k: {branches(D)[k] for D in DS} for k in ("k2", "k5", "k3", "k4")}
    assert seen == dict(k2={"v2", "generic"}, k5={"640", "1024"}, k3={"v3", "generic"}, k4={"bits20", "bits32", "bytes"}), seen
    assert branches(25) == dict(k2="v2", k5="640", k3="v3", k4="bits20") and branches(26)["k3"] == "v3"
    assert branches(27)["k3"] == "generic" and branches(26)["k5"] == "1024" and branches(32)["k4"] == "bits32"
    assert [D for D in DS if branches(D)["k3"] == "v3" and branches(D)["k4"] == "bytes"] == [D for D in DS if D <= 26 and D != 25]
    for D in DS:
        red6, blue6 = templates_for(D)
        npx = D * D
        for t in (red6, blue6):
            counts = sorted(int(v) for v in (t == 255).sum(1))
            assert counts[0] <= npx // 100 and counts[-1] == npx
        frames, boxes, off = sweep_inputs(D)
        wins, _, wo = oracle_windows(oracle, frames, boxes, off, 1.30, D)
        assert len(wins) >= 60, D
        red, blue = oracle.color_masks(wins)
        assert red.any() and blue.any(), D
    # HSV: colours on both sides of every reachable bound, in the windows of both frames sets
    for case in HSV_CASES:
        cfg = ns(**HSV_CASES[case])
        for D in (25, 32):
            frames, boxes, off = palette_frames(case, D)
            wins, _, _ = oracle_windows(oracle, frames, boxes, off, 1.0, D)
            assert len(wins) == len(boxes)
            hsv = oracle.bgr2hsv(wins).reshape(-1, 3).astype(int)
            for lo, hi in bands(cfg):
                for ch in range(3):
                    v = set(hsv[:, ch].tolist())
                    if lo[ch] > 0 and lo[ch] <= CH_MAX[ch]:
                        assert lo[ch] - 1 in v and lo[ch] in v, (case, D, lo, ch)
                    if hi[ch] < CH_MAX[ch]:
                        assert hi[ch] in v and hi[ch] + 1 in v, (case, D, hi, ch)
            r, b = oracle.color_masks(wins, cfg=cfg)
            if case != "empty_band":
                assert r.any() and (~r.astype(bool)).any()
    # aspect: boxes exactly on each bound, inside and outside, h = 0
    _, boxes, _ = aspect_inputs()
    ratios = {b[2] / b[3] for b in boxes.tolist() if b[3]}
    assert {0.75, 1.25, 0.5, 2.0, 1.0} <= ratios and any(b[3] == 0 for b in boxes.tolist())
    variants = aspect_variants()
    for k, (lo, hi) in enumerate(ASPECTS):                # moving a bound one ulp outwards admits the boxes exactly on it
        v = [oracle.expand_boxes(boxes, 1.3, aspect_lo=a, aspect_hi=b)[1] for a, b in variants[5 * k:5 * k + 5]]
        assert v[0].any() == (lo < hi)
        if lo < hi:
            assert (v[1] & ~v[0]).any() and np.array_equal(v[2], v[0]) and np.array_equal(v[3], v[0])
            assert (v[4] & ~v[0]).any() or hi == 1e300
    # far corners: d2 >= 65 536 and an oracle similarity above tol * merge_factor for every refused combination
    *_, far = dedup_inputs()
    lim = sim_limit(oracle)
    assert 0.39 < lim < 0.392
    sims = []                                             # of the pairs beyond the table (d2 >= 65 536)
    for _, a, b in far:
        d2 = (a[2] - b[2]) ** 2 + (a[3] - b[3]) ** 2
        assert a[:2] == b[:2] and 200 <= math.sqrt(d2) <= 2001
        if d2 >= 65536:
            sims.append(oracle.coord_similarity(a, b))
    assert len(sims) >= 10
    for tol in COORD_TOLS + (0.85,):
        for mf in MERGE_FACTORS:
            if refused(oracle, tol, mf):
                assert max(sims) > tol * mf, (tol, mf)
            else:
                assert max(sims) < tol * mf                               # accepted: these pairs take no action
    assert refused(oracle, 0.3) and not refused(oracle, 0.45) and not refused(oracle, 0.45, 0.8823)
    assert exact_tols(oracle) is not None
    # thresholds: a winner exactly on every tol in 0 .. 100
    red6, blue6, _ = thresh_templates()
    frames, boxes, off = thresh_inputs()
    winners = [oracle.score_window(frames[f, 5:30, 7:32], red6, blue6, 55)[2] for f in range(len(frames))]
    assert set(winners) >= {t for t in THRESH_TOLS if t >= 0}, winners
    # recognition: every label, no label within the HOG tolerance of a change at either proba_tol
    frames, boxes, off, W, b, surv = rec_inputs(oracle)
    hog = np.concatenate([h for _, h in surv])
    for tol in PROBA_TOLS:
        z, lab = oracle.lda_predict(hog, W, b, tol)
        assert rec_margin(z, hog, W, tol).min() > 1, tol
        assert len(set(lab.tolist())) >= 4, tol
    assert not np.array_equal(oracle.lda_predict(hog, W, b, 0.2)[1], oracle.lda_predict(hog, W, b, 0.8)[1])


# ---- GPU --------------------------------------------------------------------------------------------------------------
ENV_KEYS = ("TSD_KEEP_MASKS", "TSD_GRAM")


@pytest.fixture
def make_ctx(tsd, monkeypatch):
    """Contexts of a config under an environment (read at tsd_create), with the library's libm similarity table (the oracle's
    values); all closed at the end of the test."""
    made = []

    def mk(cfg, env=None):
        for k in ENV_KEYS:
            monkeypatch.delenv(k, raising=False)
        for k, v in (env or {}).items():
            monkeypatch.setenv(k, v)
        c = tsd.Context(0, config=to_ctypes(tsd, cfg), numpy_similarity=False)
        made.append(c)
        return c
    yield mk
    for c in made:
        c.close()


def run_device(ctx, frames, boxes, off):
    import torch
    dev = torch.device("cuda", 0)
    F, H, W = frames.shape[:3]
    tf, tb, to = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (frames, boxes, off))
    ctx.enqueue_frames(tf.data_ptr(), F, H, W, tb.data_ptr(), to.data_ptr(), len(boxes))
    det, counts = ctx.fetch_detections(max(len(boxes), 1))
    return records(det), counts.tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("D", DS)
def test_window_size_stages(oracle, make_ctx, D):
    """tsd_windows, tsd_hist, both tsd_dedup passes, tsd_color_masks, tsd_score_masks and tsd_score at window size D."""
    red6, blue6 = templates_for(D)
    frames, boxes, off = sweep_inputs(D)
    ctx = make_ctx(ns(window=D))
    ctx.set_templates(red6, blue6)
    wins, co, wo = ctx.windows(frames, boxes, off)
    ew, ec, eo = oracle_windows(oracle, frames, boxes, off, 1.30, D)
    assert np.array_equal(wo, eo) and np.array_equal(co, ec) and np.array_equal(wins, ew)
    assert np.array_equal(ctx.hist(ew), np.stack([oracle.hist_normalized(w) for w in ew]))
    w1, c1, o1 = ctx.dedup(ew, ec, eo, False, 0.85)
    x1, y1, z1 = oracle_dedup(oracle, ew, ec, eo, False, 0.85)
    assert np.array_equal(o1, z1) and np.array_equal(c1, y1) and np.array_equal(w1, x1)
    w2, c2, o2 = ctx.dedup(x1, y1, z1, True, 0.95)
    x2, y2, z2 = oracle_dedup(oracle, x1, y1, z1, True, 0.95)
    assert np.array_equal(o2, z2) and np.array_equal(c2, y2) and np.array_equal(w2, x2)
    red, blue = ctx.color_masks(ew)
    ored, oblue = oracle.color_masks(ew)
    assert np.array_equal(red, ored) and np.array_equal(blue, oblue)
    r = ctx.score_masks(ored, oblue)
    sc, ids, hs, em = oracle_scores(oracle, ored.reshape(len(ew), -1), oblue.reshape(len(ew), -1), red6, blue6, 55)
    assert np.array_equal(r["scores"], sc) and np.array_equal(r["id"], ids) and np.array_equal(r["hundredths"], hs)
    assert np.array_equal(r["emit"], em)
    s = ctx.score_windows(ew)
    exp = [oracle.score_window(w, red6.reshape(6, D, D), blue6.reshape(6, D, D), 55) for w in ew]
    assert [(bool(e), int(i), int(h)) for e, i, h in zip(s["emit"], s["id"], s["hundredths"])] == exp


@pytest.mark.gpu
@pytest.mark.parametrize("D", DS)
def test_window_size_chain(oracle, make_ctx, D):
    """The detection chain at window size D: host pointers (every survivor reported), device pointers, TSD_KEEP_MASKS=1 and
    TSD_GRAM=0.  The stage-by-stage expectation is the oracle's whole-frame restatement."""
    red6, blue6 = templates_for(D)
    frames, boxes, off = sweep_inputs(D)
    all_cfg, tol_cfg = ns(window=D, score_tol_hundredths=-1), ns(window=D)
    exp_all = oracle_chain(oracle, frames, boxes, off, red6, blue6, all_cfg)
    exp_tol = oracle_chain(oracle, frames, boxes, off, red6, blue6, tol_cfg)
    assert exp_all[1][2] == exp_all[1][3] > 0 and exp_tol[1][3] < exp_all[1][3]
    runs = [("host", all_cfg, {}, exp_all), ("device", tol_cfg, {}, exp_tol), ("keep_masks", all_cfg, {"TSD_KEEP_MASKS": "1"}, exp_all),
            ("gram0", all_cfg, {"TSD_GRAM": "0"}, exp_all)]
    bad = []
    for name, cfg, env, (rec, counts) in runs:
        ctx = make_ctx(cfg, env)
        ctx.set_templates(red6, blue6)
        if name == "device":
            got = run_device(ctx, frames, boxes, off)
        else:
            det, c = ctx.detect_frames(frames, boxes, off)
            got = records(det), c.tolist()
        if got != (rec, counts):
            bad.append((name, got[1], counts, sum(a != b for a, b in zip(got[0], rec))))
    assert not bad, bad


@pytest.mark.gpu
def test_window_refusals(tsd, make_ctx):
    for D in (0, 1, 33):
        with pytest.raises(tsd.TsdError):
            make_ctx(ns(window=D))
    A = tsd._capi
    frames, boxes, off = sweep_inputs(25)
    F, H, W = frames.shape[:3]
    for D in DS:
        ctx = make_ctx(ns(window=D))
        det = np.empty(len(boxes), tsd.DET_DTYPE)
        nd = np.zeros(1, np.int32)
        assert ctx._L.tsd_detect_frames(ctx._h, A.RUN_DETECT, A.ptr(frames), F, H, W, W * 3, H * W * 3, A.ptr(boxes), A.ptr(off),
                                        A.ptr(det), len(det), A.ptr(nd), None, A.MEM_HOST) == E_STATE
        ctx.set_templates(*templates_for(D))
        for Dx in (D - 1, D + 1):
            m = np.zeros((2, Dx * Dx if Dx > 0 else 1), np.uint8)
            out = np.zeros((2, 12), np.int32)
            em = np.zeros(2, np.uint8)
            assert ctx._L.tsd_score_masks(ctx._h, A.ptr(m), A.ptr(m), 2, Dx, A.ptr(out), A.ptr(out), A.ptr(out), A.ptr(em), A.MEM_HOST) == E_INVALID
            w = np.zeros((2, max(Dx, 1) ** 2 * 3), np.uint8)
            assert ctx._L.tsd_score(ctx._h, A.ptr(w), 2, Dx, A.ptr(out), A.ptr(out), A.ptr(em), A.MEM_HOST) == E_INVALID


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(HSV_CASES))
def test_hsv_bounds(oracle, make_ctx, case):
    """tsd_color_masks over all 2^24 colours (25 x 25 windows, a zero-padded tail), then the chain at D = 25 (v3 flag tables)
    and D = 32 (generic kernel) on windows of colours on both sides of every bound."""
    cfg = ns(**HSV_CASES[case])
    ctx = make_ctx(cfg)
    flat = all_colours()
    n = (len(flat) // 625) * 625
    tail = np.zeros((625, 3), np.uint8); tail[:len(flat) - n] = flat[n:]
    wins = np.concatenate([flat[:n], tail]).reshape(-1, 25, 25, 3)
    red, blue = ctx.color_masks(wins)
    ored, oblue = oracle.color_masks(wins, cfg=cfg)
    assert np.array_equal(red, ored) and np.array_equal(blue, oblue)
    for D in (25, 32):
        c = ns(window=D, enlarge=1.0, score_tol_hundredths=-1, **HSV_CASES[case])
        frames, boxes, off = palette_frames(case, D)
        red6, blue6 = templates_for(D)
        exp = oracle_chain(oracle, frames, boxes, off, red6, blue6, c)
        for env in ({}, {"TSD_KEEP_MASKS": "1"}):
            x = make_ctx(c, env)
            x.set_templates(red6, blue6)
            det, counts = x.detect_frames(frames, boxes, off)
            assert (records(det), counts.tolist()) == exp, (D, env)


@pytest.mark.gpu
def test_aspect_and_enlarge(oracle, make_ctx):
    """tsd_expand_boxes (the context's aspect bounds), tsd_windows and counts[1] of the chain."""
    frame, boxes, off = aspect_inputs()
    red6, blue6 = templates_for(25)
    for lo, hi in aspect_variants():
        for en in ENLARGES:
            cfg = ns(aspect_lo=lo, aspect_hi=hi, enlarge=en)
            ctx = make_ctx(cfg)
            ctx.set_templates(red6, blue6)
            co, v = ctx.expand_boxes(boxes, en)
            oc, ov = oracle.expand_boxes(boxes, en, cfg=cfg)
            assert np.array_equal(v, ov) and np.array_equal(co[v], oc[ov]), (lo, hi, en)
            wins, wc, wo = ctx.windows(frame, boxes, off)
            ew, ec, eo = oracle_windows(oracle, frame, boxes, off, en, 25, cfg=cfg)
            assert np.array_equal(wo, eo) and np.array_equal(wc, ec) and np.array_equal(wins, ew), (lo, hi, en)
            _, counts = ctx.detect_frames(frame, boxes, off)
            assert counts.tolist() == oracle_chain(oracle, frame, boxes, off, red6, blue6, cfg)[1], (lo, hi, en)


@pytest.mark.gpu
def test_dedup_tolerances(oracle, make_ctx, tsd):
    """The chain under every (hist_tol, coord_tol, merge_factor); tsd_create refuses a coord_tol * merge_factor the corner table
    cannot honour.  Then tsd_dedup with explicit tolerances under the default config, two of them exactly on a pair's similarity."""
    frames, boxes, off, _ = dedup_inputs()
    red6, blue6 = templates_for(25)
    for ht in HIST_TOLS:
        for ct in COORD_TOLS:
            for mf in MERGE_FACTORS:
                cfg = ns(hist_tol=ht, coord_tol=ct, merge_factor=mf, enlarge=1.0, score_tol_hundredths=-1)
                if refused(oracle, ct, mf):
                    with pytest.raises(tsd.TsdError):
                        make_ctx(cfg)
                    continue
                ctx = make_ctx(cfg)
                ctx.set_templates(red6, blue6)
                det, counts = ctx.detect_frames(frames, boxes, off)
                assert (records(det), counts.tolist()) == oracle_chain(oracle, frames, boxes, off, red6, blue6, cfg), (ht, ct, mf)
    ctx = make_ctx(ns())
    wins, co, wo = oracle_windows(oracle, frames, boxes, off, 1.0, 25)
    t_hi, t_lo = exact_tols(oracle)
    for tol in COORD_TOLS + (t_hi, t_lo):
        if refused(oracle, tol, 0.8823):
            with pytest.raises(tsd.TsdError):
                ctx.dedup(wins, co, wo, True, tol)
            continue
        got = ctx.dedup(wins, co, wo, True, tol)
        exp = oracle_dedup(oracle, wins, co, wo, True, tol)
        assert all(np.array_equal(a, b) for a, b in zip(got, exp)), tol
    for tol in HIST_TOLS:
        got = ctx.dedup(wins, co, wo, False, tol)
        exp = oracle_dedup(oracle, wins, co, wo, False, tol)
        assert all(np.array_equal(a, b) for a, b in zip(got, exp)), tol


@pytest.mark.gpu
def test_match_detections_tolerances(tsd):
    """tsd_match_detections against oracle/evaluate.py at tol 0.3 (refused: a ground truth beyond the table could match),
    0.45 and 0.85, with detections near ground truths and with one corner on a ground truth's and the other 200 .. 2000 px away."""
    from oracle import evaluate as O
    rng = np.random.default_rng(41)
    gts, dets = [], []
    for f in range(6):
        for _ in range(5):
            x, y, s, t = int(rng.integers(0, 3000)), int(rng.integers(0, 1500)), int(rng.integers(16, 90)), int(rng.integers(0, 6))
            gts.append((f, x, y, x + s, y + s, t))
            for _ in range(int(rng.integers(1, 4))):
                j = rng.integers(-15, 16, 4)
                dets.append((f, x + int(j[0]), y + int(j[1]), x + s + int(j[2]), y + s + int(j[3]), t))
            d = int(rng.integers(145, 1414))
            dets.append((f, x, y, x + s + d, y + s + d, t))
    off = np.zeros(7, np.int32)
    for g in gts:
        off[g[0] + 1] += 1
    off = np.cumsum(off).astype(np.int32)
    ctx = tsd.evaluate.context()
    for tol in (0.3, 0.45, 0.85):
        if tol < 0.3914:
            with pytest.raises(tsd.TsdError):
                ctx.match_detections(np.array(dets, np.int32), np.array(gts, np.int32), off, tol=tol)
            assert max(O.det_statistics(dets, gts, 6, tol)[0]) == 1
            continue
        st, mt, tally = ctx.match_detections(np.array(dets, np.int32), np.array(gts, np.int32), off, tol=tol)
        ost, omt, otally = O.det_statistics(dets, gts, 6, tol)
        assert st.tolist() == ost and mt.tolist() == omt and np.array_equal(tally, otally), tol


@pytest.mark.gpu
@pytest.mark.parametrize("tol", THRESH_TOLS)
def test_score_thresholds(oracle, make_ctx, tol):
    """Windows whose winner is exactly 0, 53, 54, 55, 56, 99 and 100 hundredths under score_tol_hundredths = tol: the chain
    and tsd_score_masks."""
    red6, blue6, _ = thresh_templates()
    frames, boxes, off = thresh_inputs()
    cfg = ns(enlarge=1.0, score_tol_hundredths=tol)
    ctx = make_ctx(cfg)
    ctx.set_templates(red6, blue6)
    det, counts = ctx.detect_frames(frames, boxes, off)
    assert (records(det), counts.tolist()) == oracle_chain(oracle, frames, boxes, off, red6, blue6, cfg)
    wins = frames[:, 5:30, 7:32]
    ored, oblue = oracle.color_masks(wins)
    r = ctx.score_masks(ored, oblue)
    sc, ids, hs, em = oracle_scores(oracle, ored.reshape(len(wins), -1), oblue.reshape(len(wins), -1), red6, blue6, tol)
    assert np.array_equal(r["scores"], sc) and np.array_equal(r["hundredths"], hs) and np.array_equal(r["emit"], em)
    assert np.array_equal(r["id"], ids)


@pytest.mark.gpu
@pytest.mark.parametrize("tol", PROBA_TOLS)
def test_proba_tol_chain(oracle, make_ctx, tsd, tol):
    """RUN_RECOGNIZE with proba_tol != 0.5: records equal oracle.lda_predict's labels at that tol."""
    frames, boxes, off, W, b, surv = rec_inputs(oracle)
    rec, nsurv = [], 0
    for f, (c2, hog) in enumerate(surv):
        lab = oracle.lda_predict(hog, W, b, tol)[1] if len(hog) else []
        rec += [(f,) + tuple(int(x) for x in q) + (int(l), 0) for q, l in zip(c2, lab) if l != 0]
        nsurv += len(c2)
    cfg = ns("rec", proba_tol=tol)
    ctx = make_ctx(cfg)
    ctx.set_lda(W, b)
    det, counts = ctx.detect_frames(frames, boxes, off, mode=tsd.RUN_RECOGNIZE)
    _, _, wo = oracle_windows(oracle, frames, boxes, off, 1.15, 32)
    assert records(det) == rec and counts.tolist() == [len(boxes), int(wo[-1]), nsurv, len(rec)]
