"""K5 (cleanDuplicatedDetections) route by route against the oracle, at the size limits where the producers and folds hand over.

Which kernels handle a frame depends on its window count, on its "big rows" (windows with a histogram bin holding more than 255
pixels: the tensor-core tiles keep count & 255 and those pairs are corrected exactly from the sparse lists), on the window size and
on the TSD_GRAM / TSD_FOLD_CTA_COST switches:

  producers  k5_pairs (<= 24 windows; frames k5_gram leaves; block pairs k5_gram_big hands over; everything with TSD_GRAM=0)
             k5_gram (25 .. 128 windows, <= 16 big rows), k5_gram_big (129 .. 1024 windows, 128-row block pairs, <= 32 big rows each)
  folds      k5_fold_warp (<= 256 windows), k5_fold_cta (257 .. 1024; smaller frames by merge cost with TSD_FOLD_CTA_COST),
             k5_fold (more than 1024 windows)

The input generator is seeded numpy plus the oracle's BGR -> HSV (no GPU); test_route_inputs_are_in_their_regimes checks on the
CPU that every case really is in the regime it names, so none of the GPU cases can pass vacuously.  Every GPU case compares
Context.dedup with oracle.dedup frame by frame: survivor offsets, coordinates and pixels bit for bit.
"""
import numpy as np
import pytest

# ---- the frame lists (trim here) -------------------------------------------------------------------------------------
# (a) size limits, no big rows: k5_pairs (tiny) -> k5_gram (1 / 3 / 6 / 10 blocks, second scatter rows) -> k5_gram_big (ragged
#     last block) -> warp fold -> CTA fold -> general fold
A_SIZES = (2, 24, 25, 32, 33, 96, 97, 127, 128, 129, 255, 256, 257, 384, 385, 1023, 1024, 1025)
# (b) big rows in k5_gram_big that stay on the tensor cores (<= 32 per block pair): (windows, {block: big rows in it})
B_FRAMES = (
    (129, {1: 1}),                   # the one row of the ragged block 1: (1,0) block I only, (1,1) diagonal
    (200, {0: 5}),                   # (0,0) diagonal, (1,0) block J only
    (300, {0: 16, 1: 16}),           # (1,0) both blocks, exactly 32; (2,0), (2,1) block J only
    (384, {1: 32}),                  # (1,1) exactly 32 on the diagonal; (1,0) I only, (2,1) J only
    (700, {2: 12, 3: 20, 5: 10}),    # (3,2) = 32, (5,3) = 30, (5,2) = 22 with the ragged block 5 (60 rows)
)
# (c) block pairs with more than 32 big rows, handed to k5_pairs (todo items with I != 15)
C_FRAMES = (
    (300, {2: 33}),                  # ragged last block (44 rows) with 33: (2,2) diagonal, (2,0), (2,1) off-diagonal
    (400, {0: 20, 1: 13}),           # (1,0) = 20 + 13 off-diagonal; (0,0), (1,1) and the pairs with blocks 2, 3 stay
    (320, {0: 12, 1: 20}),           # (1,0) = exactly 32: stays
    (520, {1: 33}),                  # full block with 33: (1,1), (1,0), (2,1), (3,1) and (4,1) with the ragged block 4 (8 rows)
)
CASES = {"a": tuple((n, {}) for n in A_SIZES), "b": B_FRAMES, "c": C_FRAMES}
HIST_TOLS = (0.85, 0.6, 0.4)         # histogram pass (long merge chains, merges of merged items at the lower ones)
CORNER_TOLS = (0.95, 0.6)            # corner pass
COST_FRAMES = (256, 33, 120)         # (f) frames, windows per frame between: small frames sent to k5_fold_cta by merge cost
SEEDS = {"a": 101, "b": 102, "c": 103, "cost": 104}
ROUTE_CLASSES = ((2, 24), (25, 128), (129, 256), (257, 1024), (1025, 1 << 30))     # producer / fold size classes of case a
BLOCK = 128                          # rows per block of k5_gram_big
BIG_MAX = 32                         # big rows per block pair k5_gram_big keeps on the tensor cores


# ---- input generator --------------------------------------------------------------------------------------------------
def bin_counts(oracle, wins):
    """Per-window calcHist([H, S], [50, 60]) COUNTS int64[m, 3000]: the oracle's BGR -> HSV, hue bin floor(H * 50 / 180) and
    saturation bin floor(S * 60 / 256) (the rule of hue_bin / hs_bin in the kernels)."""
    wins = np.ascontiguousarray(wins, np.uint8)
    m = len(wins)
    hsv = oracle.bgr2hsv(wins).reshape(m, -1, 3).astype(np.int64)
    b = (hsv[..., 0] * 5 // 18) * 60 + ((hsv[..., 1] * 60) >> 8)
    return np.bincount((b + 3000 * np.arange(m)[:, None]).ravel(), minlength=3000 * m).reshape(m, 3000)


def _fill(rng, D):
    """Background of a window: 8 x 8 colour blocks with +-3 jitter (tens of bins) or per-pixel noise (hundreds of bins)."""
    if rng.random() < 0.5:
        idx = np.arange(D) * 8 // D
        w = rng.integers(0, 256, (8, 8, 3))[idx][:, idx] + rng.integers(-3, 4, (D, D, 3))
    else:
        w = rng.integers(0, 256, (D, D, 3))
    return np.clip(w, 0, 255).reshape(-1, 3)


def _window(rng, D, tones, big):
    """One window.  Families share a dominant tone over k pixels; a second tone or noise fills the rest.  big: k >= 256 (flat,
    two big bins, or dominant + rest); else k in 200 .. 235 with a smaller second tone, or an ordinary noisy window."""
    npx = D * D
    px = _fill(rng, D)
    if big:
        fam = int(rng.integers(0, 3))                   # few families: many pairs big in the same bin, with different counts
        u = rng.random()
        if u < 0.25:
            k, k2 = npx, 0                              # flat: equal to every flat window of its family
        elif u < 0.5:
            k = int(rng.integers(256, npx - 255)); k2 = npx - k          # two big bins
        else:
            k = int(rng.integers(256, npx + 1)); k2 = int(rng.integers(0, min(200, npx - k) + 1))
    else:
        if rng.random() < 0.3:
            return px.reshape(D, D, 3).astype(np.uint8)                  # ordinary noisy window
        fam = int(rng.integers(0, len(tones)))
        k = int(rng.integers(200, 236)); k2 = int(rng.integers(0, 200)) if rng.random() < 0.7 else 0
    sec = (fam + 1 + int(rng.integers(0, len(tones) - 1))) % len(tones)
    px[:k] = tones[fam]
    px[k:k + k2] = tones[sec]
    return px.reshape(D, D, 3).astype(np.uint8)


def _coords(rng, n):
    """Clustered positions (half of the windows within 60 px of an earlier one) so the corner pass deletes and merges too."""
    out = []
    for i in range(n):
        if i and rng.random() < 0.5:
            p = out[int(rng.integers(0, i))]
            x, y = max(0, p[0] + int(rng.integers(-60, 61))), max(0, p[1] + int(rng.integers(-60, 61)))
        else:
            x, y = int(rng.integers(0, 1300)), int(rng.integers(0, 760))
        s = int(rng.integers(20, 80))
        out.append((x, y, x + s + int(rng.integers(-5, 6)), y + s + int(rng.integers(-5, 6))))
    return out


def big_positions(rng, n, blocks):
    """{block: count} -> sorted list positions of the big rows, drawn anywhere in their block."""
    pos = []
    for b, cnt in blocks.items():
        rows = min(BLOCK, n - b * BLOCK)
        assert 0 < cnt <= rows
        pos += (b * BLOCK + rng.choice(rows, cnt, replace=False)).tolist()
    return sorted(pos)


def make_frames(oracle, frames, D, seed):
    """frames: [(windows, {block: big rows})] -> dict(windows uint8[n,D,D,3], coords int32[n,4], offsets int32[F+1], big list of
    per-frame big-row positions).  A window whose largest bin count lands on the wrong side of 255 is drawn again; 15 % of the
    windows are exact copies of an earlier window of the same kind (pop-by-pixel-equality)."""
    rng = np.random.default_rng(seed * 100 + D)
    wins, coords, off, bigs = [], [], [0], []
    for n, blocks in frames:
        tones = rng.integers(0, 256, (8, 3))
        big = set(big_positions(rng, n, blocks))
        fw = []
        for i in range(n):
            isbig = i in big
            same = [q for q in range(i) if (q in big) == isbig]
            if same and rng.random() < 0.15:
                fw.append(fw[same[int(rng.integers(0, len(same)))]].copy())
                continue
            while True:
                w = _window(rng, D, tones, isbig)
                if (bin_counts(oracle, w[None]).max() > 255) == isbig:
                    break
            fw.append(w)
        wins += fw
        coords += _coords(rng, n)
        off.append(off[-1] + n)
        bigs.append(sorted(big))
    return dict(windows=np.stack(wins), coords=np.array(coords, np.int32), offsets=np.array(off, np.int32), big=bigs, D=D)


def make_cost_frames(oracle, D):
    F, lo, hi = COST_FRAMES
    rng = np.random.default_rng(SEEDS["cost"] * 100 + D)
    return make_frames(oracle, [(int(rng.integers(lo, hi + 1)), {}) for _ in range(F)], D, SEEDS["cost"])


_CASES, _EXPECT = {}, {}


def case(oracle, name, D):
    if (name, D) not in _CASES:
        _CASES[name, D] = make_cost_frames(oracle, D) if name == "cost" else make_frames(oracle, CASES[name], D, SEEDS[name])
    return _CASES[name, D]


def frame_slices(c):
    o = c["offsets"]
    return [slice(int(o[f]), int(o[f + 1])) for f in range(len(o) - 1)]


def expect(oracle, c, by_coords, tol, key=None):
    """Oracle survivors per frame [(windows, coords)], cached per (case, pass, tolerance) when key is given."""
    k = None if key is None else (key, c["D"], by_coords, tol)
    if k is None or k not in _EXPECT:
        r = [oracle.dedup(c["windows"][s], c["coords"][s], by_coords, tol) for s in frame_slices(c)]
        if k is None:
            return r
        _EXPECT[k] = r
    return _EXPECT[k]


def concat(per_frame, D):
    """[(windows, coords)] -> the (windows, coords, offsets) of one dedup call."""
    off = np.concatenate([[0], np.cumsum([len(c) for _, c in per_frame])]).astype(np.int32)
    w = np.concatenate([w for w, _ in per_frame]) if off[-1] else np.zeros((0, D, D, 3), np.uint8)
    c = np.concatenate([c for _, c in per_frame]).reshape(-1, 4).astype(np.int32)
    return dict(windows=w, coords=c, offsets=off, D=D)


def check(got, exp, what):
    gw, gc, go = got
    assert len(go) == len(exp) + 1, what
    for f, (ow, oc) in enumerate(exp):
        assert go[f + 1] - go[f] == len(oc), (what, f)
        assert np.array_equal(gc[go[f]:go[f + 1]], oc) and np.array_equal(gw[go[f]:go[f + 1]], ow), (what, f)


def block_pair_counts(big, n):
    """Big rows per block pair (I, J), J <= I, of k5_gram_big: block I's plus, off the diagonal, block J's."""
    nbk = (n + BLOCK - 1) // BLOCK
    per = np.bincount(np.asarray(big, np.int64) // BLOCK, minlength=nbk)
    return {(I, J): int(per[I] + (per[J] if I != J else 0)) for I in range(nbk) for J in range(I + 1)}


# ---- CPU: the inputs are in the regimes the GPU cases name --------------------------------------------------------------
def test_route_inputs_are_in_their_regimes(oracle):
    rng = np.random.default_rng(0)
    for D in (25, 32):
        for name in ("a", "b", "c"):
            c = case(oracle, name, D)
            spec = CASES[name]
            assert np.diff(c["offsets"]).tolist() == [n for n, _ in spec], (name, D)        # exact window counts
            counts = bin_counts(oracle, c["windows"])
            mx = counts.max(1)
            for f, s in enumerate(frame_slices(c)):
                n, blocks = spec[f]
                big = np.flatnonzero(mx[s] > 255)
                assert big.tolist() == c["big"][f], (name, D, f)                              # big rows exactly where placed
                nbk = (n + BLOCK - 1) // BLOCK
                assert np.bincount(big // BLOCK, minlength=nbk).tolist() == [blocks.get(b, 0) for b in range(nbk)], (name, D, f)
                pairs = block_pair_counts(big, n)
                if name == "b":
                    assert n > BLOCK and 0 < max(pairs.values()) <= BIG_MAX, (D, f, pairs)
                if name == "c":
                    assert n >= 300 and max(pairs.values()) >= BIG_MAX, (D, f, pairs)
                if name in "bc":
                    # pairs big in the SAME bin on both sides with different counts, and windows with two big bins
                    cb = counts[s][big]
                    same = [(i, j) for i in range(len(big)) for j in range(i) if np.any((cb[i] > 255) & (cb[j] > 255) & (cb[i] != cb[j]))]
                    assert same or len(big) < 5, (name, D, f)
                    # deletions and merges among the windows of this big-row frame
                    st = np.zeros(3, np.int64)
                    oracle.dedup(c["windows"][s], c["coords"][s], False, 0.85, stats=st)
                    assert st[1] > 0 and st[2] > 0, (name, D, f, st)
            if name in "bc":
                assert np.any((counts > 255).sum(1) >= 2), (name, D)                            # two big bins in one window
            if name == "b":      # big rows in block I only, in block J only, in both, on the diagonal; exactly 32 in a pair
                kinds, kept32 = set(), False
                for f, (n, blocks) in enumerate(spec):
                    for (I, J), k in block_pair_counts(c["big"][f], n).items():
                        if k:
                            kinds.add("diag" if I == J else ("both" if blocks.get(I) and blocks.get(J) else ("I" if blocks.get(I) else "J")))
                        kept32 |= k == BIG_MAX
                assert kinds == {"diag", "both", "I", "J"} and kept32, kinds
            if name == "c":      # handed over: a diagonal pair, an off-diagonal pair, one with a ragged block I; exactly 32 stays
                handed, kept32 = [], False
                for f, (n, _) in enumerate(spec):
                    for (I, J), k in block_pair_counts(c["big"][f], n).items():
                        if k > BIG_MAX:
                            handed.append((I == J, n - I * BLOCK < BLOCK))
                        kept32 |= k == BIG_MAX
                assert (True, False) in handed and (False, False) in handed and any(r for _, r in handed) and kept32, handed
            if name == "a":
                assert not np.any(mx > 255), D
                # deletions and merges in every producer / fold size class at tolerance 0.6
                for lo, hi in ROUTE_CLASSES:
                    st = np.zeros(3, np.int64)
                    for f, s in enumerate(frame_slices(c)):
                        if lo <= spec[f][0] <= hi:
                            oracle.dedup(c["windows"][s], c["coords"][s], False, 0.6, stats=st)
                    assert st[1] > 0 and st[2] > 0, (D, lo, hi, st)
            # the corner pass deletes and merges as well
            st = np.zeros(3, np.int64)
            for s in frame_slices(c):
                oracle.dedup(c["windows"][s], c["coords"][s], True, 0.95, stats=st)
            assert st[1] > 0 and st[2] > 0, (name, D, st)
            # the bin rule above is calcHist's: same occupied bins as the oracle's normalised histogram
            for i in rng.choice(len(c["windows"]), 20, replace=False):
                h = oracle.hist_normalized(c["windows"][i]).ravel()
                assert np.array_equal(np.flatnonzero(h), np.flatnonzero(counts[i])), (name, D, i)
                assert np.argmax(h) == np.argmax(counts[i])
        # (f) >= 256 frames of 33 .. 120 windows, most of them with merge-band pairs (the cost the CTA-fold routing reads)
        c = case(oracle, "cost", D)
        sizes = np.diff(c["offsets"])
        F, lo, hi = COST_FRAMES
        assert len(sizes) >= 256 and sizes.min() >= lo and sizes.max() <= hi and sizes.min() > 32
        merging = 0
        for s in frame_slices(c):
            st = np.zeros(3, np.int64)
            oracle.dedup(c["windows"][s], c["coords"][s], False, 0.85, stats=st)
            merging += st[2] > 0
        assert merging >= len(sizes) // 2, merging


# ---- GPU: every route against the oracle ----------------------------------------------------------------------------------
def _ctx(request, D):
    """The session context of the window size: 'det' for 25 x 25, 'rec' for 32 x 32 (launch_folds<640> / <1024>)."""
    return request.getfixturevalue("ctx_det" if D == 25 else "ctx_rec")


def _dedup(ctx, c, by_coords, tol):
    return ctx.dedup(c["windows"], c["coords"], c["offsets"], by_coords, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("D", (25, 32))
@pytest.mark.parametrize("name", ("a", "b", "c"))
def test_k5_routes_vs_oracle(request, oracle, name, D):
    """(a) size limits, (b) big rows kept by k5_gram_big, (c) block pairs handed to k5_pairs -- each in one call; the histogram pass
    at every tolerance, the corner pass on the raw lists (exact size limits) and on the first pass's output."""
    ctx = _ctx(request, D)
    c = case(oracle, name, D)
    for tol in HIST_TOLS:
        check(_dedup(ctx, c, False, tol), expect(oracle, c, False, tol, name), (name, D, "hist", tol))
    p1 = concat(expect(oracle, c, False, 0.85, name), D)
    for tol in CORNER_TOLS:
        check(_dedup(ctx, c, True, tol), expect(oracle, c, True, tol, name), (name, D, "corner", tol))
        check(_dedup(ctx, p1, True, tol), expect(oracle, p1, True, tol), (name, D, "corner after hist", tol))


@pytest.mark.gpu
@pytest.mark.parametrize("D", (25, 32))
def test_k5_routes_gram_off(tsd, oracle, monkeypatch, D):
    """TSD_GRAM=0: every frame's pair classes from k5_pairs -- the same survivors as the oracle (and so as the tensor-core route)."""
    monkeypatch.setenv("TSD_GRAM", "0")
    with tsd.Context(0, "det" if D == 25 else "rec") as ctx:
        for name in ("a", "b", "c"):
            c = case(oracle, name, D)
            for tol in HIST_TOLS:
                check(_dedup(ctx, c, False, tol), expect(oracle, c, False, tol, name), (name, D, "TSD_GRAM=0", tol))


@pytest.mark.gpu
@pytest.mark.parametrize("D", (25, 32))
def test_k5_fold_cta_by_cost(tsd, oracle, monkeypatch, D):
    """TSD_FOLD_CTA_COST=1 / 4 with 256 frames of 33 .. 120 windows: the frames with that many merge-band pairs go to k5_fold_cta
    instead of the warp fold; the survivors do not change."""
    c = case(oracle, "cost", D)
    for cost in ("1", "4"):
        monkeypatch.setenv("TSD_FOLD_CTA_COST", cost)
        with tsd.Context(0, "det" if D == 25 else "rec") as ctx:
            for tol in (0.85, 0.6):
                check(_dedup(ctx, c, False, tol), expect(oracle, c, False, tol, "cost"), (D, "TSD_FOLD_CTA_COST", cost, tol))


@pytest.mark.gpu
def test_chain_rec_4k_vs_oracle(ctx_rec, oracle, rec_golden, tsd):
    """Recognition flavour through the device-resident chain on two 4K frames with 2000 candidates each (~800 windows of 32 x 32
    per frame after the aspect filter, bit rows sized from max_boxes_per_frame): k5_gram_big and k5_fold_cta through the real
    chain, with large flat patches painted in so that the chain meets windows with counts above 255.  Record by record."""
    import torch
    H, W, F, N = 2160, 3840, 2, 2000
    frames = tsd.synth.make_frames(F, H, W, seed=tsd.synth.FRAME_SEED + 120)
    for f, (y, x, side) in ((0, (200, 400, 700)), (1, (900, 1800, 600)), (1, (100, 3000, 500))):
        frames[f][y:y + side, x:x + side] = np.array([30 + 70 * f, 190 - x // 40, 60 + y // 20], np.uint8)
    boxes, off = tsd.synth.make_boxes(F, N, H, W, seed=tsd.synth.BOX_SEED + 120, enlarge=1.15, D=32)
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(frames).to(dev)
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    ctx_rec.enqueue_frames(d_frames.data_ptr(), F, H, W, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), mode=tsd.RUN_RECOGNIZE,
                           max_boxes_per_frame=N)
    det, counts = ctx_rec.fetch_detections(int(off[-1]))
    got = {}
    for d in det:
        got.setdefault(int(d["frame"]), []).append((int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"])))
    r = rec_golden
    nsurv, bad = 0, []
    for f in range(F):
        cc, v = oracle.expand_boxes(boxes[off[f]:off[f + 1]], 1.15)
        cc = cc[v]
        wins = np.stack([oracle.crop_resize(frames[f], q, 32) for q in cc])
        nbig = int((bin_counts(oracle, wins).max(1) > 255).sum())
        assert 256 < len(wins) <= 1024 and nbig > BIG_MAX, (f, len(wins), nbig)       # k5_gram_big + k5_fold_cta, with big rows
        w1, c1 = oracle.dedup(wins, cc, False, 0.85)
        w2, c2 = oracle.dedup(w1, c1, True, 0.95)
        nsurv += len(c2)
        exp = []
        if len(c2):
            hog = np.stack([oracle.hog32(oracle.bgr2gray(w)) for w in w2])
            _, lab = oracle.lda_predict(hog, r["lda_W"], r["lda_b"], 0.5)
            exp = [tuple(int(x) for x in q) + (int(lab_),) for q, lab_ in zip(c2, lab) if lab_ != 0]
        if got.get(f, []) != exp:
            bad.append(f)
    assert not bad and int(counts[2]) == nsurv, (bad, counts.tolist(), nsurv)
