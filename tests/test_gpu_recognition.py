"""The recognition half (K6 grey, K7 HOG, K8 LDA, K8b KNN) against the oracle at every shape the API accepts, at angle-bin
boundaries, saturated probabilities, decision thresholds and exact distance ties.

The stored data (rec_golden.npz) leaves these to chance: 1 623 windows never make a K7 warp take a second window (tsd_hog runs
at most sm_count * 8 CTAs x 4 warps = 4 736 warps on a B200, K8 at most 9 472), real windows rarely put a gradient on a bin
boundary or the 0/360 degree wrap, real logits never tie, and real KNN queries have no distance ties.  Every case here is built
so that a kernel that is subtly wrong there gives a different answer:

  HOG        every integer gradient (dx, dy) in [-255, 255]^2 planted at interior pixels, plus ramps, steps, impulses,
             checkerboards, border-only gradients, constant and random images, in one tsd_hog call of more than 4 736
             windows; descriptors within 1e-4 relative + 1e-7 of oracle.hog32, and the same zero pattern.
  LDA        nfeat 1 .. 4096 at n = 1, 7, 20 000 (logits within the f64 summation bound, labels exact); dyadic logits
             (exact in any summation order) at ties, saturation (p == 1.0 from z ~ 36.74 on), z = 0, +-2^-k, and tol at
             0, 0.25, 0.5, 0.75, 1 - 1e-9, 1 and at expit(z) of a case: logits bit for bit, labels exact.
  KNN        k = 1..8, ntrain 1 .. 14 574, nfeat 1 .. 1500 on continuous data (labels = oracle = scikit-learn); exact ties
             on an integer lattice, pinned to the documented rule (equal distances: the smaller training index is nearer).
  composite  tsd_recognize on ~12 k BGR windows; the chain (RUN_RECOGNIZE) on 1 024 frames, ~35 k survivors, so that K6, K7
             and K8 all loop inside the chain.

test_recognition_inputs_are_in_their_regimes checks on the CPU that each case is in the regime it names.
"""
import math

import numpy as np
import pytest

HOG_WARPS_B200 = 148 * 8 * 4          # tsd_hog's largest grid on a B200 (148 SMs): sm_count * 8 CTAs x 4 warps
LDA_WARPS_B200 = 148 * 8 * 8          # dev_lda: sm_count * 8 CTAs x 8 warps
LDA_NFEAT = (1, 2, 31, 32, 33, 324, 325, 1000, 1024, 1025, 2048, 4096)
LDA_N = (1, 7, 20000)
TOLS = (0.0, 0.25, 0.5, 0.75, 1 - 1e-9, 1.0)
LADDER = (30.0, 31.0, 32.0, 33.0, 34.0, 35.0, 36.0, 36.5, 36.7, 36.73, 36.74, 36.75, 37.0, 40.0, 745.0, 750.0)
KNN_NTRAIN = (1, 3, 31, 32, 33, 1000, 14574)
KNN_NFEAT = (1, 7, 324, 1024, 1500)
KNN_QUERIES = 160
CHAIN_SEED = 41
CHAIN_LDA_SEED = 99                   # spread_lda seed that keeps every chain survivor clear of the decision (regime test)


def expit(z):
    """scipy.special.expit as the oracle computes it: 1 / (1 + exp(-z)) with the C library's exp."""
    return 1.0 / (1.0 + math.exp(-z)) if z > -709 else 0.0


# ---- HOG inputs -------------------------------------------------------------------------------------------------------
CENTRES = 2 + 3 * np.arange(10)       # stride-3 grid of plus-shaped stencils: arms at 1 .. 30, never on the border


def gradient_pairs():
    """Every (dx, dy) in [-255, 255]^2, sorted by magnitude, 100 per 32 x 32 image -> (images, (image, y, x, dx, dy))."""
    d = np.arange(-255, 256)
    dx, dy = (a.ravel() for a in np.meshgrid(d, d, indexing="ij"))
    o = np.lexsort((dy, dx, dx * dx + dy * dy))
    dx, dy = dx[o], dy[o]
    k = np.arange(len(dx))
    i, s = k // 100, k % 100
    y, x = CENTRES[s // 10], CENTRES[s % 10]
    img = np.zeros((int(i[-1]) + 1, 32, 32), np.uint8)
    img[i, y, x - 1] = np.maximum(-dx, 0); img[i, y, x + 1] = np.maximum(dx, 0)
    img[i, y - 1, x] = np.maximum(-dy, 0); img[i, y + 1, x] = np.maximum(dy, 0)
    return img, (i, y, x, dx, dy)


def hog_families(seed=71):
    """{family: uint8 [m, 32, 32]}."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:32, 0:32].astype(np.float64) - 15.5
    fam = {"pairs": gradient_pairs()[0]}
    fam["ramps"] = np.stack([np.clip(np.rint(128 + s * (xx * math.cos(math.radians(a)) + yy * math.sin(math.radians(a)))), 0, 255)
                             for a in range(0, 360, 5) for s in (0.5, 2.0, 6.0)]).astype(np.uint8)
    steps = []
    for c in range(1, 32):
        v = np.zeros((32, 32), np.uint8); v[:, c:] = 255
        steps += [v, 255 - v, v.T.copy(), 255 - v.T]
    fam["steps"] = np.stack(steps)
    imp = np.zeros((1024, 32, 32), np.uint8); imp.reshape(1024, 1024)[np.arange(1024), np.arange(1024)] = 255
    fam["impulses"] = np.concatenate([imp, 255 - imp[::3]])
    chk = []
    for p in (1, 2, 3, 4, 5, 8, 16):
        for ph in (0, 1):
            v = ((((yy + 15.5 + ph) // p) + ((xx + 15.5) // p)) % 2 * 255).astype(np.uint8)
            chk += [v, 255 - v]
    fam["checker"] = np.stack(chk)
    bord = []
    for j in range(64):
        v = np.full((32, 32), int(rng.integers(0, 256)), np.uint8)
        sides = (0, 1, 2, 3) if j < 32 else (j % 4,)
        for sd in sides:
            vals = rng.integers(0, 256, 32).astype(np.uint8)
            if sd == 0: v[0] = vals
            elif sd == 1: v[31] = vals
            elif sd == 2: v[:, 0] = vals
            else: v[:, 31] = vals
        bord.append(v)
    fam["border"] = np.stack(bord)
    fam["constant"] = np.stack([np.full((32, 32), c, np.uint8) for c in (0, 1, 127, 128, 254, 255)])
    blocky = rng.integers(0, 256, (300, 8, 8)).repeat(4, 1).repeat(4, 2)
    sparse = np.where(rng.random((300, 32, 32)) < 0.05, rng.integers(0, 256, (300, 32, 32)), 0)
    fam["random"] = np.concatenate([rng.integers(0, 256, (600, 32, 32)), blocky, sparse,
                                    rng.integers(100, 104, (100, 32, 32))]).astype(np.uint8)
    return fam


def hog_batch():
    fam = hog_families()
    return np.concatenate(list(fam.values())), {k: len(v) for k, v in fam.items()}


def bin_rule_f32(dx, dy):
    """float32 numpy copy of the orientation-bin rule (fast_atan_deg, radians, t = angle * 9 / 2pi - 0.5) -> t before floor."""
    f = np.float32
    dx, dy = dx.astype(f), dy.astype(f)
    sc = f(180.0 / math.pi)
    p1, p3, p5, p7 = f(0.9997878412794807) * sc, f(-0.3258083974640975) * sc, f(0.1555786518463281) * sc, f(-0.04432655554792128) * sc
    ax, ay = np.abs(dx), np.abs(dy)
    eps = f(np.finfo(np.float64).eps)
    with np.errstate(invalid="ignore", divide="ignore"):
        c = np.where(ax >= ay, ay / (ax + eps), ax / (ay + eps)).astype(f)
    c2 = c * c
    a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c
    a = np.where(ax >= ay, a, f(90) - a)
    a = np.where(dx < 0, f(180) - a, a)
    a = np.where(dy < 0, f(360) - a, a)
    return a * f(math.pi / 180.0) * f(9 / (2 * math.pi)) - f(0.5)


# ---- LDA inputs -------------------------------------------------------------------------------------------------------
def lda_random(nfeat, n, seed):
    """Continuous X f32 [n, nfeat] and W f64 scaled so that the logits are O(3): labels of every kind, few saturated."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, nfeat)).astype(np.float32)
    W = rng.standard_normal((nfeat, 6)) * (3.0 / math.sqrt(nfeat))
    b = rng.standard_normal(6) * 0.5
    return X, W, b


def _split(v, rng):
    """Two float32 values whose f64 sum is exactly v (v itself a float32)."""
    v = float(np.float32(v))
    for _ in range(8):
        a = float(np.float32(v * float(rng.uniform(0.2, 0.8))))
        if float(np.float32(v - a)) + a == v:
            return a, v - a
    return v, 0.0


def lda_dyadic_cases(seed=5):
    """-> dict(X f32 [n, 12], W f64 [12, 6], b f64 [6], rows {kind: slice}).  z_c = X[:, c] + X[:, 6 + c]: two float32 terms,
    so every z is exact in f64 whatever the order of summation."""
    rng = np.random.default_rng(seed)
    rows, kinds = [], {}

    def add(kind, zs):
        start = len(rows)
        for z in zs:
            rows.append([float(np.float32(v)) for v in z])
        kinds[kind] = slice(start, len(rows))

    ident = []
    for v in (0.125, 3.5, 36.75, 40.0, 2.0 ** -52, -1.5):
        for m in range(2, 7):
            z = [-2.0] * 6
            for c in rng.choice(6, m, replace=False):
                z[c] = v
            ident.append(z)
    ident.append([1.0] * 6)
    add("identical", ident)
    lad = []
    for m in range(2, 7):
        for j in range(len(LADDER)):
            vals = list(LADDER[j:j + m]) + [LADDER[-1]] * max(0, j + m - len(LADDER))
            for order in (vals, vals[::-1], list(rng.permutation(vals)), [LADDER[j]] * m):
                z = [-3.0] * 6
                for c, v in zip(rng.choice(6, m, replace=False), order):
                    z[c] = float(v)
                lad.append(z)
    add("ladder", lad)
    neg = [list(-np.array(LADDER)[rng.choice(len(LADDER), 6)]) for _ in range(40)]
    neg += [[-745.0, -750.0, -40.0, 0.5, -37.0, -36.7], [-750.0] * 6, [-36.74] * 6]
    add("negative", neg)
    small = [[0.0] * 6]
    for k in range(1, 61):
        e = 2.0 ** -k
        pool = (0.0, e, -e, e / 2, -e / 2, 2 * e, -2 * e)
        small += [[e, e / 2, 0.0, -e, 2 * e, -e / 2], [0.0, -e, e, e, 0.0, -e], [-e] * 6, [e] * 6]
        small += [[float(rng.choice(pool)) for _ in range(6)] for _ in range(3)]
    add("near_zero", small)
    Z = np.array(rows)
    X = np.zeros((len(Z), 12), np.float32)
    for r, z in enumerate(Z):
        for c, v in enumerate(z):
            X[r, c], X[r, 6 + c] = _split(v, rng)
    W = np.zeros((12, 6))
    W[np.arange(6), np.arange(6)] = 1.0
    W[6 + np.arange(6), np.arange(6)] = 1.0
    return dict(X=X, W=W, b=np.zeros(6), kinds=kinds)


def lda_tols(cases):
    """The fixed tolerances plus expit(z) of z values in the cases (a class with p exactly equal to tol)."""
    X = cases["X"]
    z = (X[:, :6].astype(np.float64) + X[:, 6:].astype(np.float64)).ravel()
    pick = [2.0 ** -1, 2.0 ** -20, 2.0 ** -52, 0.125, 3.5, 36.5, float(np.float32(36.7)), float(np.float32(36.73))]
    assert all(np.any(z == v) for v in pick)
    return TOLS + tuple(expit(v) for v in pick)


# ---- KNN inputs -------------------------------------------------------------------------------------------------------
def knn_model(nfeat, ntrain, seed, nlabels=7):
    """Continuous model: X f32 [KNN_QUERIES, nfeat], xbar, S f64 [nfeat, 6], Ztrain f64 [ntrain, 6], ytrain."""
    rng = np.random.default_rng(seed)
    xbar = rng.standard_normal(nfeat)
    S = rng.standard_normal((nfeat, 6)) / math.sqrt(nfeat)
    Zt = rng.standard_normal((ntrain, 6))
    yt = rng.integers(0, nlabels, ntrain).astype(np.int32)
    X = (xbar + rng.standard_normal((KNN_QUERIES, nfeat))).astype(np.float32)
    return X, xbar, S, Zt, yt


def knn_lattice(seed=9):
    """Exact ties: integer Ztrain in {0,1,2}^6 with every point several times under different labels, S = identity, xbar = 0,
    integer queries -> Z = X exactly and many training rows at exactly the same distance."""
    rng = np.random.default_rng(seed)
    Zt = rng.integers(0, 3, (1500, 6)).astype(np.float64)
    Zt[1000:1200] = Zt[rng.integers(0, 1000, 200)]                 # duplicates, most with another label
    Zt[1200:1260] = Zt[1200 - 32 * rng.integers(1, 30, 60)]       # duplicates in the same lane (index - 32 m)
    yt = rng.integers(0, 16, 1500).astype(np.int32)
    X = rng.integers(0, 3, (400, 6)).astype(np.float32)
    return X, np.zeros(6), np.eye(6), Zt, yt


def knn_rule(Z, Zt, yt, k, larger_index_first=False):
    """Brute-force KNN in numpy: order by (distance, index) -- or (distance, -index) -- and vote, ties to the smallest label."""
    d = ((Z[:, None, :] - Zt[None, :, :]) ** 2).sum(-1)
    idx = np.arange(len(Zt))
    out = np.empty(len(Z), np.int32)
    for q in range(len(Z)):
        o = np.lexsort((-idx if larger_index_first else idx, d[q]))[:k]
        out[q] = int(np.argmax(np.bincount(yt[o], minlength=16)))
    return out


# ---- recognition windows / chain --------------------------------------------------------------------------------------
def composite_windows(seed=13):
    """~12 k BGR windows: the HOG families as grey BGR (B = G = R), the same recoloured, and random colour windows."""
    rng = np.random.default_rng(seed)
    g, _ = hog_batch()
    g16 = g.astype(np.int16)
    recol = np.stack([g16, 255 - g16, (g16 + 85) % 256], -1).astype(np.uint8)
    return np.concatenate([np.repeat(g[..., None], 3, -1), recol, rng.integers(0, 256, (600, 32, 32, 3), dtype=np.uint8)])


def chain_inputs(tsd, U=32, F=1024, N=200, seed=CHAIN_SEED):
    """F frames x N candidates made of U unique (frame, boxes) pairs: frame f is frame f % U with the boxes of f % U."""
    uniq = tsd.synth.make_frames(U, seed=tsd.synth.FRAME_SEED + seed)
    ub, uoff = tsd.synth.make_boxes(U, N, seed=tsd.synth.BOX_SEED + seed)
    per = [ub[uoff[u]:uoff[u + 1]] for u in range(U)]
    boxes = np.concatenate([per[f % U] for f in range(F)]).astype(np.int32)
    off = np.concatenate([[0], np.cumsum([len(per[f % U]) for f in range(F)])]).astype(np.int32)
    return uniq, per, boxes, off


def oracle_rec_frame(oracle, frame, boxes):
    """Survivor coordinates and HOG descriptors of one frame (x1.15, 32 x 32, both dedup passes, grey -> HOG)."""
    c, v = oracle.expand_boxes(boxes, 1.15)
    c = c[v]
    wins = np.stack([oracle.crop_resize(frame, cc, 32) for cc in c]) if len(c) else np.zeros((0, 32, 32, 3), np.uint8)
    w1, c1 = oracle.dedup(wins, c, False, 0.85)
    w2, c2 = oracle.dedup(w1, c1, True, 0.95)
    return c2, np.stack([oracle.hog32(oracle.bgr2gray(w)) for w in w2]) if len(c2) else np.zeros((0, 324), np.float32)


def spread_lda(hog, seed, q=0.85):
    """324-feature weights under which synthetic windows get every label: random W, each b_c puts 15 % of the given descriptors
    on the positive side of classifier c.  (The reference's weights call all of them "no sign".)"""
    rng = np.random.default_rng(seed)
    W = rng.standard_normal((324, 6))
    return W, -np.quantile(hog.astype(np.float64) @ W, q, axis=0)


def decision_margin(z, hog, W):
    """Per window: how far the logits are from a change of the tol = 0.5 decision (min |z_c|, and the gap between the two
    largest positive z), in units of the largest logit change that HOG features within 1e-5 relative + 1e-7 can cause.  K7's
    descriptors differ from the oracle's by at most ~1e-6 relative (8e-7 measured on the reference's windows); the HOG test
    holds them to 1e-4."""
    guard = ((1e-5 * np.abs(hog.astype(np.float64)) + 1e-7) @ np.abs(W)).max(1)
    zs = np.sort(np.where(z > 0, z, -np.inf), 1)
    gap = np.full(len(z), np.inf)
    two = np.isfinite(zs[:, -2])
    gap[two] = zs[two, -1] - zs[two, -2]
    return np.minimum(np.abs(z).min(1), gap) / (2 * guard)


def composite_case(oracle, seed=13):
    """-> (BGR windows, W, b, oracle labels): composite_windows() under spread_lda weights, without the few windows whose label
    the HOG tolerance itself could change (decision_margin <= 1)."""
    wins = composite_windows(seed)
    hog = np.stack([oracle.hog32(oracle.bgr2gray(w)) for w in wins])
    W, b = spread_lda(hog, seed)
    z, lab = oracle.lda_predict(hog, W, b, 0.5)
    keep = decision_margin(z, hog, W) > 1
    return wins[keep], W, b, lab[keep]


# ---- CPU: every case is in its regime ---------------------------------------------------------------------------------
def test_recognition_inputs_are_in_their_regimes(oracle, tsd):
    # HOG: every pair planted, where the kernel reads it (reflect-101 never involved), in one batch with looping warps
    img, (i, y, x, dx, dy) = gradient_pairs()
    im = img.astype(np.int32)
    assert np.array_equal(im[i, y, x + 1] - im[i, y, x - 1], dx) and np.array_equal(im[i, y + 1, x] - im[i, y - 1, x], dy)
    assert len(np.unique((dx + 255) * 511 + dy + 255)) == 511 * 511 == 261121
    assert np.all(np.diff(dx * dx + dy * dy) >= 0)
    batch, sizes = hog_batch()
    assert len(batch) > HOG_WARPS_B200 and sizes["pairs"] == 2612
    t = bin_rule_f32(dx, dy)
    frac = t - np.floor(t)
    assert np.sum((frac < 1e-5) | (frac > 1 - 1e-5)) > 100                       # pairs within 1e-5 of a bin boundary
    wrap = np.floor(t).astype(int)
    assert np.sum(wrap == -1) > 100 and np.sum(wrap == 8) > 100                   # both sides of the 0 / 360 degree wrap
    # LDA: dyadic logits are exact (equal to math.fsum of the terms in any order)
    cs = lda_dyadic_cases()
    X, W = cs["X"].astype(np.float64), cs["W"]
    z, _ = oracle.lda_predict(cs["X"], W, cs["b"], 0.5)
    for r in range(len(X)):
        for c in range(6):
            assert z[r, c] == math.fsum(X[r] * W[:, c]) == math.fsum((X[r] * W[:, c])[::-1])
    lad = z[cs["kinds"]["ladder"]]
    p = np.vectorize(expit)(lad)
    sat = (p == 1.0).sum(1)
    assert np.sum(sat >= 2) > 10                                                  # p == 1.0 ties among >= 2 classes
    assert np.any([len(set(r[(r > 0) & (r < 1)])) < np.sum((r > 0) & (r < 1)) for r in p])   # equal p < 1 ties
    assert np.any((p > 0.5) & (p < 1.0)) and np.any((sat >= 2) & ((lad[:, None, :] > lad[..., None]).any((1, 2))))
    tols = lda_tols(cs)
    assert len(tols) == len(TOLS) + 8
    # LDA random: at n = 20 000 the K8 warps loop; the logits spread over every label
    assert max(LDA_N) > LDA_WARPS_B200
    _, lab = oracle.lda_predict(*lda_random(324, 2000, 1), 0.5)
    assert set(np.unique(lab)) == set(range(7))
    # KNN lattice: Z is exact, ties straddle the k-th neighbour, and a flipped tie rule changes labels at every k
    Xq, xbar, S, Zt, yt = knn_lattice()
    Zq, _ = oracle.knn_predict(Xq, xbar, S, Zt, yt, 1)
    assert np.array_equal(Zq, Xq.astype(np.float64))
    for k in range(1, 9):
        _, olab = oracle.knn_predict(Xq, xbar, S, Zt, yt, k)
        assert np.array_equal(olab, knn_rule(Zq, Zt, yt, k))
        assert np.sum(knn_rule(Zq, Zt, yt, k, larger_index_first=True) != olab) >= 1, k
    # composite windows: ~12 k of them, every label; the chain: ~35 k survivors, every label, none within reach of the HOG
    # tolerance of a different decision
    wins, W, b, lab = composite_case(oracle)
    assert 11000 < len(wins) < 13000 and set(np.unique(lab)) == set(range(7))
    uniq, per, _, off = chain_inputs(tsd)
    sv = [oracle_rec_frame(oracle, f, bx) for f, bx in zip(uniq, per)]
    hog = np.concatenate([h for _, h in sv])
    W, b = spread_lda(hog, CHAIN_LDA_SEED)
    z, lab = oracle.lda_predict(hog, W, b, 0.5)
    assert len(hog) * (len(off) - 1) // len(uniq) > 3 * LDA_WARPS_B200 and set(np.unique(lab)) == set(range(7))
    assert decision_margin(z, hog, W).min() > 1


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.gpu
def test_hog_every_gradient(ctx_rec, oracle):
    batch, sizes = hog_batch()
    assert len(batch) > _sm_count() * 8 * 4                                       # every warp of tsd_hog's grid takes > 1 window
    got = ctx_rec.hog(batch)
    exp = np.stack([oracle.hog32(g) for g in batch])
    err = np.abs(got - exp) - 1e-4 * np.abs(exp) - 1e-7
    bad = np.nonzero((err > 0).any(1) | ((got == 0) != (exp == 0)).any(1))[0]
    names = np.repeat(list(sizes), list(sizes.values()))
    assert len(bad) == 0, (len(bad), sorted(set(names[bad])), bad[:10].tolist(), float(err.max()))
    cv2 = pytest.importorskip("cv2")
    hd = cv2.HOGDescriptor((32, 32), (16, 16), (8, 8), (8, 8), 9, 1, -1, 0, 0.2, False, 64, True)
    ref = np.stack([hd.compute(g).ravel() for g in batch])
    assert np.all(np.abs(got - ref) <= 1e-4 * np.abs(ref) + 1e-7), float(np.max(np.abs(got - ref) - 1e-4 * np.abs(ref)))


@pytest.mark.gpu
@pytest.mark.parametrize("nfeat", LDA_NFEAT)
def test_lda_feature_counts(tsd, oracle, nfeat):
    X, W, b = lda_random(nfeat, max(LDA_N), 100 + nfeat)
    with tsd.Context(0, "rec") as c:
        c.set_lda(W, b)
        for n in LDA_N:
            lg, lab = c.lda_predict(X[:n])
            olg, olab = oracle.lda_predict(X[:n], W, b, 0.5)
            bound = nfeat * 2.0 ** -52 * (np.abs(X[:n].astype(np.float64)) @ np.abs(W) + np.abs(b))
            assert np.all(np.abs(lg - olg) <= bound), (n, float(np.max(np.abs(lg - olg) / bound)))
            assert np.array_equal(lab, olab), (n, int(np.sum(lab != olab)))
        # the TF32 evaluation kernel: as long as its tiles fit in one block, else a clear refusal
        if 64 * ((nfeat + 7) // 8 * 8) <= 227 * 1024:
            z3, _, _ = c.lda_predict_tf32(X[:4096], split=3)
            olg, _ = oracle.lda_predict(X[:4096], W, b, 0.5)
            assert np.all(np.abs(z3 - olg) <= 1e-5 * (np.abs(X[:4096].astype(np.float64)) @ np.abs(W) + np.abs(b)) + 1e-5)
        else:
            with pytest.raises(tsd.TsdError, match="shared memory"):
                c.lda_predict_tf32(X[:16], split=3)


@pytest.mark.gpu
def test_lda_decision_edges(tsd, oracle):
    cs = lda_dyadic_cases()
    X, W, b = cs["X"], cs["W"], cs["b"]
    bad = []
    with tsd.Context(0, "rec") as c:
        c.set_lda(W, b)
        for tol in lda_tols(cs):
            lg, lab = c.lda_predict(X, tol=tol)
            olg, olab = oracle.lda_predict(X, W, b, tol)
            assert np.array_equal(lg, olg), tol                                  # exact logits: bit for bit
            for kind, s in cs["kinds"].items():
                for r in np.nonzero(lab[s] != olab[s])[0]:
                    bad.append((tol, kind, lg[s][r].tolist(), int(lab[s][r]), int(olab[s][r])))
    assert not bad, bad[:8]


@pytest.mark.gpu
@pytest.mark.parametrize("nfeat", KNN_NFEAT)
def test_knn_sweep(tsd, oracle, nfeat):
    sk = None
    try:
        from sklearn.neighbors import KNeighborsClassifier as sk
    except ImportError:
        pass
    with tsd.Context(0, "rec") as c:
        for ntrain in KNN_NTRAIN:
            X, xbar, S, Zt, yt = knn_model(nfeat, ntrain, 1000 * nfeat + ntrain, nlabels=16 if ntrain == 1000 else 7)
            scale = np.abs(X.astype(np.float64) - xbar) @ np.abs(S)
            for k in range(1, 9):
                c.set_knn(xbar, S, Zt, yt, k)
                Z, lab = c.knn_predict(X)
                oZ, olab = oracle.knn_predict(X, xbar, S, Zt, yt, k)
                assert np.all(np.abs(Z - oZ) <= 1e-12 * scale), (ntrain, k)
                assert np.array_equal(lab, olab), (ntrain, k, int(np.sum(lab != olab)))
                if sk is not None and k <= ntrain:
                    assert np.array_equal(lab, sk(k).fit(Zt, yt).predict(oZ)), (ntrain, k)


@pytest.mark.gpu
def test_knn_exact_ties(tsd, oracle):
    """Equal distances rank by training index (the smaller one is nearer), as the oracle documents.  scikit-learn's kd-tree
    (what the reference uses) orders exact ties by its own traversal instead.  On this lattice set its labels differ from the
    rule's on 92 (k = 1), 142 (k = 3), 156 (k = 4) and 180 (k = 8) of the 400 queries; ranking the larger index first would
    change 230 to 320 of them at every k.  The reference's training set has one duplicate row and no tie of mixed labels, so
    real data is unaffected; the rule is pinned here, not sklearn's.  Labels outside 0..15 are refused."""
    Xq, xbar, S, Zt, yt = knn_lattice()
    with tsd.Context(0, "rec") as c:
        for k in range(1, 9):
            c.set_knn(xbar, S, Zt, yt, k)
            Z, lab = c.knn_predict(Xq)
            oZ, olab = oracle.knn_predict(Xq, xbar, S, Zt, yt, k)
            assert np.array_equal(Z, oZ)
            assert np.array_equal(lab, olab), (k, int(np.sum(lab != olab)))
        for y in (-1, 16):
            bad = yt.copy(); bad[7] = y
            with pytest.raises(tsd.TsdError, match="labels must be 0..15"):
                c.set_knn(xbar, S, Zt, bad, 4)


@pytest.mark.gpu
def test_recognize_composite(tsd, oracle):
    wins, W, b, olab = composite_case(oracle)
    with tsd.Context(0, "rec") as c:
        c.set_lda(W, b)
        lab = c.recognize_windows(wins)
    assert np.array_equal(lab, olab), int(np.sum(lab != olab))


@pytest.mark.gpu
def test_chain_recognition_at_scale(oracle, tsd):
    """1 024 frames x 200 candidates through RUN_RECOGNIZE: ~35 k survivors, so that K6's grid-stride loop, K7's and K8's
    persistent warps all take several windows inside the chain.  Frames repeat 32 unique (frame, boxes) pairs.  spread_lda
    weights, so that records of every label come out."""
    import torch
    uniq, per, boxes, off = chain_inputs(tsd)
    U, F = len(uniq), len(off) - 1
    sv = [oracle_rec_frame(oracle, uniq[u], per[u]) for u in range(U)]
    W, b = spread_lda(np.concatenate([h for _, h in sv]), CHAIN_LDA_SEED)
    exp, nsurv = [], 0
    for c2, hog in sv:
        lab = oracle.lda_predict(hog, W, b, 0.5)[1] if len(hog) else []
        exp.append([tuple(int(x) for x in q) + (int(l),) for q, l in zip(c2, lab) if l != 0])
        nsurv += len(c2)
    nsurv *= F // U
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(uniq).to(dev)[torch.arange(F, device=dev) % U].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    with tsd.Context(0, "rec") as c:
        c.set_lda(W, b)
        c.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), mode=tsd.RUN_RECOGNIZE,
                         max_boxes_per_frame=max(len(p) for p in per))
        det, counts = c.fetch_detections(int(off[-1]))
    got = {}
    for d in det:
        got.setdefault(int(d["frame"]), []).append((int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"])))
    assert nsurv > _sm_count() * 8 * 8 * 3                                       # K8's 9 472 warps take >= 3 windows each
    bad = [f for f in range(F) if got.get(f, []) != exp[f % U]]
    assert not bad and int(counts[2]) == nsurv, (bad[:10], counts.tolist(), nsurv)
