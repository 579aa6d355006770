"""Every entry point and the chain past 4 GiB buffers, and batches at the 2^23-frame limit, against the oracle.

Per-window addresses are computed as (int64_t)w * stride throughout; these tests are what notices when one of those widenings goes
missing.  Each case is sized so that the buffers it names exceed 2^32 bytes (test_large_cases_reach_their_sizes checks the sizes
on the CPU with the stride formulas of tsd_kernels.cuh).

Inputs repeat P pairwise different patterns, P an odd prime (4 099 windows, 127 frame patterns, 61 full-size frames,
1 000 003 pixels): the expected output of item i is the oracle's output for pattern i mod P.  An address that wraps at 2^31 or 2^32
bytes lands on another pattern or at a misaligned offset, so the comparison fails.  Outputs are compared chunk by chunk, on the
device where they live there.

  stages      tsd_recognize, tsd_hog, tsd_lda_predict, tsd_knn_predict, tsd_crop_resize, tsd_windows, tsd_hist, tsd_color_masks,
              tsd_score, tsd_score_masks, tsd_dedup (both passes), tsd_mean_windows, tsd_bgr2hsv, tsd_bgr2gray, tsd_preprocess.
  chain       two overlapped tsd_enqueue_frames batches each (detection at D = 25, recognition at D = 32), so that the second
              scratch slot's windows and histogram entries lie past 4 GiB; one fetched with fetch_previous, one with
              fetch_detections.  Host routes of tsd_detect_frames on 4.6 GB of page-locked or pageable frames.
  frame limit 2^23 - 1 frames through tsd_dedup and tsd_enqueue_frames, the last few holding frames in each K5 work-list regime;
              2^23 frames are refused.

Every case uses a fresh context.  The library's memory pool keeps what a case allocated for the rest of the process, so no case
needs more than about 26 GB of device memory; a case skips, naming the amount, when the device or the host has too little free.
"""
import ctypes as C
import functools
import os

import numpy as np
import pytest

from test_gpu_recognition import composite_case, decision_margin, oracle_rec_frame
from test_gpu_sequences import gap_bias

E_INVALID = -1
GB = 1e9
P = 4099                                    # window patterns
PF = 127                                    # frame patterns (chains, dedup)
PH = 61                                     # full-size frame patterns (preprocess, host routes)
PX = 1_000_003                              # pixel patterns (bgr2hsv, bgr2gray)

N_GREY = (1 << 22) + P                      # recognize / hog / score_masks
N_LDA = 3_400_000
N_KNN = 720_000
N_WIN32 = 1_420_000                         # crop_resize, color_masks, score, mean_windows
N_HIST = 360_000
N_DEDUP = 1_640_000                         # 205 000 frames x 8
NPX = (1 << 32) + (1 << 24) + 13
N_PRE = 3960
WIN_FRAMES, WIN_H, WIN_W = 347, 256, 256    # tsd_windows: 347 frames x P boxes
KNN_NFEAT, KNN_NTRAIN = 1500, 97
DEDUP_PER_FRAME = 8
MEAN_GROUPS = (0, 1000, 1_410_000, N_WIN32)
CH_F, CH_H, CH_W, CH_BOXES = {"det": 150_000, "rec": 100_000}, 48, 64, 8
HOST_F, HOST_H, HOST_W, HOST_BOXES = 1400, 800, 1360, 200
LIMIT = 1 << 23                             # frames a batch may not reach (K5 work-list items keep frame << 8 in an int32)
LIM_H = LIM_W = 8
LIM_COUNTS = (2, 24, 64, 200)               # windows of the last frames: tiny list, tiny list, flat (k5_pairs), k5_gram_big
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- strides and limits of the library, read from its sources -----------------------------------------------------------
def _src(name):
    return open(os.path.join(ROOT, "opencv-traffic-sign-detector_b200", "csrc", name)).read()


def win_stride(npx, ch=3):
    return (npx * ch + 15) & ~15


def ent_stride(npx):
    return (npx + 3) & ~3


def k5_constant(name):
    import re
    return int(re.search(r"constexpr int %s = (\d+);" % name, _src("tsd_k5.cuh")).group(1))


def is_prime(n):
    return n > 1 and all(n % d for d in range(2, int(n ** 0.5) + 1))


# ---- patterns ------------------------------------------------------------------------------------------------------------
def distinct_first(a, k):
    """Indices of the first k pairwise different rows of a."""
    _, first = np.unique(a.reshape(len(a), -1), axis=0, return_index=True)
    first = np.sort(first)
    assert len(first) >= k, (len(first), k)
    return first[:k]


@functools.lru_cache(None)
def _oracle():
    from oracle import oracle as O
    O.build()
    return O


@functools.lru_cache(None)
def rec_patterns():
    """-> (BGR windows [P,32,32,3], grey [P,32,32], HOG [P,324], W, b, labels): composite windows whose labels the HOG tolerance
    cannot change, pairwise different in BGR and in grey."""
    O = _oracle()
    wins, W, b, lab = composite_case(O)
    grey = np.stack([O.bgr2gray(w) for w in wins])
    keep = distinct_first(grey, P)                           # (different grey implies different BGR)
    wins, grey, lab = wins[keep], grey[keep], lab[keep]
    hog = np.stack([O.hog32(g) for g in grey])
    return wins, grey, hog, W, b, lab


@functools.lru_cache(None)
def square_boxes(n, H, W, lo, hi, seed):
    """n boxes (x, y, s, s) inside an H x W frame (every one passes the aspect test and gives a non-empty crop)."""
    rng = np.random.default_rng(seed)
    s = rng.integers(lo, hi + 1, n)
    x = (rng.random(n) * (W - s + 1)).astype(np.int64)
    y = (rng.random(n) * (H - s + 1)).astype(np.int64)
    return np.stack([x, y, s, s], 1).astype(np.int32)


@functools.lru_cache(None)
def small_frames(n, H, W, seed):
    import tsd_b200
    return tsd_b200.synth.make_frames(n, H, W, seed=tsd_b200.synth.FRAME_SEED + seed, nrect=12)


@functools.lru_cache(None)
def crop_patterns(D, enlarge):
    """P windows (frame p % PH of PH 256 x 256 frames, a square box each) -> (frames, coords [P,4], win_frame [P], windows)."""
    O = _oracle()
    frames = small_frames(PH, WIN_H, WIN_W, 900)
    boxes = square_boxes(2 * P, WIN_H, WIN_W, 6, 120, 901)
    coords, valid = O.expand_boxes(boxes, enlarge)
    assert valid.all()
    wf = np.arange(2 * P, dtype=np.int32) % PH
    wins = np.stack([O.crop_resize(frames[f], c, D) for c, f in zip(coords, wf)])
    k = distinct_first(wins, P)
    return frames, np.ascontiguousarray(coords[k]), np.ascontiguousarray(wf[k]), wins[k]


@functools.lru_cache(None)
def det32_templates():
    """32 x 32 templates from the reference's class crops (calculateMeanMasks at D = 32)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "det_crops.npz"))
    pix, shapes, off = g["pixels"], g["shapes"], g["type_offsets"]
    crops, pos = [], 0
    for h, w in shapes:
        crops.append(pix[pos:pos + h * w * 3].reshape(h, w, 3)); pos += h * w * 3
    red6, blue6, _ = _oracle().mean_masks([crops[off[t]:off[t + 1]] for t in range(6)], D=32)
    return red6, blue6


@functools.lru_cache(None)
def mask_patterns():
    """P pairwise different (red, blue) mask pairs of D = 32 windows, and the oracle's scores [P,2,6], id, hundredths, emit."""
    O = _oracle()
    frames = small_frames(PH, WIN_H, WIN_W, 902)
    boxes = square_boxes(3 * P, WIN_H, WIN_W, 6, 120, 903)
    coords, _ = O.expand_boxes(boxes, 1.15)
    wins = np.stack([O.crop_resize(frames[i % PH], c, 32) for i, c in enumerate(coords)])
    rb = np.stack([np.stack(O.color_masks(w)) for w in wins])
    k = distinct_first(rb, P)
    return wins[k], rb[k, 0].reshape(P, -1).copy(), rb[k, 1].reshape(P, -1).copy(), score_expect(rb[k, 0], rb[k, 1])


def score_expect(red, blue):
    O = _oracle()
    r6, b6 = det32_templates()
    n = len(red)
    sc = np.zeros((n, 2, 6), np.int32)
    for i in range(n):
        for k in range(6):
            sc[i, 0, k] = O.score_hundredths(red[i], r6[k])[0]
            sc[i, 1, k] = O.score_hundredths(blue[i], b6[k])[0]
    kr, kb = sc[:, 0].argmax(1), sc[:, 1].argmax(1)
    rv, bv = sc[np.arange(n), 0, kr], sc[np.arange(n), 1, kb]
    ids = np.where(rv > bv, kr + 1, kb + 1).astype(np.int32)
    hs = np.where(rv > bv, rv, bv).astype(np.int32)
    return sc, ids, hs, hs > 55


def palette_window(rng, D=32):
    """A D x D window of three random colours in random shares, with +-3 noise: windows of different palettes have unrelated
    H-S histograms."""
    cols = rng.integers(0, 256, (3, 3))
    pick = rng.choice(3, D * D, p=rng.dirichlet((1, 1, 1)))
    w = cols[pick] + rng.integers(-3, 4, (D * D, 3))
    return np.clip(w, 0, 255).astype(np.uint8).reshape(D, D, 3)


@functools.lru_cache(None)
def dedup_patterns():
    """PF frames of DEDUP_PER_FRAME D = 32 windows of their own palettes; window 1 is window 0 with 3 % of its pixels changed
    (merged by the histogram pass) and window 3 has window 2's corners moved by 1 px (merged by the coordinate pass).
    -> (windows [PF*8,...], coords, pass-1 survivors per frame, pass-2 survivors per frame)."""
    O = _oracle()
    rng = np.random.default_rng(905)
    wins, coords, s1, s2 = [], [], [], []
    for k in range(PF):
        w = np.stack([palette_window(rng) for _ in range(DEDUP_PER_FRAME)])
        ch = rng.random((32, 32)) < 0.03
        w[1] = np.where(ch[..., None], w[0] ^ 0x40, w[0])
        xy = rng.integers(0, 1200, (DEDUP_PER_FRAME, 2))
        c = np.concatenate([xy, xy + rng.integers(20, 200, (DEDUP_PER_FRAME, 1))], 1).astype(np.int32)
        c[3] = c[2] + 1
        w1, c1 = O.dedup(w, c, False, 0.85)
        w2, c2 = O.dedup(w1, c1, True, 0.95)
        wins.append(w); coords.append(c); s1.append((w1, c1)); s2.append((w2, c2))
    return np.concatenate(wins), np.concatenate(coords), s1, s2


def chain_pattern_boxes(mode, batch):
    return np.stack([square_boxes(CH_BOXES, CH_H, CH_W, 4, 30, 2000 + 1000 * batch + k + (500 if mode == "rec" else 0)) for k in range(PF)])


@functools.lru_cache(None)
def chain_patterns(mode, batch):
    """PF frames 64 x 48 with CH_BOXES square boxes each -> (frames [PF,48,64,3], boxes [PF,8,4])."""
    frames = small_frames(PF, CH_H, CH_W, 3000 + 10 * batch + (5 if mode == "rec" else 0))
    return frames, chain_pattern_boxes(mode, batch)


@functools.lru_cache(None)
def rec_chain_model():
    """(W, b) under which the recognition chain's survivors of both batches get every label, each threshold in a gap of the
    logits, and every survivor clear of the decision by more than the HOG tolerance; per (batch, pattern) the survivors."""
    O = _oracle()
    surv = {(bt, k): oracle_rec_frame(O, chain_patterns("rec", bt)[0][k], chain_patterns("rec", bt)[1][k]) for bt in (0, 1) for k in range(PF)}
    hog = np.concatenate([h for _, h in surv.values() if len(h)])
    Wl = np.random.default_rng(7321).standard_normal((324, 6))
    b = gap_bias(hog, Wl)
    return Wl, b, surv, hog


@functools.lru_cache(None)
def host_patterns():
    """PH full-size frames and HOST_BOXES synthetic boxes each (the bench's box model)."""
    import tsd_b200
    frames = tsd_b200.synth.make_frames(PH, HOST_H, HOST_W, seed=tsd_b200.synth.FRAME_SEED + 950)
    boxes, off = tsd_b200.synth.make_boxes(PH, HOST_BOXES, seed=tsd_b200.synth.BOX_SEED + 950)
    return frames, boxes.reshape(PH, HOST_BOXES, 4)


def staged_sectors(boxes, H, W, D=25, enlarge=1.30):
    """Bytes one frame's candidate ROIs make tsd_detect_frames stage: stage_mark's rows and 32-byte sectors, restated
    (test_gpu_layouts.staged_bytes)."""
    O = _oracle()
    co, v = O.expand_boxes(boxes, enlarge)
    keys = []
    nsec = (3 * W + 31) // 32
    for c in co[v]:
        cx, cy = min(c[0], W), min(c[1], H)
        cw, ch = min(c[2], W) - cx, min(c[3], H) - cy
        if cw <= 0 or ch <= 0:
            continue
        s0, s1 = (3 * cx) >> 5, (3 * (cx + cw) - 1) >> 5
        if ch <= 2 * D:
            rows = np.arange(cy, cy + ch)
        else:
            sy = np.floor(((np.arange(D) + 0.5) * (1.0 / (D / ch)) - 0.5).astype(np.float32)).astype(np.int64)
            rows = np.unique(cy + np.clip(np.concatenate([sy, sy + 1]), 0, ch - 1))
        keys.append((rows[:, None] * nsec + np.arange(s0, s1 + 1)[None, :]).ravel())
    if not keys:
        return 0
    sec = np.unique(np.concatenate(keys)) % nsec
    return int(np.sum(np.minimum(32, 3 * W - 32 * sec) & ~15))


@functools.lru_cache(None)
def limit_frames():
    """The last len(LIM_COUNTS) frames of a frame-limit batch (8 x 8) and their boxes: noise, except frame 2, whose left half is
    one colour with at least 17 of its boxes inside it (flat windows)."""
    O = _oracle()
    rng = np.random.default_rng(4242)
    fr = rng.integers(0, 256, (len(LIM_COUNTS), LIM_H, LIM_W, 3), dtype=np.uint8)
    fr[2, :, :4] = (40, 60, 200)
    cand = np.array([(x, y, s, s) for s in range(1, 9) for x in range(0, 9 - s) for y in range(0, 9 - s)], np.int32)
    co, _ = O.expand_boxes(cand, 1.30)
    flat = cand[np.minimum(co[:, 2], LIM_W) <= 4]
    other = cand[np.minimum(co[:, 2], LIM_W) > 4]
    boxes = []
    for f, n in enumerate(LIM_COUNTS):
        if f == 2:
            b = np.concatenate([flat[rng.integers(0, len(flat), 24)], other[rng.integers(0, len(other), n - 24)]])
            b = b[rng.permutation(n)]
        else:
            b = cand[rng.integers(0, len(cand), n)]
        boxes.append(b)
    return fr, boxes


@functools.lru_cache(None)
def limit_windows():
    """Per last frame: (windows D = 25, coords) as K1 + K2 make them."""
    O = _oracle()
    fr, boxes = limit_frames()
    out = []
    for f, b in enumerate(boxes):
        c, v = O.expand_boxes(b, 1.30)
        c = c[v]
        out.append((np.stack([O.crop_resize(fr[f], cc, 25) for cc in c]), c))
    return out


# ---- the cases and the buffers each must put past 2^32 bytes -------------------------------------------------------------
def chain_slot1_end(mode):
    """Bytes from the start of the windows / entries scratch to the end of the second scratch slot's windows."""
    O = _oracle()
    D = 25 if mode == "det" else 32
    en = 1.30 if mode == "det" else 1.15
    nb = CH_F[mode] * CH_BOXES
    slot_cap = (((nb + 3) & ~3) + 63) & ~63
    passing = 0
    for bt in (0, 1):
        per = [int(O.expand_boxes(b, en)[1].sum()) for b in chain_patterns(mode, bt)[1]]
        passing = max(passing, sum(per[f % PF] for f in range(CH_F[mode])))
    return {"windows": (slot_cap + passing) * win_stride(D * D), "entries": (slot_cap + passing) * ent_stride(D * D) * 4}


def case_buffers():
    """case -> {buffer: bytes}, and case -> (pattern period in items, {buffer: bytes per item})."""
    npx32, npx25 = 1024, 625
    return {
        "recognize": ({"input": N_GREY * 3072, "grey": N_GREY * 1024, "hog": N_GREY * 324 * 4}, (P, {"input": 3072, "grey": 1024, "hog": 1296})),
        "hog": ({"grey": N_GREY * 1024, "descriptors": N_GREY * 1296}, (P, {"grey": 1024, "descriptors": 1296})),
        "lda": ({"X": N_LDA * 324 * 4}, (P, {"X": 1296})),
        "knn": ({"X": N_KNN * KNN_NFEAT * 4}, (P, {"X": KNN_NFEAT * 4})),
        "crop_resize": ({"windows": N_WIN32 * 3072}, (P, {"windows": 3072})),
        "windows": ({"windows": WIN_FRAMES * P * 3072}, (P, {"windows": 3072})),
        "hist": ({"histograms": N_HIST * 3000 * 4}, (P, {"histograms": 12000})),
        "color_masks": ({"input": N_WIN32 * 3072}, (P, {"input": 3072})),
        "score": ({"input": N_WIN32 * 3072}, (P, {"input": 3072})),
        "score_masks": ({"red": N_GREY * npx32, "blue": N_GREY * npx32}, (P, {"red": 1024, "blue": 1024})),
        "dedup": ({"internal windows": N_DEDUP * win_stride(npx32), "entries": N_DEDUP * ent_stride(npx32) * 4,
                   "packed survivors": N_DEDUP // (PF * DEDUP_PER_FRAME) * sum(len(c) for _, c in dedup_patterns()[2]) * 3072},
                  (PF * DEDUP_PER_FRAME, {"internal windows": win_stride(npx32), "entries": ent_stride(npx32) * 4})),
        "mean_windows": ({"input": N_WIN32 * 3072}, (P, {"input": 3072})),
        "bgr2hsv": ({"input": NPX * 3, "output": NPX * 3}, (PX, {"input": 3, "output": 3})),
        "bgr2gray": ({"input": NPX * 3, "output": NPX}, (PX, {"input": 3, "output": 1})),
        "preprocess": ({"input": N_PRE * HOST_H * HOST_W * 3, "output": N_PRE * HOST_H * HOST_W},
                       (PH, {"input": HOST_H * HOST_W * 3, "output": HOST_H * HOST_W})),
        "host_routes": ({"frames": HOST_F * HOST_H * HOST_W * 3}, (PH, {"frames": HOST_H * HOST_W * 3})),
        "chain_det": (chain_slot1_end("det"), (PF * CH_BOXES, {"windows": win_stride(npx25), "entries": ent_stride(npx25) * 4})),
        "chain_rec": (chain_slot1_end("rec"), (PF * CH_BOXES, {"windows": win_stride(npx32), "entries": ent_stride(npx32) * 4})),
    }


# ---- CPU: the cases reach their sizes and regimes -------------------------------------------------------------------------
def test_large_cases_reach_their_sizes(oracle):
    src = _src("tsd_kernels.cuh")
    assert "inline int win_stride(int npx, int C) { return (npx * C + 15) & ~15; }" in src
    assert "inline int ent_stride(int npx) { return (npx + 3) & ~3; }" in src
    for p in (P, PF, PH, PX):
        assert p % 2 == 1 and is_prime(p), p
    for case, (bufs, (period, item)) in case_buffers().items():
        for name, nbytes in bufs.items():
            assert nbytes > 1 << 32, (case, name, nbytes)
        for name, s in item.items():                                          # a wrap never lands on the same pattern
            for k in (31, 32):
                if (1 << k) % s == 0:
                    assert ((1 << k) // s) % period != 0, (case, name, k)
    # every chain box passes K1 with a non-empty crop (the slot sizes above count only those)
    for mode, en in (("det", 1.30), ("rec", 1.15)):
        for bt in (0, 1):
            fr, bx = chain_patterns(mode, bt)
            for b in bx:
                c, v = oracle.expand_boxes(b, en)
                assert v.all() and np.all(np.minimum(c[:, 2], CH_W) > c[:, 0]) and np.all(np.minimum(c[:, 3], CH_H) > c[:, 1])
            assert len(distinct_first(fr, PF)) == PF
    # patterns pairwise different
    wins, grey, hog, W, b, lab = rec_patterns()
    assert len(set(lab.tolist())) == 7
    _, lab_b = oracle.lda_predict(hog, W, b, 0.5)
    assert np.array_equal(lab, lab_b)
    Wl, bl, surv, rhog = rec_chain_model()
    z, rl = oracle.lda_predict(rhog, Wl, bl, 0.5)
    assert set(rl.tolist()) == set(range(7)) and decision_margin(z, rhog, Wl).min() > 1
    _, _, s1, s2 = dedup_patterns()
    assert [len(c) for _, c in s1] == [DEDUP_PER_FRAME - 1] * PF and max(len(c) for _, c in s2) == DEDUP_PER_FRAME - 2


def test_frame_limit_batch_reaches_every_work_list(oracle):
    """The last frames of the frame-limit batch: two on the tiny-frame list (2 and 24 windows), one of 25..128 windows with more
    than kGramMaxBig flat rows (left to k5_pairs), one of more than kGramBM windows (k5_gram_big)."""
    tiny, big, bm = k5_constant("kGramTinyMax"), k5_constant("kGramMaxBig"), k5_constant("kGramBM")
    assert "constexpr int kMaxBatchFrames = 1 << 23;" in _src("tsd_k5.cuh") and LIMIT == 1 << 23
    assert (LIMIT - 1) << 8 < 1 << 31 <= LIMIT << 8
    wins = [w for w, _ in limit_windows()]
    n = [len(w) for w in wins]
    assert n == list(LIM_COUNTS)                                              # square boxes inside the frame: all pass K1
    assert 2 <= n[0] <= tiny and n[1] == tiny
    flat = int(np.sum([np.all(w == w[:1, :1]) for w in wins[2]]))
    assert tiny < n[2] <= bm and flat > big, (n[2], flat)
    assert n[3] > bm


# ---- GPU helpers -------------------------------------------------------------------------------------------------------------
_HELD = [0.0]                                # device bytes the library's memory pool keeps from earlier cases of this process


def room(device_gb, host_gb=0.0, lib_gb=None):
    """Skip unless the device (counting what the pool already holds) and the host have the memory a case needs."""
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info()[0] / GB
    if free + _HELD[0] < device_gb:
        pytest.skip("needs %.1f GB of device memory, %.1f GB free" % (device_gb, free + _HELD[0]))
    if host_gb:
        avail = 0.0
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024 / GB
        if avail < host_gb:
            pytest.skip("needs %.1f GB of host memory, %.1f GB available" % (host_gb, avail))
    _HELD[0] = max(_HELD[0], device_gb if lib_gb is None else lib_gb)


def _A():
    from tsd_b200 import _capi
    return _capi


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", 0))


def dev_tile(pat, n):
    """[n, ...] on the device: item i = pat[i % len(pat)] (pat numpy or a device tensor)."""
    import torch
    t = pat if isinstance(pat, torch.Tensor) else dev(pat)
    reps = -(-n // len(t))
    return t.repeat((reps,) + (1,) * (t.dim() - 1))[:n]


def host_tile(pat, n):
    """[n, ...] in host memory: item i = pat[i % len(pat)], written 256 MB at a time (mode="wrap": np.take does not buffer)."""
    out = np.empty((n,) + pat.shape[1:], pat.dtype)
    step = max(1, (1 << 28) // max(1, pat[:1].nbytes))
    for a in range(0, n, step):
        np.take(pat, np.arange(a, min(a + step, n)), axis=0, out=out[a:a + step], mode="wrap")
    return out


def periodic_bad(got, exp, differ=None, chunk=1 << 28):
    """Up to 10 indices i where got[i] differs from exp[i % len(exp)] (both numpy, or both device tensors).
    differ(a, b) -> elementwise bool; default !=."""
    torch_ = not isinstance(got, np.ndarray)
    n, p = len(got), len(exp)
    item = max(1, int(np.prod(got.shape[1:])) * (got.element_size() if torch_ else got.itemsize))
    step = p * max(1, chunk // (p * item))
    reps = -(-min(step, n) // p)
    tiled = exp.repeat((reps,) + (1,) * (exp.dim() - 1)) if torch_ else np.tile(exp, (reps,) + (1,) * (exp.ndim - 1))
    out = []
    for a in range(0, n, step):
        blk = got[a:a + step]
        e = tiled[:len(blk)]
        d = differ(blk, e) if differ else blk != e
        d = d.reshape(len(blk), -1).any(1)
        idx = d.nonzero().flatten()[:10].tolist() if torch_ else np.flatnonzero(d)[:10].tolist()
        out += [a + i for i in idx]
        if len(out) >= 10:
            break
    return out[:10]


def rel_differ(rel, floor):
    return lambda g, e: (g - e).abs() > rel * e.abs().clamp_min(floor)


def records(det):
    return np.stack([det[k] for k in ("frame", "x1", "y1", "x2", "y2", "id", "hundredths")], 1) if len(det) else np.zeros((0, 7), np.int64)


def tile_records(per, nframes, f_of=lambda f: f):
    """Expected records of nframes frames, frame f carrying pattern f % len(per): per = list of int arrays [m, 6] (no frame)."""
    cnt = np.array([len(r) for r in per], np.int64)
    flat = np.concatenate([np.asarray(r, np.int64).reshape(-1, 6) for r in per])
    starts = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    k = np.arange(nframes) % len(per)
    c = cnt[k]
    fr = np.repeat(np.arange(nframes), c)
    pos = np.arange(int(c.sum())) - np.repeat(np.cumsum(c) - c, c)
    return np.concatenate([f_of(fr)[:, None], flat[np.repeat(starts[k], c) + pos]], 1)


def det_pattern_records(O, frames, boxes, red6, blue6):
    per, counts = [], []
    for f in range(len(frames)):
        o = O.detect_frame(frames[f], boxes[f], red6, blue6)
        per.append(np.concatenate([o["coords"], o["ids"][:, None], o["hundredths"][:, None]], 1) if len(o["ids"]) else np.zeros((0, 6), np.int64))
        counts.append(o["stage_counts"].astype(np.int64))
    return per, np.array(counts)


def pattern_counts(counts, nframes):
    return (counts[np.arange(nframes) % len(counts)]).sum(0).tolist()


# ---- GPU: stage entry points -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_recognize_past_4gib(tsd, oracle):
    """tsd_recognize on 2^22 + 4 099 windows: input 12.9 GB, grey 4.3 GB, HOG 5.4 GB."""
    wins, _, _, W, b, lab = rec_patterns()
    room(23.0, host_gb=14.5)
    x = host_tile(wins, N_GREY)
    with tsd.Context(0, "rec") as ctx:
        ctx.set_lda(W, b)
        got = ctx.recognize_windows(x, 0.5)
    del x
    bad = periodic_bad(got, lab)
    assert not bad, [(i, int(got[i]), int(lab[i % P])) for i in bad]


@pytest.mark.gpu
def test_hog_past_4gib(tsd, oracle):
    """tsd_hog (device pointers) on 2^22 + 4 099 grey windows: grey 4.3 GB, descriptors 5.4 GB."""
    import torch
    _, grey, hog, _, _, _ = rec_patterns()
    room(11.0)
    A = _A()
    g = dev_tile(grey, N_GREY)
    out = torch.empty((N_GREY, 324), dtype=torch.float32, device="cuda")
    with tsd.Context(0, "rec") as ctx:
        A.check(ctx._L.tsd_hog(ctx._h, A.ptr(g.data_ptr()), N_GREY, A.ptr(out.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    del g
    bad = periodic_bad(out, dev(hog), rel_differ(1e-4, 1e-2))
    assert not bad, bad


@pytest.mark.gpu
def test_lda_past_4gib(tsd, oracle):
    """tsd_lda_predict (324 features, logits on, device pointers) on 3 400 000 rows: X 4.4 GB."""
    import torch
    _, _, hog, W, b, lab = rec_patterns()
    z, olab = oracle.lda_predict(hog, W, b, 0.5)
    assert np.array_equal(olab, lab)
    room(6.0)
    A = _A()
    X = dev_tile(hog, N_LDA)
    lg = torch.empty((N_LDA, 6), dtype=torch.float64, device="cuda")
    lb = torch.empty(N_LDA, dtype=torch.int32, device="cuda")
    with tsd.Context(0, "rec") as ctx:
        ctx.set_lda(W, b)
        A.check(ctx._L.tsd_lda_predict(ctx._h, A.ptr(X.data_ptr()), N_LDA, 0.5, A.ptr(lg.data_ptr()), A.ptr(lb.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    del X
    tol = 1e-12 * float((np.abs(hog.astype(np.float64)) @ np.abs(W) + np.abs(b)).max())
    bad = periodic_bad(lg, dev(z), lambda g, e: (g - e).abs() > tol)
    assert not bad, bad
    bad = periodic_bad(lb, dev(lab))
    assert not bad, bad


@pytest.mark.gpu
def test_knn_past_4gib(tsd, oracle):
    """tsd_knn_predict (1 500 features, 97 training rows, device pointers) on 720 000 rows: X 4.3 GB."""
    import torch
    rng = np.random.default_rng(61)
    xbar = rng.standard_normal(KNN_NFEAT)
    S = rng.standard_normal((KNN_NFEAT, 6)) / np.sqrt(KNN_NFEAT)
    Zt = rng.standard_normal((KNN_NTRAIN, 6))
    yt = rng.integers(0, 7, KNN_NTRAIN).astype(np.int32)
    Xp = (xbar + rng.standard_normal((P, KNN_NFEAT))).astype(np.float32)
    oZ, olab = oracle.knn_predict(Xp, xbar, S, Zt, yt, 4)
    assert len(set(olab.tolist())) > 3
    room(5.5)
    A = _A()
    X = dev_tile(Xp, N_KNN)
    Z = torch.empty((N_KNN, 6), dtype=torch.float64, device="cuda")
    lb = torch.empty(N_KNN, dtype=torch.int32, device="cuda")
    with tsd.Context(0, "rec") as ctx:
        ctx.set_knn(xbar, S, Zt, yt, 4)
        A.check(ctx._L.tsd_knn_predict(ctx._h, A.ptr(X.data_ptr()), N_KNN, A.ptr(Z.data_ptr()), A.ptr(lb.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    del X
    assert not periodic_bad(Z, dev(oZ), lambda g, e: (g - e).abs() > 1e-9)
    bad = periodic_bad(lb, dev(olab))
    assert not bad, bad


@pytest.mark.gpu
def test_crop_resize_and_windows_past_4gib(tsd, oracle):
    """tsd_crop_resize (D = 32, BGR, device pointers) of 1 420 000 windows and tsd_windows (host pointers) of 347 x 4 099: the
    windows reach 4.4 GB."""
    import torch
    A = _A()
    frames, coords, wf, exp = crop_patterns(32, 1.15)
    room(6.0, host_gb=11.0)
    d_frames = dev(frames)
    co, fr = dev_tile(coords, N_WIN32), dev_tile(wf, N_WIN32)
    out = torch.empty((N_WIN32, 32, 32, 3), dtype=torch.uint8, device="cuda")
    with tsd.Context(0, "rec") as ctx:
        A.check(ctx._L.tsd_crop_resize(ctx._h, A.ptr(d_frames.data_ptr()), PH, WIN_H, WIN_W, WIN_W * 3, WIN_H * WIN_W * 3, 3,
                                       A.ptr(co.data_ptr()), A.ptr(fr.data_ptr()), N_WIN32, 32, A.ptr(out.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    bad = periodic_bad(out, dev(exp))
    assert not bad, bad
    del out, co, fr, d_frames
    # tsd_windows: every frame the same 256 x 256 frame with the P pattern boxes
    one = np.ascontiguousarray(np.broadcast_to(frames[:1], (WIN_FRAMES, WIN_H, WIN_W, 3)))
    boxes = square_boxes(2 * P, WIN_H, WIN_W, 6, 120, 901)
    bk = boxes[distinct_first(np.stack([oracle.crop_resize(frames[0], c, 32) for c in oracle.expand_boxes(boxes, 1.15)[0]]), P)]
    wexp = np.stack([oracle.crop_resize(frames[0], c, 32) for c in oracle.expand_boxes(bk, 1.15)[0]])
    off = (np.arange(WIN_FRAMES + 1) * P).astype(np.int32)
    with tsd.Context(0, "rec") as ctx:
        wins, wco, woff = ctx.windows(one, host_tile(bk, WIN_FRAMES * P), off)
    assert np.array_equal(woff, off)
    assert not periodic_bad(wco, oracle.expand_boxes(bk, 1.15)[0])
    bad = periodic_bad(wins, wexp)
    assert not bad, bad


@pytest.mark.gpu
def test_hist_past_4gib(tsd, oracle):
    """tsd_hist (D = 25, device pointers) on 360 000 windows: histograms 4.3 GB."""
    import torch
    A = _A()
    _, _, _, w25 = crop_patterns(25, 1.30)
    exp = np.stack([oracle.hist_normalized(w) for w in w25])
    room(6.0)
    x = dev_tile(w25, N_HIST)
    out = torch.empty((N_HIST, 50, 60), dtype=torch.float32, device="cuda")
    with tsd.Context(0, "det") as ctx:
        A.check(ctx._L.tsd_hist(ctx._h, A.ptr(x.data_ptr()), N_HIST, 25, A.ptr(out.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    bad = periodic_bad(out, dev(exp))
    assert not bad, bad


@pytest.mark.gpu
def test_color_masks_and_score_past_4gib(tsd, oracle):
    """tsd_color_masks (device pointers) and tsd_score (host pointers) at D = 32 on 1 420 000 windows: input 4.4 GB."""
    import torch
    A = _A()
    wins, red, blue, (_, ids, hs, em) = mask_patterns()
    room(8.0, host_gb=6.0)
    x = dev_tile(wins, N_WIN32)
    r = torch.empty((N_WIN32, 1024), dtype=torch.uint8, device="cuda")
    bl = torch.empty_like(r)
    with tsd.Context(0, "rec") as ctx:
        A.check(ctx._L.tsd_color_masks(ctx._h, A.ptr(x.data_ptr()), N_WIN32, 32, A.ptr(r.data_ptr()), A.ptr(bl.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    assert not periodic_bad(r, dev(red))
    assert not periodic_bad(bl, dev(blue))
    del x, r, bl
    hx = host_tile(wins, N_WIN32)
    with tsd.Context(0, "rec") as ctx:
        ctx.set_templates(*det32_templates())
        got = ctx.score_windows(hx)
    assert not periodic_bad(got["id"], ids)
    assert not periodic_bad(got["hundredths"], hs)
    assert not periodic_bad(got["emit"], em)


@pytest.mark.gpu
def test_score_masks_past_4gib(tsd, oracle):
    """tsd_score_masks (D = 32, device pointers) on 2^22 + 4 099 mask pairs: each mask array 4.3 GB."""
    import torch
    A = _A()
    _, red, blue, (sc, ids, hs, em) = mask_patterns()
    assert len(set(ids.tolist())) > 1 and len(set(hs.tolist())) > 10
    room(9.5)
    r, b = dev_tile(red, N_GREY), dev_tile(blue, N_GREY)
    o_sc = torch.empty((N_GREY, 2, 6), dtype=torch.int32, device="cuda")
    o_id, o_h = torch.empty(N_GREY, dtype=torch.int32, device="cuda"), torch.empty(N_GREY, dtype=torch.int32, device="cuda")
    o_em = torch.empty(N_GREY, dtype=torch.uint8, device="cuda")
    with tsd.Context(0, "rec") as ctx:
        ctx.set_templates(*det32_templates())
        A.check(ctx._L.tsd_score_masks(ctx._h, A.ptr(r.data_ptr()), A.ptr(b.data_ptr()), N_GREY, 32, A.ptr(o_sc.data_ptr()), A.ptr(o_id.data_ptr()),
                                       A.ptr(o_h.data_ptr()), A.ptr(o_em.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    del r, b
    for got, exp in ((o_sc, sc), (o_id, ids), (o_h, hs), (o_em, em.astype(np.uint8))):
        bad = periodic_bad(got, dev(exp))
        assert not bad, bad


def dedup_call(ctx, windows, coords, offsets, by_coords, tol):
    """tsd_dedup into preallocated outputs -> views (windows, coords, offsets) of the survivors (no host copy)."""
    A = _A()
    nf = len(offsets) - 1
    ow, oc = np.empty_like(windows), np.empty_like(coords)
    oo = np.zeros(nf + 1, np.int32); tot = C.c_int32()
    A.check(ctx._L.tsd_dedup(ctx._h, A.ptr(windows), A.ptr(coords), A.ptr(offsets), nf, 32, int(by_coords), tol, A.ptr(ow), A.ptr(oc),
                             A.ptr(oo), C.byref(tot), A.MEM_HOST))
    return ow[:tot.value], oc[:tot.value], oo


@pytest.mark.gpu
def test_dedup_past_4gib(tsd, oracle):
    """tsd_dedup (D = 32) by histograms then by coordinates on 205 000 frames x 8 windows: the internal windows reach 5.0 GB, the
    histogram entries 6.7 GB and the packed survivors of the first pass 4.4 GB."""
    wins, coords, s1, s2 = dedup_patterns()
    nf = N_DEDUP // DEDUP_PER_FRAME
    room(18.5, host_gb=15.0)
    x = host_tile(wins, N_DEDUP)
    c = host_tile(coords, N_DEDUP)
    off = (np.arange(nf + 1) * DEDUP_PER_FRAME).astype(np.int32)
    with tsd.Context(0, "rec") as ctx:
        w1, c1, o1 = dedup_call(ctx, x, c, off, False, 0.85)
        del x, c
        for got_w, got_c, got_o, exp in ((w1, c1, o1, s1),):
            cnt = np.array([len(cc) for _, cc in exp])
            assert np.array_equal(np.diff(got_o), cnt[np.arange(nf) % PF])
            assert not periodic_bad(got_c, np.concatenate([cc for _, cc in exp]))
            bad = periodic_bad(got_w, np.concatenate([ww for ww, _ in exp]))
            assert not bad, bad
        w2, c2, o2 = dedup_call(ctx, w1, c1, o1, True, 0.95)
    cnt = np.array([len(cc) for _, cc in s2])
    assert np.array_equal(np.diff(o2), cnt[np.arange(nf) % PF])
    assert not periodic_bad(c2, np.concatenate([cc for _, cc in s2]))
    assert not periodic_bad(w2, np.concatenate([ww for ww, _ in s2]))


def mean_expected(wins, a, b):
    """calculateMeanMasks' running average of windows a .. b-1 (item i = wins[i % P]).  avg_rne is monotone in the running
    mean, so runs from all-0 and all-255 over the last windows that meet give the exact result whatever came before."""
    def run(m, lo):
        for i in range(lo, b):
            s = wins[i % len(wins)].astype(np.int32) + m
            m = (s >> 1) + ((s & 1) & ((s >> 1) & 1))
        return m
    lo = max(a + 1, b - 4 * P)
    first = wins[a % len(wins)].astype(np.int32)
    if lo == a + 1:
        return run(first, lo).astype(np.uint8)
    m0, m1 = run(np.zeros_like(first), lo), run(np.full_like(first, 255), lo)
    assert np.array_equal(m0, m1), "the sandwich did not close"
    return m0.astype(np.uint8)


@pytest.mark.gpu
def test_mean_windows_past_4gib(tsd, oracle):
    """tsd_mean_windows (D = 32) of 1 420 000 windows in 3 groups; the second spans 2 GiB and 4 GiB, the third lies past 4 GiB."""
    _, _, _, wins = crop_patterns(32, 1.15)
    g = np.array(MEAN_GROUPS, np.int32)
    assert int(g[1]) * 3072 < 1 << 31 < 1 << 32 < int(g[2]) * 3072 < N_WIN32 * 3072
    exp = np.stack([mean_expected(wins, a, b) for a, b in zip(g[:-1], g[1:])])
    room(5.0, host_gb=5.5)
    x = host_tile(wins, N_WIN32)
    with tsd.Context(0, "rec") as ctx:
        got = ctx.mean_windows(x, g)
    assert np.array_equal(got, exp), [int(np.sum(got[k] != exp[k])) for k in range(3)]


@pytest.mark.gpu
def test_bgr2hsv_and_bgr2gray_past_4gib(tsd, oracle):
    """tsd_bgr2hsv and tsd_bgr2gray (device pointers) on 2^32 + 2^24 + 13 pixels: input 12.9 GB, outputs 12.9 and 4.3 GB."""
    import torch
    A = _A()
    base = np.random.default_rng(88).integers(0, 256, (PX, 3), dtype=np.uint8)
    ehsv, egray = oracle.bgr2hsv(base), oracle.bgr2gray(base)
    room(26.0)
    x = dev_tile(base, NPX)
    with tsd.Context(0, "det") as ctx:
        out = torch.empty((NPX, 3), dtype=torch.uint8, device="cuda")
        A.check(ctx._L.tsd_bgr2hsv(ctx._h, A.ptr(x.data_ptr()), NPX, A.ptr(out.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
        bad = periodic_bad(out, dev(ehsv))
        assert not bad, bad
        del out
        torch.cuda.empty_cache()
        g = torch.empty(NPX, dtype=torch.uint8, device="cuda")
        A.check(ctx._L.tsd_bgr2gray(ctx._h, A.ptr(x.data_ptr()), NPX, A.ptr(g.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    bad = periodic_bad(g, dev(egray))
    assert not bad, bad


@pytest.mark.gpu
def test_preprocess_past_4gib(tsd, oracle):
    """tsd_preprocess (device pointers) on 3 960 frames of 1360 x 800: input 12.9 GB, grey and output 4.3 GB."""
    import torch
    A = _A()
    frames = host_patterns()[0]
    exp = np.stack([oracle.preprocess(f) for f in frames])
    room(22.0)
    x = dev_tile(frames, N_PRE)
    out = torch.empty((N_PRE, HOST_H, HOST_W), dtype=torch.uint8, device="cuda")
    with tsd.Context(0, "det") as ctx:
        table = oracle.gamma_table(2)
        A.check(ctx._L.tsd_set_gamma_table(ctx._h, A.ptr(table)))
        A.check(ctx._L.tsd_preprocess(ctx._h, A.ptr(x.data_ptr()), N_PRE, HOST_H, HOST_W, HOST_W * 3, HOST_H * HOST_W * 3, 2.0, 8, 8,
                                      A.ptr(out.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
    del x
    bad = periodic_bad(out, dev(exp))
    assert not bad, bad


# ---- GPU: the chain ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("det", "rec"))
def test_chain_second_slot_past_4gib(tsd, oracle, monkeypatch, templates, mode):
    """Two overlapped tsd_enqueue_frames batches (device pointers) of 64 x 48 frames x 8 square boxes with different contents:
    more than 65 535 frames a batch, and the second scratch slot's windows and entries past 4 GiB (detection D = 25: 1.2 M boxes a
    batch; recognition D = 32: 800 000).  Batch 1 fetched with fetch_previous, batch 2 with fetch_detections."""
    A = _A()
    nf = CH_F[mode]
    nb = nf * CH_BOXES
    exp = []
    if mode == "det":
        for bt in (0, 1):
            fr, bx = chain_patterns(mode, bt)
            per, cnt = det_pattern_records(oracle, fr, bx, *templates)
            exp.append((tile_records(per, nf), pattern_counts(cnt, nf)))
    else:
        Wl, bl, surv, _ = rec_chain_model()
        for bt in (0, 1):
            per, cnt = [], []
            for k in range(PF):
                c2, hog = surv[(bt, k)]
                lab = oracle.lda_predict(hog, Wl, bl, 0.5)[1] if len(c2) else np.zeros(0, np.int32)
                per.append(np.array([list(cc) + [int(l), 0] for cc, l in zip(c2, lab) if l != 0], np.int64).reshape(-1, 6))
                cnt.append([CH_BOXES, CH_BOXES, len(c2), int(np.sum(lab != 0))])
            exp.append((tile_records(per, nf), pattern_counts(np.array(cnt), nf)))
    room(22.0 if mode == "det" else 21.0)
    monkeypatch.delenv("TSD_OVERLAP", raising=False)
    with tsd.Context(0, mode) as ctx:
        if mode == "det":
            ctx.set_templates(*templates)
        else:
            ctx.set_lda(Wl, bl)
        run = A.RUN_DETECT if mode == "det" else A.RUN_RECOGNIZE
        keep = []
        for bt in (0, 1):
            fr, bx = chain_patterns(mode, bt)
            d_fr, d_bx = dev_tile(fr, nf), dev_tile(bx, nf).reshape(nb, 4)
            d_off = dev((np.arange(nf + 1) * CH_BOXES).astype(np.int32))
            keep.append((d_fr, d_bx, d_off))
            ctx.enqueue_frames(d_fr.data_ptr(), nf, CH_H, CH_W, d_bx.data_ptr(), d_off.data_ptr(), nb, mode=run, max_boxes_per_frame=CH_BOXES)
        got = [ctx.fetch_detections(nb, previous=True), ctx.fetch_detections(nb)]
    for bt in (0, 1):
        det, counts = got[bt]
        erec, ecounts = exp[bt]
        assert counts.tolist() == ecounts, (bt, counts.tolist(), ecounts)
        g = records(det)
        assert g.shape == erec.shape and np.array_equal(g, erec), (bt, g.shape, erec.shape)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ("staged", "staged_chunks", "gather", "pageable"))
def test_host_routes_past_4gib(tsd, oracle, monkeypatch, templates, route):
    """tsd_detect_frames on 1 400 frames of 1360 x 800 (4.6 GB) in host memory, 200 boxes each: page-locked and staged whole
    (the mirror exceeds 4 GiB) or in chunks (chunk sources past 4 GiB), page-locked and read by K2 over PCIe (TSD_STAGE=0), and
    pageable.  Records and stage counts equal the oracle's; the staged routes stage exactly stage_mark's bytes."""
    frames, boxes = host_patterns()
    per, cnt = det_pattern_records(oracle, frames, boxes, *templates)
    erec, ecounts = tile_records(per, HOST_F), pattern_counts(cnt, HOST_F)
    room(12.0, host_gb=7.0)
    env = {"staged": {"TSD_STAGE_CHUNK": "0"}, "staged_chunks": {}, "gather": {"TSD_STAGE": "0"}, "pageable": {}}[route]
    for k in ("TSD_STAGE", "TSD_STAGE_CHUNK", "TSD_CHUNK_FRAMES", "TSD_ZEROCOPY"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x = host_tile(frames, HOST_F)
    bx = host_tile(boxes, HOST_F).reshape(-1, 4)
    off = (np.arange(HOST_F + 1) * HOST_BOXES).astype(np.int32)
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(*templates)
        pinned = route != "pageable"
        if pinned:
            ctx.pin(x)
        try:
            ctx.stat_staged_bytes(reset=True)
            det, counts = ctx.detect_frames(x, bx, off)
            staged = ctx.stat_staged_bytes(reset=True)
        finally:
            if pinned:
                ctx.unpin(x)
    assert counts.tolist() == ecounts, (counts.tolist(), ecounts)
    g = records(det)
    assert g.shape == erec.shape and np.array_equal(g, erec), (g.shape, erec.shape)
    if route.startswith("staged"):
        per_frame = [staged_sectors(b, HOST_H, HOST_W) for b in boxes]
        assert staged == sum(per_frame[f % PH] for f in range(HOST_F)), staged
    else:
        assert staged == 0


# ---- GPU: the frame-count limit ------------------------------------------------------------------------------------------------
def limit_expected(oracle, templates, nframes):
    fr, boxes = limit_frames()
    k0 = nframes - len(LIM_COUNTS)
    recs, counts = [], np.zeros(4, np.int64)
    for j in range(len(LIM_COUNTS)):
        o = oracle.detect_frame(fr[j], boxes[j], *templates)
        counts += o["stage_counts"]
        recs += [[k0 + j] + list(map(int, c)) + [int(i), int(h)] for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    return np.array(recs, np.int64).reshape(-1, 7), counts.tolist()


@pytest.mark.gpu
def test_dedup_at_the_frame_limit(tsd, oracle):
    """tsd_dedup, both passes, on 2^23 - 1 frames, all empty but the last four (2 and 24 windows: tiny-frame list; 64 with more
    than kGramMaxBig flat windows: k5_pairs; 200: k5_gram_big).  2^23 frames are refused with TSD_E_INVALID."""
    A = _A()
    lw = limit_windows()
    nf = LIMIT - 1
    counts = np.zeros(nf, np.int32)
    counts[-len(LIM_COUNTS):] = [len(c) for _, c in lw]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    wins = np.concatenate([w for w, _ in lw]); co = np.concatenate([c for _, c in lw])
    e1 = [oracle.dedup(w, c, False, 0.85) for w, c in lw]
    e2 = [oracle.dedup(w, c, True, 0.95) for w, c in e1]
    room(4.0, host_gb=1.0)
    with tsd.Context(0, "det") as ctx:
        for by, tol, exp in ((False, 0.85, e1), (True, 0.95, e2)):
            ow, oc, oo = ctx.dedup(wins, co, off, by, tol)
            n = np.diff(oo)
            assert not n[:-len(LIM_COUNTS)].any() and n[-len(LIM_COUNTS):].tolist() == [len(c) for _, c in exp], (by, n[-len(LIM_COUNTS):])
            assert np.array_equal(ow, np.concatenate([w for w, _ in exp])) and np.array_equal(oc, np.concatenate([c for _, c in exp])), by
            wins, co, off = ow, oc, oo
        big = np.concatenate([off, off[-1:]]).astype(np.int32)
        out_off = np.zeros(LIMIT + 1, np.int32); tot = C.c_int32(-7)
        rc = ctx._L.tsd_dedup(ctx._h, A.ptr(wins), A.ptr(co), A.ptr(big), LIMIT, 25, 0, 0.85, A.ptr(np.empty_like(wins)), A.ptr(np.empty_like(co)),
                              A.ptr(out_off), C.byref(tot), A.MEM_HOST)
        assert rc == E_INVALID and b"2^23" in ctx._L.tsd_last_error() and tot.value == -7
        ctx.synchronize()


@pytest.mark.gpu
def test_enqueue_at_the_frame_limit(tsd, oracle, templates):
    """tsd_enqueue_frames (D = 25, device pointers) on 2^23 - 1 frames of 8 x 8 (1.6 GB), all without boxes but the last four
    (see test_dedup_at_the_frame_limit): records and stage counts equal the oracle's.  2^23 frames are refused with
    TSD_E_INVALID before any device work."""
    A = _A()
    fr, boxes = limit_frames()
    nf = LIMIT - 1
    erec, ecounts = limit_expected(oracle, templates, nf)
    room(6.0)
    fb = LIM_H * LIM_W * 3
    import torch
    d_fr = torch.zeros(LIMIT * fb, dtype=torch.uint8, device="cuda")
    d_fr[(nf - len(LIM_COUNTS)) * fb:nf * fb] = dev(fr.reshape(-1))
    counts = np.zeros(LIMIT, np.int32)
    counts[nf - len(LIM_COUNTS):nf] = LIM_COUNTS
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    d_off = dev(off)
    bx = np.concatenate(boxes).astype(np.int32)
    d_bx = dev(bx)
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(*templates)
        ctx.enqueue_frames(d_fr.data_ptr(), nf, LIM_H, LIM_W, d_bx.data_ptr(), d_off.data_ptr(), len(bx), max_boxes_per_frame=max(LIM_COUNTS))
        det, cnt = ctx.fetch_detections(len(bx))
        assert cnt.tolist() == ecounts, (cnt.tolist(), ecounts)
        assert np.array_equal(records(det), erec)
        launches = ctx.launch_count
        rc = ctx._L.tsd_enqueue_frames(ctx._h, A.RUN_DETECT, A.ptr(d_fr.data_ptr()), LIMIT, LIM_H, LIM_W, LIM_W * 3, fb, A.ptr(d_bx.data_ptr()),
                                       A.ptr(d_off.data_ptr()), len(bx), max(LIM_COUNTS))
        assert rc == E_INVALID and b"2^23" in ctx._L.tsd_last_error()
        assert ctx.launch_count == launches
        det2, cnt2 = ctx.fetch_detections(len(bx))                 # the refused call left the last batch in place
        assert cnt2.tolist() == ecounts and np.array_equal(records(det2), erec)
