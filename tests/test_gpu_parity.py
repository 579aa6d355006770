"""GPU (-m gpu): the CUDA path, called through the C ABI, against the oracle and the reference-generated goldens.
Bit-exact for every integer / byte / index artefact; HOG within 1e-4 relative; LDA logits within 1e-9."""
import numpy as np
import pytest

from conftest import STORED

pytestmark = pytest.mark.gpu


# ---- K1 -------------------------------------------------------------------------------------------------------------
def test_k1_expand(ctx_det, ctx_rec, oracle, det_frames):
    rng = np.random.default_rng(11)
    n = 20000
    w = rng.integers(1, 400, n); h = np.maximum(1, np.rint(w / rng.uniform(0.6, 1.6, n))).astype(np.int64)
    boxes = np.stack([rng.integers(0, 3840, n), rng.integers(0, 2160, n), w, h], 1).astype(np.int32)
    boxes[:50, 3] = 0                                                    # h == 0 -> inf/nan ratio -> rejected
    for ctx, p in ((ctx_det, 1.30), (ctx_rec, 1.15)):
        c, v = ctx.expand_boxes(boxes)
        oc, ov = oracle.expand_boxes(boxes, p)
        assert np.array_equal(v, ov) and np.array_equal(c[v], oc[ov])
    for k in STORED:
        c, v = ctx_det.expand_boxes(det_frames[k + "_boxes"])
        assert np.array_equal(v, det_frames[k + "_valid"]) and np.array_equal(c[v], det_frames[k + "_coords"][v])
    c, v = ctx_det.expand_boxes(np.zeros((0, 4), np.int32))
    assert c.shape == (0, 4) and v.shape == (0,)


# ---- K2 -------------------------------------------------------------------------------------------------------------
def test_k2_resize_sweep(ctx_det, ctx_rec, oracle):
    """Size sweep incl. the same-size copy, the 2x AREA path, upscales, 1-px crops and frame-edge clipping."""
    rng = np.random.default_rng(5)
    frame = rng.integers(0, 256, (2, 420, 640, 3), dtype=np.uint8)
    for ctx, D in ((ctx_det, 25), (ctx_rec, 32)):
        coords, wf = [], []
        for h in list(range(1, 90)) + [2 * D, 2 * D + 1, 128, 257, 400]:
            for w in (1, 2, 3, D - 1, D, D + 1, 2 * D - 1, 2 * D, 2 * D + 1, 37, 100, 300, h):
                x0 = int(rng.integers(0, 640 - min(w, 600))); y0 = int(rng.integers(0, 420 - min(h, 400)))
                coords.append((x0, y0, x0 + w, y0 + h)); wf.append(int(rng.integers(0, 2)))
        coords += [(600, 400, 700, 480), (630, 0, 660, 30), (0, 410, 40, 450), (639, 419, 700, 500)]   # clipped by the frame
        wf += [0, 1, 0, 1]
        coords = np.array(coords, np.int32); wf = np.array(wf, np.int32)
        got = ctx.crop_resize(frame, coords, wf, D)
        for i, (c, f) in enumerate(zip(coords, wf)):
            assert np.array_equal(got[i], oracle.crop_resize(frame[f], c, D)), (D, c)
        # a frame whose rows are not 4-byte aligned (637 px = 1911 bytes): the aligned 32-bit tap loads of the general path do
        # not apply, every window takes the byte loads
        odd = np.ascontiguousarray(frame[:, :, :637])
        keep = np.flatnonzero(coords[:, 0] < 630)[::5]                       # (crops that start inside the narrower frame)
        got_odd = ctx.crop_resize(odd, coords[keep], wf[keep], D)
        for i, (c, f) in enumerate(zip(coords[keep], wf[keep])):
            assert np.array_equal(got_odd[i], oracle.crop_resize(odd[f], c, D)), (D, c, "odd width")
        gray = np.ascontiguousarray(frame[..., 1])
        got1 = ctx.crop_resize(gray, coords[::3], wf[::3], D)
        for i, (c, f) in enumerate(zip(coords[::3], wf[::3])):
            assert np.array_equal(got1[i], oracle.crop_resize(gray[f], c, D)), (D, c, "grey")


def test_k2_golden_frames(ctx_det, det_frames, frames3):
    for k in STORED:
        v = det_frames[k + "_valid"]
        got = ctx_det.crop_resize(frames3[k], det_frames[k + "_coords"][v])
        assert np.array_equal(got, det_frames[k + "_windows"])


def test_k1k2_windows_batch(ctx_det, det_frames, frames3, oracle, tsd):
    frames = np.stack([frames3[k] for k in STORED])
    boxes = [det_frames[k + "_boxes"] for k in STORED]
    off = np.concatenate([[0], np.cumsum([len(b) for b in boxes])]).astype(np.int32)
    wins, coords, woff = ctx_det.windows(frames, np.concatenate(boxes), off)
    exp_w = np.concatenate([det_frames[k + "_windows"] for k in STORED])
    exp_c = np.concatenate([det_frames[k + "_coords"][det_frames[k + "_valid"]] for k in STORED])
    assert np.array_equal(woff, np.concatenate([[0], np.cumsum([det_frames[k + "_valid"].sum() for k in STORED])]))
    assert np.array_equal(coords, exp_c) and np.array_equal(wins, exp_w)
    # a frame without boxes in the middle, and an empty batch of boxes
    off2 = np.array([0, len(boxes[0]), len(boxes[0]), len(boxes[0]) + len(boxes[2])], np.int32)
    w2, c2, wo2 = ctx_det.windows(frames, np.concatenate([boxes[0], boxes[2]]), off2)
    assert wo2[1] == wo2[2] and np.array_equal(w2[wo2[2]:], det_frames[STORED[2] + "_windows"])
    w3, c3, wo3 = ctx_det.windows(frames[:1], np.zeros((0, 4), np.int32), np.array([0, 0], np.int32))
    assert len(w3) == 0 and wo3.tolist() == [0, 0]


# ---- K3 -------------------------------------------------------------------------------------------------------------
def test_k3_exhaustive_colours(ctx_det, oracle):
    """All 2^24 BGR colours: HSV bytes and both masks bit-exact (SURVEY A.3)."""
    g, r = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    for b0 in range(0, 256, 32):
        img = np.stack([np.stack([np.full_like(g, b), g, r], -1) for b in range(b0, b0 + 32)])      # [32,256,256,3]
        assert np.array_equal(ctx_det.bgr2hsv(img), oracle.bgr2hsv(img))
        # masks kernel works on DxD windows: view the colours as 25x25 windows (pad the tail)
        flat = img.reshape(-1, 3)
        n = (len(flat) // 625) * 625
        wins = flat[:n].reshape(-1, 25, 25, 3)
        red, blue = ctx_det.color_masks(wins)
        ored, oblue = oracle.color_masks(wins)
        assert np.array_equal(red, ored) and np.array_equal(blue, oblue)
        tail = np.zeros((1, 25, 25, 3), np.uint8); tail.reshape(-1, 3)[:len(flat) - n] = flat[n:]
        red, blue = ctx_det.color_masks(tail)
        ored, oblue = oracle.color_masks(tail)
        assert np.array_equal(red, ored) and np.array_equal(blue, oblue)
        assert np.array_equal(ctx_det.bgr2gray(img), oracle.bgr2gray(img))


def test_k3_golden(ctx_det, det_frames):
    for k in STORED:
        wins = det_frames[k + "_p2_windows"]
        assert np.array_equal(ctx_det.bgr2hsv(wins), det_frames[k + "_hsv"])
        red, blue = ctx_det.color_masks(wins)
        assert np.array_equal(red, det_frames[k + "_red"]) and np.array_equal(blue, det_frames[k + "_blue"])


# ---- K4 -------------------------------------------------------------------------------------------------------------
def test_k4_scores_golden_and_random(ctx_det, oracle, det_frames, templates, tsd):
    red6, blue6 = templates
    for k in STORED:
        r = ctx_det.score_masks(det_frames[k + "_red"], det_frames[k + "_blue"])
        assert np.array_equal(r["scores"], np.rint(det_frames[k + "_scores"] * 100).astype(np.int32))
    rng = np.random.default_rng(2)
    n = 3000
    red = (rng.random((n, 25, 25)) < rng.random((n, 1, 1))).astype(np.uint8) * 255
    blue = (rng.random((n, 25, 25)) < rng.random((n, 1, 1))).astype(np.uint8) * 255
    red[0] = 0; blue[0] = 0; red[1] = 255; blue[1] = 255; red[2] = red6[2]; blue[2] = blue6[5]
    r = ctx_det.score_masks(red, blue)
    for i in range(n):
        for ci, (m, t6) in enumerate(((red[i], red6), (blue[i], blue6))):
            for ti in range(6):
                assert r["scores"][i, ci, ti] == oracle.score_hundredths(m, t6[ti])[0]
    # random templates (incl. degenerate ones with <= 6 pixels set), decision rule vs the oracle's window scorer
    with tsd.Context(device=0, flavour="det") as c2:
        t_r = (rng.random((6, 25, 25)) < np.array([0.0, 0.005, 0.01, 0.2, 0.5, 1.0])[:, None, None]).astype(np.uint8) * 255
        t_b = (rng.random((6, 25, 25)) < np.array([0.3, 0.3, 0.009, 0.0, 0.7, 0.1])[:, None, None]).astype(np.uint8) * 255
        c2.set_templates(t_r, t_b)
        wins = rng.integers(0, 256, (500, 25, 25, 3), dtype=np.uint8)
        wins[:250, :, :, 2] = 255; wins[:250, :, :, :2] //= 3                     # reddish
        wins[250:400, :, :, 0] = 250; wins[250:400, :, :, 1:] //= 3               # bluish
        mr, mb = c2.color_masks(wins)
        r = c2.score_masks(mr, mb)
        for i in range(len(wins)):
            ok, oid, oh = oracle.score_window(wins[i], t_r, t_b, 55)
            assert (bool(r["emit"][i]), int(r["id"][i]), int(r["hundredths"][i])) == (ok, oid, oh)


# ---- K5 -------------------------------------------------------------------------------------------------------------
def test_k5_hist(ctx_det, ctx_rec, oracle, det_frames):
    for k in STORED:
        got = ctx_det.hist(det_frames[k + "_windows"])
        assert np.array_equal(got, det_frames[k + "_hists"])
    rng = np.random.default_rng(9)
    w32 = rng.integers(0, 256, (40, 32, 32, 3), dtype=np.uint8)
    w32[0] = 200; w32[1, :16] = (10, 200, 30)
    got = ctx_rec.hist(w32)
    for i in range(len(w32)):
        assert np.array_equal(got[i], oracle.hist_normalized(w32[i]))


def test_k5_dedup_golden_50_frames(ctx_det, det_windows50):
    g = det_windows50
    w1, c1, o1 = ctx_det.dedup(g["windows"], g["coords"], g["offsets"], False, 0.85)
    assert np.array_equal(o1, g["p1_offsets"]) and np.array_equal(c1, g["p1_coords"])
    w2, c2, o2 = ctx_det.dedup(w1, c1, o1, True, 0.95)
    assert np.array_equal(o2, g["surv_offsets"])
    assert np.array_equal(c2, g["surv_coords"]) and np.array_equal(w2, g["surv_windows"])


def test_k5_dedup_per_frame_golden(ctx_det, det_frames):
    for k in STORED:
        wins = det_frames[k + "_windows"]; coords = det_frames[k + "_coords"][det_frames[k + "_valid"]]
        off = np.array([0, len(wins)], np.int32)
        w1, c1, o1 = ctx_det.dedup(wins, coords, off, False, 0.85)
        assert np.array_equal(w1, det_frames[k + "_p1_windows"]) and np.array_equal(c1, det_frames[k + "_p1_coords"])
        w2, c2, o2 = ctx_det.dedup(w1, c1, o1, True, 0.95)
        assert np.array_equal(w2, det_frames[k + "_p2_windows"]) and np.array_equal(c2, det_frames[k + "_p2_coords"])


def test_k5_dedup_adversarial(ctx_det, oracle):
    """Duplicates, identical pixels at different places, merge chains, empty and single-item frames."""
    rng = np.random.default_rng(21)
    base = rng.integers(0, 256, (12, 25, 25, 3), dtype=np.uint8)
    wins, coords, off = [], [], [0]
    for f in range(40):
        n = int(rng.integers(0, 60)) if f not in (3, 4) else (0 if f == 3 else 1)
        for i in range(n):
            b = base[int(rng.integers(0, 12))].astype(np.int16)
            mode = rng.random()
            if mode < 0.3:
                w = b                                                    # exact duplicate pixels
            elif mode < 0.7:
                w = b + rng.integers(-12, 13, b.shape)                   # near duplicate -> delete / merge bands
            else:
                w = rng.integers(0, 256, b.shape)
            wins.append(np.clip(w, 0, 255).astype(np.uint8))
            x, y = int(rng.integers(0, 1300)), int(rng.integers(0, 760))
            if coords and rng.random() < 0.5 and len(coords) > off[-1]:
                px = coords[int(rng.integers(off[-1], len(coords)))]
                x, y = max(0, px[0] + int(rng.integers(-30, 31))), max(0, px[1] + int(rng.integers(-30, 31)))
            s = int(rng.integers(20, 80))
            coords.append((x, y, x + s + int(rng.integers(-5, 6)), y + s + int(rng.integers(-5, 6))))
        off.append(len(coords))
    wins = np.stack(wins); coords = np.array(coords, np.int32); off = np.array(off, np.int32)
    for by_coords, tol in ((False, 0.85), (True, 0.95), (False, 0.5), (True, 0.6)):
        gw, gc, go = ctx_det.dedup(wins, coords, off, by_coords, tol)
        for f in range(len(off) - 1):
            ow, oc = oracle.dedup(wins[off[f]:off[f + 1]], coords[off[f]:off[f + 1]], by_coords, tol)
            assert go[f + 1] - go[f] == len(oc), (by_coords, tol, f)
            assert np.array_equal(gc[go[f]:go[f + 1]], oc) and np.array_equal(gw[go[f]:go[f + 1]], ow), (by_coords, tol, f)


def test_k5_dedup_flat_windows_32(ctx_rec, oracle):
    """32 x 32 windows (1024 pixels: bin counts up to 1024) with a few flat or two-tone windows per frame: the tensor-core pair
    kernel keeps counts modulo 256 and corrects the pairs of such windows exactly -- also when BOTH windows of a pair exceed 255 in
    the same bin -- for 2 .. 128 windows per frame; frames with more than 16 such windows go to k5_pairs, frames of more than 128
    windows to k5_gram_big (the same correction per pair of 128-row blocks)."""
    rng = np.random.default_rng(33)
    tones = rng.integers(0, 256, (5, 3), dtype=np.uint8)
    wins, coords, off = [], [], [0]
    for f, n in enumerate((2, 9, 33, 64, 65, 96, 97, 128, 129, 40, 40, 70)):
        nflat = (0, 3, 8, 16, 2, 5, 12, 16, 4, 17, 40, 1)[f]
        for i in range(n):
            if i < nflat:
                w = np.empty((32, 32, 3), np.int16)
                w[:] = tones[int(rng.integers(0, 5))]
                kind = rng.random()
                if kind < 0.4:
                    w[:, int(rng.integers(4, 28)):] = tones[int(rng.integers(0, 5))]         # two-tone
                elif kind < 0.7:
                    w[int(rng.integers(8, 24)):] += rng.integers(-6, 7, 3)                   # slightly different lower part
            else:
                w = rng.integers(0, 256, (8, 8, 3)).repeat(4, 0).repeat(4, 1).astype(np.int16) + rng.integers(-3, 4, (32, 32, 3))
            wins.append(np.clip(w, 0, 255).astype(np.uint8))
            x, y, sd = int(rng.integers(0, 1300)), int(rng.integers(0, 760)), int(rng.integers(20, 80))
            coords.append((x, y, x + sd, y + sd))
        order = rng.permutation(n) + off[-1]                              # flat windows anywhere in the list
        wins[off[-1]:] = [wins[k] for k in order]
        off.append(len(coords))
    wins = np.stack(wins); coords = np.array(coords, np.int32); off = np.array(off, np.int32)
    for tol in (0.85, 0.6):
        gw, gc, go = ctx_rec.dedup(wins, coords, off, False, tol)
        for f in range(len(off) - 1):
            ow, oc = oracle.dedup(wins[off[f]:off[f + 1]], coords[off[f]:off[f + 1]], False, tol)
            assert go[f + 1] - go[f] == len(oc), (tol, f)
            assert np.array_equal(gc[go[f]:go[f + 1]], oc) and np.array_equal(gw[go[f]:go[f + 1]], ow), (tol, f)


def test_k5_dedup_large_frames(ctx_det, oracle):
    """Frames with 300 / 700 / 1300 windows in one call: the 1024-window warp-per-frame fold, and the frame that exceeds it
    (flagged and redone by the general block-synchronous fold)."""
    rng = np.random.default_rng(5)
    base = rng.integers(0, 256, (40, 25, 25, 3), dtype=np.uint8)
    wins, coords, off = [], [], [0]
    for n in (300, 1300, 700):
        for i in range(n):
            b = base[int(rng.integers(0, 40))].astype(np.int16)
            w = b + rng.integers(-10, 11, b.shape) if rng.random() < 0.7 else rng.integers(0, 256, b.shape)
            wins.append(np.clip(w, 0, 255).astype(np.uint8))
            x, y, s = int(rng.integers(0, 1300)), int(rng.integers(0, 760)), int(rng.integers(20, 80))
            coords.append((x, y, x + s, y + s))
        off.append(len(coords))
    wins = np.stack(wins); coords = np.array(coords, np.int32); off = np.array(off, np.int32)
    for by_coords, tol in ((False, 0.85), (True, 0.95)):
        gw, gc, go = ctx_det.dedup(wins, coords, off, by_coords, tol)
        for f in range(len(off) - 1):
            ow, oc = oracle.dedup(wins[off[f]:off[f + 1]], coords[off[f]:off[f + 1]], by_coords, tol)
            assert go[f + 1] - go[f] == len(oc), (by_coords, f)
            assert np.array_equal(gc[go[f]:go[f + 1]], oc) and np.array_equal(gw[go[f]:go[f + 1]], ow), (by_coords, f)


def test_template_builder_golden(tsd, det_crops, templates, oracle):
    """SURVEY 8(f) N2: calculateMeanMasks on the GPU (K2 on every class crop, order-dependent running average, K3) gives the
    reference's 6 + 6 template masks bit for bit; the mean images equal the oracle's."""
    red6, blue6 = templates
    red, blue, mean6 = tsd.source_det.meanMasksFromCrops(det_crops)
    assert np.array_equal(np.stack([m for m, _ in red]), red6) and np.array_equal(np.stack([m for m, _ in blue]), blue6)
    assert [n for _, n in red] == tsd.source_det.SIGNALLIST
    assert np.array_equal(mean6, oracle.mean_masks(det_crops)[2])


def test_composite_entry_points(ctx_det, ctx_rec, det_frames, rec_frames):
    """tsd_score (K3+K4) and tsd_recognize (K6+K7+K8) against the reference's stored outputs for the real frames."""
    for k in STORED:
        r = ctx_det.score_windows(det_frames[k + "_p2_windows"])
        sc = det_frames[k + "_scores"]                                    # [n][2][6] per-template scores of the reference
        best_r, best_b = sc[:, 0].max(1), sc[:, 1].max(1)
        win = np.where(best_r > best_b, best_r, best_b)
        assert np.array_equal(r["hundredths"], np.round(win * 100).astype(np.int32))
        assert np.array_equal(r["emit"], win > 0.55)
        exp_id = np.where(best_r > best_b, sc[:, 0].argmax(1), sc[:, 1].argmax(1)) + 1
        assert np.array_equal(r["id"], exp_id.astype(np.int32))
        lab = ctx_rec.recognize_windows(rec_frames[k + "_windows"])
        assert np.array_equal(lab, rec_frames[k + "_pred_lda"])


# ---- whole chain ------------------------------------------------------------------------------------------------------
def _records(det):
    return [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]


def test_chain_golden_frames(ctx_det, det_frames, frames3):
    frames = np.stack([frames3[k] for k in STORED])
    boxes = [det_frames[k + "_boxes"] for k in STORED]
    off = np.concatenate([[0], np.cumsum([len(b) for b in boxes])]).astype(np.int32)
    det, counts = ctx_det.detect_frames(frames, np.concatenate(boxes), off)
    exp = []
    for f, k in enumerate(STORED):
        for c, i, s in zip(det_frames[k + "_det_coords"], det_frames[k + "_det_ids"], det_frames[k + "_det_scores"]):
            exp.append((f,) + tuple(int(v) for v in c) + (int(i), int(round(s * 100))))
    assert _records(det) == exp
    assert counts.tolist() == [int(off[-1]), int(sum(det_frames[k + "_valid"].sum() for k in STORED)),
                               int(sum(len(det_frames[k + "_p2_coords"]) for k in STORED)), len(exp)]


def test_chain_synthetic_vs_oracle(ctx_det, oracle, templates, tsd):
    """BASELINE config 3 shape (1360x800, 200 candidates/frame) on 64 frames, plus 4K frames with 500 and 2000 candidates
    (BASELINE config 5 sweep ends: ~800 windows per frame after the aspect filter, the 1024-window fold variant)."""
    red6, blue6 = templates
    for (H, W, F, N) in ((800, 1360, 64, 200), (2160, 3840, 1, 500), (2160, 3840, 2, 2000)):
        frames = tsd.synth.make_frames(F, H, W)
        boxes, off = tsd.synth.make_boxes(F, N, H, W)
        det, counts = ctx_det.detect_frames(frames, boxes, off)
        exp, tot = [], np.zeros(4, np.int64)
        for f in range(F):
            o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
            tot += o["stage_counts"]
            exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
        assert counts.tolist() == tot.tolist()
        assert _records(det) == exp


def test_chain_gram_block_variants_vs_oracle(ctx_det, oracle, templates, tsd):
    """Frames of ~12, ~45, ~75, ~110 and ~135 windows after the aspect filter in ONE batch: the tensor-core pair kernel (k5_gram)
    runs with 1, 3, 6 and 10 blocks of its lower triangle (K split over 12, 4, 2 and 1 warps; second rows of the first 32 lane
    groups above 96 windows) and hands the frames above 128 windows to k5_pairs through its todo list."""
    red6, blue6 = templates
    H, W = 800, 1360
    per_frame = [30, 110, 185, 270, 335, 30, 270, 110, 335, 185, 250, 300]
    F = len(per_frame)
    frames = tsd.synth.make_frames(F, H, W, seed=tsd.synth.FRAME_SEED + 5)
    for f, (y, x, side) in ((2, (100, 200, 260)), (3, (300, 700, 200)), (6, (50, 50, 420)), (9, (400, 900, 300))):
        frames[f][y:y + side, x:x + side] = np.array([40 + 20 * f, 60, 210 - 15 * f], np.uint8)   # flat patches: some windows with counts > 255
    bl, off = [], [0]
    for f, nbx in enumerate(per_frame):
        b, _ = tsd.synth.make_boxes(1, nbx, H, W, seed=tsd.synth.BOX_SEED + 100 + f)
        bl.append(b)
        off.append(off[-1] + len(b))
    boxes, off = np.concatenate(bl), np.asarray(off, np.int32)
    det, counts = ctx_det.detect_frames(frames, boxes, off)
    exp, tot, nwin = [], np.zeros(4, np.int64), []
    for f in range(F):
        o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
        tot += o["stage_counts"]
        nwin.append(int(o["stage_counts"][1]))
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    assert min(nwin) <= 32 and any(32 < v <= 64 for v in nwin) and any(64 < v <= 96 for v in nwin)
    assert any(96 < v <= 128 for v in nwin) and max(nwin) > 128, nwin
    assert counts.tolist() == tot.tolist()
    assert _records(det) == exp


def test_chain_flat_frames_vs_oracle(ctx_det, oracle, templates, tsd):
    """Frames made of large flat patches (windows whose histogram puts all 625 pixels into one or two bins, many exactly equal
    windows -> the pop-by-pixel-equality rule, degenerate correlations), mixed with ordinary frames in one batch."""
    red6, blue6 = templates
    rng = np.random.default_rng(17)
    F, H, W = 10, 800, 1360
    frames = tsd.synth.make_frames(F)
    for f in (1, 4, 7):                                               # flat / two-tone / coarse-block frames
        frames[f] = np.array([30, 40, 200], np.uint8)
    frames[4][:, W // 2:] = np.array([200, 60, 20], np.uint8)
    blocks = rng.integers(0, 256, (H // 40, W // 40, 3), dtype=np.uint8)
    frames[7] = np.repeat(np.repeat(blocks, 40, 0), 40, 1)
    boxes, off = tsd.synth.make_boxes(F, 200, seed=tsd.synth.BOX_SEED + 3)
    det, counts = ctx_det.detect_frames(frames, boxes, off)
    exp, tot = [], np.zeros(4, np.int64)
    for f in range(F):
        o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
        tot += o["stage_counts"]
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    assert counts.tolist() == tot.tolist()
    assert _records(det) == exp


def test_chain_256_frames_vs_oracle(ctx_det, oracle, templates, tsd):
    """A full-sized batch (256 frames x 200 candidates = 51 200 windows) through the device-resident asynchronous chain, record
    by record against the oracle: rare paths of the fold (merges of already merged items, pruning against rewritten
    histograms, twins) only show up at this scale."""
    import torch
    red6, blue6 = templates
    F = 256
    uniq = tsd.synth.make_frames(16)
    boxes, off = tsd.synth.make_boxes(F, 200, seed=tsd.synth.BOX_SEED + 7)
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(uniq).to(dev)[torch.arange(F, device=dev) % 16].contiguous()
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    ctx_det.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), max_boxes_per_frame=200)
    det, counts = ctx_det.fetch_detections(int(off[-1]))
    exp, tot = [], np.zeros(4, np.int64)
    for f in range(F):
        o = oracle.detect_frame(uniq[f % 16], boxes[off[f]:off[f + 1]], red6, blue6)
        tot += o["stage_counts"]
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    assert counts.tolist() == tot.tolist()
    assert _records(det) == exp


def test_too_small_box_bound_is_harmless(ctx_det, oracle, templates, tsd):
    """tsd_enqueue_frames with a max_boxes_per_frame that is SMALLER than the truth (a caller bug): frames that do not fit the
    bit rows sized from it are flagged by the warp fold and redone by the general fold -- same records as the oracle."""
    import torch
    red6, blue6 = templates
    F = 6
    frames = tsd.synth.make_frames(F)
    boxes, off = tsd.synth.make_boxes(F, 200)
    dev = torch.device("cuda", 0)
    d_frames = torch.from_numpy(frames).to(dev)
    d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
    ctx_det.enqueue_frames(d_frames.data_ptr(), F, 800, 1360, d_boxes.data_ptr(), d_off.data_ptr(), int(off[-1]), max_boxes_per_frame=64)
    det, counts = ctx_det.fetch_detections(int(off[-1]))
    exp = []
    for f in range(F):
        o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    assert _records(det) == exp


def test_chain_properties_full_size(ctx_det, tsd):
    """Size-independent properties at a larger batch: idempotence of the fold, determinism, frame independence."""
    F = 48
    frames = tsd.synth.make_frames(8)
    frames = np.concatenate([frames] * (F // 8))
    boxes, off = tsd.synth.make_boxes(F, 200)
    det, counts = ctx_det.detect_frames(frames, boxes, off)
    det2, counts2 = ctx_det.detect_frames(frames, boxes, off)
    assert np.array_equal(det, det2) and np.array_equal(counts, counts2)            # deterministic
    # frame independence: a frame processed alone gives the same records as inside the batch
    for f in (0, 17, 47):
        d1, _ = ctx_det.detect_frames(frames[f], boxes[off[f]:off[f + 1]], np.array([0, off[f + 1] - off[f]], np.int32))
        sel = det[det["frame"] == f]
        assert [r[1:] for r in _records(d1)] == [r[1:] for r in _records(sel)]
    # the coordinate pass is idempotent on its own output
    wins, coords, woff = ctx_det.windows(frames[:4], boxes[:off[4]], off[:5])
    w1, c1, o1 = ctx_det.dedup(wins, coords, woff, False, 0.85)
    w2, c2, o2 = ctx_det.dedup(w1, c1, o1, True, 0.95)
    w3, c3, o3 = ctx_det.dedup(w2, c2, o2, True, 0.95)
    assert np.array_equal(o2, o3) and np.array_equal(c2, c3) and np.array_equal(w2, w3)
    assert counts[0] == F * 200 and counts[0] >= counts[1] >= counts[2] >= counts[3]


def test_host_paths_agree(tsd, templates, oracle, monkeypatch):
    """tsd_detect_frames with host buffers: pageable frames (copied whole, in chunks that overlap the chain; 3 frames per
    chunk here so several chunks and a ragged tail are exercised), page-locked frames (the sectors the ROIs touch staged once
    into a device mirror; or, TSD_STAGE=0, gathered from host memory by K2 itself) and whole-frame copies (TSD_ZEROCOPY=0) must
    give identical records, equal to the oracle's."""
    red6, blue6 = templates
    F = 10
    frames = tsd.synth.make_frames(F)
    boxes, off = tsd.synth.make_boxes(F, 200)
    exp = []
    for f in range(F):
        o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
        exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    monkeypatch.setenv("TSD_CHUNK_FRAMES", "3")
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)
        d_pageable, c_pageable = ctx.detect_frames(frames, boxes, off)
        pinned = np.ascontiguousarray(frames.copy())
        ctx.pin(pinned)
        try:
            ctx.stat_staged_bytes(reset=True)
            d_pinned, c_pinned = ctx.detect_frames(pinned, boxes, off)
            staged = ctx.stat_staged_bytes()
        finally:
            ctx.unpin(pinned)
    # page-locked frames: only the sectors the ROIs touch cross the bus -- far fewer bytes than the frames, at least the ROIs' own
    assert 0 < staged < pinned.nbytes // 3
    # the same frames in CHUNKS through the two scratch slots (staging of chunk k+1 beside the chain of chunk k, records of chunk k
    # read after chunk k+1 is enqueued; TSD_STAGE_CHUNK=3 -> 3 chunks of 4, 4 and 2 frames), called twice (graph replay)
    monkeypatch.setenv("TSD_STAGE_CHUNK", "3")
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)
        ctx.pin(pinned)
        try:
            for _ in range(3):
                d_chunked, c_chunked = ctx.detect_frames(pinned, boxes, off)
                assert _records(d_chunked) == exp and c_chunked.tolist() == c_pinned.tolist()
        finally:
            ctx.unpin(pinned)
    monkeypatch.setenv("TSD_STAGE", "0")                                  # round 1's path: K2 itself gathers from host memory
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)
        ctx.pin(pinned)
        try:
            d_gather, c_gather = ctx.detect_frames(pinned, boxes, off)
            assert ctx.stat_staged_bytes() == 0                           # (nothing staged on this path)
        finally:
            ctx.unpin(pinned)
    monkeypatch.setenv("TSD_ZEROCOPY", "0")
    with tsd.Context(0, "det") as ctx:
        ctx.set_templates(red6, blue6)
        d_copy, c_copy = ctx.detect_frames(frames, boxes, off)
    assert _records(d_pageable) == exp and _records(d_pinned) == exp and _records(d_copy) == exp and _records(d_gather) == exp
    assert c_pageable.tolist() == c_pinned.tolist() == c_copy.tolist() == c_gather.tolist()


def test_back_to_back_batches_overlap_slots(tsd, templates, oracle, monkeypatch):
    """Consecutive enqueue_frames calls alternate between two scratch slots and two internal streams (the fold of one batch
    overlaps the kernels of the next).  Different batches enqueued back to back without a host sync in between, of different
    sizes (the second one forces the slot layout to grow), must each give the oracle's records; fetch returns the LAST batch;
    flush + an event on the context's stream covers everything enqueued; TSD_OVERLAP=0 gives the same records."""
    import torch
    red6, blue6 = templates
    dev = torch.device("cuda", 0)
    batches = []
    for k, (F, N) in enumerate(((6, 200), (9, 260), (4, 120))):
        frames = tsd.synth.make_frames(F, seed=tsd.synth.FRAME_SEED + 40 + k)
        boxes, off = tsd.synth.make_boxes(F, N, seed=tsd.synth.BOX_SEED + 40 + k)
        exp = []
        for f in range(F):
            o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6)
            exp += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
        batches.append((torch.from_numpy(frames).to(dev), torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev), F, int(off[-1]), N, exp))
    for overlap in ("1", "0"):
        monkeypatch.setenv("TSD_OVERLAP", overlap)
        with tsd.Context(0, "det") as ctx:
            ctx.set_templates(red6, blue6)

            def enqueue(b):
                ctx.enqueue_frames(b[0].data_ptr(), b[3], 800, 1360, b[1].data_ptr(), b[2].data_ptr(), b[4], max_boxes_per_frame=b[5])
            for last in (0, 1, 2, 1, 0):                                  # ... A B | A B C | ... : the fetched batch sits in either slot
                for b in batches[:last + 1]:
                    enqueue(b)
                det, _ = ctx.fetch_detections(batches[last][4])
                assert _records(det) == batches[last][6], (overlap, last)
            if overlap == "1":                                            # streaming: read batch k while batch k+1 runs
                enqueue(batches[0]); enqueue(batches[1])
                prev, _ = ctx.fetch_detections(batches[0][4], previous=True)
                assert _records(prev) == batches[0][6]
                enqueue(batches[2])
                prev, _ = ctx.fetch_detections(batches[1][4], previous=True)
                assert _records(prev) == batches[1][6]
                with pytest.raises(tsd.TsdError):
                    ctx.fetch_detections(batches[1][4], previous=True)   # already taken
                det, _ = ctx.fetch_detections(batches[2][4])
                assert _records(det) == batches[2][6]
            for b in batches:                                             # stream order: flush, then an event on the context's stream
                enqueue(b)
            ctx.flush()
            ev = torch.cuda.Event()
            ev.record(torch.cuda.ExternalStream(ctx.stream, device=dev))
            ev.synchronize()
            det, _ = ctx.fetch_detections(batches[2][4])
            assert _records(det) == batches[2][6]


# ---- recognition --------------------------------------------------------------------------------------------------------
def test_k6_k7_k8_recognition_golden(ctx_rec, rec_golden, rec_frames, oracle):
    g = rec_golden
    hog = ctx_rec.hog(g["gray"])
    ref = g["hog"]
    rel = np.abs(hog - ref) / np.maximum(np.abs(ref), 1e-2)
    assert rel.max() < 1e-4, rel.max()                                   # north_star: HOG within 1e-4 relative (measured: 8e-7)
    # the same bound WITHOUT the 1e-2 floor: purely relative down to features of 1e-3, plus 1e-7 absolute below that
    assert np.all(np.abs(hog - ref) <= 1e-4 * np.abs(ref) + 1e-7), float(np.max(np.abs(hog - ref) - 1e-4 * np.abs(ref)))
    assert np.abs(ctx_rec.hog(np.full((1, 32, 32), 9, np.uint8))).max() == 0.0    # constant image -> all zeros, no NaN
    lg, lab = ctx_rec.lda_predict(g["hog"])
    assert np.max(np.abs(lg - g["logits"])) < 1e-9
    assert np.array_equal(lab, g["pred_lda"])
    lg2, lab2 = ctx_rec.lda_predict(hog)                                  # our own descriptors: labels still exact
    assert np.array_equal(lab2, g["pred_lda"])
    Z, lk = ctx_rec.knn_predict(g["hog"])
    assert np.max(np.abs(Z - g["knn_Zq"])) < 1e-9
    assert np.array_equal(lk, g["pred_knn"])
    # saturation tie rule: logits this large make p == 1.0 for several classifiers -> lowest class wins
    X = np.zeros((3, 324), np.float32)
    with_big = type(ctx_rec)(device=0, flavour="rec")
    W = np.zeros((324, 6)); b = np.array([-50.0, 40.0, 45.0, -1.0, 60.0, 0.0])
    with_big.set_lda(W, b)
    _, lab = with_big.lda_predict(X)
    _, olab = oracle.lda_predict(X, W, b)
    assert np.array_equal(lab, olab) and lab[0] == 2
    with_big.close()
    for k in STORED:
        assert np.array_equal(ctx_rec.bgr2gray(rec_frames[k + "_windows"]), rec_frames[k + "_gray"])


def test_recognition_window_extraction_golden(ctx_rec, rec_frames, frames3):
    """x1.15 / 32x32 flavour of K1+K2+K5 (REC:47-64) reproduces the reference's survivors."""
    for k in STORED:
        boxes = rec_frames[k + "_boxes"]
        wins, coords, woff = ctx_rec.windows(frames3[k], boxes, np.array([0, len(boxes)], np.int32))
        w1, c1, o1 = ctx_rec.dedup(wins, coords, woff, False, 0.85)
        w2, c2, o2 = ctx_rec.dedup(w1, c1, o1, True, 0.95)
        assert np.array_equal(c2, rec_frames[k + "_coords"]) and np.array_equal(w2, rec_frames[k + "_windows"])


def test_recognition_chain(ctx_rec, rec_frames, frames3, tsd):
    """detect -> recognise composition (SURVEY 3.4): labels of the surviving windows equal the reference's."""
    for k in STORED:
        boxes = rec_frames[k + "_boxes"]
        det, counts = ctx_rec.detect_frames(frames3[k], boxes, np.array([0, len(boxes)], np.int32), mode=tsd.RUN_RECOGNIZE)
        lab = rec_frames[k + "_pred_lda"]
        exp = [tuple(int(v) for v in c) + (int(l),) for c, l in zip(rec_frames[k + "_coords"], lab) if l != 0]
        got = [(int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"])) for d in det]
        assert got == exp and counts[2] == len(lab)


# ---- error behaviour ------------------------------------------------------------------------------------------------------
def test_errors_are_reported_not_thrown(tsd, templates):
    with tsd.Context(device=0, flavour="det") as c:
        with pytest.raises(tsd.TsdError, match="templates not set"):
            c.score_masks(np.zeros((1, 25, 25), np.uint8), np.zeros((1, 25, 25), np.uint8))
        with pytest.raises(tsd.TsdError):
            c.set_templates(np.full((6, 25, 25), 7, np.uint8), np.zeros((6, 25, 25), np.uint8))
        with pytest.raises(tsd.TsdError):
            c.lda_predict(np.zeros((1, 324), np.float32))
    with pytest.raises(tsd.TsdError):
        tsd.Context(device=99)


def test_lda_tensor_core_evaluation(ctx_rec, rec_golden):
    """The TF32 evaluation kernels (not on the product path): 3xTF32 reproduces the f64 labels on the reference's held-out set and
    its logits agree to 1e-3; plain TF32 logits are off by up to ~0.1 -- larger than the smallest label margin of the data,
    which is why the product path stays f64 (DESIGN.md)."""
    X = rec_golden["hog"].astype(np.float32)
    z64, lab64 = ctx_rec.lda_predict(X)
    z3, lab3, _ = ctx_rec.lda_predict_tf32(X, split=3)
    z1, lab1, _ = ctx_rec.lda_predict_tf32(X, split=1)
    assert np.array_equal(lab3, lab64) and np.abs(z3 - z64).max() < 1e-3
    assert np.abs(z1 - z64).max() < 0.5 and np.abs(z1 - z64).max() > 1e-3


def test_k2_more_windows_than_persistent_warps(ctx_det, oracle):
    """More windows than the persistent K2 grid has warps (256 CTAs x 4 warps per SM): the 25x25 kernel strides over them; a window
    size without a specialised kernel (16x16) takes the generic kernel, which keeps one window per warp.  Sampled against the oracle
    (incl. the first and last windows)."""
    rng = np.random.default_rng(77)
    frame = rng.integers(0, 256, (1, 96, 128, 3), dtype=np.uint8)
    n = 160000
    x0 = rng.integers(0, 100, n); y0 = rng.integers(0, 70, n)
    coords = np.stack([x0, y0, x0 + rng.integers(3, 28, n), y0 + rng.integers(3, 26, n)], 1).astype(np.int32)
    pick = np.unique(np.concatenate([[0, 1, n - 2, n - 1], rng.integers(0, n, 300), np.arange(151500, 151600)]))
    for D in (25, 16):
        got = ctx_det.crop_resize(frame, coords, np.zeros(n, np.int32), D)
        for i in pick:
            assert np.array_equal(got[i], oracle.crop_resize(frame[0], coords[i], D)), (D, i)
