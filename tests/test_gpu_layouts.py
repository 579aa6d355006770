"""Every frame layout and host-memory route of the C ABI against the oracle, and tsd_preprocess at every shape and parameter.

The engine always passes contiguous frames (row_stride = 3 W, frame_stride = 3 H W).  The C ABI takes any row_stride,
frame_stride and base pointer, and the layout picks the kernel variant that reads the frames:

  K2 wide       aligned 32-bit tap loads: BGR, base, row_stride, frame_stride all multiples of 4 (D = 25 / 32)
  K2 bytes      byte loads: any other layout, and grey
  K2 tma        TSD_K2=tma: base and both strides multiples of 16
  K2 generic    any D other than 25 / 32
  staged        page-locked frames, 16-byte legal (base, strides, 3 W): stage_mark -> stage_copy -> device mirror
  gather        page-locked frames otherwise (or TSD_STAGE=0): K2 reads host memory over PCIe
  pageable      pageable frames: chunked whole-frame copies (TSD_CHUNK_FRAMES)
  staged chunks staged, nframes >= 2 TSD_STAGE_CHUNK: chunks through both scratch slots

Each batch here is a strided view into a larger canvas of noise (host numpy for the host routes, torch device memory for the
device routes), with a padded row, a padded frame and a base offset chosen on a named side of every rule above.  Widths are
1360 (3 W % 32 = 16: the last sector of a row is half a sector), 1366 (3 W even, not a multiple of 4), 1376 (3 W % 32 = 0)
and tiny ones (1, 5, 16, 21, D - 1, D, D + 1); heights 800, 1, 7, 9 and D +- 1.  Boxes clamp at x = 0 / y = 0, cross the
right or bottom edge, lie wholly outside, end on the last row of the last frame, give exact D x D and 2D x 2D crops at an
edge, 1-px crops, crops of 33 .. 2D rows and crops taller than 2D.

  per stage   tsd_crop_resize (host / device, C = 3 / 1, D = 25 / 32 / 20, plus TSD_K2=tma) and tsd_windows, bit-exact against
              oracle.crop_resize / expand_boxes; strides below the minimum refused by every entry point.
  chain       RUN_DETECT and RUN_RECOGNIZE through device pointers (and tma), pageable chunks, staging at TSD_STAGE_GRAN =
              32 / 64 / 128 and in chunks, TSD_STAGE=0 and TSD_ZEROCOPY=0: records and stage counts equal the oracle's, the
              staged byte count equals the marking rule restated in numpy, and the mirrors hold other pixels first (poison).
  det_cap     TSD_E_NOMEM with *ndet and the counts filled on the unchunked, pageable-chunked and staged-chunked routes.
  preprocess  host / device, contiguous / strided, tiles (1,1) (8,8) (3,5) (16,2) and larger than the image, H or W = 1, 2,
              3, (3, 300), 4K, clip 0 / 0.01 / 2 / 40, gamma 1 / 2 / 0.5 and a caller's table; more than 65 535 frames.

test_layout_inputs_are_in_their_regimes checks on the CPU that every route row is reached at both D, that every box class
occurs and that the staged-byte model marks half sectors and granules clamped at the row end.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from test_gpu_recognition import decision_margin, oracle_rec_frame, spread_lda

F = 5                                 # frames per batch: 2 pageable chunks + a ragged one, 2 staged chunks (3 + 2)
SLACK = 64                            # canvas bytes after the last frame
REC_LDA_SEED = 20                     # spread_lda seed that keeps every survivor clear of the decision (regime test)
FLAVOURS = {25: 1.30, 32: 1.15}       # D -> enlargement of the chain's flavour (det / rec)
MODES = {"det": 25, "rec": 32}

# name: (H, W, row_stride, frame_stride, base offset).  (frame_stride None = the minimum, row_stride * (H - 1) + 3 W.)
LAYOUTS = {
    "1360_contiguous":  (800, 1360, 4080, 4080 * 800, 0),          # all %16: staged, tma, wide; half last sector
    "1360_padded":      (800, 1360, 4096, 4096 * 800 + 32, 16),    # all %16 with padding
    "1366_odd":         (800, 1366, 4101, 4101 * 800 + 3, 1),      # nothing %4: bytes, gather
    "1366_contiguous":  (800, 1366, 4098, 4098 * 800, 0),          # 3 W % 4 = 2: bytes
    "1376_rs4":         (7, 1376, 4132, 4132 * 7, 4),              # rs, fs, base %4 only: wide, no tma, gather
    "1376_minimal":     (7, 1376, 4160, None, 16),                 # 3 W % 32 = 0, minimal frame_stride (29 088, %16 = 0): staged
    "1360_rs16x4":      (9, 1360, 4084, 4084 * 9 + 12, 16),        # only rs %16 = 4
    "1360_fs16x8":      (9, 1360, 4096, 4096 * 9 + 8, 16),         # only fs %16 = 8
    "1360_base4":       (9, 1360, 4096, 4096 * 9, 4),              # only base %16 = 4
    "1360_base1":       (9, 1360, 4096, 4096 * 9, 1),              # only base %4 = 1
    "1360_h1":          (1, 1360, 4083, 4085, 0),                  # one row; rs %4 = 3
    "w1_h26":           (26, 1, 16, 16 * 26, 16),                  # %16 everywhere but 3 W = 3: tma, wide, gather
    "w5_h24":           (24, 5, 20, None, 4),                      # fs = 475
    "w16_h33":          (33, 16, 48, 48 * 33, 0),                  # 3 W = 48: staged
    "w21_h31":          (31, 21, 63, 63 * 31, 1),
    "w24_h26":          (26, 24, 80, 80 * 26, 16),                 # D - 1 of 25, 3 W = 72
    "w25_h25":          (25, 25, 75, None, 0),
    "w26_h24":          (24, 26, 80, 80 * 24, 0),                  # 3 W = 78
    "w31_h33":          (33, 31, 96, 96 * 33 + 4, 4),
    "w32_h32":          (32, 32, 96, 96 * 32, 16),                 # 3 W = 96: staged
    "w33_h31":          (31, 33, 112, 112 * 31, 0),
}
ROUTES = {                            # name: (memory, environment)
    "device":        ("device", {}),
    "device_tma":    ("device", {"TSD_K2": "tma"}),
    "pageable":      ("pageable", {"TSD_CHUNK_FRAMES": "2"}),
    "staged32":      ("pinned", {"TSD_STAGE_GRAN": "32", "TSD_STAGE_CHUNK": "0"}),
    "staged64":      ("pinned", {"TSD_STAGE_GRAN": "64", "TSD_STAGE_CHUNK": "0"}),
    "staged128":     ("pinned", {"TSD_STAGE_GRAN": "128", "TSD_STAGE_CHUNK": "0"}),
    "staged_chunks": ("pinned", {"TSD_STAGE_CHUNK": "2"}),
    "staged_tma":    ("pinned", {"TSD_K2": "tma", "TSD_STAGE_CHUNK": "0"}),
    "gather":        ("pinned", {"TSD_STAGE": "0"}),
    "zerocopy_off":  ("pinned", {"TSD_ZEROCOPY": "0"}),
}
BOX_CLASSES = ("clamp_x0", "clamp_y0", "cross_right", "cross_bottom", "outside", "last_row_last_frame", "exact_D_edge",
               "exact_2D_edge", "one_px", "rows_33_to_2D", "taller_than_2D")


def layout(name):
    H, W, rs, fs, base = LAYOUTS[name]
    return H, W, rs, rs * (H - 1) + 3 * W if fs is None else fs, base


def grey_layout(name):
    """The same padding for one channel: row_stride - W and frame_stride - minimum as in the BGR layout."""
    H, W, rs, fs, base = layout(name)
    rg = W + (rs - 3 * W)
    return H, W, rg, rg * (H - 1) + W + (fs - rs * (H - 1) - 3 * W), base


# ---- inputs ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def source_frames():
    import tsd_b200
    return tsd_b200.synth.make_frames(F, 800, 1376, seed=tsd_b200.synth.FRAME_SEED + 77)


def frames_of(name, C=3):
    H, W = LAYOUTS[name][:2]
    f = source_frames()[:, :H, :W]
    return np.ascontiguousarray(f if C == 3 else f[..., 1])


def canvas_for(name, C=3, seed=0):
    """-> (canvas uint8 1-D, page aligned, noise outside the frames; view [F,H,W(,3)] into it; (H, W, rs, fs, base))."""
    H, W, rs, fs, base = layout(name) if C == 3 else grey_layout(name)
    n = base + fs * (F - 1) + rs * (H - 1) + W * C + SLACK
    raw = np.empty(n + 4096, np.uint8)
    a = (-raw.ctypes.data) % 4096
    canvas = raw[a:a + n]
    canvas[:] = np.random.default_rng(seed + n).integers(0, 256, n, dtype=np.uint8)
    shape, strides = ((F, H, W, 3), (fs, rs, 3, 1)) if C == 3 else ((F, H, W), (fs, rs, 1))
    view = np.lib.stride_tricks.as_strided(canvas[base:], shape, strides)
    view[...] = frames_of(name, C)
    return canvas, view, (H, W, rs, fs, base)


def expand(b, enlarge):
    """K1 / oracle.expand_box in float64 (DET:155-174) -> (x1, y1, x2, y2) or None."""
    x, y, w, h = (int(v) for v in b)
    r = float(w) / float(h)
    if not (0.8 < r < 1.2):
        return None
    pm1 = enlarge - 1.0
    dw, dh = float(w) * pm1 * 0.5, float(h) * pm1 * 0.5
    return tuple(int(max(v, 0.0)) for v in (x - dw, y - dh, (x + w) + dw, (y + h) + dh))


def clipped(c, H, W):
    """-> (cx, cy, cw, ch) of the crop clipped to the frame (cw or ch <= 0: empty)."""
    cx, cy = min(c[0], W), min(c[1], H)
    return cx, cy, min(c[2], W) - cx, min(c[3], H) - cy


def edge_box(H, W, enlarge, size):
    """A square box whose clipped crop is exactly size x size at the bottom-right corner (x2 >= W, y2 >= H), or None."""
    if size > min(H, W):
        return None
    for s in range(max(1, int(size / enlarge) - 3), size + 3):
        d = int(s * (enlarge - 1) * 0.5)
        for x in range(W - size + d - 2, W - size + d + 3):
            for y in range(H - size + d - 2, H - size + d + 3):
                c = expand((x, y, s, s), enlarge)
                if c and c[0] == W - size and c[1] == H - size and c[2] >= W and c[3] >= H:
                    return (x, y, s, s)
    return None


def sized_box(H, W, enlarge, lo, hi, rng):
    """A square interior box whose crop has between lo and hi rows (and as many columns), or None."""
    for s in range(max(1, int(lo / enlarge) - 2), int(hi / enlarge) + 3):
        if s + 4 > min(H, W):
            break
        x, y = int(rng.integers(0, W - s + 1)), int(rng.integers(0, H - s + 1))
        c = expand((x, y, s, s), enlarge)
        cw, ch = clipped(c, H, W)[2:]
        if lo <= ch <= hi:
            return (x, y, s, s)
    return None


@functools.lru_cache(maxsize=None)
def boxes_for(name, D):
    """-> (boxes int32 [n, 4], offsets int32 [F + 1]) for the flavour of window size D, every class that fits the frame."""
    H, W = LAYOUTS[name][:2]
    en = FLAVOURS[D]
    rng = np.random.default_rng([D, H, W, sum(map(ord, name))])
    out = []
    for f in range(F):
        bx = []
        for _ in range(20):                                                    # random, mostly square, anywhere
            s = int(rng.integers(1, max(2, min(H, W, 140)) + 1))
            w = max(1, int(round(s * rng.uniform(0.85, 1.15))))
            bx.append((int(rng.integers(0, W)), int(rng.integers(0, H)), w, s))
        s = int(rng.integers(4, 40))
        bx += [(0, 0, s, s), (0, int(rng.integers(0, H)), s, s), (int(rng.integers(0, W)), 0, s, s)]        # clamp at 0
        bx += [(W - s // 2, int(rng.integers(0, H)), s, s), (int(rng.integers(0, W)), H - s // 2, s, s),    # cross the edges
               (W - s // 3, H - s // 3, s, s)]
        bx += [(W + 3 + s, int(rng.integers(0, H)), s, s), (int(rng.integers(0, W)), H + 3 + s, s, s)]     # wholly outside
        bx += [(W, int(rng.integers(0, H)), 1, 1), (int(rng.integers(0, W)), H, 1, 1), (W, H, 1, 1)]     # 1-px crops
        for b in (edge_box(H, W, en, D), edge_box(H, W, en, 2 * D), sized_box(H, W, en, 33, 2 * D, rng),
                  sized_box(H, W, en, 2 * D + 1, 4 * D, rng)):
            if b is not None:
                bx.append(b)
        rng.shuffle(bx)
        out.append(bx)
    boxes = np.array([b for bx in out for b in bx], np.int32).reshape(-1, 4)
    off = np.concatenate([[0], np.cumsum([len(bx) for bx in out])]).astype(np.int32)
    return boxes, off


def box_classes(name, D):
    """{class: number of boxes of that class} (regime test)."""
    H, W = LAYOUTS[name][:2]
    boxes, off = boxes_for(name, D)
    got = dict.fromkeys(BOX_CLASSES, 0)
    for f in range(F):
        for b in boxes[off[f]:off[f + 1]]:
            x, y, w, h = (int(v) for v in b)
            c = expand(b, FLAVOURS[D])
            if c is None:
                continue
            cx, cy, cw, ch = clipped(c, H, W)
            if cw <= 0 or ch <= 0:
                got["outside"] += 1
                continue
            got["clamp_x0"] += x - (w * (FLAVOURS[D] - 1) * 0.5) < 0
            got["clamp_y0"] += y - (h * (FLAVOURS[D] - 1) * 0.5) < 0
            got["cross_right"] += c[2] > W
            got["cross_bottom"] += c[3] > H
            got["last_row_last_frame"] += f == F - 1 and cy + ch == H
            got["exact_D_edge"] += cw == ch == D and (c[2] >= W or c[3] >= H)
            got["exact_2D_edge"] += cw == ch == 2 * D and (c[2] >= W or c[3] >= H)
            got["one_px"] += cw == 1 or ch == 1
            got["rows_33_to_2D"] += 32 < ch <= 2 * D
            got["taller_than_2D"] += ch > 2 * D
    return got


def windows_of(name, D):
    """K1-passing windows in chain order -> (coords int32 [n, 4], frame int32 [n], clipped crop int32 [n, 4])."""
    H, W = LAYOUTS[name][:2]
    boxes, off = boxes_for(name, D)
    co, fr, cl = [], [], []
    for f in range(F):
        for b in boxes[off[f]:off[f + 1]]:
            c = expand(b, FLAVOURS[D])
            if c is not None and min(clipped(c, H, W)[2:]) > 0:
                co.append(c); fr.append(f); cl.append(clipped(c, H, W))
    return np.array(co, np.int32).reshape(-1, 4), np.array(fr, np.int32), np.array(cl, np.int32).reshape(-1, 4)


# ---- the staged-byte model: stage_mark + stage_copy restated ----------------------------------------------------------
def staged_bytes(name, D, gran):
    """-> (bytes one batch stages, number of half sectors copied, number of spans clamped at the row end)."""
    H, W = LAYOUTS[name][:2]
    _, fr, cl = windows_of(name, D)
    g = gran // 32
    last = (3 * W + 31) // 32 - 1
    sectors, clamped = set(), 0
    for f, (cx, cy, cw, ch) in zip(fr.tolist(), cl.tolist()):
        s0 = ((3 * cx) >> 5) & ~(g - 1)
        s1u = ((3 * (cx + cw) - 1) >> 5) | (g - 1)
        s1 = min(s1u, last)
        clamped += s1u > last
        if ch <= 2 * D:
            rows = range(cy, cy + ch)
        else:
            rows = set()
            for dy in range(D):
                sy = int(np.floor(np.float32((dy + 0.5) * (1.0 / (D / ch)) - 0.5)))
                rows |= {cy + min(max(sy, 0), ch - 1), cy + min(max(sy + 1, 0), ch - 1)}
        for r in rows:
            for s in range(s0, s1 + 1):
                sectors.add((f, r, s))
    nbytes = half = 0
    for _, _, s in sectors:
        b = min(32, 3 * W - 32 * s) & ~15
        nbytes += b
        half += b == 16
    return nbytes, half, clamped


def stages(name, route):
    """Whether tsd_detect_frames stages this layout on this route (the rule of tsd_detect_frames)."""
    H, W, rs, fs, base = layout(name)
    mem, env = ROUTES[route]
    return mem == "pinned" and env.get("TSD_STAGE") != "0" and env.get("TSD_ZEROCOPY") != "0" and \
        base % 16 == 0 and rs % 16 == 0 and fs % 16 == 0 and (3 * W) % 16 == 0


def k2_rows(name, route, D):
    """Route-table rows one chain call reaches."""
    H, W, rs, fs, base = layout(name)
    mem, env = ROUTES[route]
    pinned_legal = base % 16 == 0 and rs % 16 == 0 and fs % 16 == 0 and (3 * W) % 16 == 0
    rows = set()
    if mem == "device" or (mem == "pinned" and env.get("TSD_ZEROCOPY") != "0" and not stages(name, route)):
        b = base                                                              # K2 reads the caller's memory
        if mem == "pinned":
            rows.add("gather_stage0" if env.get("TSD_STAGE") == "0" else "gather_unaligned")
            assert env.get("TSD_STAGE") == "0" or not pinned_legal
    else:
        b = 0                                                                 # K2 reads the library's copy / mirror
        if stages(name, route):
            rows.add("staged_chunks" if 0 < int(env.get("TSD_STAGE_CHUNK", "256")) <= F // 2
                     else "staged")
        else:
            rows.add("pageable_chunked" if int(env.get("TSD_CHUNK_FRAMES", "32")) < F else "pageable")
    rows.add("wide" if b % 4 == 0 and rs % 4 == 0 and fs % 4 == 0 else "bytes")
    if env.get("TSD_K2") == "tma" and b % 16 == 0 and rs % 16 == 0 and fs % 16 == 0:
        rows.add("tma")
    return rows


# ---- oracle expectations -------------------------------------------------------------------------------------------
def _lib_expand_check(oracle, name, D):
    boxes, _ = boxes_for(name, D)
    oc, ov = oracle.expand_boxes(boxes, FLAVOURS[D])
    for b, c, v in zip(boxes, oc, ov):
        e = expand(b, FLAVOURS[D])
        assert (e is not None) == bool(v) and (e is None or e == tuple(int(q) for q in c)), (name, b.tolist())


def expected_det(oracle, red6, blue6):
    """{layout: (records, stage counts)} of RUN_DETECT under the given templates."""
    out = {}
    for name in LAYOUTS:
        boxes, off = boxes_for(name, 25)
        fr = frames_of(name)
        rec, counts = [], np.zeros(4, np.int64)
        for f in range(F):
            o = oracle.detect_frame(fr[f], boxes[off[f]:off[f + 1]], red6, blue6)
            rec += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
            counts += o["stage_counts"]
        out[name] = (rec, counts.tolist())
    return out


@pytest.fixture(scope="module")
def det_expected(oracle, templates):
    return expected_det(oracle, *templates)


@functools.lru_cache(maxsize=None)
def rec_survivors(oracle):
    out = {}
    for name in LAYOUTS:
        boxes, off = boxes_for(name, 32)
        fr = frames_of(name)
        H, W = LAYOUTS[name][:2]
        keep = np.array([(c := expand(b, 1.15)) is None or min(clipped(c, H, W)[2:]) > 0 for b in boxes], bool)   # (K1 drops empty crops)
        out[name] = [oracle_rec_frame(oracle, fr[f], boxes[off[f]:off[f + 1]][keep[off[f]:off[f + 1]]]) for f in range(F)]
    return out


@functools.lru_cache(maxsize=None)
def expected_rec(oracle):
    sv = rec_survivors(oracle)
    W, b = spread_lda(np.concatenate([h for v in sv.values() for _, h in v]), REC_LDA_SEED)
    out = {}
    for name in LAYOUTS:
        rec, nsurv = [], 0
        for f, (c2, hog) in enumerate(sv[name]):
            lab = oracle.lda_predict(hog, W, b, 0.5)[1] if len(hog) else []
            rec += [(f,) + tuple(int(x) for x in q) + (int(l), 0) for q, l in zip(c2, lab) if l != 0]
            nsurv += len(c2)
        boxes, _ = boxes_for(name, 32)
        out[name] = (rec, [len(boxes), len(windows_of(name, 32)[0]), nsurv, len(rec)])
    return W, b, out


def _records(det):
    return [(int(d["frame"]), int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]


# ---- CPU: every case is in its regime -------------------------------------------------------------------------------
def test_layout_inputs_are_in_their_regimes(oracle, det_expected):
    for name in LAYOUTS:
        H, W, rs, fs, base = layout(name)
        assert rs >= 3 * W and fs >= rs * (H - 1) + 3 * W, name
        Hg, Wg, rg, fg, _ = grey_layout(name)
        assert rg >= Wg and fg >= rg * (Hg - 1) + Wg, name
        canvas, view, _ = canvas_for(name)
        assert np.array_equal(view, frames_of(name)) and view.ctypes.data == canvas.ctypes.data + base
        for D in FLAVOURS:
            _lib_expand_check(oracle, name, D)
    # every side of every rule: row_stride, frame_stride and base each not %4, %4 but not %16, %16
    for k in (2, 3, 4):
        vals = [layout(n)[k] for n in LAYOUTS]
        assert any(v % 4 for v in vals) and any(v % 4 == 0 and v % 16 for v in vals) and any(v % 16 == 0 for v in vals), k
    assert {layout(n)[4] for n in LAYOUTS} == {0, 1, 4, 16}
    widths, heights = {LAYOUTS[n][1] for n in LAYOUTS}, {LAYOUTS[n][0] for n in LAYOUTS}
    wide = [W for W in widths if W >= 1360]
    assert any(3 * W % 32 == 16 for W in wide)                                    # the last sector of a row is half a sector
    assert any(3 * W % 2 == 0 and 3 * W % 4 for W in wide)                        # 3 W even, not a multiple of 4
    assert any(3 * W % 32 == 0 for W in wide)                                     # 3 W a whole number of sectors
    assert {1, 5, 16, 21, 24, 25, 26, 31, 32, 33} <= widths and {800, 1, 7, 24, 26, 31, 33} <= heights
    # every route row at both D (the generic kernel: D = 20 through tsd_crop_resize)
    for D in FLAVOURS:
        rows = set()
        for route in ROUTES:
            for name in LAYOUTS:
                rows |= k2_rows(name, route, D)
        assert rows >= {"wide", "bytes", "tma", "staged", "staged_chunks", "gather_unaligned", "gather_stage0",
                        "pageable_chunked"}, (D, rows)
    # every box class, at both D
    for D in FLAVOURS:
        tot = dict.fromkeys(BOX_CLASSES, 0)
        for name in LAYOUTS:
            for k, v in box_classes(name, D).items():
                tot[k] += v
        assert all(v > 0 for v in tot.values()), (D, tot)
        assert sum(box_classes(name, D)["last_row_last_frame"] > 0 for name in LAYOUTS) >= len(LAYOUTS) - 2
    # the staged-byte model: half sectors and granules clamped at the row end both occur on staged layouts
    staged = [n for n in LAYOUTS if stages(n, "staged32")]
    assert len(staged) >= 5
    for D in FLAVOURS:
        assert sum(staged_bytes(n, D, 32)[1] for n in staged) > 0
        assert sum(staged_bytes(n, D, g)[2] for n in staged for g in (64, 128)) > 0
        for n in staged:
            b32, b64, b128 = (staged_bytes(n, D, g)[0] for g in (32, 64, 128))
            assert 0 < b32 <= b64 <= b128, n
    # the chain's expectations have detections on big frames and every recognition label
    det = det_expected
    assert sum(len(det[n][0]) for n in LAYOUTS) > 20
    _, _, rec = expected_rec(oracle)
    labels = {r[5] for n in LAYOUTS for r in rec[n][0]}
    assert labels == set(range(1, 7)), labels
    hog = np.concatenate([h for v in rec_survivors(oracle).values() for _, h in v])
    Wl, bl, _ = expected_rec(oracle)
    assert decision_margin(oracle.lda_predict(hog, Wl, bl, 0.5)[0], hog, Wl).min() > 1


def test_preprocess_oracle_matches_cv2(oracle):
    """The oracle's grayAndEnhanceContrast equals live cv2 (createCLAHE + GaussianBlur + LUT) at every case the GPU test runs."""
    cv2 = pytest.importorskip("cv2")
    for img, clip, tiles, gamma in preprocess_cases():
        for f in range(len(img)):
            g = cv2.cvtColor(img[f], cv2.COLOR_BGR2GRAY)
            c = cv2.createCLAHE(clipLimit=clip, tileGridSize=tiles).apply(g)
            ref = cv2.LUT(cv2.GaussianBlur(c, (3, 3), 0), oracle.gamma_table(gamma) if np.isscalar(gamma) else gamma)
            assert np.array_equal(pre_oracle(oracle, img[f], clip, tiles, gamma), ref), (img.shape, clip, tiles, f)


# ---- preprocess cases ----------------------------------------------------------------------------------------------
PRE_SIZES = ((1, 1), (1, 7), (7, 1), (2, 2), (2, 9), (3, 3), (3, 300), (5, 3), (64, 64), (97, 131))
PRE_TILES = ((1, 1), (8, 8), (3, 5), (16, 2), (40, 40))
PRE_CLIPS = (0.0, 0.01, 2.0, 40.0)


def custom_gamma():
    return np.random.default_rng(5).permutation(256).astype(np.uint8)


@functools.lru_cache(maxsize=None)
def _pre_cases():
    rng = np.random.default_rng(8)
    gam = (1, 2, 0.5, "custom")
    out, k = [], 0
    for H, W in PRE_SIZES:
        for tiles in PRE_TILES:
            for clip in PRE_CLIPS:
                img = np.clip(rng.normal(120, 50, (2, H, W, 3)), 0, 255).astype(np.uint8)
                out.append((img, clip, tiles, gam[k % 4])); k += 1
    img = np.clip(rng.normal(120, 40, (1, 2160, 3840, 3)), 0, 255).astype(np.uint8)
    out += [(img, 2.0, (8, 8), 2), (img, 40.0, (3, 5), "custom")]
    return out


def preprocess_cases():
    return [(i, c, t, custom_gamma() if g == "custom" else g) for i, c, t, g in _pre_cases()]


def pre_oracle(oracle, img, clip, tiles, gamma):
    if np.isscalar(gamma):
        return oracle.preprocess(img, clip, tiles, gamma)
    return gamma[oracle.gauss3(oracle.clahe(oracle.bgr2gray(img), clip, tiles))]


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _lib():
    import tsd_b200
    return tsd_b200._capi


@pytest.fixture
def make_ctx(tsd, monkeypatch):
    """Contexts created under an environment (read at tsd_create); all closed at the end of the test."""
    made = []

    def mk(flavour="det", env=None):
        for k in ("TSD_K2", "TSD_STAGE", "TSD_STAGE_GRAN", "TSD_STAGE_CHUNK", "TSD_CHUNK_FRAMES", "TSD_ZEROCOPY"):
            monkeypatch.delenv(k, raising=False)
        for k, v in (env or {}).items():
            monkeypatch.setenv(k, v)
        c = tsd.Context(0, flavour)
        made.append(c)
        return c
    yield mk
    for c in made:
        c.close()


def _to_device(canvas):
    import torch
    return torch.from_numpy(canvas).to(torch.device("cuda", 0))


def _crop_expect(oracle, name, C, D):
    """-> (coords, win_frame, expected windows) of every non-empty K1 crop of the layout for window size D."""
    co, fr, _ = windows_of(name, 25 if D == 20 else D)
    fx = frames_of(name, C)
    shape = (D, D, 3) if C == 3 else (D, D)
    exp = np.stack([oracle.crop_resize(fx[f], c, D) for c, f in zip(co, fr)]) if len(co) else np.zeros((0,) + shape, np.uint8)
    return co, fr, exp


@pytest.mark.gpu
@pytest.mark.parametrize("tma", (False, True))
def test_crop_resize_layouts(oracle, make_ctx, tma):
    """tsd_crop_resize on every layout, host and device pointers, C = 3 / 1, D = 25 / 32 / 20, against oracle.crop_resize on the
    contiguous frame.  Device calls add crops that are empty after clipping: their windows must be all zero.  With TSD_K2=tma the
    TMA kernel runs only at D = 32 here: tsd_crop_resize writes packed windows, and the 1 875-byte stride of D = 25 is not a
    multiple of 16.  The chain routes (internal 16-byte window stride) run it at D = 25."""
    A = _lib()
    ctx = make_ctx("det", {"TSD_K2": "tma"} if tma else {})
    bad = []
    for name in LAYOUTS:
        for Cn in (3, 1):
            canvas, _, (H, W, rs, fs, base) = canvas_for(name, Cn)
            d_canvas = _to_device(canvas)
            for D in (25, 32, 20):
                co, fr, exp = _crop_expect(oracle, name, Cn, D)
                n = len(co)
                got = np.empty_like(exp)
                A.check(ctx._L.tsd_crop_resize(ctx._h, A.ptr(canvas.ctypes.data + base), F, H, W, rs, fs, Cn, A.ptr(co), A.ptr(fr), n, D,
                                               A.ptr(got), A.MEM_HOST))
                if not np.array_equal(got, exp):
                    bad.append((name, Cn, D, "host", int(np.sum(np.any((got != exp).reshape(n, -1), 1)))))
                # device: the same crops plus empty ones (wholly outside), interleaved
                ec = np.array([[W + 1, 0, W + 9, H], [0, H, W, H + 5]] * 2, np.int32)
                dco = np.concatenate([co, ec]); dfr = np.concatenate([fr, np.array([0, F - 1, 1, 2], np.int32)])
                perm = np.random.default_rng(n).permutation(len(dco))
                import torch
                dev = torch.device("cuda", 0)
                t_co, t_fr = torch.from_numpy(dco[perm].copy()).to(dev), torch.from_numpy(dfr[perm].copy()).to(dev)
                t_out = torch.full((len(dco) * D * D * Cn,), 77, dtype=torch.uint8, device=dev)
                A.check(ctx._L.tsd_crop_resize(ctx._h, A.ptr(d_canvas.data_ptr() + base), F, H, W, rs, fs, Cn, A.ptr(t_co.data_ptr()),
                                               A.ptr(t_fr.data_ptr()), len(dco), D, A.ptr(t_out.data_ptr()), A.MEM_DEVICE))
                ctx.synchronize()
                got = t_out.cpu().numpy().reshape((len(dco),) + exp.shape[1:])
                full = np.concatenate([exp, np.zeros((len(ec),) + exp.shape[1:], np.uint8)])[perm]
                if not np.array_equal(got, full):
                    bad.append((name, Cn, D, "device", int(np.sum(np.any((got != full).reshape(len(dco), -1), 1)))))
    assert not bad, bad[:12]


@pytest.mark.gpu
def test_windows_layouts(oracle, make_ctx):
    """tsd_windows (K1 + K2, host pointers) on every BGR layout at both flavours: offsets, coords and windows equal
    oracle.expand_boxes + crop_resize with the empty clipped crops dropped."""
    A = _lib()
    ctx = make_ctx("det")
    for name in LAYOUTS:
        canvas, _, (H, W, rs, fs, base) = canvas_for(name)
        for D, en in FLAVOURS.items():
            boxes, off = boxes_for(name, D)
            co, fr, _ = windows_of(name, D)
            exp = _crop_expect(oracle, name, 3, D)[2]
            eoff = np.searchsorted(fr, np.arange(F + 1)).astype(np.int32)
            nb = len(boxes)
            win = np.empty((nb, D, D, 3), np.uint8); coords = np.empty((nb, 4), np.int32)
            woff = np.empty(F + 1, np.int32); tot = C.c_int32()
            A.check(ctx._L.tsd_windows(ctx._h, A.ptr(canvas.ctypes.data + base), F, H, W, rs, fs, A.ptr(boxes), A.ptr(off), en, D,
                                       A.ptr(win), A.ptr(coords), A.ptr(woff), C.byref(tot), A.MEM_HOST))
            n = tot.value
            assert n == len(co) and np.array_equal(woff, eoff), (name, D)
            assert np.array_equal(coords[:n], co), (name, D)
            assert np.array_equal(win[:n], exp), (name, D, int(np.sum(np.any((win[:n] != exp).reshape(n, -1), 1))))


@pytest.mark.gpu
def test_strides_refused(tsd, make_ctx):
    """A row_stride below W * C or a frame_stride below row_stride * (H - 1) + W * C is refused by every entry point that takes
    frames, before any launch; the minimum itself is accepted (the layouts above use it)."""
    import torch
    A = _lib()
    ctx = make_ctx("det")
    H, W = 6, 10
    buf = np.zeros(4096, np.uint8)
    d_buf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    boxes = np.array([[1, 1, 4, 4]], np.int32); off = np.array([0, 1], np.int32)
    co = np.array([[0, 0, 5, 5]], np.int32); wf = np.zeros(1, np.int32)
    d_boxes, d_off = torch.from_numpy(boxes).cuda(), torch.from_numpy(off).cuda()
    out = np.zeros(65536, np.uint8); det = np.zeros(4, A.DET_DTYPE); nd = C.c_int32(); cnt = np.zeros(4, np.int32)
    hb = A.ptr(buf)
    for Cn in (3, 1):
        for rs, fs in ((W * Cn - 1, 100 * W), (W * Cn, W * Cn * (H - 1) + W * Cn - 1), (W * Cn + 5, (W * Cn + 5) * (H - 1) + W * Cn - 1)):
            calls = {"crop_resize": lambda m, p: ctx._L.tsd_crop_resize(ctx._h, p, 2, H, W, rs, fs, Cn, A.ptr(co), A.ptr(wf), 1, 25, A.ptr(out), m)}
            if Cn == 3:
                calls.update({
                    "windows": lambda m, p: ctx._L.tsd_windows(ctx._h, p, 2, H, W, rs, fs, A.ptr(boxes), A.ptr(np.array([0, 1, 1], np.int32)), 1.3, 25,
                                                               A.ptr(out), A.ptr(np.zeros(4, np.int32)), A.ptr(np.zeros(3, np.int32)), None, m),
                    "preprocess": lambda m, p: ctx._L.tsd_preprocess(ctx._h, p, 2, H, W, rs, fs, 2.0, 8, 8, A.ptr(out) if m == A.MEM_HOST else A.ptr(d_buf.data_ptr()), m),
                    "detect_frames": lambda m, p: ctx._L.tsd_detect_frames(ctx._h, 1, p, 1, H, W, rs, fs, A.ptr(boxes) if m == A.MEM_HOST else A.ptr(d_boxes.data_ptr()),
                                                                           A.ptr(off) if m == A.MEM_HOST else A.ptr(d_off.data_ptr()), A.ptr(det), 4, C.byref(nd), A.ptr(cnt), m),
                    "enqueue_frames": lambda m, p: ctx._L.tsd_enqueue_frames(ctx._h, 1, A.ptr(d_buf.data_ptr()), 1, H, W, rs, fs, A.ptr(d_boxes.data_ptr()),
                                                                             A.ptr(d_off.data_ptr()), 1, 1),
                })
            for what, fn in calls.items():
                for m, p in ((A.MEM_HOST, hb), (A.MEM_DEVICE, A.ptr(d_buf.data_ptr()))):
                    if what == "windows" and m == A.MEM_DEVICE:
                        continue
                    assert fn(m, p) == -1, (what, Cn, rs, fs, m)
                    assert b"stride" in ctx._L.tsd_last_error(), (what, ctx._L.tsd_last_error())
    ctx.synchronize()


def _det_call(ctx, mode, p, lay, boxes, off, cap):
    A = _lib()
    H, W, rs, fs, _ = lay
    det = np.zeros(max(cap, 1), A.DET_DTYPE); nd = C.c_int32(-1); counts = np.full(4, -1, np.int32)
    rc = ctx._L.tsd_detect_frames(ctx._h, mode, A.ptr(p), F, H, W, rs, fs, A.ptr(boxes), A.ptr(off), A.ptr(det), cap, C.byref(nd),
                                  A.ptr(counts), A.MEM_HOST)
    return rc, det[:max(nd.value, 0)], nd.value, counts.tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("mode", list(MODES))
def test_chain_layouts(oracle, templates, det_expected, make_ctx, mode, route):
    """The whole chain on every layout through one route: records (frame by frame, in order) and the four stage counts equal the
    oracle's.  Page-locked routes: the staged byte count is the marking rule's exactly where the layout is staged and 0
    elsewhere, and each staged layout first runs twice on other pixels (255 - canvas) so that both slots' mirrors hold stale
    bytes wherever stage_mark does not mark."""
    import torch
    A = _lib()
    D = MODES[mode]
    mem, env = ROUTES[route]
    ctx = make_ctx(mode, env)
    if mode == "det":
        red6, blue6 = templates
        ctx.set_templates(red6, blue6)
        exp_all = det_expected
        run_mode = A.RUN_DETECT
    else:
        Wl, bl, exp_all = expected_rec(oracle)
        ctx.set_lda(Wl, bl)
        run_mode = A.RUN_RECOGNIZE
    gran = int(env.get("TSD_STAGE_GRAN", "32"))
    bad = []
    for name in LAYOUTS:
        boxes, off = boxes_for(name, D)
        exp, ecounts = exp_all[name]
        canvas, _, lay = canvas_for(name)
        H, W, rs, fs, base = lay
        if mem == "device":
            dev = torch.device("cuda", 0)
            d_canvas = _to_device(canvas)
            d_boxes, d_off = torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev)
            A.check(ctx._L.tsd_enqueue_frames(ctx._h, run_mode, A.ptr(d_canvas.data_ptr() + base), F, H, W, rs, fs, A.ptr(d_boxes.data_ptr()),
                                              A.ptr(d_off.data_ptr()), len(boxes), 0))
            det, counts = ctx.fetch_detections(len(boxes))
            got, gcounts = _records(det), counts.tolist()
        elif mem == "pageable":
            rc, det, _, gcounts = _det_call(ctx, run_mode, canvas.ctypes.data + base, lay, boxes, off, len(boxes))
            A.check(rc)
            got = _records(det)
        else:
            ctx.pin(canvas)
            try:
                real = canvas.copy()
                if stages(name, route):
                    canvas[:] = 255 - real                                    # poison both slots' mirrors
                    for _ in range(2):
                        A.check(_det_call(ctx, run_mode, canvas.ctypes.data + base, lay, boxes, off, len(boxes))[0])
                    canvas[:] = real
                    A.check(_det_call(ctx, run_mode, canvas.ctypes.data + base, lay, boxes, off, len(boxes))[0])
                ctx.stat_staged_bytes(reset=True)
                rc, det, _, gcounts = _det_call(ctx, run_mode, canvas.ctypes.data + base, lay, boxes, off, len(boxes))
                A.check(rc)
                staged = ctx.stat_staged_bytes(reset=True)
            finally:
                ctx.unpin(canvas)
            got = _records(det)
            want = staged_bytes(name, D, gran)[0] if stages(name, route) else 0
            if staged != want:
                bad.append((name, "staged bytes", staged, want))
        if got != exp or gcounts != list(ecounts):
            diff = [f for f in range(F) if [r for r in got if r[0] == f] != [r for r in exp if r[0] == f]]
            bad.append((name, "frames", diff, gcounts, list(ecounts)))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("route", ("staged32", "staged_chunks", "pageable", "device"))
def test_det_cap(oracle, make_ctx, route):
    """det_cap = 0 and n - 1: TSD_E_NOMEM with *ndet = n and the counts filled in (summed over chunks); det_cap = n: the oracle's
    records; the next call on the same context is still right."""
    import torch
    A = _lib()
    mem, env = ROUTES[route]
    ctx = make_ctx("rec", env)
    Wl, bl, exp_all = expected_rec(oracle)
    ctx.set_lda(Wl, bl)
    name = "1360_padded"
    boxes, off = boxes_for(name, 32)
    exp, ecounts = exp_all[name]
    n = len(exp)
    assert n >= 2 and len({r[0] for r in exp}) >= 2
    canvas, _, lay = canvas_for(name)
    H, W, rs, fs, base = lay
    p = canvas.ctypes.data + base
    if mem == "pinned":
        ctx.pin(canvas)
    try:
        if mem == "device":
            d_canvas = _to_device(canvas)
            d_boxes, d_off = torch.from_numpy(boxes).cuda(), torch.from_numpy(off).cuda()
            for cap in (0, n - 1, n, n):
                A.check(ctx._L.tsd_enqueue_frames(ctx._h, A.RUN_RECOGNIZE, A.ptr(d_canvas.data_ptr() + base), F, H, W, rs, fs,
                                                  A.ptr(d_boxes.data_ptr()), A.ptr(d_off.data_ptr()), len(boxes), 0))
                det = np.zeros(max(cap, 1), A.DET_DTYPE); nd = C.c_int32(-1); counts = np.full(4, -1, np.int32)
                rc = ctx._L.tsd_fetch_detections(ctx._h, A.ptr(det), cap, C.byref(nd), A.ptr(counts))
                assert nd.value == n and counts.tolist() == list(ecounts), (cap, nd.value, counts.tolist())
                assert rc == (-4 if cap < n else 0), cap
                if cap == n:
                    assert _records(det[:n]) == exp
            return
        for cap in (0, n - 1, n, n):
            rc, det, nd, counts = _det_call(ctx, A.RUN_RECOGNIZE, p, lay, boxes, off, cap)
            assert nd == n and counts == list(ecounts), (route, cap, nd, counts)
            assert rc == (-4 if cap < n else 0), (route, cap, rc)
            if cap == n:
                assert _records(det) == exp, route
    finally:
        if mem == "pinned":
            ctx.unpin(canvas)


def _preprocess(ctx, img, clip, tiles, gamma, strided, device, seed):
    """tsd_preprocess on img [F,H,W,3], as a strided view of a noise canvas when asked, through host or device pointers."""
    import torch
    A = _lib()
    Fn, H, W = img.shape[:3]
    table = oracle_gamma(gamma)
    A.check(ctx._L.tsd_set_gamma_table(ctx._h, A.ptr(table)))
    if strided:
        rs = 3 * W + 1 + seed % 7
        fs = rs * H + 3 + seed % 5
        base = 1 + seed % 13
    else:
        rs, fs, base = 3 * W, 3 * W * H, 0
    n = base + fs * (Fn - 1) + rs * (H - 1) + 3 * W
    canvas = np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)
    np.lib.stride_tricks.as_strided(canvas[base:], img.shape, (fs, rs, 3, 1))[...] = img
    if device:
        d_in = torch.from_numpy(canvas).cuda()
        d_out = torch.full((Fn * H * W,), 7, dtype=torch.uint8, device="cuda")
        A.check(ctx._L.tsd_preprocess(ctx._h, A.ptr(d_in.data_ptr() + base), Fn, H, W, rs, fs, float(clip), tiles[0], tiles[1],
                                      A.ptr(d_out.data_ptr()), A.MEM_DEVICE))
        ctx.synchronize()
        return d_out.cpu().numpy().reshape(Fn, H, W)
    out = np.empty((Fn, H, W), np.uint8)
    A.check(ctx._L.tsd_preprocess(ctx._h, A.ptr(canvas.ctypes.data + base), Fn, H, W, rs, fs, float(clip), tiles[0], tiles[1], A.ptr(out),
                                  A.MEM_HOST))
    return out


def oracle_gamma(gamma):
    from oracle import oracle as O
    return O.gamma_table(gamma) if np.isscalar(gamma) else np.ascontiguousarray(gamma, np.uint8)


@pytest.mark.gpu
def test_preprocess_shapes_and_parameters(oracle, make_ctx):
    """tsd_preprocess against oracle.preprocess at every size / tiles / clip / gamma case, each through host and device pointers,
    contiguous and strided."""
    ctx = make_ctx("det")
    bad = []
    for k, (img, clip, tiles, gamma) in enumerate(preprocess_cases()):
        exp = np.stack([pre_oracle(oracle, im, clip, tiles, gamma) for im in img])
        for strided in (False, True):
            for device in (False, True):
                got = _preprocess(ctx, img, clip, tiles, gamma, strided, device, k)
                if not np.array_equal(got, exp):
                    bad.append((img.shape[1:3], clip, tiles, "gamma" if not np.isscalar(gamma) else gamma, strided, device,
                                int(np.sum(got != exp))))
    assert not bad, bad[:12]


@pytest.mark.gpu
def test_preprocess_more_than_65535_frames(oracle, make_ctx):
    """65 537 frames of 8 x 8 in one call (frames past gridDim.y / gridDim.z's 65 535): the first and last 500 and a seeded
    sample equal the oracle's."""
    ctx = make_ctx("det")
    Fn = 65537
    rng = np.random.default_rng(65537)
    img = rng.integers(0, 256, (Fn, 8, 8, 3), dtype=np.uint8)
    got = _preprocess(ctx, img, 2.0, (8, 8), 2, False, False, 0)
    idx = np.unique(np.concatenate([np.arange(500), np.arange(Fn - 500, Fn), rng.integers(0, Fn, 500)]))
    bad = [int(f) for f in idx if not np.array_equal(got[f], oracle.preprocess(img[f], 2.0, (8, 8), 2))]
    assert not bad, (len(bad), bad[:10])
