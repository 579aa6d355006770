"""Frames of different sizes in one batch: the *_ragged entry points (one base pointer + a tsd_frame_desc table) against the
oracle, frame by frame, bit-exact.

  per stage   tsd_crop_resize_ragged (host / device, C = 3 / 1, D = 25 / 32 / 20) and tsd_windows_ragged on one table that
              mixes 1360x800, 1920x1080, 3840x2160, 7 rows x 1376, 26 rows x 1 and 1 x 1 frames, an aliased entry (entry 0 again)
              and a sub-rectangle view of the 4K frame, whose last row ends the buffer although it is a middle entry of the table.
              Three layouts of that table: every offset and row stride a multiple of 16, a multiple of 4 only, and odd.
  chain       RUN_DETECT and RUN_RECOGNIZE x {HOG, GRAY} x {LDA, KNN} through device pointers, page-locked staging, page-locked
              gather (one misaligned entry), pageable chunks and staged chunks: records and counts equal the oracle's in table
              order; the staged byte count equals the marking rule restated per frame; TSD_E_NOMEM fills *ndet and the counts.
  uniform     a uniform batch written as a table gives what the uniform entry point gives, on every route.
  sequences   ragged and uniform enqueues alternate; two ragged tables that differ only in their offsets share a CUDA graph
              (replays), fetched with tsd_fetch_previous.
  real        the 24 JPEG and 3 PNG golden frames plus rescaled copies (cv2.resize, boxes from cv2.MSER) in one batch.
  drop-ins    extractMSERDetectionsGray, orderCroppedImagesByImageFile, detectBatch, recognizeBatch on mixed sizes equal the
              same functions called one frame at a time.
  limits      every invalid table field is refused before any device work; offsets past 4 GiB on the device.
"""
import ctypes as C
import functools
import os

import numpy as np
import pytest

from test_gpu_layouts import _records, clipped, edge_box, expand, sized_box
from test_gpu_rec_modes import feats, knn_model, lda_model, oracle_survivors, predict, robust, set_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAVOURS = {25: 1.30, 32: 1.15}                   # D -> enlargement of the chain's flavour (det / rec)
STAGE_SIZES = ((800, 1360), (1080, 1920), (2160, 3840), (7, 1376))      # per-stage table, plus the tiny frames below
TINY = ((26, 1), (1, 1))
CHAIN_SIZES = ((800, 1360), (1080, 1920), (2160, 3840), (7, 1376), (33, 16), (480, 640))   # 3 W % 16 == 0: stageable
KINDS = ("a16", "a4", "odd")
REC_MODES = {"hog_lda": (2, False), "hog_knn": (2 | 8, False), "gray_lda": (2 | 4, True), "gray_knn": (2 | 4 | 8, True)}
ROUTES = {                                          # name: (memory, environment, table kind)
    "device":        ("device", {}, "a4"),
    "staged":        ("pinned", {"TSD_STAGE_CHUNK": "0"}, "a16"),
    "gather":        ("pinned", {"TSD_STAGE_CHUNK": "0"}, "a4"),
    "pageable":      ("pageable", {"TSD_CHUNK_FRAMES": "3"}, "odd"),
    "staged_chunks": ("pinned", {"TSD_STAGE_CHUNK": "2"}, "a16"),
}


def _lib():
    import tsd_b200
    return tsd_b200._capi


# ---- tables --------------------------------------------------------------------------------------------------------------
def _pixels(H, W, seed):
    import tsd_b200
    if min(H, W) >= 16:
        return tsd_b200.synth.make_frames(1, H, W, seed=seed)[0]
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


@functools.lru_cache(maxsize=None)
def batch(sizes, kind, C=3, seed=0):
    """-> (canvas uint8 [extent] page-aligned, table FRAME_DESC_DTYPE, frames: list of [H,W(,3)] arrays in table order).
    Entries: the frames of `sizes` (the largest last in memory, so that its last row ends the buffer), entry 0 again (alias) and a
    sub-rectangle view of the largest frame.  kind a16: offsets and row strides multiples of 16; a4: multiples of 4, some not of
    16; odd: the first entry at an odd offset with an odd row stride."""
    from tsd_b200._capi import FRAME_DESC_DTYPE
    rng = np.random.default_rng([seed, C, KINDS.index(kind), len(sizes)])
    al = {"a16": 16, "a4": 4, "odd": 1}[kind]
    up = lambda v: -(-v // al) * al
    order = sorted(range(len(sizes)), key=lambda i: sizes[i][0] * sizes[i][1])
    ent = [None] * len(sizes)
    o = up(int(rng.integers(0, 40)))
    for k, i in enumerate(order):
        H, W = sizes[i]
        rs = up(W * C + (int(rng.integers(0, 3)) * al if k % 2 else 0))
        if kind == "a4" and rs % 16 == 0:
            rs += 4
        if kind == "odd" and i == 0:
            o += 1 - o % 2
            rs += 1 - rs % 2
        ent[i] = (o, rs, H, W)
        o = up(o + rs * (H - 1) + W * C + int(rng.integers(0, 24)))
    big = order[-1]                                                  # the frame placed last in memory
    bo, brs, bH, bW = ent[big]
    vy, vx = bH // 3, up(bW // 5) if C == 3 and al > 1 else bW // 5
    view = (bo + vy * brs + vx * C, brs, bH // 2, up(bW // 3))
    table = np.array(ent + [ent[0], view], FRAME_DESC_DTYPE)
    extent = max(int(e["offset"]) + int(e["row_stride"]) * (int(e["H"]) - 1) + int(e["W"]) * C for e in table)
    assert extent == bo + brs * (bH - 1) + bW * C                    # the largest frame ends the buffer; it is not the last entry
    raw = np.empty(extent + 4096, np.uint8)
    canvas = raw[(-raw.ctypes.data) % 4096:][:extent]
    canvas[:] = rng.integers(0, 256, extent, dtype=np.uint8)
    for i, (H, W) in enumerate(sizes):
        px = _pixels(H, W, 1000 + 17 * i + seed)
        view_i = frame_view(canvas, table[i], C)
        view_i[...] = px if C == 3 else px[..., 1]
    frames = [np.array(frame_view(canvas, e, C)) for e in table]
    return canvas, table, frames


def frame_view(canvas, e, C):
    o, rs, H, W = int(e["offset"]), int(e["row_stride"]), int(e["H"]), int(e["W"])
    shape, strides = ((H, W, 3), (rs, 3, 1)) if C == 3 else ((H, W), (rs, 1))
    return np.lib.stride_tricks.as_strided(canvas[o:], shape, strides)


@functools.lru_cache(maxsize=None)
def boxes_for(shapes, D, seed=0):
    """-> (boxes int32 [n, 4], offsets) per frame shape (H, W): random, edge, outside, 1-px, D x D / 2D x 2D edge crops."""
    import tsd_b200
    en = FLAVOURS[D]
    rng = np.random.default_rng([seed, D, len(shapes)])
    out = []
    for k, (H, W) in enumerate(shapes):
        bx = [(W, H, 1, 1), (0, 0, 1, 1), (W + 5, 0, 3, 3)]
        if min(H, W) >= 64:
            b, _ = tsd_b200.synth.make_boxes(1, 60, H, W, seed=int(rng.integers(1 << 30)), enlarge=en, D=D)
            bx += [tuple(int(v) for v in r) for r in b]
            s = int(rng.integers(4, 40))
            bx += [(W - s // 2, int(rng.integers(0, H)), s, s), (int(rng.integers(0, W)), H - s // 2, s, s), (0, 0, s, s)]
            for b in (edge_box(H, W, en, D), edge_box(H, W, en, 2 * D), sized_box(H, W, en, 2 * D + 1, 4 * D, rng)):
                if b is not None:
                    bx.append(b)
        else:
            m = min(H, W)
            bx += [(0, 0, m, m), (W - m, H - m, m, m), (W // 2, H // 2, 1, 1), (0, H - 1, 1, 1)]
        rng.shuffle(bx)
        out.append(bx)
    boxes = np.array([b for bx in out for b in bx], np.int32).reshape(-1, 4)
    off = np.concatenate([[0], np.cumsum([len(bx) for bx in out])]).astype(np.int32)
    return boxes, off


def shapes_of(table):
    return tuple((int(e["H"]), int(e["W"])) for e in table)


def k1_windows(table, boxes, off, D):
    """K1-passing windows in chain order -> (coords, frame, clipped crops)."""
    co, fr, cl = [], [], []
    for f, (H, W) in enumerate(shapes_of(table)):
        for b in boxes[off[f]:off[f + 1]]:
            c = expand(b, FLAVOURS[D])
            if c is not None and min(clipped(c, H, W)[2:]) > 0:
                co.append(c); fr.append(f); cl.append(clipped(c, H, W))
    return np.array(co, np.int32).reshape(-1, 4), np.array(fr, np.int32), np.array(cl, np.int32).reshape(-1, 4)


def staged_bytes(table, boxes, off, D):
    """stage_mark + stage_copy restated per table entry: bytes of every distinct (entry, row, 32-byte sector) the ROIs touch."""
    _, fr, cl = k1_windows(table, boxes, off, D)
    sectors = set()
    for f, (cx, cy, cw, ch) in zip(fr.tolist(), cl.tolist()):
        s0, s1 = (3 * cx) >> 5, (3 * (cx + cw) - 1) >> 5
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
    W = [w for _, w in shapes_of(table)]
    return sum(min(32, 3 * W[f] - 32 * s) & ~15 for f, _, s in sectors)


# ---- oracle expectations ---------------------------------------------------------------------------------------------------
def expected_det(oracle, templates, frames, boxes, off):
    red6, blue6 = templates
    rec, counts = [], np.zeros(4, np.int64)
    for f, fr in enumerate(frames):
        o = oracle.detect_frame(np.ascontiguousarray(fr), boxes[off[f]:off[f + 1]], red6, blue6)
        rec += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
        counts += o["stage_counts"]
    return rec, counts.tolist()


def survivors(oracle, frames, boxes, off):
    out = []
    for f, fr in enumerate(frames):
        H, W = fr.shape[:2]
        b = boxes[off[f]:off[f + 1]]
        keep = np.array([(c := expand(x, 1.15)) is None or min(clipped(c, H, W)[2:]) > 0 for x in b], bool)   # (K1 drops empty crops)
        out.append(oracle_survivors(oracle, np.ascontiguousarray(fr), b[keep]))
    return out


def rec_model(sv, mode):
    gray = REC_MODES[mode][1]
    X = feats(sv, gray)
    return lda_model(X, gray) if mode.endswith("lda") else knn_model(X, gray, seed=23, ntrain=2000)


def expected_rec(sv, model, gray, boxes, table):
    rec, nsurv = [], 0
    for f, s in enumerate(sv):
        X = feats([s], gray)
        lab = predict(model, X)
        rec += [(f,) + tuple(int(x) for x in q) + (int(l), 0) for q, l in zip(s[0], lab) if l != 0]
        nsurv += len(s[0])
    return rec, nsurv


@functools.lru_cache(maxsize=None)
def chain_case(kind, seed=0):
    canvas, table, frames = batch(CHAIN_SIZES, kind, 3, seed)
    return canvas, table, frames


# ---- CPU: the inputs are in their regimes ----------------------------------------------------------------------------------
def test_ragged_inputs_are_in_their_regimes(oracle):
    for C in (3, 1):
        for kind in KINDS:
            canvas, table, frames = batch(STAGE_SIZES + TINY, kind, C)
            ext = [int(e["offset"]) + int(e["row_stride"]) * (int(e["H"]) - 1) + int(e["W"]) * C for e in table]
            assert max(ext) == len(canvas) and int(np.argmax(ext)) not in (0, len(table) - 1)
            assert np.array_equal(frames[0], frames[len(STAGE_SIZES) + len(TINY)])              # the alias
            off, rs = table["offset"], table["row_stride"]
            if kind == "a16":
                assert np.all(off % 16 == 0) and np.all(rs % 16 == 0)
            elif kind == "a4":
                assert np.all(off % 4 == 0) and np.all(rs % 4 == 0) and np.any(rs % 16)
            else:
                assert np.any(off % 2) and np.any(rs % 2)
    for kind in ("a16", "a4", "odd"):
        _, table, _ = chain_case(kind)
        stage16 = np.all(table["offset"] % 16 == 0) and np.all(table["row_stride"] % 16 == 0) and np.all(3 * table["W"] % 16 == 0)
        assert stage16 == (kind == "a16"), kind
    # the recognition models decide every survivor clear of the chain's descriptor error
    _, table, frames = chain_case("a4")
    boxes, off = boxes_for(shapes_of(table), 32)
    sv = survivors(oracle, frames, boxes, off)
    for mode, (_, gray) in REC_MODES.items():
        model = rec_model(sv, mode)
        assert robust(model, feats(sv, gray), gray), mode
        rec, _ = expected_rec(sv, model, gray, boxes, table)
        assert len(rec) > 5 and len({r[0] for r in rec}) >= 3, mode


def test_frame_table_packing(tsd):
    """The engine's packing: 16-byte aligned offsets, rows back to back, same-shape lists and ndarrays take the uniform call."""
    from tsd_b200 import engine
    assert C.sizeof(tsd._capi.FrameDesc) == 24 and tsd.FRAME_DESC_DTYPE.itemsize == 24
    assert [tsd._capi.FrameDesc.offset.offset, tsd._capi.FrameDesc.row_stride.offset, tsd._capi.FrameDesc.H.offset,
            tsd._capi.FrameDesc.W.offset] == [0, 8, 16, 20]
    assert [tsd.FRAME_DESC_DTYPE.fields[k][1] for k in ("offset", "row_stride", "H", "W")] == [0, 8, 16, 20]
    t, n = engine.frame_table([(2, 3), (1, 1), (5, 7)], 3)
    assert t["offset"].tolist() == [0, 32, 48] and t["row_stride"].tolist() == [9, 3, 21] and n == 48 + 112
    t, n = engine.frame_table([(2, 3), (1, 1)], 1)
    assert t["offset"].tolist() == [0, 16] and t["row_stride"].tolist() == [3, 1] and n == 32
    a, b = np.zeros((4, 5, 3), np.uint8), np.zeros((4, 6, 3), np.uint8)
    assert not engine.is_mixed([a, a.copy()]) and not engine.is_mixed(np.stack([a, a])) and engine.is_mixed([a, b])
    assert isinstance(engine.stack_if_uniform([a, a]), np.ndarray) and isinstance(engine.stack_if_uniform([a, b]), list)
    assert engine.as_frame_table([(0, 9, 2, 3)]).tolist() == [(0, 9, 2, 3)]


# ---- GPU -------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def make_ctx(tsd, monkeypatch):
    made = []

    def mk(flavour="det", env=None):
        for k in ("TSD_STAGE", "TSD_STAGE_CHUNK", "TSD_CHUNK_FRAMES", "TSD_ZEROCOPY", "TSD_OVERLAP", "TSD_GRAPH"):
            monkeypatch.delenv(k, raising=False)
        for k, v in (env or {}).items():
            monkeypatch.setenv(k, v)
        c = tsd.Context(0, flavour)
        made.append(c)
        return c
    yield mk
    for c in made:
        c.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", 0))


@pytest.mark.gpu
def test_crop_resize_and_windows_ragged(oracle, make_ctx):
    """tsd_crop_resize_ragged (host / device, C = 3 / 1, D = 25 / 32 / 20) and tsd_windows_ragged (both flavours) on every table
    layout: windows, coords and offsets equal oracle.crop_resize / expand_boxes frame by frame.  Device calls add empty crops."""
    import torch
    A = _lib()
    ctx = make_ctx("det")
    bad = []
    for kind in KINDS:
        for Cn in (3, 1):
            canvas, table, frames = batch(STAGE_SIZES + TINY, kind, Cn)
            d_canvas = _dev(canvas)
            F = len(table)
            for D in (25, 32, 20):
                boxes, off = boxes_for(shapes_of(table), 25 if D == 20 else D)
                co, fr, _ = k1_windows(table, boxes, off, 25 if D == 20 else D)
                exp = np.stack([oracle.crop_resize(np.ascontiguousarray(frames[f]), c, D) for c, f in zip(co, fr)])
                got = np.empty_like(exp)
                A.check(ctx._L.tsd_crop_resize_ragged(ctx._h, A.ptr(canvas), A.ptr(table), F, Cn, A.ptr(co), A.ptr(fr), len(co), D,
                                                      A.ptr(got), A.MEM_HOST))
                if not np.array_equal(got, exp):
                    bad.append((kind, Cn, D, "host", sorted(set(fr[np.any((got != exp).reshape(len(co), -1), 1)].tolist()))))
                H, W = table["H"], table["W"]
                ec = np.array([[W[f] + 1, 0, W[f] + 9, H[f]] for f in (0, 2)] + [[0, H[f], W[f], H[f] + 5] for f in (3, F - 1)], np.int32)
                dco = np.concatenate([co, ec]); dfr = np.concatenate([fr, np.array([0, 2, 3, F - 1], np.int32)])
                perm = np.random.default_rng(len(co)).permutation(len(dco))
                t_out = torch.full((len(dco) * D * D * Cn,), 77, dtype=torch.uint8, device="cuda")
                t_co, t_fr = _dev(dco[perm]), _dev(dfr[perm])
                A.check(ctx._L.tsd_crop_resize_ragged(ctx._h, A.ptr(d_canvas.data_ptr()), A.ptr(table), F, Cn, A.ptr(t_co.data_ptr()),
                                                      A.ptr(t_fr.data_ptr()), len(dco), D, A.ptr(t_out.data_ptr()), A.MEM_DEVICE))
                ctx.synchronize()
                gd = t_out.cpu().numpy().reshape((len(dco),) + exp.shape[1:])
                full = np.concatenate([exp, np.zeros((len(ec),) + exp.shape[1:], np.uint8)])[perm]
                if not np.array_equal(gd, full):
                    bad.append((kind, Cn, D, "device"))
                if Cn == 3 and D != 20:
                    nb = len(boxes)
                    win = np.empty((nb, D, D, 3), np.uint8); coords = np.empty((nb, 4), np.int32)
                    woff = np.empty(F + 1, np.int32); tot = C.c_int32()
                    A.check(ctx._L.tsd_windows_ragged(ctx._h, A.ptr(canvas), A.ptr(table), F, A.ptr(boxes), A.ptr(off), FLAVOURS[D], D,
                                                      A.ptr(win), A.ptr(coords), A.ptr(woff), C.byref(tot), A.MEM_HOST))
                    n = tot.value
                    eoff = np.searchsorted(fr, np.arange(F + 1)).astype(np.int32)
                    if not (n == len(co) and np.array_equal(woff, eoff) and np.array_equal(coords[:n], co) and np.array_equal(win[:n], exp)):
                        bad.append((kind, D, "windows"))
    assert not bad, bad


def _ragged_call(ctx, mode, mem, base, table, boxes, off, cap, d_keep):
    """One tsd_detect_frames_ragged / enqueue call -> (rc, records, ndet, counts)."""
    A = _lib()
    det = np.zeros(max(cap, 1), A.DET_DTYPE); nd = C.c_int32(-1); counts = np.full(4, -1, np.int32)
    if mem == "device":
        d_base, d_boxes, d_off = d_keep
        rc = ctx._L.tsd_detect_frames_ragged(ctx._h, mode, A.ptr(d_base.data_ptr()), A.ptr(table), len(table), A.ptr(d_boxes.data_ptr()),
                                             A.ptr(d_off.data_ptr()), A.ptr(det), cap, C.byref(nd), A.ptr(counts), A.MEM_DEVICE)
    else:
        rc = ctx._L.tsd_detect_frames_ragged(ctx._h, mode, A.ptr(base), A.ptr(table), len(table), A.ptr(boxes), A.ptr(off), A.ptr(det), cap,
                                             C.byref(nd), A.ptr(counts), A.MEM_HOST)
    return rc, _records(det[:max(nd.value, 0)]), nd.value, counts.tolist()


def _route_inputs(ctx, route, canvas, boxes, off):
    mem = ROUTES[route][0]
    if mem == "pinned":
        ctx.pin(canvas)
    return (_dev(canvas), _dev(boxes), _dev(off)) if mem == "device" else None


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("mode", ["det"] + list(REC_MODES))
def test_chain_ragged(oracle, templates, make_ctx, mode, route):
    """The whole chain on one mixed table (aliased entry, sub-rectangle view, buffer-ending middle entry) through one route: records
    and counts equal the oracle's in table order; page-locked routes stage exactly the marked sectors (gather: none); det_cap = 0
    gives TSD_E_NOMEM with *ndet and the counts filled, and the next call is right."""
    A = _lib()
    mem, env, kind = ROUTES[route]
    D = 25 if mode == "det" else 32
    ctx = make_ctx("det" if mode == "det" else "rec", env)
    canvas, table, frames = chain_case(kind)
    if route == "gather":
        assert not np.all(table["offset"] % 16 == 0) or not np.all(table["row_stride"] % 16 == 0)
    boxes, off = boxes_for(shapes_of(table), D)
    if mode == "det":
        ctx.set_templates(*templates)
        exp, ecounts = expected_det(oracle, templates, frames, boxes, off)
        run_mode = A.RUN_DETECT
    else:
        run_mode, gray = REC_MODES[mode]
        sv = survivors(oracle, frames, boxes, off)
        model = rec_model(sv, mode)
        set_model(ctx, model)
        exp, nsurv = expected_rec(sv, model, gray, boxes, table)
        ecounts = [len(boxes), len(k1_windows(table, boxes, off, D)[0]), nsurv, len(exp)]
    keep = _route_inputs(ctx, route, canvas, boxes, off)
    try:
        if mem == "pinned":
            ctx.stat_staged_bytes(reset=True)
        rc, got, nd, counts = _ragged_call(ctx, run_mode, mem, canvas, table, boxes, off, len(boxes), keep)
        A.check(rc)
        assert counts == list(ecounts), (counts, ecounts)
        if got != exp:
            diff = [f for f in range(len(table)) if [r for r in got if r[0] == f] != [r for r in exp if r[0] == f]]
            pytest.fail("frames differ: %s" % diff)
        if mem == "pinned":
            want = staged_bytes(table, boxes, off, D) if route != "gather" else 0
            assert ctx.stat_staged_bytes(reset=True) == want
        if len(exp):
            rc, _, nd, counts = _ragged_call(ctx, run_mode, mem, canvas, table, boxes, off, 0, keep)
            assert rc == -4 and nd == len(exp) and counts == list(ecounts), (rc, nd, counts)
            rc, got, _, _ = _ragged_call(ctx, run_mode, mem, canvas, table, boxes, off, len(exp), keep)
            assert rc == 0 and got == exp
    finally:
        if mem == "pinned":
            ctx.unpin(canvas)


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(ROUTES))
def test_uniform_batch_as_table(oracle, templates, make_ctx, route):
    """A uniform batch (5 frames of 1360 x 800 at a padded frame stride) written as a table: the same records and counts as
    tsd_detect_frames / tsd_enqueue_frames, the same windows as tsd_windows and tsd_crop_resize, the same staged bytes."""
    import tsd_b200
    A = _lib()
    mem, env, _ = ROUTES[route]
    ctx = make_ctx("det", dict(env, TSD_STAGE_CHUNK="2") if route == "staged_chunks" else env)
    ctx.set_templates(*templates)
    F, H, W = 5, 800, 1360
    rs = 4096 if route != "gather" else 4084
    fs = rs * H + (32 if route != "gather" else 12)
    raw = np.empty(fs * F + 8192, np.uint8)
    canvas = raw[(-raw.ctypes.data) % 4096:][:fs * (F - 1) + rs * (H - 1) + 3 * W]
    canvas[:] = 0
    for f, img in enumerate(tsd_b200.synth.make_frames(F, H, W, seed=99)):
        np.lib.stride_tricks.as_strided(canvas[f * fs:], (H, W, 3), (rs, 3, 1))[...] = img
    table = np.array([(f * fs, rs, H, W) for f in range(F)], A.FRAME_DESC_DTYPE)
    boxes, off = tsd_b200.synth.make_boxes(F, 150, H, W)
    keep = _route_inputs(ctx, route, canvas, boxes, off)
    try:
        for rep in range(2):
            if mem == "pinned":
                ctx.stat_staged_bytes(reset=True)
            det = np.zeros(len(boxes), A.DET_DTYPE); nd = C.c_int32(); cu = np.zeros(4, np.int32)
            if mem == "device":
                d_base, d_boxes, d_off = keep
                A.check(ctx._L.tsd_detect_frames(ctx._h, A.RUN_DETECT, A.ptr(d_base.data_ptr()), F, H, W, rs, fs, A.ptr(d_boxes.data_ptr()),
                                                 A.ptr(d_off.data_ptr()), A.ptr(det), len(det), C.byref(nd), A.ptr(cu), A.MEM_DEVICE))
            else:
                A.check(ctx._L.tsd_detect_frames(ctx._h, A.RUN_DETECT, A.ptr(canvas), F, H, W, rs, fs, A.ptr(boxes), A.ptr(off), A.ptr(det),
                                                 len(det), C.byref(nd), A.ptr(cu), A.MEM_HOST))
            uni = _records(det[:nd.value])
            su = ctx.stat_staged_bytes(reset=True) if mem == "pinned" else 0
            rc, rag, _, rcounts = _ragged_call(ctx, A.RUN_DETECT, mem, canvas, table, boxes, off, len(boxes), keep)
            A.check(rc)
            sr = ctx.stat_staged_bytes(reset=True) if mem == "pinned" else 0
            assert rag == uni and rcounts == cu.tolist() and sr == su, (rep, rcounts, cu.tolist(), sr, su)
        assert len(uni) > 0
        exp, _ = expected_det(oracle, templates, [np.lib.stride_tricks.as_strided(canvas[f * fs:], (H, W, 3), (rs, 3, 1)) for f in range(F)], boxes, off)
        assert uni == exp
        if route == "pageable":                              # the per-stage calls
            co = np.array([[0, 0, 30, 30], [100, 90, 190, 200], [W - 50, H - 40, W + 9, H + 3]], np.int32)
            wf = np.array([0, 2, 4], np.int32)
            a = np.empty((3, 25, 25, 3), np.uint8); b = np.empty_like(a)
            A.check(ctx._L.tsd_crop_resize(ctx._h, A.ptr(canvas), F, H, W, rs, fs, 3, A.ptr(co), A.ptr(wf), 3, 25, A.ptr(a), A.MEM_HOST))
            A.check(ctx._L.tsd_crop_resize_ragged(ctx._h, A.ptr(canvas), A.ptr(table), F, 3, A.ptr(co), A.ptr(wf), 3, 25, A.ptr(b), A.MEM_HOST))
            assert np.array_equal(a, b)
            outs = []
            for fn in ("u", "r"):
                win = np.empty((len(boxes), 25, 25, 3), np.uint8); cc = np.empty((len(boxes), 4), np.int32); wo = np.empty(F + 1, np.int32); t = C.c_int32()
                if fn == "u":
                    A.check(ctx._L.tsd_windows(ctx._h, A.ptr(canvas), F, H, W, rs, fs, A.ptr(boxes), A.ptr(off), 1.3, 25, A.ptr(win), A.ptr(cc), A.ptr(wo), C.byref(t), A.MEM_HOST))
                else:
                    A.check(ctx._L.tsd_windows_ragged(ctx._h, A.ptr(canvas), A.ptr(table), F, A.ptr(boxes), A.ptr(off), 1.3, 25, A.ptr(win), A.ptr(cc), A.ptr(wo), C.byref(t), A.MEM_HOST))
                outs.append((win[:t.value], cc[:t.value], wo))
            assert all(np.array_equal(x, y) for x, y in zip(*outs))
    finally:
        if mem == "pinned":
            ctx.unpin(canvas)


@pytest.mark.gpu
def test_ragged_sequences(oracle, templates, make_ctx):
    """Ragged and uniform enqueues alternate on one context (two-slot overlap, CUDA graphs); two tables that differ only in their
    offsets (frames of equal sizes swapped) share a captured graph, so replays run with another table's contents.  Every batch is
    fetched with tsd_fetch_previous while the next runs (the last with tsd_fetch_detections) and equals the oracle."""
    import tsd_b200
    A = _lib()
    ctx = make_ctx("det")
    ctx.set_templates(*templates)
    sizes = ((800, 1360), (1080, 1920), (800, 1360), (1080, 1920))
    canvas, base_t, frames = batch(sizes, "a4", 3, 5)
    t1 = base_t[:4].copy()
    t2 = t1[[2, 3, 0, 1]].copy()                                   # same sizes per entry, same extent: the same graph key
    boxes, off = boxes_for(shapes_of(t1), 25, 7)
    exp1, _ = expected_det(oracle, templates, [frames[i] for i in range(4)], boxes, off)
    exp2, _ = expected_det(oracle, templates, [frames[i] for i in (2, 3, 0, 1)], boxes, off)
    Fu, Hu, Wu = 3, 480, 640
    uni = tsd_b200.synth.make_frames(Fu, Hu, Wu, seed=8)
    ub, uo = tsd_b200.synth.make_boxes(Fu, 80, Hu, Wu, seed=9)
    expu, _ = expected_det(oracle, templates, list(uni), ub, uo)
    d_canvas, d_boxes, d_off, d_uni, d_ub, d_uo = (_dev(x) for x in (canvas, boxes, off, uni, ub, uo))
    maxb = int(np.diff(off).max())
    plan = ["r1", "r2", "u"] * 5
    want = {"r1": exp1, "r2": exp2, "u": expu}
    g0 = ctx.stat_graphs()
    got = []
    for i, k in enumerate(plan):
        if k == "u":
            ctx.enqueue_frames(d_uni.data_ptr(), Fu, Hu, Wu, d_ub.data_ptr(), d_uo.data_ptr(), len(ub), max_boxes_per_frame=80)
        else:
            ctx.enqueue_frames_ragged(d_canvas.data_ptr(), t1 if k == "r1" else t2, d_boxes.data_ptr(), d_off.data_ptr(), len(boxes),
                                      max_boxes_per_frame=maxb)
        if i:
            got.append(_records(ctx.fetch_detections(len(boxes) + len(ub), previous=True)[0]))
    got.append(_records(ctx.fetch_detections(len(boxes) + len(ub))[0]))
    bad = [(i, k) for i, k in enumerate(plan) if got[i] != want[k]]
    assert not bad, bad
    cap, rep = ctx.stat_graphs()
    assert cap - g0[0] >= 2 and rep - g0[1] >= 4, (cap, rep)


@pytest.mark.gpu
def test_real_frames_ragged(oracle, templates, make_ctx, det_full150, jpeg24, frames3, det_frames, resultado150):
    """The 24 JPEG and 3 PNG golden frames plus rescaled copies of some (cv2.resize; boxes from cv2.MSER with the reference's
    parameters) in one batch, pageable and page-locked: every frame equals the oracle; the unscaled frames give their lines of
    the reference's resultado.txt."""
    import cv2
    import tsd_b200
    from conftest import STORED
    ctx = make_ctx("det")
    ctx.set_templates(*templates)
    g = det_full150
    frames, boxes, files = [], [], []
    for i, f in enumerate(jpeg24["index"]):
        frames.append(jpeg24["frames"][i]); boxes.append(g["boxes"][g["box_offsets"][f]:g["box_offsets"][f + 1]]); files.append(jpeg24["files"][i])
    for k in STORED:
        frames.append(frames3[k]); boxes.append(det_frames[k + "_boxes"]); files.append(k + ".jpg")
    mser = cv2.MSER_create(delta=7, min_area=200, max_area=2000, max_variation=0.15)
    n_orig = len(frames)
    for i, size in ((0, (1920, 1080)), (5, (680, 400)), (24, (2040, 1200)), (11, (1000, 700))):
        img = cv2.resize(frames[i], size)
        frames.append(img); boxes.append(tsd_b200.source_det.proposals(img, mser)); files.append("scaled_%d.jpg" % i)
    order = np.random.default_rng(3).permutation(len(frames))
    frames = [frames[i] for i in order]; boxes = [boxes[i] for i in order]; files = [files[i] for i in order]
    off = np.concatenate([[0], np.cumsum([len(b) for b in boxes])]).astype(np.int32)
    allb = np.concatenate(boxes).astype(np.int32)
    exp, ecounts = expected_det(oracle, templates, frames, allb, off)
    det, counts = ctx.detect_frames(frames, allb, off)
    assert _records(det) == exp and counts.tolist() == ecounts
    lines = ["%s;%d;%d;%d;%d;%d;%s" % (files[r[0]], r[1], r[2], r[3], r[4], r[5], str(r[6] / 100)) for r in exp if order[r[0]] < n_orig]
    mine = set(files[i] for i in range(len(files)) if order[i] < n_orig)
    assert sorted(lines) == sorted(ln for ln in resultado150 if ln.split(";")[0] in mine)
    assert sum(1 for r in exp if order[r[0]] >= n_orig) > 0
    # pageable: the same list as one contiguous-per-frame host buffer through the pageable route
    canvas = np.concatenate([f.reshape(-1) for f in frames])
    table = np.zeros(len(frames), tsd_b200.FRAME_DESC_DTYPE)
    table["offset"] = np.concatenate([[0], np.cumsum([f.size for f in frames])[:-1]])
    table["row_stride"] = [f.shape[1] * 3 for f in frames]; table["H"] = [f.shape[0] for f in frames]; table["W"] = [f.shape[1] for f in frames]
    rc, got, _, gcounts = _ragged_call(ctx, 1, "pageable", canvas, table, allb, off, len(allb), None)
    assert rc == 0 and got == exp and gcounts == ecounts


@pytest.mark.gpu
def test_dropins_mixed_sizes(tsd, templates, frames3, det_frames):
    """extractMSERDetectionsGray, orderCroppedImagesByImageFile, detectBatch and recognizeBatch on frames of mixed sizes equal the same
    functions called one frame at a time."""
    import cv2
    S, R = tsd.source_det, tsd.source_rec
    base = [frames3[k] for k in sorted(frames3)]
    imgs = [base[0], cv2.resize(base[1], (1920, 1080)), base[2], cv2.resize(base[0], (800, 600))]
    names = ["f%d.jpg" % i for i in range(len(imgs))]
    train = dict(zip(names, imgs))
    mser = cv2.MSER_create(delta=7, min_area=200, max_area=2000, max_variation=1.0)
    whole = R.extractMSERDetectionsGray(train, mser)
    for n in names:
        one = R.extractMSERDetectionsGray({n: train[n]}, mser)[n]
        assert [d[1] for d in whole[n]] == [d[1] for d in one] and all(np.array_equal(a[0], b[0]) for a, b in zip(whole[n], one)), n
    results = [(n, 5 + i, 7, 60 + 3 * i, 70, 1 + i % 6) for i, n in enumerate(names)] + [(names[1], 1500, 900, 1900, 1070, 2)]
    whole = R.orderCroppedImagesByImageFile(train, results)
    for n in names:
        one = R.orderCroppedImagesByImageFile({n: train[n]}, [r for r in results if r[0] == n])[n]
        assert [d[1:] for d in whole[n]] == [d[1:] for d in one] and all(np.array_equal(a[0], b[0]) for a, b in zip(whole[n], one)), n
    red6, blue6 = templates
    red = [(red6[k], S.SIGNALLIST[k]) for k in range(6)]; blue = [(blue6[k], S.SIGNALLIST[k]) for k in range(6)]
    mser_d = cv2.MSER_create(delta=7, min_area=200, max_area=2000, max_variation=0.15)
    bx = [S.proposals(im, mser_d) for im in imgs]
    off = np.concatenate([[0], np.cumsum([len(b) for b in bx])]).astype(np.int32)
    allb = np.concatenate(bx)
    out, counts = S.detectBatch(imgs, allb, off, names, red, blue)
    one = []
    for i in range(len(imgs)):
        o, _ = S.detectBatch(imgs[i][None], bx[i], np.array([0, len(bx[i])], np.int32), [names[i]], red, blue)
        one += o
    assert out == one
    rg = np.load(os.path.join(ROOT, "tests", "golden", "rec_golden.npz"))
    R.context().set_lda(rg["lda_W"], rg["lda_b"])
    clf = [type("LDA", (), {"coef_": rg["lda_W"][:, c][None], "intercept_": rg["lda_b"][c:c + 1]})() for c in range(6)]
    out, _ = R.recognizeBatch(imgs, allb, off, names, (clf, "LDABAYES"), None, (None, "HOG"))
    one = []
    for i in range(len(imgs)):
        o, _ = R.recognizeBatch(imgs[i][None], bx[i], np.array([0, len(bx[i])], np.int32), [names[i]], (clf, "LDABAYES"), None, (None, "HOG"))
        one += o
    assert out == one


@pytest.mark.gpu
def test_ragged_limits(oracle, templates, make_ctx):
    """Every invalid table field: TSD_E_INVALID before any device work from every ragged entry point, and the next valid call is
    right.  A device table whose offsets reach past 4 GiB works."""
    import torch
    import tsd_b200
    A = _lib()
    ctx = make_ctx("det")
    ctx.set_templates(*templates)
    frames = tsd_b200.synth.make_frames(2, 480, 640, seed=4)
    canvas = np.ascontiguousarray(frames).reshape(-1)
    good = np.array([(0, 1920, 480, 640), (480 * 1920, 1920, 480, 640)], A.FRAME_DESC_DTYPE)
    boxes, off = tsd_b200.synth.make_boxes(2, 80, 480, 640, seed=5)
    exp, ecounts = expected_det(oracle, templates, list(frames), boxes, off)
    d_canvas, d_boxes, d_off = _dev(canvas), _dev(boxes), _dev(off)
    bads = {"H0": ("H", 0), "W0": ("W", 0), "Hneg": ("H", -3), "rs_small": ("row_stride", 1919), "offset_neg": ("offset", -16),
            "2GiB": ("row_stride", (1 << 31) // 480 + 16)}
    co = np.array([[0, 0, 30, 30]], np.int32); wf = np.zeros(1, np.int32); out = np.zeros(25 * 25 * 3, np.uint8)
    det = np.zeros(8, A.DET_DTYPE); nd = C.c_int32(); cnt = np.zeros(4, np.int32); tot = C.c_int32(); woff = np.zeros(3, np.int32)
    for name, (field, v) in bads.items():
        t = good.copy(); t[1][field] = v
        calls = {
            "crop_resize": lambda m, p: ctx._L.tsd_crop_resize_ragged(ctx._h, p, A.ptr(t), 2, 3, A.ptr(co), A.ptr(wf), 1, 25, A.ptr(out), m),
            "windows": lambda m, p: ctx._L.tsd_windows_ragged(ctx._h, p, A.ptr(t), 2, A.ptr(boxes), A.ptr(off), 1.3, 25, A.ptr(out), A.ptr(co),
                                                              A.ptr(woff), C.byref(tot), m),
            "detect": lambda m, p: ctx._L.tsd_detect_frames_ragged(ctx._h, 1, p, A.ptr(t), 2, A.ptr(boxes) if m == A.MEM_HOST else A.ptr(d_boxes.data_ptr()),
                                                                   A.ptr(off) if m == A.MEM_HOST else A.ptr(d_off.data_ptr()), A.ptr(det), 8, C.byref(nd), A.ptr(cnt), m),
            "enqueue": lambda m, p: ctx._L.tsd_enqueue_frames_ragged(ctx._h, 1, A.ptr(d_canvas.data_ptr()), A.ptr(t), 2, A.ptr(d_boxes.data_ptr()),
                                                                     A.ptr(d_off.data_ptr()), len(boxes), 80),
        }
        for what, fn in calls.items():
            for m, p in ((A.MEM_HOST, A.ptr(canvas)), (A.MEM_DEVICE, A.ptr(d_canvas.data_ptr()))):
                if what in ("windows", "enqueue") and m == A.MEM_DEVICE:
                    continue
                assert fn(m, p) == -1, (name, what, m)
    for n in (0, 1 << 23):
        assert ctx._L.tsd_enqueue_frames_ragged(ctx._h, 1, A.ptr(d_canvas.data_ptr()), A.ptr(good), n, A.ptr(d_boxes.data_ptr()),
                                                A.ptr(d_off.data_ptr()), len(boxes), 80) == -1
    assert ctx._L.tsd_detect_frames_ragged(ctx._h, 1, A.ptr(canvas), None, 2, A.ptr(boxes), A.ptr(off), A.ptr(det), 8, C.byref(nd), A.ptr(cnt), A.MEM_HOST) == -1
    det, counts = ctx.detect_frames([frames[0], frames[1][:400, :600]], np.concatenate([boxes[:80], boxes[80:]]), off)
    exp2, ecounts2 = expected_det(oracle, templates, [frames[0], frames[1][:400, :600]], boxes, off)
    assert _records(det) == exp2 and counts.tolist() == ecounts2
    # offsets past 4 GiB: three 4K frames at 0, 4 GiB + 16 and the end of a 5.2 GiB device buffer
    H, W = 2160, 3840
    big = tsd_b200.synth.make_frames(3, H, W, seed=6)
    fb = H * W * 3
    offs = [0, (1 << 32) + 16, 5_200_000_000 - fb]
    d_big = torch.zeros(5_200_000_000, dtype=torch.uint8, device="cuda")
    for o, img in zip(offs, big):
        d_big[o:o + fb].copy_(torch.from_numpy(img.reshape(-1)))
    t = np.array([(o, W * 3, H, W) for o in offs], A.FRAME_DESC_DTYPE)
    bb, bo = tsd_b200.synth.make_boxes(3, 120, H, W, seed=7)
    expb, ecb = expected_det(oracle, templates, list(big), bb, bo)
    d_bb, d_bo = _dev(bb), _dev(bo)
    ctx.enqueue_frames_ragged(d_big.data_ptr(), t, d_bb.data_ptr(), d_bo.data_ptr(), len(bb))
    det, counts = ctx.fetch_detections(len(bb))
    assert _records(det) == expb and counts.tolist() == ecb
    del d_big
