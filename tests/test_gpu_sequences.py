"""Call sequences on long-lived contexts against the oracle.

A context keeps state between calls: two scratch slots and two internal streams, a cache of CUDA graphs keyed by batch shape and
scratch pointers, grow-only scratch, per-slot tickets, work lists, order arrays, staging maps and mirrors, the batch before the
last one (tsd_fetch_previous), and setters that join the running batch.  A kernel that reads a word no producer of its batch
rewrote gives the right answer whenever the previous batch had the same contents, so every test here changes the contents
between batches and checks each fetched batch, record by record and with its stage counts, against the oracle for the model
state in effect when it was enqueued.

  pool          seeded synth frames with boxes cut per frame to ragged counts: frames of 0, 1, 31, 32, 33 and 200 boxes, a
                batch of no boxes, a batch whose boxes all fail the aspect test, a single frame, a 4K batch with a frame of more
                than 1024 aspect-passing windows (the general fold), a batch large enough to grow the slot layout.
  streaming     fixed device buffers rewritten with new frames and new boxes every step (same nb and max_boxes_per_frame,
                other per-frame counts), fetched directly and through fetch_detections(previous=True), for TSD_GRAPH x
                TSD_OVERLAP x TSD_STAGGER x {detect, recognise}; the exact graph captures and replays the capture rule implies.
                Page-locked frames rewritten in place (staged, 2 and 3 chunks) and pageable frames in chunks.
  interleaved   a seeded sequence of ~60 operations on one overlapped context: enqueues from the pool, fetch last / previous,
                flush, synchronize, host-pointer stage calls, device-pointer crop_resize, template and similarity-table
                changes, profiling modes, stat_hist_entries.  A plain model decides when fetch previous must succeed.
  modes         RUN_DETECT and RUN_RECOGNIZE alternating on one D = 32 context; two contexts interleaved.
  recovery      refused calls (bad strides, no templates, det_cap too small, max_boxes_per_frame too small) in a stream.

test_sequences_reach_their_regimes checks on the CPU that the pool and the sequences reach every case named above.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from test_gpu_recognition import decision_margin, oracle_rec_frame

E_INVALID, E_STATE, E_NOMEM = -1, -3, -4
H, W = 800, 1360
H4, W4 = 2160, 3840
GRAPH_CAP = 8                                                # graphs kept = keys remembered from eager runs (tsd_capi.cu)


# ---- models of the library's host state ---------------------------------------------------------------------------
def pair_row_words(m):
    return (max(min(m, 1024), 1) + 31) // 32


def todo_capacity(nf, m):
    nbk = (min(m, 1024) + 127) // 128
    return nf * max(1, nbk * (nbk + 1) // 2) + 2


class SlotModel:
    """enqueue_impl's slot choice and slot-layout growth (sticky maxima) in overlap mode."""

    def __init__(self):
        self.slot, self.cap, self.fcap, self.rw, self.todo = 0, 0, 0, 1, 0

    def enqueue(self, nf, nb, maxb):
        self.slot ^= 1
        need_w = (max(nb, 1) + 3) & ~3
        sw, sf = (need_w + 63) & ~63, (nf + 2 + 63) & ~63
        rw, todo = pair_row_words(maxb), 2 * todo_capacity(nf, maxb)
        grew = sw > self.cap or sf > self.fcap or rw > self.rw or todo > self.todo
        self.cap, self.fcap, self.rw, self.todo = max(self.cap, sw), max(self.fcap, sf), max(self.rw, rw), max(self.todo, todo)
        return self.slot, grew


class GraphModel:
    """run_chain's capture rule: eager on a key's first sighting, captured when it comes back while among the last GRAPH_CAP
    eagerly run keys, replayed while cached (GRAPH_CAP graphs, least recently used evicted)."""

    def __init__(self, on=True):
        self.on, self.graphs, self.seen, self.captured, self.replayed = on, [], [], 0, 0

    def run(self, key):
        if not self.on:
            return
        if key in self.graphs:
            self.graphs.remove(key); self.graphs.append(key); self.replayed += 1
        elif key in self.seen:
            self.seen.remove(key); self.captured += 1
            if len(self.graphs) >= GRAPH_CAP:
                self.graphs.pop(0)
            self.graphs.append(key)
        else:
            if len(self.seen) >= GRAPH_CAP:
                self.seen.pop(0)
            self.seen.append(key)


# ---- inputs ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(None)
def base_frames():
    from tsd_b200 import synth
    return synth.make_frames(8, seed=synth.FRAME_SEED + 700)


@functools.lru_cache(None)
def frames_4k():
    from tsd_b200 import synth
    return synth.make_frames(2, H=H4, W=W4, seed=synth.FRAME_SEED + 701, nrect=96)


def ragged_boxes(counts, seed, H_=H, W_=W, square=False):
    """Per frame f the first counts[f] boxes of a synth.make_boxes frame of max(counts) boxes (ragged CSR)."""
    from tsd_b200 import synth
    m = max(max(counts), 1)
    b, _ = synth.make_boxes(len(counts), m, H=H_, W=W_, seed=synth.BOX_SEED + seed)
    b = b.reshape(len(counts), m, 4)
    if square:                                               # every box passes the aspect test
        b[:, :, 3] = b[:, :, 2]
        b[:, :, 1] = np.minimum(b[:, :, 1], H_ - b[:, :, 3])
    boxes = np.concatenate([b[f, :c] for f, c in enumerate(counts)] + [np.zeros((0, 4), np.int32)]).astype(np.int32)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    return boxes, off


# name -> (frame source, frame indices, per-frame box counts, box seed, options)
POOL = {
    "ragged":   ("base", (0, 1, 2, 3, 4, 5), (0, 1, 31, 32, 33, 200), 11, {}),
    "ragged_b": ("base", (6, 7, 0, 1, 2), (33, 200, 1, 0, 32), 12, {}),
    "empty":    ("base", (3, 4, 5), (0, 0, 0), 13, {}),
    "aspect":   ("base", (1, 2), (40, 40), 14, {"aspect_fail": True}),
    "single":   ("base", (5,), (57,), 15, {}),
    "big4k":    ("4k", (0, 1), (1150, 3), 16, {"square": True}),
    "grow":     ("base", (0, 1, 2, 3, 4, 5, 6, 7), (300, 250, 17, 300, 0, 120, 300, 64), 17, {}),
    "c1":       ("base", (2, 6), (5, 9), 18, {}),
    "c2":       ("base", (7, 3, 4), (17, 0, 64), 19, {}),
    "c3":       ("base", (1, 2, 3, 4), (2, 2, 2, 2), 20, {}),
}


@functools.lru_cache(None)
def pool_batch(name):
    """-> (frames uint8[F,H,W,3], boxes int32[nb,4], offsets int32[F+1])."""
    src, idx, counts, seed, opt = POOL[name]
    fr = (frames_4k() if src == "4k" else base_frames())[list(idx)]
    Hh, Ww = fr.shape[1:3]
    boxes, off = ragged_boxes(counts, seed, Hh, Ww, square=opt.get("square", False))
    if opt.get("aspect_fail"):                               # w / h = 1/2 before and after any enlargement
        boxes[:, 3] = boxes[:, 2] * 2
        boxes[:, 1] = np.minimum(boxes[:, 1], Hh - boxes[:, 3])
    return fr, boxes, off


def maxb(off):
    return int(max(np.diff(off).max(initial=0), 1))


# ---- expected records -------------------------------------------------------------------------------------------------
def tuples(det, f0=0):
    return [(int(d["frame"]) + f0, int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"])) for d in det]


def expect_det(oracle, frames, boxes, off, red6, blue6, D=25, enlarge=1.30, cfg=None):
    """Records and stage counts of the detection chain, frame by frame from oracle.detect_frame."""
    recs, counts = [], np.zeros(4, np.int64)
    for f in range(len(frames)):
        kw = dict(cfg=cfg) if cfg is not None else {}
        o = oracle.detect_frame(frames[f], boxes[off[f]:off[f + 1]], red6, blue6, percentage=enlarge, D=D, **kw)
        counts += o["stage_counts"]
        recs += [(f,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
    return recs, counts.tolist()


def rec_survivors(oracle, frames, boxes, off):
    """Per frame: (aspect-passing count, survivor coords, survivor HOG descriptors) of the recognition flavour."""
    out = []
    for f in range(len(frames)):
        bb = boxes[off[f]:off[f + 1]]
        _, v = oracle.expand_boxes(bb, 1.15)
        c2, hog = oracle_rec_frame(oracle, frames[f], bb)
        out.append((int(np.sum(v)), c2, hog))
    return out


def expect_rec(oracle, frames, boxes, off, Wl, bl):
    recs, counts = [], [int(off[-1]), 0, 0, 0]
    for f, (npass, c2, hog) in enumerate(rec_survivors(oracle, frames, boxes, off)):
        counts[1] += npass; counts[2] += len(c2)
        if len(c2):
            _, lab = oracle.lda_predict(hog, Wl, bl, 0.5)
            recs += [(f,) + tuple(int(x) for x in cc) + (int(l), 0) for cc, l in zip(c2, lab) if l != 0]
    counts[3] = len(recs)
    return recs, counts


@functools.lru_cache(None)
def rec_weights():
    """324-feature LDA weights under which the streaming windows get every label, with every threshold placed in a gap of the
    logits: no window's decision is within reach of K7's rounding (checked by test_sequences_reach_their_regimes)."""
    rng = np.random.default_rng(77)
    Wl = rng.standard_normal((324, 6))
    return Wl, rng.standard_normal(6)


def gap_bias(hog, Wl, q=0.85):
    """b_c = -(midpoint of the widest gap between sorted logits of classifier c between the q-0.1 and q+0.1 quantiles)."""
    z = np.sort(hog.astype(np.float64) @ Wl, axis=0)
    n = len(z)
    lo, hi = int(n * (q - 0.1)), max(int(n * (q + 0.1)), int(n * (q - 0.1)) + 2)
    b = np.empty(6)
    for c in range(6):
        g = np.diff(z[lo:hi, c])
        k = int(np.argmax(g))
        b[c] = -(z[lo + k, c] + z[lo + k + 1, c]) / 2
    return b


# ---- streaming steps ----------------------------------------------------------------------------------------------------
SF, SNB, SMAX, SSTEPS = 4, 240, 100, 10
SCOUNTS = [(100, 40, 0, 100), (100, 100, 20, 20), (0, 100, 100, 40), (40, 100, 100, 0), (100, 0, 40, 100),
           (20, 20, 100, 100), (100, 70, 70, 0), (60, 100, 0, 80), (100, 1, 39, 100), (33, 100, 7, 100)]


@functools.lru_cache(None)
def stream_step(k, mode="det"):
    """Step k: SF new frames (pool frames rolled and permuted), SNB boxes with at most SMAX per frame, counts SCOUNTS[k]."""
    base = base_frames()
    perm = np.random.default_rng(500 + k).permutation(8)[:SF]
    frames = np.ascontiguousarray(np.roll(base[perm], 37 * k + 11, axis=2))
    boxes, off = ragged_boxes(SCOUNTS[k], 200 + k)
    assert int(off[-1]) == SNB and maxb(off) == SMAX
    return frames, boxes, off


@functools.lru_cache(None)
def stream_expected(k, mode):
    from tsd_b200 import synth  # noqa: F401  (frames come from synth via base_frames)
    import oracle.oracle as O
    O.build()
    frames, boxes, off = stream_step(k)
    if mode == "det":
        return expect_det(O, frames, boxes, off, *det_templates())
    return expect_rec(O, frames, boxes, off, *rec_model())


@functools.lru_cache(None)
def det_templates():
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "det_templates.npz"))
    return g["red6"], g["blue6"]


@functools.lru_cache(None)
def rec_model():
    """(W, b) of the recognition streams: random W, each threshold in a gap of the logits over every streaming window."""
    import oracle.oracle as O
    O.build()
    Wl, _ = rec_weights()
    hogs = [h for k in range(SSTEPS) for _, _, h in rec_survivors(O, *stream_step(k)) if len(h)]
    return Wl, gap_bias(np.concatenate(hogs), Wl)


def _lib():
    from tsd_b200 import _capi
    return _capi


def _ctx(tsd, monkeypatch, flavour, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ctx = tsd.Context(0, flavour)
    for k in env:
        monkeypatch.delenv(k)
    return ctx


def _setup(ctx, mode):
    if mode == "det":
        ctx.set_templates(*det_templates())
    else:
        ctx.set_lda(*rec_model())


def _run_mode(mode, tsd):
    return tsd.RUN_DETECT if mode == "det" else tsd.RUN_RECOGNIZE


class DeviceStream:
    """Fixed device buffers (frames, boxes, offsets) rewritten on the context's stream before each enqueue."""

    def __init__(self, ctx, nsets=1):
        import torch
        self.torch, self.ctx = torch, ctx
        dev = torch.device("cuda", 0)
        self.sets = [(torch.empty((SF, H, W, 3), dtype=torch.uint8, device=dev), torch.empty((SNB, 4), dtype=torch.int32, device=dev),
                      torch.empty((SF + 1,), dtype=torch.int32, device=dev)) for _ in range(nsets)]
        self.s = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def write(self, i, frames, boxes, off):
        fr, bx, of = self.sets[i]
        with self.torch.cuda.stream(self.s):                 # ordered before the next batch (it forks from the context's stream)
            fr.copy_(self.torch.from_numpy(frames)); bx.copy_(self.torch.from_numpy(boxes)); of.copy_(self.torch.from_numpy(off))

    def enqueue(self, i, mode, maxb_=SMAX):
        fr, bx, of = self.sets[i]
        self.ctx.enqueue_frames(fr.data_ptr(), SF, H, W, bx.data_ptr(), of.data_ptr(), SNB, mode=mode, max_boxes_per_frame=maxb_)


# ---- CPU: the pool and the sequences reach their regimes -----------------------------------------------------------------
def test_sequences_reach_their_regimes(oracle):
    counts = set()
    for name in POOL:
        fr, boxes, off = pool_batch(name)
        counts |= set(np.diff(off).tolist())
        assert len(boxes) == off[-1] and (np.diff(off) >= 0).all()
    assert {0, 1, 31, 32, 33, 200} <= counts                 # ragged and empty frames
    assert pool_batch("empty")[2][-1] == 0 and len(pool_batch("single")[0]) == 1
    fr, boxes, off = pool_batch("aspect")
    assert not oracle.expand_boxes(boxes, 1.30)[1].any() and not oracle.expand_boxes(boxes, 1.15)[1].any()
    fr, boxes, off = pool_batch("big4k")
    assert fr.shape[1:3] == (H4, W4) and oracle.expand_boxes(boxes[off[0]:off[1]], 1.30)[1].sum() > 1024     # general fold
    # streaming: same nb and maximum, other per-frame counts every step
    offs = {tuple(stream_step(k)[2].tolist()) for k in range(SSTEPS)}
    assert len(offs) == SSTEPS
    # recognition streams: every label occurs, no decision within reach of K7's rounding
    Wl, bl = rec_model()
    labs, margins = set(), []
    for k in range(SSTEPS):
        for _, c2, hog in rec_survivors(oracle, *stream_step(k)):
            if len(hog):
                z, lab = oracle.lda_predict(hog, Wl, bl, 0.5)
                labs |= set(lab.tolist()); margins.append(decision_margin(z, hog, Wl).min())
    assert labs == set(range(7)) and min(margins) > 1, (labs, min(margins))
    # the interleaved sequence: growth while the other slot is busy, a stage call between two batches of one slot, > 8 keys,
    # fetch previous both succeeding and refused, every operation kind
    ops = interleaved_ops()
    m = interleaved_model(ops)
    assert m["grew_busy"] and m["stage_between_same_slot"] and len(m["keys"]) > GRAPH_CAP
    assert m["prev_ok"] >= 3 and m["prev_refused"] >= 3
    assert {o[0] for o in ops} == set(OP_KINDS)
    r = [i for i, o in enumerate(ops) if o[0] == "replays"]     # the replayed batches: in slots, no layout change, fetch previous allowed
    assert r and all(m["out"][i + 1][0] == "prev" and m["out"][i - 1][1][2] is not None for i in r)
    # mode switching: a mode's scratch is first allocated while the other slot runs a batch of the other mode
    assert MODE_SEQ[0] != MODE_SEQ[1] and len(set(MODE_SEQ)) == 2


# ---- streaming with fixed pointers -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("det", "rec"))
@pytest.mark.parametrize("stagger", ("1", "0"))
@pytest.mark.parametrize("overlap", ("1", "0"))
@pytest.mark.parametrize("graph", ("1", "0"))
def test_streaming_fixed_buffers(tsd, monkeypatch, graph, overlap, stagger, mode):
    """SSTEPS steps of new frames and boxes in the same device buffers (same nb, same max_boxes_per_frame, other per-frame
    counts: the offsets are device data, not part of the graph key).  Every step is fetched and compared with the oracle; the
    captures and replays must be those the capture rule gives for the key sequence."""
    env = {"TSD_GRAPH": graph, "TSD_OVERLAP": overlap, "TSD_STAGGER": stagger}
    run = _run_mode(mode, tsd)
    flavour = "det" if mode == "det" else "rec"
    # direct: write, enqueue, fetch the last batch (one buffer set)
    ctx = _ctx(tsd, monkeypatch, flavour, env)
    try:
        _setup(ctx, mode)
        ds = DeviceStream(ctx)
        gm, slot = GraphModel(graph == "1"), 0
        for k in range(SSTEPS):
            ds.write(0, *stream_step(k))
            ds.enqueue(0, run)
            slot ^= overlap == "1"
            gm.run(slot)
            det, counts = ctx.fetch_detections(SNB)
            exp, ecounts = stream_expected(k, mode)
            assert tuples(det) == exp and counts.tolist() == ecounts, (env, mode, k)
        assert ctx.stat_graphs() == (gm.captured, gm.replayed)
        if graph == "1":
            assert gm.replayed == SSTEPS - (4 if overlap == "1" else 2)
    finally:
        ctx.close()
    if overlap == "0":
        return
    # streaming: enqueue(k); enqueue(k+1); fetch previous -> k while k+1 runs (two buffer sets, one per slot)
    ctx = _ctx(tsd, monkeypatch, flavour, env)
    try:
        _setup(ctx, mode)
        ds = DeviceStream(ctx, 2)
        gm = GraphModel(graph == "1")
        for k in range(SSTEPS):
            ds.write(k & 1, *stream_step(k))
            ds.enqueue(k & 1, run)
            gm.run(k & 1)
            if k:
                det, counts = ctx.fetch_detections(SNB, previous=True)
                exp, ecounts = stream_expected(k - 1, mode)
                assert tuples(det) == exp and counts.tolist() == ecounts, (env, mode, k - 1)
        det, counts = ctx.fetch_detections(SNB)
        assert tuples(det) == stream_expected(SSTEPS - 1, mode)[0]
        assert ctx.stat_graphs() == (gm.captured, gm.replayed)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_no_graphs_while_profiling(tsd, monkeypatch):
    """set_profiling(1) and (2) launch every batch eagerly; after set_profiling(0) the capture rule applies again."""
    ctx = _ctx(tsd, monkeypatch, "det", {})
    try:
        _setup(ctx, "det")
        ds = DeviceStream(ctx)
        k = 0
        for prof in (1, 2):
            ctx.set_profiling(prof)
            for _ in range(5):
                ds.write(0, *stream_step(k % SSTEPS)); ds.enqueue(0, tsd.RUN_DETECT)
                det, counts = ctx.fetch_detections(SNB)
                assert tuples(det) == stream_expected(k % SSTEPS, "det")[0]
                k += 1
            assert ctx.stat_graphs() == (0, 0), prof
        ctx.set_profiling(0)
        for _ in range(6):
            ds.write(0, *stream_step(k % SSTEPS)); ds.enqueue(0, tsd.RUN_DETECT)
            det, counts = ctx.fetch_detections(SNB)
            assert tuples(det) == stream_expected(k % SSTEPS, "det")[0]
            k += 1
        assert ctx.stat_graphs() == (2, 2)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("route,F,env", (("pinned", 4, {"TSD_STAGE_CHUNK": "2"}), ("pinned", 6, {"TSD_STAGE_CHUNK": "2"}),
                                         ("pageable", 4, {"TSD_CHUNK_FRAMES": "2"})))
def test_host_frames_rewritten(tsd, oracle, monkeypatch, route, F, env):
    """detect_frames on one host buffer rewritten in place between calls: page-locked and staged in chunks (4 frames: 2 chunks;
    6 frames: 3 chunks, so the slot parity flips between calls), and pageable in chunks.  Frame contents and boxes change,
    per-frame counts stay, so every chunk's key comes back: the calls must reach replay and match the oracle."""
    red6, blue6 = det_templates()
    ctx = _ctx(tsd, monkeypatch, "det", env)
    buf = np.empty((F, H, W, 3), np.uint8)
    if route == "pinned":
        ctx.pin(buf)
    try:
        ctx.set_templates(red6, blue6)
        counts_f = (100, 37, 0, 64, 100, 5)[:F]
        chunk = 2
        nch = F // chunk
        gm, slot, reps, used = GraphModel(), 0, [], set()
        for call in range(5):
            frames = np.roll(base_frames()[[(call + i) % 8 for i in range(F)]], 53 * call, axis=1)
            boxes, off = ragged_boxes(counts_f, 300 + call)
            buf[:] = frames
            det, counts = ctx.detect_frames(buf, boxes, off)
            exp, ecounts = expect_det(oracle, frames, boxes, off, red6, blue6)
            assert tuples(det) == exp and counts.tolist() == ecounts, (route, F, call)
            for c in range(nch):
                slot ^= 1
                used.add(slot)                               # (the first use of a slot's staging mirror reallocates: new key)
                gm.run((c, slot, len(used) if route == "pinned" else 0))
            reps.append(ctx.stat_graphs())
            assert reps[-1] == (gm.captured, gm.replayed), (call, reps)
        # 2 chunks keep their slots: replays from call 3 on (pinned: the first use of a slot's staging mirror reallocates it, so one
        # chunk's key settles a call later); 3 chunks change slots every call, so a key comes back every other call: from call 5
        assert reps[2][1] > 0 if nch == 2 else (reps[3][1] == 0 and reps[4][1] > 0), reps
    finally:
        if route == "pinned":
            ctx.unpin(buf)
        ctx.close()


# ---- interleaved calls ---------------------------------------------------------------------------------------------------
OP_KINDS = ("enqueue", "fetch_last", "fetch_prev", "flush", "sync", "stage", "crop_dev", "templates", "simtab", "profiling", "hist_entries",
            "graphs_mark", "replays")
STAGES = ("windows", "dedup_hist", "dedup_coords", "hist", "score", "color_masks")
SMALL_NAMES = ("ragged", "ragged_b", "empty", "aspect", "single", "c1", "c2", "c3")


@functools.lru_cache(None)
def interleaved_ops(seed=2024, n=60):
    """Seeded sequence: random operations, with scripted pieces that must occur (a cycle through more than 8 batch shapes, the
    'grow' and 4K batches enqueued right after another batch, a stage call between two batches of the same slot)."""
    rng = np.random.default_rng(seed)
    kinds = ("enqueue",) * 8 + ("fetch_last", "fetch_prev", "fetch_prev", "flush", "sync", "stage", "stage", "crop_dev", "templates",
                                "simtab", "profiling", "hist_entries")
    ops = []
    for i in range(n):
        if i == 12:                                          # > 8 distinct shapes in a cycle, twice
            ops += [("enqueue", nm) for nm in SMALL_NAMES + ("c1", "c2")] * 2
        if i == 24:
            ops += [("enqueue", "ragged"), ("enqueue", "grow"), ("fetch_prev",)]
        if i == 36:
            ops += [("enqueue", "c3"), ("enqueue", "big4k"), ("stage", "dedup_hist"), ("enqueue", "c1"), ("fetch_prev",)]
        if i == 48:                                          # replays after a stage call wrote slot 0's scratch, new templates
            ops += [("profiling", 0)] + [("enqueue", "c1")] * 4 + [("stage", "dedup_hist"), ("templates",), ("graphs_mark",),
                                                                    ("enqueue", "c1"), ("enqueue", "c1"), ("replays", 2), ("fetch_prev",),
                                                                    ("fetch_last",)]
        k = kinds[int(rng.integers(len(kinds)))]
        if k == "enqueue":
            ops.append((k, SMALL_NAMES[int(rng.integers(len(SMALL_NAMES)))]))
        elif k == "stage":
            ops.append((k, STAGES[int(rng.integers(len(STAGES)))]))
        elif k == "profiling":
            ops.append((k, int(rng.choice([1, 2, 0, 0]))))
        else:
            ops.append((k,))
    ops += [("enqueue", "ragged"), ("enqueue", "ragged_b"), ("fetch_prev",), ("fetch_last",), ("hist_entries",), ("profiling", 0),
            ("templates",), ("enqueue", "c2"), ("enqueue", "c2"), ("fetch_prev",), ("templates",)]
    return tuple(ops)


def interleaved_model(ops):
    """Walks the sequence as the library's host state does.  Per op: what it must return.  A fetch previous succeeds only when
    the last enqueue ran in a slot without a layout change and followed another slotted enqueue, and no call since then joined
    the batches (everything but device-pointer crop_resize and stat_graphs joins) or fetched the previous batch."""
    sm = SlotModel()
    prof, tmpl = 0, 0
    last = prev = None                                       # (batch name, template set, slot) of the last / previous batch
    pending, prev_valid = False, False
    out, keys = [], set()
    slot_batches = {}                                        # slot -> index of its last batch
    grew_busy = stage_between = False
    stage_since = {0: False, 1: False}
    nprev_ok = nprev_bad = 0
    for op in ops:
        k = op[0]
        if k == "enqueue":
            fr, boxes, off = pool_batch(op[1])
            in_slot = prof != 1
            prev, prev_valid = last, last is not None and last[2] is not None and in_slot
            if in_slot:
                slot, grew = sm.enqueue(len(fr), len(boxes), maxb(off))
                if grew:
                    prev_valid = False
                    grew_busy |= pending
                if stage_since[slot] and slot in slot_batches:
                    stage_between = True
                stage_since[slot] = False
                slot_batches[slot] = len(out)
                keys.add((op[1], slot))
            else:
                slot = None
            last, pending = (op[1], tmpl, slot), in_slot
            out.append(("enqueued", last))
            continue
        if k == "fetch_prev":
            ok = prev_valid and pending
            nprev_ok += ok; nprev_bad += not ok
            out.append(("prev", prev) if ok else ("refused",))
            prev_valid = False
            continue
        if k in ("crop_dev", "graphs_mark", "replays"):           # device-pointer crop_resize and stat_graphs do not join
            out.append((k,))
            continue
        pending = False                                      # every other call joins the batches
        if k == "stage":
            stage_since = {0: True, 1: True}
        if k == "templates":
            tmpl ^= 1
        if k == "profiling":
            prof = op[1]
        out.append((k, last))
    return dict(out=out, keys=keys, grew_busy=grew_busy, stage_between_same_slot=stage_between, prev_ok=nprev_ok, prev_refused=nprev_bad)


@functools.lru_cache(None)
def alt_templates():
    red6, blue6 = det_templates()
    return 255 - red6[::-1].copy(), 255 - blue6[::-1].copy()


@functools.lru_cache(None)
def pool_expected(name, tmpl):
    import oracle.oracle as O
    fr, boxes, off = pool_batch(name)
    return expect_det(O, fr, boxes, off, *(alt_templates() if tmpl else det_templates()))


def hist_nnz(oracle, name):
    """What tsd_stat_hist_entries counts for a pool batch: non-zero H-S bins summed over its aspect-passing windows, each window
    as the first duplicate-removal pass leaves it.  An item that absorbed an earlier near duplicate holds the merged pixels (the
    fold rebuilds its histogram in place); cleanDuplicatedDetections appends item i last, so that is the last survivor of the
    pass over the first i + 1 windows."""
    fr, boxes, off = pool_batch(name)
    n = 0
    for f in range(len(fr)):
        c, v = oracle.expand_boxes(boxes[off[f]:off[f + 1]], 1.30)
        c = c[v]
        w = np.stack([oracle.crop_resize(fr[f], cc, 25) for cc in c]) if len(c) else None
        for i in range(len(c)):
            item = oracle.dedup(w[:i + 1], c[:i + 1], False, 0.85)[0][-1]
            n += int(np.count_nonzero(oracle.hist_normalized(item)))
    return n


def check_stage(ctx, oracle, which, red6, blue6):
    """One host-pointer stage call on a small batch, checked against the oracle."""
    fr, boxes, off = pool_batch("c2")
    ew, ec, eo = [], [], [0]
    for f in range(len(fr)):
        c, v = oracle.expand_boxes(boxes[off[f]:off[f + 1]], 1.30)
        ew += [oracle.crop_resize(fr[f], cc, 25) for cc in c[v]]; ec += list(c[v]); eo.append(len(ec))
    ew, ec, eo = np.stack(ew), np.array(ec, np.int32), np.array(eo, np.int32)
    if which == "windows":
        w, c, o = ctx.windows(fr, boxes, off)
        assert np.array_equal(w, ew) and np.array_equal(c, ec) and np.array_equal(o, eo)
    elif which.startswith("dedup"):
        by_coords = which == "dedup_coords"
        tol = 0.95 if by_coords else 0.85
        w, c, o = ctx.dedup(ew, ec, eo, by_coords, tol)
        xw, xc, xo = [], [], [0]
        for f in range(len(fr)):
            if eo[f + 1] > eo[f]:
                a, b = oracle.dedup(ew[eo[f]:eo[f + 1]], ec[eo[f]:eo[f + 1]], by_coords, tol)
                xw += list(a); xc += list(b)
            xo.append(len(xc))
        assert np.array_equal(w, np.stack(xw)) and np.array_equal(c, np.array(xc, np.int32)) and np.array_equal(o, xo), which
    elif which == "hist":
        assert np.array_equal(ctx.hist(ew), np.stack([oracle.hist_normalized(w) for w in ew]))
    elif which == "score":
        s = ctx.score_windows(ew)
        o = [oracle.score_window(w, red6, blue6) for w in ew]
        assert s["emit"].tolist() == [a for a, _, _ in o] and s["id"].tolist() == [b for _, b, _ in o]
        assert s["hundredths"].tolist() == [h for _, _, h in o]
    else:
        r, b = ctx.color_masks(ew)
        o = [oracle.color_masks(w) for w in ew]
        assert np.array_equal(r, np.stack([a for a, _ in o]).reshape(r.shape)) and np.array_equal(b, np.stack([x for _, x in o]).reshape(b.shape))


@pytest.mark.gpu
def test_interleaved_calls(tsd, oracle, monkeypatch):
    """interleaved_ops on one overlapped detection context: every fetched batch equals the oracle for the templates in effect
    when it was enqueued; fetch previous succeeds or returns TSD_E_STATE as interleaved_model says; stage calls and
    stat_hist_entries are right in between."""
    import torch
    A = _lib()
    dev = torch.device("cuda", 0)
    ops = interleaved_ops()
    model = interleaved_model(ops)["out"]
    ctx = _ctx(tsd, monkeypatch, "det", {"TSD_OVERLAP": "1", "TSD_GRAPH": "1"})
    dbuf = {}
    for name in POOL:
        fr, boxes, off = pool_batch(name)
        dbuf[name] = (torch.from_numpy(fr).to(dev), torch.from_numpy(boxes.reshape(-1, 4) if len(boxes) else np.zeros((1, 4), np.int32)).to(dev),
                      torch.from_numpy(off).to(dev))
    crop_fr, crop_boxes, crop_off = pool_batch("ragged")
    cc, cv = oracle.expand_boxes(crop_boxes[crop_off[5]:crop_off[6]], 1.30)
    cc = cc[cv][:40]
    d_cc, d_cf = torch.from_numpy(np.ascontiguousarray(cc)).to(dev), torch.full((len(cc),), 5, dtype=torch.int32, device=dev)
    d_cw = torch.empty((len(cc), 25, 25, 3), dtype=torch.uint8, device=dev)
    exp_crop = np.stack([oracle.crop_resize(crop_fr[5], c, 25) for c in cc])
    simtab = tsd.engine.similarity_table()
    tsets = (det_templates(), alt_templates())
    tmpl = 0
    try:
        ctx.set_templates(*tsets[0])
        for i, (op, m) in enumerate(zip(ops, model)):
            k = op[0]
            where = (i, op)
            if k == "enqueue":
                fr, boxes, off = pool_batch(op[1])
                d_fr, d_b, d_o = dbuf[op[1]]
                ctx.enqueue_frames(d_fr.data_ptr(), len(fr), fr.shape[1], fr.shape[2], d_b.data_ptr(), d_o.data_ptr(), int(off[-1]),
                                   max_boxes_per_frame=maxb(off))
            elif k == "fetch_prev":
                det = np.empty(4096, A.DET_DTYPE); nd = C.c_int32(-1); counts = np.zeros(4, np.int32)
                rc = ctx._L.tsd_fetch_previous(ctx._h, A.ptr(det), len(det), C.byref(nd), A.ptr(counts))
                if m[0] == "refused":
                    assert rc == E_STATE, where
                else:
                    assert rc == 0, (where, A.lib().tsd_last_error())
                    exp, ecounts = pool_expected(m[1][0], m[1][1])
                    assert tuples(det[:nd.value]) == exp and counts.tolist() == ecounts, where
            elif k in ("fetch_last", "hist_entries") and m[1] is None:
                with pytest.raises(A.TsdError, match="error -3"):
                    ctx.fetch_detections(4096) if k == "fetch_last" else ctx.stat_hist_entries()
            elif k == "fetch_last":
                det, counts = ctx.fetch_detections(4096)
                exp, ecounts = pool_expected(m[1][0], m[1][1])
                assert tuples(det) == exp and counts.tolist() == ecounts, where
            elif k == "hist_entries":
                assert ctx.stat_hist_entries() == hist_nnz(oracle, m[1][0]), where
            elif k == "flush":
                ctx.flush()
            elif k == "sync":
                ctx.synchronize()
            elif k == "stage":
                check_stage(ctx, oracle, op[1], *tsets[tmpl])
            elif k == "crop_dev":
                d_cw.fill_(77)
                d_crop = dbuf["ragged"][0]
                A.check(ctx._L.tsd_crop_resize(ctx._h, A.ptr(d_crop.data_ptr()), 6, H, W, W * 3, H * W * 3, 3, A.ptr(d_cc.data_ptr()),
                                               A.ptr(d_cf.data_ptr()), len(cc), 25, A.ptr(d_cw.data_ptr()), A.MEM_DEVICE))
                torch.cuda.synchronize()
                assert np.array_equal(d_cw.cpu().numpy(), exp_crop), where
            elif k == "templates":
                tmpl ^= 1
                ctx.set_templates(*tsets[tmpl])
            elif k == "simtab":
                A.check(ctx._L.tsd_set_similarity_table(ctx._h, A.ptr(simtab), len(simtab)))
            elif k == "profiling":
                ctx.set_profiling(op[1])
            elif k == "graphs_mark":
                rep0 = ctx.stat_graphs()[1]
            elif k == "replays":                             # the batches since the mark were replayed graphs
                assert ctx.stat_graphs()[1] - rep0 == op[1], where
    finally:
        ctx.close()


# ---- mode switching and two contexts ---------------------------------------------------------------------------------------
MODE_SEQ = ("rec", "det", "rec", "det", "det", "rec", "rec", "det", "rec", "det")


@functools.lru_cache(None)
def templates32():
    rng = np.random.default_rng(32)
    return (rng.random((6, 1024)) < 0.4).astype(np.uint8) * 255, (rng.random((6, 1024)) < 0.4).astype(np.uint8) * 255


@pytest.mark.gpu
def test_mode_switching(tsd, oracle):
    """RUN_RECOGNIZE and RUN_DETECT alternating on one overlapped D = 32 context: each mode's scratch is first allocated while the
    other slot's batch of the other mode is still running.  Detection at D = 32 / enlarge 1.15 against
    oracle.detect_frame(cfg=), recognition against the HOG + LDA composition."""
    import torch
    dev = torch.device("cuda", 0)
    Wl, bl = rec_model()
    red, blue = templates32()
    names = ("grow", "ragged", "c1", "grow", "ragged_b", "single", "c3", "ragged", "grow", "c2")     # (the largest first: no layout growth)
    with tsd.Context(0, "rec") as ctx:
        ctx.set_templates(red, blue)
        ctx.set_lda(Wl, bl)
        cfg = ctx.cfg
        bufs, exp = [], []
        for mode, name in zip(MODE_SEQ, names):
            fr, boxes, off = pool_batch(name)
            bufs.append((torch.from_numpy(fr).to(dev), torch.from_numpy(boxes if len(boxes) else np.zeros((1, 4), np.int32)).to(dev),
                         torch.from_numpy(off).to(dev)))
            if mode == "det":
                exp.append(expect_det(oracle, fr, boxes, off, red, blue, D=32, enlarge=1.15, cfg=cfg))
            else:
                exp.append(expect_rec(oracle, fr, boxes, off, Wl, bl))
        for i, (mode, name) in enumerate(zip(MODE_SEQ, names)):
            fr, boxes, off = pool_batch(name)
            d_fr, d_b, d_o = bufs[i]
            ctx.enqueue_frames(d_fr.data_ptr(), len(fr), H, W, d_b.data_ptr(), d_o.data_ptr(), int(off[-1]), mode=_run_mode(mode, tsd),
                               max_boxes_per_frame=maxb(off))
            if i:
                det, counts = ctx.fetch_detections(4096, previous=i % 3 != 0)
                j = i - 1 if i % 3 != 0 else i
                assert tuples(det) == exp[j][0] and counts.tolist() == exp[j][1], (i, j)
        det, counts = ctx.fetch_detections(4096)
        assert tuples(det) == exp[-1][0] and counts.tolist() == exp[-1][1]


@pytest.mark.gpu
def test_two_contexts(tsd, oracle):
    """A detection and a recognition context on one device, enqueues interleaved, fetched out of order."""
    import torch
    dev = torch.device("cuda", 0)
    Wl, bl = rec_model()
    red6, blue6 = det_templates()
    steps = [("det", "grow"), ("rec", "grow"), ("det", "ragged"), ("rec", "c2"), ("det", "c1"), ("rec", "ragged_b"), ("det", "ragged_b"),
             ("rec", "ragged")]                              # (the largest first: no layout growth, so fetch previous is allowed)
    dbuf = {n: tuple(torch.from_numpy(a if len(a) else np.zeros((1, 4), np.int32)).to(dev) for a in pool_batch(n)) for _, n in steps}
    with tsd.Context(0, "det") as cd, tsd.Context(0, "rec") as cr:
        cd.set_templates(red6, blue6)
        cr.set_lda(Wl, bl)
        ctxs = {"det": cd, "rec": cr}
        done = {"det": [], "rec": []}
        for i, (mode, name) in enumerate(steps):
            fr, boxes, off = pool_batch(name)
            d_fr, d_b, d_o = dbuf[name]
            ctxs[mode].enqueue_frames(d_fr.data_ptr(), len(fr), fr.shape[1], fr.shape[2], d_b.data_ptr(), d_o.data_ptr(), int(off[-1]),
                                      mode=_run_mode(mode, tsd), max_boxes_per_frame=maxb(off))
            done[mode].append(name)
            if i in (3, 7):                                  # the other context's previous batch first, then both last ones
                for mm in ("rec", "det"):
                    prev, last = done[mm][-2], done[mm][-1]
                    for nm, previous in ((prev, True), (last, False)):
                        fr2, b2, o2 = pool_batch(nm)
                        e = expect_det(oracle, fr2, b2, o2, red6, blue6) if mm == "det" else expect_rec(oracle, fr2, b2, o2, Wl, bl)
                        det, counts = ctxs[mm].fetch_detections(8192, previous=previous)
                        assert tuples(det) == e[0] and counts.tolist() == e[1], (i, mm, nm)


# ---- recovery after refused calls --------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_recovery_after_refusals(tsd, monkeypatch):
    """Refused calls in the middle of a replayed stream leave the context usable: bad strides, RUN_DETECT before templates,
    det_cap too small (TSD_E_NOMEM with the count, then the records on a second fetch), and a max_boxes_per_frame below the
    real maximum (the general fold redoes the flagged frames)."""
    A = _lib()
    ctx = _ctx(tsd, monkeypatch, "det", {})
    try:
        ds = DeviceStream(ctx)
        fr, bx, of = ds.sets[0]
        ds.write(0, *stream_step(0))
        rc = ctx._L.tsd_enqueue_frames(ctx._h, tsd.RUN_DETECT, A.ptr(fr.data_ptr()), SF, H, W, W * 3, H * W * 3, A.ptr(bx.data_ptr()),
                                       A.ptr(of.data_ptr()), SNB, SMAX)
        assert rc == E_STATE                                 # no templates yet
        _setup(ctx, "det")
        for k in range(SSTEPS):
            ds.write(0, *stream_step(k))
            if k == 2:
                rc = ctx._L.tsd_enqueue_frames(ctx._h, tsd.RUN_DETECT, A.ptr(fr.data_ptr()), SF, H, W, W * 3 - 1, H * W * 3, A.ptr(bx.data_ptr()),
                                               A.ptr(of.data_ptr()), SNB, SMAX)
                assert rc == E_INVALID
            ds.enqueue(0, tsd.RUN_DETECT, maxb_=10 if k == 6 else SMAX)
            exp, ecounts = stream_expected(k, "det")
            if k in (4, 7):
                assert len(exp) >= 2
                det = np.empty(len(exp), A.DET_DTYPE); nd = C.c_int32(-1); counts = np.zeros(4, np.int32)
                rc = ctx._L.tsd_fetch_detections(ctx._h, A.ptr(det), len(exp) - 1, C.byref(nd), A.ptr(counts))
                assert rc == E_NOMEM and nd.value == len(exp) and counts.tolist() == ecounts
            det, counts = ctx.fetch_detections(SNB)
            assert tuples(det) == exp and counts.tolist() == ecounts, k
        cap, rep = ctx.stat_graphs()
        assert rep > 0
    finally:
        ctx.close()
