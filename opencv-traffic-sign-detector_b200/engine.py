"""Host-side engine: one `Context` per (process, GPU) over the C-ABI library.

numpy arrays in, numpy arrays out; every method is one call into libtsd_b200.so (CUDA kernels).  Nothing here
computes a stage on the CPU and nothing imports the oracle.  Citations name the reference function each method
stands in for (DET = "Deteción de Objetos/source.py", REC = "Reconocimiento de Objetos/source.py").
"""
import ctypes as C

import numpy as np

from . import _capi
from ._capi import DET_DTYPE, HOG_LEN, MEM_DEVICE, MEM_HOST, RUN_DETECT, RUN_RECOGNIZE, Config, TsdError, check, ptr

_SIMTAB = None


def similarity_table(n=1 << 16):
    """f(d2) for d2 = 0..n-1 evaluated with the reference's own expression and numpy scalar calls
    (EuclDSimilarity, DET:459-462), so the in-process reference and the GPU fold use bit-identical values."""
    global _SIMTAB
    if _SIMTAB is None or len(_SIMTAB) < n:
        f = np.empty(n, np.float64)
        f[0] = 1.0
        for d2 in range(1, n):
            dist = np.sqrt(np.float64(d2))
            f[d2] = 1 / (1 + np.power(np.e, (((0.154 * np.power(dist, 1.2)) - 31.8) / (0.2 * dist))))
        _SIMTAB = f
    return _SIMTAB[:n]


def default_config(flavour="det"):
    cfg = Config()
    check(_capi.lib().tsd_config_default(C.byref(cfg), 1 if flavour == "rec" else 0))
    return cfg


def _u8(a):
    return np.ascontiguousarray(a, np.uint8)


def _i32(a):
    return np.ascontiguousarray(a, np.int32)


class Context:
    """tsd_ctx wrapper.  flavour 'det' = x1.30 / 25x25 (DET:119,124); 'rec' = x1.15 / 32x32 (REC:54,57)."""

    def __init__(self, device=0, flavour="det", config=None, numpy_similarity=True):
        self._L = _capi.lib()
        self.cfg = config if config is not None else default_config(flavour)
        h = C.c_void_p()
        check(self._L.tsd_create(C.byref(h), int(device), C.byref(self.cfg)))
        self._h = h
        self.device = int(device)
        self.D = int(self.cfg.window)
        if numpy_similarity:
            t = similarity_table()
            check(self._L.tsd_set_similarity_table(self._h, ptr(t), len(t)))

    # -- lifetime ------------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.tsd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def stream(self):
        return self._L.tsd_stream(self._h)

    def synchronize(self):
        check(self._L.tsd_synchronize(self._h))

    def flush(self):
        """Make the context's stream wait for every batch enqueued so far (no host block): consecutive enqueue_frames calls run on
        two internal streams and their join to `stream` is deferred by one call (TSD_OVERLAP=0 disables the overlap)."""
        check(self._L.tsd_flush(self._h))

    def pin(self, array):
        """Page-lock a caller-owned C-contiguous numpy array so that detect_frames reads it in place over PCIe
        (only candidate ROIs are transferred).  Call unpin(array) before the array is freed."""
        check(self._L.tsd_host_register(ptr(array), int(array.nbytes)))

    def unpin(self, array):
        check(self._L.tsd_host_unregister(ptr(array)))

    @property
    def launch_count(self):
        return int(self._L.tsd_launch_count(self._h))

    # -- state ---------------------------------------------------------------------------------------------------
    def set_templates(self, red6, blue6):
        """6 red + 6 blue template masks {0,255} from calculateMeanMasks (DET:24-59)."""
        red6, blue6 = _u8(red6).reshape(6, -1), _u8(blue6).reshape(6, -1)
        if red6.shape[1] != self.D * self.D or blue6.shape != red6.shape:
            raise TsdError("templates must be 6 x %d x %d" % (self.D, self.D))
        check(self._L.tsd_set_templates(self._h, ptr(red6), ptr(blue6)))

    def set_lda(self, W, b):
        """W f64 [nfeat,6] (column c = classifiers[c].coef_[0]), b f64 [6] (REC:551-562)."""
        W = np.ascontiguousarray(W, np.float64); b = np.ascontiguousarray(b, np.float64)
        if W.ndim != 2 or W.shape[1] != 6 or b.shape != (6,):
            raise TsdError("W must be [nfeat,6] and b [6]")
        check(self._L.tsd_set_lda(self._h, ptr(W), ptr(b), W.shape[0]))
        self._lda_nfeat = W.shape[0]

    def set_knn(self, xbar, scalings, Ztrain, ytrain, k=4):
        """7-class LDA reducer (xbar_, scalings_[:, :6]) + KNN training set (REC:586-589)."""
        xbar = np.ascontiguousarray(xbar, np.float64); S = np.ascontiguousarray(scalings, np.float64)
        Z = np.ascontiguousarray(Ztrain, np.float64); y = _i32(ytrain)
        if S.shape != (len(xbar), 6) or Z.ndim != 2 or Z.shape[1] != 6 or len(y) != len(Z):
            raise TsdError("bad KNN model shapes")
        check(self._L.tsd_set_knn(self._h, ptr(xbar), ptr(S), len(xbar), ptr(Z), ptr(y), len(y), int(k)))
        self._knn_nfeat = len(xbar)

    # -- stages --------------------------------------------------------------------------------------------------
    def expand_boxes(self, boxes, enlarge=None):
        """K1: makeWindowBiggerOrDiscardFakeDetections per box (DET:155-174).  -> (coords int32[n,4], valid bool[n])."""
        boxes = _i32(boxes).reshape(-1, 4)
        n = len(boxes)
        coords = np.zeros((n, 4), np.int32); valid = np.zeros(n, np.uint8)
        check(self._L.tsd_expand_boxes(self._h, ptr(boxes), n, float(self.cfg.enlarge if enlarge is None else enlarge),
                                       ptr(coords), ptr(valid), MEM_HOST))
        return coords, valid.astype(bool)

    def crop_resize(self, frames, coords, win_frame=None, D=None):
        """K2: cv2.resize(cropImageByCoords(coords, frame), (D, D)) (DET:123-124).  frames uint8 [F,H,W,3], [H,W,3],
        [F,H,W] or [H,W] (grey, REC:253-254)."""
        frames = np.asarray(frames)
        grey = frames.ndim == 2 or (frames.ndim == 3 and frames.shape[-1] != 3)
        if (frames.ndim == 2) or (frames.ndim == 3 and not grey):
            frames = frames[None]
        frames = _u8(frames)
        F, H, W = frames.shape[:3]
        ch = 1 if grey else 3
        coords = _i32(coords).reshape(-1, 4)
        n = len(coords)
        wf = np.zeros(n, np.int32) if win_frame is None else _i32(win_frame)
        D = self.D if D is None else int(D)
        out = np.empty((n, D, D) if grey else (n, D, D, 3), np.uint8)
        check(self._L.tsd_crop_resize(self._h, ptr(frames), F, H, W, W * ch, H * W * ch, ch, ptr(coords), ptr(wf), n, D, ptr(out), MEM_HOST))
        return out

    def windows(self, frames, boxes, box_offsets):
        """K1+K2 on whole frames: the candidate loop of MSERTrafficSignDetector (DET:116-124).
        -> (windows uint8[m,D,D,3], coords int32[m,4], win_offsets int32[F+1])."""
        frames = _u8(frames)
        if frames.ndim == 3:
            frames = frames[None]
        F, H, W = frames.shape[:3]
        boxes = _i32(boxes).reshape(-1, 4); box_offsets = _i32(box_offsets)
        nb = int(box_offsets[-1])
        wins = np.empty((max(nb, 1), self.D, self.D, 3), np.uint8); coords = np.empty((max(nb, 1), 4), np.int32)
        woff = np.zeros(F + 1, np.int32); tot = C.c_int32()
        check(self._L.tsd_windows(self._h, ptr(frames), F, H, W, W * 3, H * W * 3, ptr(boxes), ptr(box_offsets), float(self.cfg.enlarge),
                                  self.D, ptr(wins), ptr(coords), ptr(woff), C.byref(tot), MEM_HOST))
        return wins[:tot.value].copy(), coords[:tot.value].copy(), woff

    def dedup(self, windows, coords, offsets, by_coords, tol):
        """K5: cleanDuplicatedDetections per frame (DET:177-223).  -> (windows, coords, offsets) of the survivors."""
        windows = _u8(windows); coords = _i32(coords).reshape(-1, 4); offsets = _i32(offsets)
        n = len(coords); F = len(offsets) - 1
        D = windows.shape[1] if n else self.D
        ow = np.empty_like(windows) if n else windows; oc = np.empty_like(coords)
        ooff = np.zeros(F + 1, np.int32); tot = C.c_int32()
        check(self._L.tsd_dedup(self._h, ptr(windows), ptr(coords), ptr(offsets), F, D, int(bool(by_coords)), float(tol),
                                ptr(ow), ptr(oc), ptr(ooff), C.byref(tot), MEM_HOST))
        return ow[:tot.value].copy(), oc[:tot.value].copy(), ooff

    def hist(self, windows):
        """calculateHistAndNormalize (DET:575-586) -> float32 [n,50,60]."""
        windows = _u8(windows)
        n, D = windows.shape[0], windows.shape[1]
        out = np.empty((n, 50, 60), np.float32)
        check(self._L.tsd_hist(self._h, ptr(windows), n, D, ptr(out), MEM_HOST))
        return out

    def color_masks(self, windows):
        """K3: getColorMaskRedOrBlue(img,'r'), (img,'b') (DET:63-89) -> (red, blue) uint8 [n,D,D]."""
        windows = _u8(windows)
        n, D = windows.shape[0], windows.shape[1]
        red = np.empty((n, D, D), np.uint8); blue = np.empty((n, D, D), np.uint8)
        check(self._L.tsd_color_masks(self._h, ptr(windows), n, D, ptr(red), ptr(blue), MEM_HOST))
        return red, blue

    def bgr2hsv(self, bgr):
        bgr = _u8(bgr)
        out = np.empty_like(bgr)
        check(self._L.tsd_bgr2hsv(self._h, ptr(bgr), bgr.size // 3, ptr(out), MEM_HOST))
        return out

    def score_masks(self, red, blue, want_scores=True):
        """K4 (DET:229-261,545-567) -> dict(scores int32[n,2,6] hundredths, id, hundredths, emit)."""
        red, blue = _u8(red), _u8(blue)
        n, D = red.shape[0], red.shape[1]
        sc = np.zeros((n, 2, 6), np.int32) if want_scores else None
        ids = np.zeros(n, np.int32); hs = np.zeros(n, np.int32); em = np.zeros(n, np.uint8)
        check(self._L.tsd_score_masks(self._h, ptr(red), ptr(blue), n, D, ptr(sc), ptr(ids), ptr(hs), ptr(em), MEM_HOST))
        return dict(scores=sc, id=ids, hundredths=hs, emit=em.astype(bool))

    def score_windows(self, windows):
        """K3 + K4 in one call (detectionsMaskCorrelation, DET:229-245) -> dict(id, hundredths, emit)."""
        windows = _u8(windows)
        n, D = windows.shape[0], windows.shape[1]
        ids = np.zeros(n, np.int32); hs = np.zeros(n, np.int32); em = np.zeros(n, np.uint8)
        check(self._L.tsd_score(self._h, ptr(windows), n, D, ptr(ids), ptr(hs), ptr(em), MEM_HOST))
        return dict(id=ids, hundredths=hs, emit=em.astype(bool))

    def recognize_windows(self, windows, tol=None):
        """K6 + K7 + K8 in one call on uint8 [n,32,32,3] BGR windows -> labels int32[n] (0 = no sign)."""
        windows = _u8(windows).reshape(-1, 32, 32, 3)
        lab = np.zeros(len(windows), np.int32)
        check(self._L.tsd_recognize(self._h, ptr(windows), len(windows), float(self.cfg.proba_tol if tol is None else tol), ptr(lab), MEM_HOST))
        return lab

    def lda_predict_tf32(self, X, split=3, tol=None):
        """Evaluation only: K8 on the tensor cores (mma.sync TF32; split 1 = plain, 3 = 3xTF32) -> (logits f32[n,6], labels, kernel ms)."""
        X = np.ascontiguousarray(X, np.float32)
        n = len(X)
        lg = np.zeros((n, 6), np.float32); lab = np.zeros(n, np.int32); ms = C.c_float()
        check(self._L.tsd_lda_predict_tf32(self._h, ptr(X), n, float(self.cfg.proba_tol if tol is None else tol), int(split), ptr(lg), ptr(lab),
                                           C.byref(ms), MEM_HOST))
        return lg, lab, float(ms.value)

    def bgr2gray(self, bgr):
        """K6: cv2.cvtColor(BGR2GRAY) (REC:388)."""
        bgr = _u8(bgr)
        out = np.empty(bgr.shape[:-1], np.uint8)
        check(self._L.tsd_bgr2gray(self._h, ptr(bgr), bgr.size // 3, ptr(out), MEM_HOST))
        return out

    def hog(self, gray):
        """K7: cv2.HOGDescriptor.compute (REC:519) on uint8 [n,32,32] -> float32 [n,324]."""
        gray = _u8(gray).reshape(-1, 32, 32)
        out = np.empty((len(gray), HOG_LEN), np.float32)
        check(self._L.tsd_hog(self._h, ptr(gray), len(gray), ptr(out), MEM_HOST))
        return out

    def lda_predict(self, X, tol=None, want_logits=True):
        """K8 (REC:565-577,627-641) -> (logits f64[n,6] or None, labels int32[n])."""
        X = np.ascontiguousarray(X, np.float32)
        if X.ndim != 2 or X.shape[1] != getattr(self, "_lda_nfeat", -1):
            raise TsdError("X must be [n,%d]" % getattr(self, "_lda_nfeat", -1))
        n = len(X)
        lg = np.empty((n, 6), np.float64) if want_logits else None
        lab = np.zeros(n, np.int32)
        check(self._L.tsd_lda_predict(self._h, ptr(X), n, float(self.cfg.proba_tol if tol is None else tol), ptr(lg), ptr(lab), MEM_HOST))
        return lg, lab

    def knn_predict(self, X, want_Z=True):
        """K8b (REC:592-596) -> (Z f64[n,6] or None, labels int32[n])."""
        X = np.ascontiguousarray(X, np.float32)
        if X.ndim != 2 or X.shape[1] != getattr(self, "_knn_nfeat", -1):
            raise TsdError("X must be [n,%d]" % getattr(self, "_knn_nfeat", -1))
        n = len(X)
        Z = np.empty((n, 6), np.float64) if want_Z else None
        lab = np.zeros(n, np.int32)
        check(self._L.tsd_knn_predict(self._h, ptr(X), n, ptr(Z), ptr(lab), MEM_HOST))
        return Z, lab

    # -- whole path ------------------------------------------------------------------------------------------------
    def detect_frames(self, frames, boxes, box_offsets, mode=RUN_DETECT):
        """The whole post-MSER chain on HOST frames (H2D copy inside): DET:116-131 + DET:708-716.
        -> (records structured array DET_DTYPE, counts int32[4] = raw / aspect-passing / survivors / detections)."""
        frames = _u8(frames)
        if frames.ndim == 3:
            frames = frames[None]
        F, H, W = frames.shape[:3]
        boxes = _i32(boxes).reshape(-1, 4); box_offsets = _i32(box_offsets)
        cap = max(int(box_offsets[-1]), 1)
        det = np.empty(cap, DET_DTYPE); nd = C.c_int32(); counts = np.zeros(4, np.int32)      # (only det[:nd] is ever read)
        check(self._L.tsd_detect_frames(self._h, int(mode), ptr(frames), F, H, W, W * 3, H * W * 3, ptr(boxes), ptr(box_offsets),
                                        ptr(det), cap, C.byref(nd), ptr(counts), MEM_HOST))
        return det[:nd.value].copy(), counts

    def enqueue_frames(self, d_frames, nframes, H, W, d_boxes, d_box_offsets, nboxes_total, mode=RUN_DETECT,
                       row_stride=None, frame_stride=None, max_boxes_per_frame=0):
        """Asynchronous, device-resident chain (integer device pointers, e.g. torch tensor .data_ptr()).
        max_boxes_per_frame: largest per-frame candidate count (0 = let the library read the offsets back)."""
        rs = W * 3 if row_stride is None else int(row_stride)
        fs = H * rs if frame_stride is None else int(frame_stride)
        check(self._L.tsd_enqueue_frames(self._h, int(mode), ptr(int(d_frames)), int(nframes), int(H), int(W), rs, fs,
                                         ptr(int(d_boxes)), ptr(int(d_box_offsets)), int(nboxes_total), int(max_boxes_per_frame)))

    def fetch_detections(self, cap, previous=False):
        """Records + stage counts of the last enqueue_frames call; previous=True: of the call before it, while the last batch
        keeps running (streaming use of the two scratch slots: enqueue(k); enqueue(k+1); fetch(previous=True) -> batch k)."""
        det = np.empty(max(int(cap), 1), DET_DTYPE); nd = C.c_int32(); counts = np.zeros(4, np.int32)
        fn = self._L.tsd_fetch_previous if previous else self._L.tsd_fetch_detections
        check(fn(self._h, ptr(det), len(det), C.byref(nd), ptr(counts)))
        return det[:nd.value].copy(), counts

    def stat_hist_entries(self):
        """Total non-zero histogram bins over the windows of the last enqueue_frames call (measurement helper)."""
        t = C.c_int64()
        check(self._L.tsd_stat_hist_entries(self._h, C.byref(t)))
        return int(t.value)

    def stat_unsure_pairs(self, reset=False):
        """Pairs decided by the exact float64 compareHist evaluation (within 2e-6 of a threshold) since process start / the last reset."""
        t = C.c_int64()
        check(self._L.tsd_stat_unsure_pairs(self._h, C.byref(t), int(bool(reset))))
        return int(t.value)

    def stat_staged_bytes(self, reset=False):
        """Bytes the ROI staging of detect_frames (page-locked host frames) moved over PCIe since process start / the last reset."""
        t = C.c_int64()
        check(self._L.tsd_stat_staged_bytes(self._h, C.byref(t), int(bool(reset))))
        return int(t.value)

    def stat_graphs(self):
        """(captured, replayed): CUDA graphs of the chain instantiated, and cached graphs launched again, since the context was
        created (host-side counters, no synchronisation)."""
        cap, rep = C.c_int64(), C.c_int64()
        check(self._L.tsd_stat_graphs(self._h, C.byref(cap), C.byref(rep)))
        return int(cap.value), int(rep.value)

    def preprocess(self, frames, clip_limit=2.0, tiles=(8, 8), gamma=2):
        """grayAndEnhanceContrast (DET:135-152) for a batch: BGR2GRAY -> CLAHE -> GaussianBlur 3x3 -> gamma LUT.
        frames uint8 [F,H,W,3] or [H,W,3] -> uint8 [F,H,W] (or [H,W])."""
        frames = _u8(frames)
        single = frames.ndim == 3
        if single:
            frames = frames[None]
        F, H, W = frames.shape[:3]
        if getattr(self, "_gamma", None) != gamma:
            inv = 1 / gamma
            table = np.array([((i / 255) ** inv) * 255 for i in range(256)], np.uint8)      # the reference's own expression (DET:602-603)
            check(self._L.tsd_set_gamma_table(self._h, ptr(table)))
            self._gamma = gamma
        out = np.empty((F, H, W), np.uint8)
        check(self._L.tsd_preprocess(self._h, ptr(frames), F, H, W, W * 3, H * W * 3, float(clip_limit), int(tiles[0]), int(tiles[1]), ptr(out), MEM_HOST))
        return out[0] if single else out

    def mean_windows(self, windows, group_offsets):
        """calculateMeanMasks' running average (DET:44-52) per group of windows (CSR offsets, caller's order).
        -> uint8 [ngroups, D, D, 3]."""
        windows = _u8(windows); group_offsets = _i32(group_offsets)
        ng = len(group_offsets) - 1
        D = windows.shape[1]
        out = np.zeros((ng, D, D, 3), np.uint8)
        check(self._L.tsd_mean_windows(self._h, ptr(windows), ptr(group_offsets), ng, D, ptr(out), MEM_HOST))
        return out

    def match_detections(self, det, gt, gt_offsets, tol=0.85):
        """The matching loops of generateStatistics (DET:401-450) for all files and types at once.  det / gt: int32 [n, 6] =
        (frame, x1, y1, x2, y2, type bucket 0..5), gt grouped by frame (CSR gt_offsets).  -> status int32 [ndet] (1 correct),
        match int32 [ndet] (gt row or -1), tally int32 [nframes, 6, 4] = (correct, incorrect, not detected, expected)."""
        det = _i32(det).reshape(-1, 6); gt = _i32(gt).reshape(-1, 6); gt_offsets = _i32(gt_offsets)
        nf = len(gt_offsets) - 1
        status = np.zeros(len(det), np.int32); match = np.full(len(det), -1, np.int32); tally = np.zeros((nf, 6, 4), np.int32)
        check(self._L.tsd_match_detections(self._h, ptr(det), len(det), ptr(gt), ptr(gt_offsets), nf, float(tol), ptr(status), ptr(match), ptr(tally)))
        return status, match, tally

    def match_iou(self, det, det_offsets, gt, gt_offsets, ovr=0.5):
        """The loop of precision_recall_curve (evaluar_resultados.py:224-262).  det int32 [ndet, 5] = (left, top, right, bottom,
        index in the score-descending list) grouped by image (CSR det_offsets, list order inside an image); gt int32 [ngt, 5] =
        (left, top, right, bottom, class; -1 = ignore) grouped by image.  -> tp, fp uint8 [ndet] by list position."""
        det = _i32(det).reshape(-1, 5); gt = _i32(gt).reshape(-1, 5); det_offsets = _i32(det_offsets); gt_offsets = _i32(gt_offsets)
        ni = len(det_offsets) - 1
        tp = np.zeros(len(det), np.uint8); fp = np.zeros(len(det), np.uint8)
        check(self._L.tsd_match_iou(self._h, ptr(det), ptr(det_offsets), ptr(gt), ptr(gt_offsets), ni, float(ovr), ptr(tp), ptr(fp)))
        return tp, fp

    def set_profiling(self, on=True):
        """1 / True: per-stage times (batches serialised); 2: timeline of the overlapped batches (timeline())."""
        check(self._L.tsd_set_profiling(self._h, int(on)))

    def timeline(self, cap=4096):
        names = (C.c_char_p * cap)(); ms = (C.c_float * cap)()
        n = self._L.tsd_timeline(self._h, names, ms, cap)
        return [(names[i].decode(), float(ms[i])) for i in range(n)]

    def stage_times(self):
        names = (C.c_char_p * 32)(); ms = (C.c_float * 32)()
        n = self._L.tsd_stage_times(self._h, names, ms, 32)
        return [(names[i].decode(), float(ms[i])) for i in range(n)]
