"""ctypes front-end of the CPU oracle (oracle/tsd_oracle.c).

TEST INFRASTRUCTURE ONLY -- the checker the CUDA path is compared with.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module;
the product package (opencv-traffic-sign-detector_b200/) never does.

Every wrapper names the reference call site it restates (DET = "Deteción de Objetos/source.py",
REC = "Reconocimiento de Objetos/source.py").
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libtsd_oracle.so")

_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")


def build(force=False):
    """Compile the C restatement (gcc) -- building the checker is not using it."""
    src = os.path.join(_HERE, "tsd_oracle.c")
    if force or not os.path.isfile(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.orc_expand_box.argtypes = [C.c_int32] * 4 + [C.c_double, C.c_double, C.c_double, _i32p]
        L.orc_expand_box.restype = C.c_int
        L.orc_resize_linear_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, C.c_int]
        L.orc_resize_linear_u8.restype = None
        L.orc_crop_resize.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, _i32p, _u8p, C.c_int]
        L.orc_crop_resize.restype = C.c_int
        L.orc_bgr2hsv.argtypes = [_u8p, C.c_int, _u8p]
        L.orc_color_masks.argtypes = [_u8p, C.c_int, _u8p, _u8p, _u8p, _u8p]
        L.orc_score_hundredths.argtypes = [_u8p, _u8p, C.c_int, _i32p]
        L.orc_score_hundredths.restype = C.c_int
        L.orc_best_template.argtypes = [_u8p, _u8p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.orc_score_window.argtypes = [_u8p, C.c_int, _u8p, _u8p, C.c_int, _u8p, _u8p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.orc_score_window.restype = C.c_int
        L.orc_hist_normalized.argtypes = [_u8p, C.c_int, _f32p]
        L.orc_hist_correl.argtypes = [_f32p, _f32p]
        L.orc_hist_correl.restype = C.c_double
        L.orc_eucl_similarity_d2.argtypes = [C.c_int64]
        L.orc_eucl_similarity_d2.restype = C.c_double
        L.orc_coord_similarity.argtypes = [_i32p, _i32p]
        L.orc_coord_similarity.restype = C.c_double
        L.orc_dedup.argtypes = [_u8p, _i32p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.orc_dedup.restype = C.c_int
        L.orc_bgr2gray.argtypes = [_u8p, C.c_int, _u8p]
        L.orc_clahe.argtypes = [_u8p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, _u8p]
        L.orc_gauss3.argtypes = [_u8p, C.c_int, C.c_int, _u8p]
        L.orc_preprocess.argtypes = [_u8p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, _u8p, _u8p]
        L.orc_hog_32.argtypes = [_u8p, _f32p]
        L.orc_lda_predict.argtypes = [_f32p, C.c_int, C.c_int, _f64p, _f64p, C.c_double, _f64p, _i32p]
        L.orc_knn_predict.argtypes = [_f32p, C.c_int, C.c_int, _f64p, _f64p, _f64p, _i32p, C.c_int, C.c_int, _f64p, _i32p]
        L.orc_detect_frame.argtypes = [_u8p, C.c_int, C.c_int, _i32p, C.c_int, C.c_double, C.c_int, _u8p, _u8p, C.c_int,
                                       C.c_double, C.c_double, _u8p, _u8p, C.c_double, C.c_double, C.c_double,
                                       _i32p, _i32p, _i32p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_detect_frame.restype = C.c_int
        _lib = L
    return _lib


# ---- the tsd_config fields the oracle takes ------------------------------------------------------------------------
# The reference's constants (DET:119-129,164,70-87,712); `cfg` below is a tsd_config (ctypes) or any object with these field names.
DEFAULTS = dict(aspect_lo=0.8, aspect_hi=1.20, hist_tol=0.85, coord_tol=0.95, merge_factor=0.8823,
                red_lo=((0, 50, 10), (160, 50, 10)), red_hi=((10, 255, 255), (179, 255, 255)), blue_lo=(90, 70, 10),
                blue_hi=(128, 255, 255))


def _config(cfg, kw, names):
    """-> {name: value} for `names`: keyword argument, else cfg's field, else the reference's constant."""
    unknown = set(kw) - set(DEFAULTS)
    if unknown:
        raise TypeError("unknown config fields %s" % sorted(unknown))
    return {k: kw[k] if k in kw else getattr(cfg, k) if cfg is not None else DEFAULTS[k] for k in names}


def _hsv_bounds(cfg, kw):
    """-> (lo, hi) uint8 [3][3] (red band 0, red band 1, blue) x (H, S, V)."""
    v = _config(cfg, kw, ("red_lo", "red_hi", "blue_lo", "blue_hi"))
    lo = np.array([list(v["red_lo"][0]), list(v["red_lo"][1]), list(v["blue_lo"])], np.uint8)
    hi = np.array([list(v["red_hi"][0]), list(v["red_hi"][1]), list(v["blue_hi"])], np.uint8)
    return lo.reshape(-1), hi.reshape(-1)


# ---- A.1  DET:155-174 / REC:88-107 -------------------------------------------------------------------------------
def expand_box(box, percentage, cfg=None, **kw):
    """(x,y,w,h) int32 -> (x1,y1,x2,y2) tuple or None.  Aspect bounds: aspect_lo / aspect_hi (cfg or keywords)."""
    a = _config(cfg, kw, ("aspect_lo", "aspect_hi"))
    out = np.zeros(4, np.int32)
    ok = lib().orc_expand_box(int(box[0]), int(box[1]), int(box[2]), int(box[3]), float(percentage), float(a["aspect_lo"]),
                              float(a["aspect_hi"]), out)
    return tuple(int(v) for v in out) if ok else None


def expand_boxes(boxes, percentage, cfg=None, **kw):
    """boxes int32[n,4] -> (coords int32[n,4], valid bool[n])."""
    a = _config(cfg, kw, ("aspect_lo", "aspect_hi"))
    boxes = np.ascontiguousarray(boxes, np.int32).reshape(-1, 4)
    coords = np.zeros_like(boxes)
    valid = np.zeros(len(boxes), bool)
    out = np.zeros(4, np.int32)
    L = lib()
    for i, b in enumerate(boxes):
        if L.orc_expand_box(int(b[0]), int(b[1]), int(b[2]), int(b[3]), float(percentage), float(a["aspect_lo"]),
                            float(a["aspect_hi"]), out):
            coords[i] = out
            valid[i] = True
    return coords, valid


# ---- A.2  DET:123-124 --------------------------------------------------------------------------------------------
def resize_linear(src, D):
    """cv2.resize(src, (D, D)) for uint8 [h,w] or [h,w,C] (any row stride)."""
    src = np.asarray(src)
    assert src.dtype == np.uint8
    h, w = src.shape[:2]
    ch = 1 if src.ndim == 2 else src.shape[2]
    if not (src.strides[-1] == 1 and (src.ndim == 2 or src.strides[1] == ch)):
        src = np.ascontiguousarray(src)
    dst = np.empty((D, D) if src.ndim == 2 else (D, D, ch), np.uint8)
    lib().orc_resize_linear_u8(src.ctypes.data, h, w, src.strides[0], ch, dst, D)
    return dst


def crop_resize(frame, coords, D):
    """cv2.resize(frame[y1:y2, x1:x2], (D, D)) -- crop clipped to the frame like a numpy slice."""
    frame = np.ascontiguousarray(frame)
    H, W = frame.shape[:2]
    ch = 1 if frame.ndim == 2 else frame.shape[2]
    dst = np.empty((D, D) if frame.ndim == 2 else (D, D, ch), np.uint8)
    ok = lib().orc_crop_resize(frame.reshape(-1), H, W, ch, np.asarray(coords, np.int32), dst.reshape(-1), D)
    if not ok:
        raise ValueError("empty crop")
    return dst


# ---- A.3  DET:63-89 ----------------------------------------------------------------------------------------------
def bgr2hsv(bgr):
    bgr = np.ascontiguousarray(bgr, np.uint8)
    out = np.empty_like(bgr)
    lib().orc_bgr2hsv(bgr.reshape(-1), bgr.size // 3, out.reshape(-1))
    return out


def color_masks(window, cfg=None, **kw):
    """-> (red uint8[D,D], blue uint8[D,D]) in {0,255}; getColorMaskRedOrBlue(img,'r'/'b').  HSV bounds: red_lo, red_hi
    [2][3], blue_lo, blue_hi [3] (cfg or keywords)."""
    window = np.ascontiguousarray(window, np.uint8)
    shp = window.shape[:-1]
    red = np.empty(shp, np.uint8)
    blue = np.empty(shp, np.uint8)
    lo, hi = _hsv_bounds(cfg, kw)
    lib().orc_color_masks(window.reshape(-1), window.size // 3, lo, hi, red.reshape(-1), blue.reshape(-1))
    return red, blue


# ---- A.4  DET:545-567, 248-261, 229-245 --------------------------------------------------------------------------
def score_hundredths(mask, templ):
    """calculateScoreBetweenMatrixs(mask*templ, templ) in hundredths, plus (TP,FP,FN,TN)."""
    counts = np.zeros(4, np.int32)
    s = lib().orc_score_hundredths(np.ascontiguousarray(mask, np.uint8).reshape(-1),
                                   np.ascontiguousarray(templ, np.uint8).reshape(-1), int(np.asarray(mask).size), counts)
    return s, tuple(int(c) for c in counts)


def score_window(window, red6, blue6, tol_hundredths=55, cfg=None, **kw):
    """detectionsMaskCorrelation -> (emitted, id, hundredths).  HSV bounds as in color_masks."""
    D = window.shape[0]
    i, h = C.c_int(), C.c_int()
    lo, hi = _hsv_bounds(cfg, kw)
    ok = lib().orc_score_window(np.ascontiguousarray(window, np.uint8).reshape(-1), D,
                                np.ascontiguousarray(red6, np.uint8).reshape(-1),
                                np.ascontiguousarray(blue6, np.uint8).reshape(-1), int(tol_hundredths), lo, hi, C.byref(i), C.byref(h))
    return bool(ok), i.value, h.value


# ---- A.5  DET:575-586, 200-202, 459-468, 177-223 -----------------------------------------------------------------
def hist_normalized(window):
    window = np.ascontiguousarray(window, np.uint8)
    h = np.empty(3000, np.float32)
    lib().orc_hist_normalized(window.reshape(-1), window.size // 3, h)
    return h.reshape(50, 60)


def hist_correl(h1, h2):
    return lib().orc_hist_correl(np.ascontiguousarray(h1, np.float32).reshape(-1),
                                 np.ascontiguousarray(h2, np.float32).reshape(-1))


def eucl_similarity_d2(d2):
    return lib().orc_eucl_similarity_d2(int(d2))


def coord_similarity(a, b):
    return lib().orc_coord_similarity(np.asarray(a, np.int32), np.asarray(b, np.int32))


def dedup(windows, coords, by_coords, tol, merge_factor=0.8823, stats=None):
    """cleanDuplicatedDetections on one frame's list.  -> (windows[m], coords[m]) survivors in list order."""
    windows = np.array(windows, np.uint8, copy=True, order="C")
    coords = np.array(coords, np.int32, copy=True, order="C").reshape(-1, 4)
    n = len(coords)
    if n == 0:
        return windows[:0], coords[:0]
    D = windows.shape[1]
    sp = stats.ctypes.data if stats is not None else None
    m = lib().orc_dedup(windows.reshape(-1), coords.reshape(-1), n, D, int(bool(by_coords)), float(tol),
                        float(merge_factor), sp)
    return windows[:m], coords[:m]


def mean_masks(crops_per_type, D=25):
    """calculateMeanMasks (DET/source.py:24-59): per sign type, every crop resized to DxD (cv2.resize INTER_LINEAR, A.2),
    mask = first crop (addWeighted(img, 1, zeros, 0)), then mask = addWeighted(img, .5, mask, .5) = round-half-even of the mean
    (A.5 avg_rne) in list order; then the red / blue masks of the mean image (A.3).  -> (red6, blue6, mean6)."""
    red6, blue6, mean6 = [], [], []
    for crops in crops_per_type:
        mask = np.zeros((D, D, 3), np.uint8)
        for k, c in enumerate(crops):
            r = resize_linear(np.ascontiguousarray(c, np.uint8), D).astype(np.int32)
            if k == 0:
                mask = r.astype(np.uint8)
            else:
                s_ = r + mask.astype(np.int32)
                mask = ((s_ >> 1) + ((s_ & 1) & ((s_ >> 1) & 1))).astype(np.uint8)
        rm, bm = color_masks(mask)
        red6.append(rm); blue6.append(bm); mean6.append(mask)
    return np.stack(red6), np.stack(blue6), np.stack(mean6)


# ---- A.6 / A.7 / A.8  REC:388, 519, 565-641, 592-596 -------------------------------------------------------------
def bgr2gray(bgr):
    bgr = np.ascontiguousarray(bgr, np.uint8)
    out = np.empty(bgr.shape[:-1], np.uint8)
    lib().orc_bgr2gray(bgr.reshape(-1), bgr.size // 3, out.reshape(-1))
    return out


def gamma_table(gamma=2):
    """gammaCorrection's table exactly as the reference builds it (DET/source.py:599-603)."""
    inv = 1 / gamma
    return np.array([((i / 255) ** inv) * 255 for i in range(256)], np.uint8)


def clahe(gray, clip_limit=2.0, tiles=(8, 8)):
    gray = np.ascontiguousarray(gray, np.uint8)
    out = np.empty_like(gray)
    lib().orc_clahe(gray.reshape(-1), gray.shape[0], gray.shape[1], float(clip_limit), int(tiles[0]), int(tiles[1]), out.reshape(-1))
    return out


def gauss3(gray):
    gray = np.ascontiguousarray(gray, np.uint8)
    out = np.empty_like(gray)
    lib().orc_gauss3(gray.reshape(-1), gray.shape[0], gray.shape[1], out.reshape(-1))
    return out


def preprocess(bgr, clip_limit=2.0, tiles=(8, 8), gamma=2):
    """grayAndEnhanceContrast (DET/source.py:135-152): BGR2GRAY -> CLAHE(clip 2, 8x8) -> GaussianBlur 3x3 -> gamma LUT."""
    bgr = np.ascontiguousarray(bgr, np.uint8)
    out = np.empty(bgr.shape[:2], np.uint8)
    lib().orc_preprocess(bgr.reshape(-1), bgr.shape[0], bgr.shape[1], float(clip_limit), int(tiles[0]), int(tiles[1]),
                         gamma_table(gamma), out.reshape(-1))
    return out


def hog32(gray):
    gray = np.ascontiguousarray(gray, np.uint8)
    assert gray.shape == (32, 32)
    d = np.empty(324, np.float32)
    lib().orc_hog_32(gray.reshape(-1), d)
    return d


def lda_predict(X, W, b, tol=0.5):
    """-> (logits f64[n,6], labels int32[n]); W f64[nfeat,6] (column c = classifier c's coef_), b f64[6]."""
    X = np.ascontiguousarray(X, np.float32)
    n, nf = X.shape
    logits = np.empty((n, 6), np.float64)
    labels = np.empty(n, np.int32)
    lib().orc_lda_predict(X.reshape(-1), n, nf, np.ascontiguousarray(W, np.float64).reshape(-1),
                          np.ascontiguousarray(b, np.float64), float(tol), logits.reshape(-1), labels)
    return logits, labels


def knn_predict(X, xbar, S, Ztrain, ytrain, k=4):
    """-> (Z f64[n,6], labels int32[n])."""
    X = np.ascontiguousarray(X, np.float32)
    n, nf = X.shape
    Z = np.empty((n, 6), np.float64)
    labels = np.empty(n, np.int32)
    Zt = np.ascontiguousarray(Ztrain, np.float64)
    lib().orc_knn_predict(X.reshape(-1), n, nf, np.ascontiguousarray(xbar, np.float64),
                          np.ascontiguousarray(S, np.float64).reshape(-1), Zt.reshape(-1),
                          np.ascontiguousarray(ytrain, np.int32), len(Zt), int(k), Z.reshape(-1), labels)
    return Z, labels


# ---- whole frame: DET:116-131 + 708-716 --------------------------------------------------------------------------
def detect_frame(frame, boxes, red6, blue6, percentage=1.30, D=25, tol_hundredths=55, want_survivors=False, cfg=None, **kw):
    """-> dict(coords int32[nd,4], ids, hundredths, stage_counts[4] [, surv_windows, surv_coords]).
    cfg (or keywords): aspect_lo / aspect_hi, the HSV bounds, hist_tol, coord_tol, merge_factor."""
    a = _config(cfg, kw, ("aspect_lo", "aspect_hi", "hist_tol", "coord_tol", "merge_factor"))
    lo, hi = _hsv_bounds(cfg, kw)
    frame = np.ascontiguousarray(frame, np.uint8)
    boxes = np.ascontiguousarray(boxes, np.int32).reshape(-1, 4)
    n = len(boxes)
    H, W = frame.shape[:2]
    cap = max(n, 1)
    dc = np.zeros((cap, 4), np.int32)
    di = np.zeros(cap, np.int32)
    dh = np.zeros(cap, np.int32)
    sc = np.zeros(4, np.int32)
    sw = np.zeros((cap, D, D, 3), np.uint8) if want_survivors else None
    sco = np.zeros((cap, 4), np.int32) if want_survivors else None
    nd = lib().orc_detect_frame(frame.reshape(-1), H, W, boxes.reshape(-1), n, float(percentage), D,
                                np.ascontiguousarray(red6, np.uint8).reshape(-1),
                                np.ascontiguousarray(blue6, np.uint8).reshape(-1), int(tol_hundredths),
                                float(a["aspect_lo"]), float(a["aspect_hi"]), lo, hi, float(a["hist_tol"]), float(a["coord_tol"]),
                                float(a["merge_factor"]), dc.reshape(-1), di, dh,
                                sw.ctypes.data if sw is not None else None,
                                sco.ctypes.data if sco is not None else None, sc.ctypes.data)
    out = dict(coords=dc[:nd].copy(), ids=di[:nd].copy(), hundredths=dh[:nd].copy(), stage_counts=sc)
    if want_survivors:
        out["surv_windows"] = sw[:sc[2]].copy()
        out["surv_coords"] = sco[:sc[2]].copy()
    return out
