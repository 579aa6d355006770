"""Drop-in mirror of the hot-path functions of "Deteción de Objetos/source.py" (DET).

Same names, argument meaning, return conventions and error behaviour as the reference functions, so the reference's
drivers (`test()`, DET:611-853) run unchanged when these are patched in (see INTEGRATION.md: `install(source)`).
Every stage runs on the GPU through engine.Context; cv2 is used ONLY for what BASELINE.json keeps on the
reference's cv2 path: the MSER region proposals and their pre-processing (DET:112-114,135-152), and image decode.
"""
import os

import numpy as np

from . import engine
from ._capi import TsdError

SIGNALLIST = ['prohibicion', 'peligro', 'stop', 'direccionProhibida', 'cedaPaso', 'direccionObligatoria']  # DET/constants.py:1

_ctx = None
_templates_key = None
_installed_into = None            # the reference module install() patched last


def context():
    """Process-wide detection-flavour context (x1.30, 25x25) on cuda:0 (or $TSD_DEVICE)."""
    global _ctx
    if _ctx is None:
        _ctx = engine.Context(device=int(os.environ.get("TSD_DEVICE", "0")), flavour="det")
    return _ctx


def _use_templates(signalsMasksRed, signalsMasksBlue):
    """Upload the 6+6 template masks produced by calculateMeanMasks (DET:24-59) once per distinct set."""
    global _templates_key
    red = np.stack([np.asarray(m, np.uint8) for m, _ in signalsMasksRed])
    blue = np.stack([np.asarray(m, np.uint8) for m, _ in signalsMasksBlue])
    key = (red.tobytes(), blue.tobytes())
    if key != _templates_key:
        context().set_templates(red, blue)
        _templates_key = key


# ---- proposal stage ---------------------------------------------------------------------------------------------------
def grayAndEnhanceContrast(image):
    """DET:135-152 -- the pre-processing that feeds MSER (SURVEY 8(f) N1), on the GPU: BGR2GRAY, CLAHE(clip 2, 8x8), Gaussian
    3x3 and the gamma-2 table, bit-identical to the four cv2 calls of the reference."""
    return context().preprocess(np.asarray(image, np.uint8))


def gammaCorrection(src, gamma):
    """DET:599-605 (a 256-entry table lookup; host-side numpy, kept for callers that use it on its own)."""
    table = np.array([((i / 255) ** (1 / gamma)) * 255 for i in range(256)], np.uint8)
    return table[np.asarray(src, np.uint8)]


def proposals(image, mser):
    """int32 [n,4] (x,y,w,h) MSER boxes exactly as DET:112-114 produces them: GPU pre-processing, then cv2's MSER (which stays
    on the reference's cv2 path by north_star)."""
    boxes = mser.detectRegions(grayAndEnhanceContrast(image))[1]
    return np.asarray(boxes, np.int32).reshape(-1, 4)


# ---- template masks (SURVEY 8(f) N2) -----------------------------------------------------------------------------
SIGN_GROUPS = (['00', '01', '02', '03', '04', '05', '07', '08', '09', '10', '15', '16'],                       # DET/constants.py:2-7
               ['11', '18', '19', '20', '21', '22', '23', '24', '25', '26', '27', '28', '29', '30', '31'],
               ['14'], ['17'], ['13'], ['38'])


def meanMasksFromCrops(crops_per_type):
    """The arithmetic of calculateMeanMasks (DET:24-59) on the GPU: every class crop resized to 25x25 (K2), the
    order-dependent running average per sign type (tsd_mean_windows), then the red / blue masks of the six mean images
    (K3).  crops_per_type: 6 lists of BGR uint8 images in the reference's iteration order.
    -> (signalsMasksRed, signalsMasksBlue, mean6) with the reference's [(mask, name)] * 6 convention."""
    ctx = context()
    crops = [np.asarray(c, np.uint8) for t in crops_per_type for c in t]
    off = np.concatenate([[0], np.cumsum([len(t) for t in crops_per_type])]).astype(np.int32)
    Hm, Wm = max(c.shape[0] for c in crops), max(c.shape[1] for c in crops)
    Wm = (Wm + 15) // 16 * 16
    # One "frame" per crop; the crop is the ROI (0, 0, w, h).  Context.crop_resize would take the crops as a list of frames of
    # different sizes, but the atlas stays: the reference's driver test runs this function through an oracle-backed stand-in
    # of the Context that takes ndarrays only.
    atlas = np.zeros((len(crops), Hm, Wm, 3), np.uint8)
    coords = np.zeros((len(crops), 4), np.int32)
    for i, c in enumerate(crops):
        atlas[i, :c.shape[0], :c.shape[1]] = c
        coords[i] = (0, 0, c.shape[1], c.shape[0])
    wins = ctx.crop_resize(atlas, coords, np.arange(len(crops), dtype=np.int32))
    mean6 = ctx.mean_windows(wins, off)
    red, blue = ctx.color_masks(mean6)
    return [(red[k], SIGNALLIST[k]) for k in range(6)], [(blue[k], SIGNALLIST[k]) for k in range(6)], mean6


def calculateMeanMasks(train_path=None):
    """DET:24-59 drop-in: same directory walk (os.listdir order, DET:42-43) and image decode (cv2.imread) as the reference;
    resize, running average and masks on the GPU."""
    import cv2
    if train_path is None:
        # the reference reads its module global constants.TRAIN_PATH (set by test(), DET:612): the `constants` the patched
        # module itself imported, or -- called without install() from the reference's directory -- the importable one
        consts = getattr(_installed_into, "constants", None)
        if consts is None:
            import constants as consts
        train_path = consts.TRAIN_PATH
    crops = []
    for dirs in SIGN_GROUPS:
        t = []
        for d in dirs:
            for f in os.listdir(train_path + '/' + d):
                t.append(cv2.imread(train_path + '/' + d + '/' + f))
        crops.append(t)
    red, blue, _ = meanMasksFromCrops(crops)
    return red, blue


# ---- K1 -----------------------------------------------------------------------------------------------------------
def makeWindowBiggerOrDiscardFakeDetections(window, percentage):
    """DET:155-174 -> (x1, y1, x2, y2) Python ints, or None."""
    coords, valid = context().expand_boxes(np.asarray(window, np.int32).reshape(1, 4), percentage)
    return tuple(int(v) for v in coords[0]) if valid[0] else None


def cropImageByCoords(coords, image):
    """DET:570-572 (a numpy view; no arithmetic)."""
    x1, y1, x2, y2 = coords
    return image[y1:y2, x1:x2]


# ---- K1+K2+K5: MSERTrafficSignDetector ---------------------------------------------------------------------------
def windowsFromBoxes(image, boxes, file):
    """Candidate loop DET:116-124 on the GPU -> list of (uint8[25,25,3], (x1,y1,x2,y2), file)."""
    ctx = context()
    boxes = np.asarray(boxes, np.int32).reshape(-1, 4)
    wins, coords, _ = ctx.windows(image, boxes, np.array([0, len(boxes)], np.int32))
    return [(wins[i], tuple(int(v) for v in coords[i]), file) for i in range(len(coords))]


def cleanDuplicatedDetections(imageDetections, isSimilarityByEuclideanDistanceON, tolerance):
    """DET:177-189 on one frame's list of (window, coords, file[, label]) tuples."""
    items = list(imageDetections)
    if not items:
        return []
    wins = np.stack([np.asarray(i[0], np.uint8) for i in items])
    coords = np.array([i[1] for i in items], np.int32)
    ow, oc, _ = context().dedup(wins, coords, np.array([0, len(items)], np.int32), isSimilarityByEuclideanDistanceON, tolerance)
    # A survivor keeps its own (file[, label]); a merged one takes them from the absorbing (incoming) item (DET:219-221).  The
    # reference only ever calls this with one frame's list, where every tail is the same -- anything else is refused rather
    # than answered with the wrong tail.
    tail = tuple(items[0][2:])
    if any(tuple(i[2:]) != tail for i in items):
        raise ValueError("cleanDuplicatedDetections: items of one call must share (file[, label]) -- one frame's list per call")
    return [(ow[i], tuple(int(v) for v in oc[i])) + tail for i in range(len(oc))]


def MSERTrafficSignDetector(image, mser, file):
    """DET:111-131: cv2 MSER proposals, then K1+K2 and both K5 passes on the GPU."""
    boxes = proposals(image, mser)
    dets = windowsFromBoxes(image, boxes, file)
    dets = cleanDuplicatedDetections(dets, False, 0.85)      # DET:127
    dets = cleanDuplicatedDetections(dets, True, 0.95)       # DET:129
    return dets


def createImageWithWindows(image, windowsBorders):
    """DET:589-594 (drawing; cv2, not on the hot path)."""
    import cv2
    for det in windowsBorders:
        x1, y1, x2, y2 = det[1]
        image = cv2.rectangle(image, (x1, y1), (x2, y2), (0, 0, 255), 1)
    return image


def detectSignsOnDirectory(path, mser):
    """DET:95-108 -> (detections per file, [(file, count)], [(file, image with windows)])."""
    import cv2
    directoryDetections, numberOfDetections, imagesWithWindows = [], [], []
    for file in os.listdir(path):
        if not file.endswith('.txt'):
            image = cv2.imread(path + '/' + file)
            detections = MSERTrafficSignDetector(image, mser, file)
            directoryDetections.append(detections)
            numberOfDetections.append((file, len(detections)))
            imagesWithWindows.append((file, createImageWithWindows(image.copy(), detections)))
    return directoryDetections, numberOfDetections, imagesWithWindows


# ---- K5 pieces ----------------------------------------------------------------------------------------------------
def calculateHistAndNormalize(image):
    """DET:575-586 -> float32 [50,60]."""
    return context().hist(np.asarray(image, np.uint8)[None])[0]


# ---- K3 -----------------------------------------------------------------------------------------------------------
def getColorMaskRedOrBlue(image, color):
    """DET:63-89 -> uint8 [25,25] in {0,255} ('r' or 'b'); None for any other colour, like the reference."""
    image = np.asarray(image, np.uint8)
    D = context().D
    if image.shape[:2] != (D, D):
        # DET:64 resizes to 25x25 first (identity on the hot path, where windows are already 25x25)
        image = context().crop_resize(image, np.array([[0, 0, image.shape[1], image.shape[0]]], np.int32))[0]
    red, blue = context().color_masks(image[None])
    if color == 'r':
        return red[0]
    if color == 'b':
        return blue[0]
    return None


# ---- K4 -----------------------------------------------------------------------------------------------------------
def getSimilarSignalType(imageMask, signalsMasks):
    """DET:248-261 -> (score float, id 1..6): best of the 6 templates, first maximum wins."""
    _use_templates(signalsMasks, signalsMasks)
    m = np.asarray(imageMask, np.uint8)[None]
    r = context().score_masks(m, m)
    sc = r["scores"][0, 0]
    best, bid = -1, ''
    for k in range(6):
        if sc[k] > best:
            best, bid = int(sc[k]), SIGNALLIST.index(signalsMasks[k][1]) + 1
    return best / 100, bid


def calculateScoreBetweenMatrixs(matrix1, matrix2):
    """DET:545-567 for the reference's call shape: matrix1 = mask*template (uint8 wrap -> {0,1}), matrix2 = template.
    Returns a float rounded to 2 dp, the int 0 for a degenerate template, None on shape mismatch."""
    matrix1 = np.asarray(matrix1); matrix2 = np.asarray(matrix2, np.uint8)
    if matrix1.shape != matrix2.shape:
        return None
    ones = matrix1 == 1
    if np.any(ones & (matrix2 != 255)):
        raise TsdError("matrix1 has ones outside the template: not producible by DET:254 (mask*template)")
    tm = [(matrix2, SIGNALLIST[k]) for k in range(6)]
    _use_templates(tm, tm)
    mask = np.where(ones, 255, 0).astype(np.uint8)[None]
    r = context().score_masks(mask, mask)
    T = int((matrix2 == 255).sum())
    npx = matrix2.size
    if npx + npx * 0.01 >= npx - T >= npx - npx * 0.01:
        return 0
    return int(r["scores"][0, 0, 0]) / 100


def detectionsMaskCorrelation(detection, signalsMasksRed, signalsMasksBlue, tolerance):
    """DET:229-245 -> (file, x1, y1, x2, y2, id, score) or None."""
    _use_templates(signalsMasksRed, signalsMasksBlue)
    ctx = context()
    red, blue = ctx.color_masks(np.asarray(detection[0], np.uint8)[None])
    r = ctx.score_masks(red, blue, want_scores=False)
    score = int(r["hundredths"][0]) / 100
    if score > tolerance:
        x1, y1, x2, y2 = detection[1]
        return detection[2], x1, y1, x2, y2, int(r["id"][0]), score
    return None


# ---- batched entry point (what bench.py and a production caller use) ------------------------------------------------
def detectBatch(frames, boxes, box_offsets, files, signalsMasksRed, signalsMasksBlue):
    """Whole chain for a batch of frames in ONE library call: DET:116-131 per frame + DET:708-716.
    -> list of (file, x1, y1, x2, y2, id, score) in frame order then list order, and the stage counts."""
    _use_templates(signalsMasksRed, signalsMasksBlue)
    det, counts = context().detect_frames(frames, boxes, box_offsets)
    out = [(files[int(d["frame"])], int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"]), int(d["hundredths"]) / 100)
           for d in det]
    return out, counts


def createDetectionsStrings(detections):
    """DET:501-508: `file;x1;y1;x2;y2;type;score` (formatting only)."""
    return [";".join([d[0]] + [str(v) for v in d[1:]]) for d in detections]


_PATCHED = ("calculateMeanMasks", "grayAndEnhanceContrast", "makeWindowBiggerOrDiscardFakeDetections", "cleanDuplicatedDetections", "MSERTrafficSignDetector",
            "detectSignsOnDirectory", "calculateHistAndNormalize", "getColorMaskRedOrBlue", "getSimilarSignalType",
            "calculateScoreBetweenMatrixs", "detectionsMaskCorrelation")


def install(reference_source_module):
    """Monkey-patch the reference's DET `source` module so its own `test()` driver runs the GPU path."""
    global _installed_into
    _installed_into = reference_source_module
    for name in _PATCHED:
        setattr(reference_source_module, name, globals()[name])
    return reference_source_module
