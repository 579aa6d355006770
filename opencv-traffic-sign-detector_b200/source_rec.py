"""Drop-in mirror of the hot-path functions of "Reconocimiento de Objetos/source.py" (REC).

Window extraction (x1.15, 32x32 -- REC:47-64), grey conversion (REC:388), HOG (REC:517-521) and the LDA / KNN
decisions (REC:565-641, 592-596) run on the GPU.  Fitting stays scikit-learn on the host (REC:526-616, out of scope);
its fitted objects are read for their weights only.
"""
import os

import numpy as np

from . import engine
from . import source_det as _det
from ._capi import REC_GRAY, REC_KNN, RUN_RECOGNIZE, TsdError

_ctx = None
_lda_key = None
_knn_key = None


def context():
    """Process-wide recognition-flavour context (x1.15, 32x32)."""
    global _ctx
    if _ctx is None:
        _ctx = engine.Context(device=int(os.environ.get("TSD_DEVICE", "0")), flavour="rec")
    return _ctx


grayAndEnhanceContrast = _det.grayAndEnhanceContrast     # REC:67-84 is the same code as DET:135-152
proposals = _det.proposals
cropImageByCoords = _det.cropImageByCoords


def makeWindowBiggerOrDiscardFakeDetections(window, percentage):
    """REC:88-107."""
    coords, valid = context().expand_boxes(np.asarray(window, np.int32).reshape(1, 4), percentage)
    return tuple(int(v) for v in coords[0]) if valid[0] else None


def cleanDuplicatedDetections(imageDetections, isSimilarityByEuclideanDistanceON, tolerance):
    """REC:110-122 on one frame's list of (window, coords, file, label) tuples."""
    items = list(imageDetections)
    if not items:
        return []
    wins = np.stack([np.asarray(i[0], np.uint8) for i in items])
    coords = np.array([i[1] for i in items], np.int32)
    ow, oc, _ = context().dedup(wins, coords, np.array([0, len(items)], np.int32), isSimilarityByEuclideanDistanceON, tolerance)
    # A survivor keeps its own (file[, label]); a merged one takes them from the absorbing (incoming) item (REC:151-153).  The
    # reference only ever calls this with one frame's list, where every tail is the same -- anything else is refused rather
    # than answered with the wrong tail.
    tail = tuple(items[0][2:])
    if any(tuple(i[2:]) != tail for i in items):
        raise ValueError("cleanDuplicatedDetections: items of one call must share (file[, label]) -- one frame's list per call")
    return [(ow[i], tuple(int(v) for v in oc[i])) + tail for i in range(len(oc))]


def MSERTrafficSignDetector(image, mser, file):
    """REC:47-64 -> list of (uint8[32,32,3], (x1,y1,x2,y2), file, 0)."""
    ctx = context()
    boxes = proposals(image, mser)
    wins, coords, _ = ctx.windows(image, boxes, np.array([0, len(boxes)], np.int32))
    dets = [(wins[i], tuple(int(v) for v in coords[i]), file, 0) for i in range(len(coords))]
    dets = cleanDuplicatedDetections(dets, False, 0.85)
    dets = cleanDuplicatedDetections(dets, True, 0.95)
    return dets


def windowsToGray(detections):
    """The per-window cv2.cvtColor(BGR2GRAY) loop of REC:386-389, batched."""
    if not detections:
        return []
    g = context().bgr2gray(np.stack([np.asarray(d[0], np.uint8) for d in detections]))
    return [(g[i],) + tuple(d[1:]) for i, d in enumerate(detections)]


# ---- training-set window extraction (SURVEY 8(f) N3) ------------------------------------------------------------------
def orderCroppedImagesByImageFile(trainImages, trainResults):
    """REC:247-258: positives = ground-truth boxes cropped from the GREY frame and resized to 32x32 (1-channel K6 + K2),
    -> {file: [(uint8[32,32], (x1,y1,x2,y2), file, signType)]}.  One grey conversion per frame that has ground truth, one
    batched crop+resize call for all boxes."""
    ctx = context()
    out = dict((name, []) for name in trainImages.keys())
    files = sorted(set(r[0] for r in trainResults))
    if not files:
        return out
    index = {f: i for i, f in enumerate(files)}
    grey = engine.stack_if_uniform([ctx.bgr2gray(np.asarray(trainImages[f], np.uint8)) for f in files])     # (frames of different sizes: a list)
    coords = np.array([r[1:5] for r in trainResults], np.int32)
    wf = np.array([index[r[0]] for r in trainResults], np.int32)
    wins = ctx.crop_resize(grey, coords, wf)
    for i, r in enumerate(trainResults):
        out[r[0]].append((wins[i], (r[1], r[2], r[3], r[4]), r[0], r[5]))
    return out


def intersectionOverUnion(imageACoords, imageBCoords):
    """REC:263-280 (inclusive-pixel IoU; a handful of Python ints per call, host side like the reference)."""
    xA, yA = max(imageACoords[0], imageBCoords[0]), max(imageACoords[1], imageBCoords[1])
    xB, yB = min(imageACoords[2], imageBCoords[2]), min(imageACoords[3], imageBCoords[3])
    inter = max(0, xB - xA + 1) * max(0, yB - yA + 1)
    areaA = (imageACoords[2] - imageACoords[0] + 1) * (imageACoords[3] - imageACoords[1] + 1)
    areaB = (imageBCoords[2] - imageBCoords[0] + 1) * (imageBCoords[3] - imageBCoords[1] + 1)
    return inter / float(areaA + areaB - inter)


def computeNegativeTrainResults(trainImages, positiveTrainResults, allImagesMSERDetections):
    """REC:365-377: MSER windows whose best IoU with the frame's ground truth is <= 0.5 are negatives."""
    negatives = dict((name, []) for name in trainImages.keys())
    for name in trainImages.keys():
        for det in allImagesMSERDetections[name]:
            best = -float("inf")
            for pos in positiveTrainResults[name]:
                best = max(best, intersectionOverUnion(det[1], pos[1]))
            if best <= 0.5:
                negatives[name].append(det)
    return negatives


def extractMSERDetectionsGray(trainImages, mser, frames_per_call=64):
    """The body of REC:383-389 for ALL frames: MSERTrafficSignDetector (x1.15, 32x32, both de-duplication passes) followed by the
    per-window BGR2GRAY, batched: cv2.MSER per frame on the host (north_star), then K1+K2, K5 x2 and K6 in four library calls
    per `frames_per_call` frames.  -> {file: [(uint8[32,32] grey, (x1,y1,x2,y2), file, 0)]} -- the content of MSERTrain.val."""
    ctx = context()
    names = list(trainImages.keys())
    out = dict((name, []) for name in names)
    for c0 in range(0, len(names), frames_per_call):
        chunk = names[c0:c0 + frames_per_call]
        imgs = engine.stack_if_uniform([np.asarray(trainImages[n], np.uint8) for n in chunk])
        boxes = [proposals(trainImages[n], mser) for n in chunk]
        off = np.concatenate([[0], np.cumsum([len(b) for b in boxes])]).astype(np.int32)
        allb = np.concatenate(boxes) if off[-1] else np.zeros((0, 4), np.int32)
        wins, coords, woff = ctx.windows(imgs, allb, off)
        w1, c1, o1 = ctx.dedup(wins, coords, woff, False, 0.85)      # REC:59
        w2, c2, o2 = ctx.dedup(w1, c1, o1, True, 0.95)               # REC:61
        grey = ctx.bgr2gray(w2) if len(w2) else np.zeros((0, 32, 32), np.uint8)
        for f, n in enumerate(chunk):
            out[n] = [(grey[i], tuple(int(v) for v in c2[i]), n, 0) for i in range(int(o2[f]), int(o2[f + 1]))]
    return out


def calculateNegativeTrainResults(trainImages, positiveTrainResults, mser):
    """REC:380-398 drop-in, same cwd-relative pickle cache `MSERTrain.val` with the same layout."""
    import pickle
    if not os.path.exists('MSERTrain.val'):
        allImagesMSERDetections = extractMSERDetectionsGray(trainImages, mser)
        with open("MSERTrain.val", "wb") as outfile:
            pickle.dump(allImagesMSERDetections, outfile)
    else:
        with open("MSERTrain.val", "rb") as infile:
            allImagesMSERDetections = pickle.load(infile)
    return computeNegativeTrainResults(trainImages, positiveTrainResults, allImagesMSERDetections)


# ---- descriptors ---------------------------------------------------------------------------------------------------
def computeDescriptors(image, featureDescriptor):
    """REC:517-521: 'HOG' -> float32[324] (cv2.HOGDescriptor.compute), 'GRAY' -> image.ravel()."""
    if featureDescriptor[1] == 'HOG':
        return context().hog(np.asarray(image, np.uint8)[None])[0]
    elif featureDescriptor[1] == 'GRAY':
        return np.asarray(image).ravel()


def calculateDescriptors(trainImages, featureDescriptor):
    """REC:507-514, one GPU call per class list instead of one cv2 call per window."""
    out = dict((signType, []) for signType in range(0, 7))
    for signType in trainImages.keys():
        dets = trainImages[signType]
        if not dets:
            continue
        if featureDescriptor[1] == 'HOG':
            descs = context().hog(np.stack([np.asarray(d[0], np.uint8) for d in dets]))
        else:
            descs = [np.asarray(d[0]).ravel() for d in dets]
        out[signType] = [(descs[i], d[1], d[2], d[3]) for i, d in enumerate(dets)]
    return out


# ---- classifiers -----------------------------------------------------------------------------------------------------
def extractDescriptorsAndRealSignTypes(detectionsDescriptors):
    """REC:307-313."""
    return [d[0] for d in detectionsDescriptors], [d[3] for d in detectionsDescriptors]


def _use_lda(LDAClassifiers):
    global _lda_key
    W = np.stack([np.asarray(c.coef_, np.float64)[0] for c in LDAClassifiers], 1)
    b = np.array([np.asarray(c.intercept_, np.float64)[0] for c in LDAClassifiers])
    key = (W.tobytes(), b.tobytes())
    if key != _lda_key:
        context().set_lda(W, b)
        _lda_key = key


def predictProbabilityLDAClassifiers(LDAClassifiers, detectionsDescriptors, tolerance):
    """REC:565-577 + extractBestPredictions REC:627-641 -> (predicted labels list, true labels list)."""
    X, true = extractDescriptorsAndRealSignTypes(detectionsDescriptors)
    if not X:
        return [], true
    _use_lda(LDAClassifiers)
    _, labels = context().lda_predict(np.stack(X).astype(np.float32), tol=tolerance, want_logits=False)
    return [int(v) for v in labels], true


def _use_knn(KNNClassifier, reducer):
    global _knn_key
    lda = reducer[0]
    Zt = np.asarray(KNNClassifier._fit_X, np.float64)
    yt = np.asarray(KNNClassifier.classes_)[np.asarray(KNNClassifier._y)].astype(np.int32)
    key = (lda.xbar_.tobytes(), Zt.tobytes(), yt.tobytes(), KNNClassifier.n_neighbors)
    if key != _knn_key:
        ncomp = Zt.shape[1]
        if ncomp != 6:
            raise TsdError("KNN path expects the 6-component LDA reducer of REC:586-589")
        context().set_knn(lda.xbar_, lda.scalings_[:, :ncomp], Zt, yt, KNNClassifier.n_neighbors)
        _knn_key = key


def predictProbabilityKNNClassifiers(KNNClassifier, reducer, detectionDescriptors):
    """REC:592-596 -> (predicted labels ndarray, true labels list)."""
    X, true = extractDescriptorsAndRealSignTypes(detectionDescriptors)
    _use_knn(KNNClassifier, reducer)
    if not X:
        return np.zeros(0, np.int64), true
    _, labels = context().knn_predict(np.stack(X).astype(np.float32), want_Z=False)
    return labels.astype(np.int64), true


def predictProbability(classifiers, reducer, testDataDescriptors, tolerance):
    """REC:619-624 dispatcher."""
    if classifiers[1] == 'LDABAYES':
        return predictProbabilityLDAClassifiers(classifiers[0], testDataDescriptors, tolerance)
    elif classifiers[1] == 'KNN':
        return predictProbabilityKNNClassifiers(classifiers[0], reducer, testDataDescriptors)


def recognizeBatch(frames, boxes, box_offsets, files, classifiers, reducer, featureDescriptor):
    """Whole recognition chain for a batch of frames in ONE library call, the counterpart of source_det.detectBatch: per frame
    MSERTrafficSignDetector (REC:47-64) -> windowsToGray -> calculateDescriptors (featureDescriptor[1] = 'HOG' or 'GRAY') ->
    predictProbability (classifiers[1] = 'LDABAYES' with the context's proba_tol, 0.5 as at REC:760, or 'KNN' with `reducer`).
    -> list of (file, x1, y1, x2, y2, label) for every survivor whose label is not 0, in frame order then list order, and the
    stage counts (raw boxes, aspect-passing windows, survivors, records)."""
    mode = RUN_RECOGNIZE
    if featureDescriptor[1] == 'GRAY':
        mode |= REC_GRAY
    elif featureDescriptor[1] != 'HOG':
        raise TsdError("featureDescriptor must be (_, 'HOG') or (_, 'GRAY'), not %r" % (featureDescriptor[1],))
    if classifiers[1] == 'KNN':
        mode |= REC_KNN
        _use_knn(classifiers[0], reducer)
    elif classifiers[1] == 'LDABAYES':
        _use_lda(classifiers[0])
    else:
        raise TsdError("classifiers must be (_, 'LDABAYES') or (_, 'KNN'), not %r" % (classifiers[1],))
    det, counts = context().detect_frames(frames, boxes, box_offsets, mode=mode)
    return [(files[int(d["frame"])], int(d["x1"]), int(d["y1"]), int(d["x2"]), int(d["y2"]), int(d["id"])) for d in det], counts


_PATCHED = ("grayAndEnhanceContrast", "makeWindowBiggerOrDiscardFakeDetections", "cleanDuplicatedDetections", "MSERTrafficSignDetector",
            "orderCroppedImagesByImageFile", "calculateNegativeTrainResults", "computeDescriptors", "calculateDescriptors", "predictProbabilityLDAClassifiers",
            "predictProbabilityKNNClassifiers", "predictProbability")


def install(reference_source_module):
    """Monkey-patch the reference's REC `source` module so `testValidation()` runs the GPU path."""
    for name in _PATCHED:
        setattr(reference_source_module, name, globals()[name])
    return reference_source_module
