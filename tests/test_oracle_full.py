"""CPU (-m "not gpu"): the oracle and the timed CPU port (oracle/ref_port.py) against the full-dataset goldens -- every one of the
150 test frames of the reference (tests/golden/make_golden.py full) -- and against the GRAY-descriptor classifiers
(make_golden.py gray).  This is the known-answer test BASELINE.json's north_star names: the reference's resultado.txt, 192 lines."""
import os
import sys

import numpy as np
import pytest

from conftest import STORED

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import refload  # noqa: E402

needs_reference = pytest.mark.skipif(not refload.reference_available(), reason="needs the reference's source tree (TSD_REFERENCE_ROOT)")


def _lines(files, records):
    """resultado.txt lines (DET/source.py:501-508): file;x1;y1;x2;y2;type;score with str() of the 2-decimal score."""
    return ["%s;%d;%d;%d;%d;%d;%s" % (files[f], x1, y1, x2, y2, t, str(h / 100)) for (f, x1, y1, x2, y2, t, h) in records]


def test_full_dataset_kat_oracle(oracle, det_full150, resultado150, templates):
    """All 150 frames: K1 on every MSER box, then both de-duplication passes and the template scores on the reference's
    post-resize windows -> the reference's resultado.txt byte for byte."""
    g = det_full150
    red6, blue6 = templates
    files = [str(f) for f in g["files"]]
    coords, valid = oracle.expand_boxes(g["boxes"], 1.30)
    assert np.array_equal(valid, g["valid"]) and np.array_equal(coords[valid], g["coords_all"][g["valid"]])
    assert np.array_equal(coords[valid], g["coords"])
    records = []
    for f in range(len(files)):
        a, b = g["offsets"][f], g["offsets"][f + 1]
        w1, c1 = oracle.dedup(g["windows"][a:b], g["coords"][a:b], False, 0.85)
        assert np.array_equal(c1, g["p1_coords"][g["p1_offsets"][f]:g["p1_offsets"][f + 1]]), files[f]
        w2, c2 = oracle.dedup(w1, c1, True, 0.95)
        sa, sb = g["surv_offsets"][f], g["surv_offsets"][f + 1]
        assert np.array_equal(w2, g["surv_windows"][sa:sb]) and np.array_equal(c2, g["surv_coords"][sa:sb]), files[f]
        for w, c in zip(w2, c2):
            ok, i, h = oracle.score_window(w, red6, blue6)
            if ok:
                records.append((f,) + tuple(int(v) for v in c) + (i, h))
    assert _lines(files, records) == resultado150


def test_real_frames_k2_oracle(oracle, det_full150, jpeg24, templates, resultado150):
    """24 real frames from their JPEG bytes: crop + resize of every aspect-passing box equals the reference's windows, and the
    whole restated chain gives exactly the frames' lines of resultado.txt."""
    g = det_full150
    red6, blue6 = templates
    for k, f in enumerate(jpeg24["index"]):
        a, b = g["offsets"][f], g["offsets"][f + 1]
        wins = np.stack([oracle.crop_resize(jpeg24["frames"][k], c, 25) for c in g["coords"][a:b]])
        assert np.array_equal(wins, g["windows"][a:b]), jpeg24["files"][k]
        o = oracle.detect_frame(jpeg24["frames"][k], g["boxes"][g["box_offsets"][f]:g["box_offsets"][f + 1]], red6, blue6)
        recs = [(0,) + tuple(int(v) for v in c) + (int(i), int(h)) for c, i, h in zip(o["coords"], o["ids"], o["hundredths"])]
        assert _lines([jpeg24["files"][k]], recs) == [ln for ln in resultado150 if ln.startswith(jpeg24["files"][k])]


def test_ref_port_all_stored_frames(det_full150, jpeg24, templates, resultado150, det_frames, frames3):
    """oracle/ref_port.py -- what bench.py times as the CPU baseline and what the headline ratio divides by -- on every stored real
    frame (24 JPEG + 3 PNG): survivors and detections equal the reference's own outputs."""
    pytest.importorskip("cv2")
    from oracle import ref_port
    g = det_full150
    red, blue = ref_port.templates_as_lists(*templates)
    for k, f in enumerate(jpeg24["index"]):
        name = jpeg24["files"][k]
        boxes = g["boxes"][g["box_offsets"][f]:g["box_offsets"][f + 1]]
        items = ref_port.frame_windows(jpeg24["frames"][k], boxes, name)
        sa, sb = g["surv_offsets"][f], g["surv_offsets"][f + 1]
        assert len(items) == sb - sa
        if items:
            assert np.array_equal(np.stack([i[0] for i in items]), g["surv_windows"][sa:sb])
            assert np.array_equal(np.array([i[1] for i in items]), g["surv_coords"][sa:sb])
        dets = ref_port.detect_frame(jpeg24["frames"][k], boxes, name, red, blue)
        got = ["%s;%d;%d;%d;%d;%d;%s" % (d[0], d[1], d[2], d[3], d[4], d[5], str(d[6])) for d in dets]
        assert got == [ln for ln in resultado150 if ln.startswith(name)]
    for k in STORED:
        dets = ref_port.detect_frame(frames3[k], det_frames[k + "_boxes"], k, red, blue)
        assert [d[1:5] for d in dets] == [tuple(c) for c in det_frames[k + "_det_coords"].tolist()]


@needs_reference
def test_ref_port_vs_live_reference_synthetic(templates, tsd):
    """Where the reference's source tree is available: ref_port against the unmodified reference functions on 6 synthetic bench
    frames (1360x800, 200 candidates: the workload both bench arms time) -- same survivors, same detection tuples -- and its cost
    stays within a factor 1.5 of the reference's (it must cost what the reference costs to be a fair baseline)."""
    import time
    import cv2
    from oracle import ref_port
    src, _ = refload.load_det()
    src.tqdm = lambda it=None, *a, **k: it
    red6, blue6 = templates
    red, blue = ref_port.templates_as_lists(red6, blue6)
    F = 6
    frames = tsd.synth.make_frames(F)
    boxes, off = tsd.synth.make_boxes(F, 200)
    t_ref = t_port = 0.0
    for f in range(F):
        name = "%05d.jpg" % f
        bx = boxes[off[f]:off[f + 1]]
        t0 = time.perf_counter()
        items = []
        for b in bx:                                                     # DET/source.py:116-129 without the MSER call
            c = src.makeWindowBiggerOrDiscardFakeDetections(b, 1.30)
            if c is not None:
                items.append((cv2.resize(src.cropImageByCoords(c, frames[f]), (25, 25)), c, name))
        items = src.cleanDuplicatedDetections(items, False, 0.85)
        items = src.cleanDuplicatedDetections(items, True, 0.95)
        ref_dets = [d for d in (src.detectionsMaskCorrelation(i, red, blue, 0.55) for i in items) if d is not None]
        t1 = time.perf_counter()
        port_items = ref_port.frame_windows(frames[f], bx, name)
        port_dets = [d for d in (ref_port.classify_window(i, red, blue) for i in port_items) if d is not None]
        t2 = time.perf_counter()
        t_ref += t1 - t0; t_port += t2 - t1
        assert len(items) == len(port_items)
        assert all(np.array_equal(a[0], b[0]) and tuple(a[1]) == tuple(b[1]) for a, b in zip(items, port_items))
        assert [tuple(d) for d in ref_dets] == [tuple(d) for d in port_dets]
    assert 1 / 1.5 < t_port / t_ref < 1.5, (t_port, t_ref)


def test_gray_descriptor_classifiers_oracle(oracle, rec_golden, rec_gray_golden):
    """GRAY_LDA_LDABAYES / GRAY_LDA_KNN (REC/constants.py:10-12): the 1024 raw grey pixels (REC/source.py:520-521 image.ravel())
    through the oracle's LDA decision and 4-NN equal sklearn's logits / labels as the reference computed them."""
    g = rec_gray_golden
    X = rec_golden["gray"].reshape(-1, 1024).astype(np.float32)
    lg, lab = oracle.lda_predict(X, g["lda_W"], g["lda_b"])
    assert np.max(np.abs(lg - g["logits"]) / np.maximum(1.0, np.abs(g["logits"]))) < 1e-9 and np.array_equal(lab, g["pred_lda"])
    Z, lk = oracle.knn_predict(X[:300], g["knn_xbar"], g["knn_scalings"], g["knn_Ztrain"], g["knn_ytrain"])
    assert np.max(np.abs(Z - g["knn_Zq"][:300]) / np.maximum(1.0, np.abs(g["knn_Zq"][:300]))) < 1e-9 and np.array_equal(lk, g["pred_knn"][:300])


def test_install_rebinds_exactly_the_patched_names(tsd, monkeypatch):
    """install() on stand-in modules: every name in _PATCHED is rebound to the mirror's own function and every other attribute is
    left as it was.  (That the reference's modules define and call those names is checked where the reference tree is available.)"""
    import types
    monkeypatch.setattr(tsd.source_det, "_installed_into", None)          # install() records its target; restored afterwards
    for mirror in (tsd.source_det, tsd.source_rec):
        mod = types.ModuleType("stand_in_source")
        before = {name: object() for name in mirror._PATCHED + ("test", "testValidation", "constants", "tqdm")}
        vars(mod).update(before)
        assert mirror.install(mod) is mod
        for name, obj in before.items():
            assert getattr(mod, name) is (getattr(mirror, name) if name in mirror._PATCHED else obj), name
        assert set(vars(mod)) == set(before) | set(vars(types.ModuleType("x")))


@needs_reference
def test_install_rebinds_the_reference_modules_call_compatibly():
    """The drop-in boundary on the live reference modules (no GPU needed: nothing is called): every name source_det / source_rec
    patch exists in the reference's own `source` module with the same positional parameters, is really looked up through the module's
    globals by the reference's code (so rebinding it reroutes the reference's own drivers and helpers), and install() rebinds
    exactly those names and nothing else."""
    import inspect
    import tsd_b200
    for load, mirror in ((refload.load_det, tsd_b200.source_det), (refload.load_rec, tsd_b200.source_rec)):
        ref, _ = load()
        before = dict(vars(ref))
        used = set()
        for obj in before.values():
            if inspect.isfunction(obj) and obj.__module__ == ref.__name__:
                used |= set(obj.__code__.co_names)
        for name in mirror._PATCHED:
            assert name in before and inspect.isfunction(before[name]), name
            ours = getattr(mirror, name)
            p_ref = list(inspect.signature(before[name]).parameters.values())
            p_our = list(inspect.signature(ours).parameters.values())
            required = [p for p in p_our if p.default is inspect.Parameter.empty]
            # callable exactly the way the reference calls its own function (positionally, with its number of arguments)
            assert len(required) <= len(p_ref) <= len(p_our), (name, [p.name for p in p_ref], [p.name for p in p_our])
            assert name in used, name + " is not called through the module's globals"
        mirror.install(ref)
        after = vars(ref)
        for name in mirror._PATCHED:
            assert after[name] is getattr(mirror, name)
        changed = {k for k in after if k in before and after[k] is not before[k]}
        assert changed == set(mirror._PATCHED)
        for name, obj in before.items():                                          # (restore: the loader caches the modules)
            setattr(ref, name, obj)


@needs_reference
def test_reference_driver_through_install(tmp_path, monkeypatch, resultado150):
    """The reference's OWN driver `test()` (DET/source.py:611-853) run through source_det.install(), on the 150 test frames, without
    a GPU: the engine behind the mirrors is a test double answered by the CPU oracle (tests/oracle_context.py).  What this pins is everything between the driver and the engine: the patched
    names, their argument / return conventions as the driver uses them (Python-int tuples, float scores, [(mask, name)] lists,
    (detections, counts, images) triples), the directory walks.  resultado.txt must equal the reference's own, line for line."""
    sys.path.insert(0, os.path.dirname(__file__))
    import tsd_b200
    from oracle_context import OracleContext
    src, _ = refload.load_det()
    before = dict(vars(src))
    fake = OracleContext()
    monkeypatch.setattr(tsd_b200.source_det, "_ctx", fake)
    monkeypatch.setattr(tsd_b200.source_det, "_templates_key", None)
    for d in ("train_jpg", "test_alumnos_jpg"):
        os.symlink(os.path.join(refload.DET_DIR, d), tmp_path / d)
    monkeypatch.chdir(tmp_path)
    try:
        tsd_b200.source_det.install(src)
        src.tqdm = lambda it=None, *a, **k: it
        src.sleep = lambda *_: None
        src.test("train_jpg", "test_alumnos_jpg", (7, 200, 2000, 0.15))
    finally:
        for name, obj in before.items():
            setattr(src, name, obj)
    got = (tmp_path / "resultado.txt").read_text().splitlines()
    assert sorted(got) == sorted(resultado150) and len(got) == 192
    # the driver really went through the mirrors
    assert fake.calls["windows"] == 150 and fake.calls["dedup"] >= 150 and fake.calls["score_masks"] >= 192 and fake.calls["mean_windows"] == 1
    assert len(os.listdir(tmp_path / "resultado_imgs")) == 150


@needs_reference
@pytest.mark.parametrize("descriptor,classifier", [("HOG", "LDABAYES"), ("HOG", "KNN"), ("GRAY", "LDABAYES"), ("GRAY", "KNN")])
def test_reference_recognition_driver_through_install(tmp_path, monkeypatch, descriptor, classifier):
    """The reference's own `testValidation()` (REC/source.py:646-809) on a reduced training directory (8 real train frames that
    hold at least three signs of every type + their gt.txt lines; MSER (7, 200, 2000, 1.0) as in the reference), run twice from
    the same seeds: UNPATCHED (pure reference: cv2 + scikit-learn) and through source_rec.install() with the engine behind the
    mirrors replaced by the oracle-backed test double (no GPU in the container that holds the reference tree).  The training-window
    cache MSERTrain.val (grey 32x32 pixels and coordinates, in order) and the predicted / true labels of the validation split
    must be identical: this pins the glue of every patched REC function as the driver uses it (window extraction, negatives,
    descriptors, weights read out of the fitted sklearn objects, the LDA-Bayes and KNN decisions), for the four classifier strings
    of REC/constants.py:10-12 (HOG / GRAY descriptor x LDA-Bayes / KNN)."""
    import pickle
    import random
    sys.path.insert(0, os.path.dirname(__file__))
    import tsd_b200
    from oracle_context import OracleContext
    src, _ = refload.load_rec()
    files = ["00073.jpg", "00177.jpg", "00307.jpg", "00097.jpg", "00200.jpg", "00004.jpg", "00010.jpg", "00020.jpg"]
    train = tmp_path / "train_small"
    train.mkdir()
    for f in files:
        os.symlink(os.path.join(refload.REC_DIR, "train_jpg", f), train / f)
    stems = {f.split(".")[0] for f in files}
    with open(train / "gt.txt", "w") as out:
        for line in open(os.path.join(refload.REC_DIR, "train_jpg", "gt.txt")):
            if line.split(".")[0] in stems:
                out.write(line)
    before = dict(vars(src))
    fakes = {}

    def run(patched):
        cwd = tmp_path / ("patched" if patched else "reference")
        cwd.mkdir()
        monkeypatch.chdir(cwd)                               # (MSERTrain.val is a cwd-relative cache: one directory per run)
        for k, v in before.items():
            setattr(src, k, v)
        src.tqdm = lambda it=None, *a, **k: it
        src.sleep = lambda *_: None
        if patched:
            fakes["det"], fakes["rec"] = OracleContext("det"), OracleContext("rec")
            monkeypatch.setattr(tsd_b200.source_det, "_ctx", fakes["det"])
            monkeypatch.setattr(tsd_b200.source_rec, "_ctx", fakes["rec"])
            monkeypatch.setattr(tsd_b200.source_rec, "_lda_key", None)
            monkeypatch.setattr(tsd_b200.source_rec, "_knn_key", None)
            tsd_b200.source_rec.install(src)
        rec = {}
        inner = src.predictProbability

        def spy(*a, **k):
            r = inner(*a, **k)
            rec["pred"], rec["true"] = [int(v) for v in r[0]], [int(v) for v in r[1]]
            return r
        src.predictProbability = spy
        random.seed(0); np.random.seed(0)
        src.testValidation(str(train), (7, 200, 2000, 1.0), (descriptor, "LDA", classifier), 0.1, 0.5)
        rec["val"] = pickle.load(open("MSERTrain.val", "rb"))
        return rec
    try:
        ref, got = run(False), run(True)
    finally:
        for k, v in before.items():
            setattr(src, k, v)
    assert len(ref["pred"]) > 20 and got["pred"] == ref["pred"] and got["true"] == ref["true"]
    assert list(got["val"].keys()) == list(ref["val"].keys())
    for k in ref["val"]:
        assert len(got["val"][k]) == len(ref["val"][k]) > 0
        for a, b in zip(got["val"][k], ref["val"][k]):
            assert np.array_equal(a[0], b[0]) and tuple(a[1]) == tuple(b[1]) and a[2:] == b[2:]
    assert fakes["rec"].calls["windows"] >= 1 and (descriptor == "GRAY" or fakes["rec"].calls["hog"] >= 2)
    assert fakes["rec"].calls.get("lda_predict" if classifier == "LDABAYES" else "knn_predict", 0) == 1
