"""B200-native candidate-window scoring and recognition path of cfkr-dev/OpenCV-Traffic-Sign-Detector.

Layout
  csrc/            hand-written sm_100a kernels + the C-ABI library (include/tsd_b200.h)
  _capi.py         ctypes binding (fails loudly when the CUDA extension is missing)
  engine.py        Context: numpy-in / numpy-out stage calls and the batched chain
  source_det.py    drop-in mirror of the hot-path functions of "Deteción de Objetos/source.py"
  source_rec.py    drop-in mirror of the hot-path functions of "Reconocimiento de Objetos/source.py"
  sharding.py      frame sharding across ranks (one process per GPU) + the reporting gather
  synth.py         synthetic frames / candidate boxes of SURVEY.md section 8(d)
  evaluate.py      the two evaluators (generateStatistics, precision_recall_curve / AP) with their matching loops on the GPU
"""
from . import _capi, synth  # noqa: F401
from ._capi import DET_DTYPE, FRAME_DESC_DTYPE, HOG_LEN, MEM_DEVICE, MEM_HOST, REC_GRAY, REC_KNN, RUN_DETECT, RUN_RECOGNIZE, TsdError, build  # noqa: F401
from .engine import Context, default_config, similarity_table  # noqa: F401
from . import evaluate, sharding, source_det, source_rec  # noqa: F401,E402

__all__ = ["Context", "default_config", "similarity_table", "TsdError", "build", "DET_DTYPE", "HOG_LEN",
           "RUN_DETECT", "RUN_RECOGNIZE", "REC_GRAY", "REC_KNN", "MEM_HOST", "MEM_DEVICE", "synth"]
