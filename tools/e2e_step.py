"""e2e timing of Context.detect_frames (host pinned frames -> H2D -> chain -> D2H records).
Environment: TSD_STAGE (0 = K2 gathers from host memory itself), TSD_STAGE_CHUNK, TSD_STAGE_CTAS, TSD_ZEROCOPY, TSD_CHUNK_FRAMES."""
import argparse, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import tsd_b200
ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=256)
ap.add_argument("--steps", type=int, default=5)
a = ap.parse_args()
g = np.load(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "det_templates.npz"))
uniq = tsd_b200.synth.make_frames(16)
boxes, off = tsd_b200.synth.make_boxes(a.frames, 200)
h = torch.empty((a.frames, 800, 1360, 3), dtype=torch.uint8).pin_memory()
h.copy_(torch.from_numpy(uniq)[torch.arange(a.frames) % 16])
hf = h.numpy()
ctx = tsd_b200.Context(0, "det")
ctx.set_templates(g["red6"], g["blue6"])
for _ in range(2):
    det, counts = ctx.detect_frames(hf, boxes, off)
ctx.stat_staged_bytes(reset=True)
t0 = time.perf_counter()
for _ in range(a.steps):
    det, counts = ctx.detect_frames(hf, boxes, off)
dt = (time.perf_counter() - t0) / a.steps
staged = ctx.stat_staged_bytes() / a.steps
ctx.set_profiling(True)
ctx.detect_frames(hf, boxes, off)
print({k: round(v, 3) for k, v in ctx.stage_times()})
ctx.set_profiling(False)
print("stage=%s zerocopy=%s frames=%d ms=%.2f windows/s=%.2fM staged=%.1f MB (%.1f GB/s) counts=%s" % (
    os.environ.get("TSD_STAGE", "1"), os.environ.get("TSD_ZEROCOPY", "1"), a.frames, dt * 1e3,
    a.frames * 200 / dt / 1e6, staged / 1e6, staged / dt / 1e9, counts.tolist()))
