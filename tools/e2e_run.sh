#!/bin/bash
# e2e experiments on the GPU box: Context.detect_frames on page-locked host frames, chunked / unchunked staging, copy-kernel grid.
cd "$(dirname "$0")/.."; mkdir -p gpurun_out; L=gpurun_out/${NAME:-e2e}.log; : > $L
(python -m pytest tests -m gpu -x -q -k "host or e2e or detect_frames or pinned or zero or stage" 2>&1 | tail -2) >> $L
for rep in 1 2; do
for cfg in "TSD_STAGE_CHUNK=0" "TSD_STAGE_CHUNK=256" "TSD_STAGE_CHUNK=0 TSD_STAGE_CTAS=8" "TSD_STAGE_CHUNK=256 TSD_STAGE_CTAS=8"; do
  echo "== $cfg" >> $L
  env $cfg python tools/e2e_step.py --frames 1024 --steps 10 2>&1 | tail -2 >> $L
done; done
cat $L
