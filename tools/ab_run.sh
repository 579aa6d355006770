#!/bin/bash
# A/B on the GPU box: GPU tests selected by $TESTS (pytest -k expression) with the default library, then per-stage times of the
# device-resident detection step for the default library and every build/libtsd_*.so (tools/build_variants.sh).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
N=${NAME:-ab}
if [ -n "$TESTS" ]; then (python -m pytest tests -m gpu -x -q -k "$TESTS" 2>&1 | tail -3) > gpurun_out/$N.tests.log 2>&1; fi
: > gpurun_out/$N.log
for lib in "" build/libtsd_*.so; do
  [ -n "$lib" ] && [ ! -f "$lib" ] && continue
  echo "== ${lib:-default}" >> gpurun_out/$N.log
  TSD_LIB=${lib:+$PWD/$lib} python tools/prof_step.py --frames 4096 --steps 5 --times 2>&1 | tail -2 | head -1 >> gpurun_out/$N.log
  TSD_LIB=${lib:+$PWD/$lib} python tools/prof_step.py --frames 4096 --steps 10 --wall 2>&1 | head -1 >> gpurun_out/$N.log
  [ -n "$REC" ] && TSD_LIB=${lib:+$PWD/$lib} python tools/prof_step.py --mode rec --frames 1024 --steps 5 --times 2>&1 | tail -2 | head -1 >> gpurun_out/$N.log
done
cat gpurun_out/$N.tests.log gpurun_out/$N.log 2>/dev/null
