"""k5_hist alone, two trees alternated: the per-stage CUDA-event time of the histogram kernel in the device-resident detection chain
(tools/prof_step.py --times: batches serialised; 4096 frames x 200 candidates = bench.py's 332 505 windows by default).

    python tools/hist_ab.py --base-root DIR [--rounds 3] [--frames 4096] [--steps 10]

DIR is a checkout of the reference commit with its library built; the other arm is this tree.  Each arm runs its own
tools/prof_step.py, so the two need not share an API.  Prints one line per run and a JSON summary with the GPU's name and power limit.
"""
import argparse
import ast
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def stage_ms(root, frames, steps):
    env = dict(os.environ)
    env.pop("TSD_LIB", None)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "prof_step.py"), "--frames", str(frames), "--steps", str(steps), "--times"],
                         env=env, capture_output=True, text=True, check=True).stdout
    return ast.literal_eval(next(l for l in out.splitlines() if l.startswith("{")))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-root", required=True, help="tree of the reference arm (library built)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    res = {"gpu": q.strip().splitlines()[0] if q.strip() else "unknown", "frames": a.frames, "base": [], "this": []}
    for r in range(a.rounds):
        for arm, root in (("base", os.path.abspath(a.base_root)), ("this", ROOT)):
            st = stage_ms(root, a.frames, a.steps)
            res[arm].append(st["k5_hist"])
            print("round %d %-4s k5_hist %.4f ms  (stages %s)" % (r, arm, st["k5_hist"], st), flush=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
