"""Cost of Keras gradient clipping on the GPU: the Criteo-shape DeepFM step without clipping and with clipvalue, clipnorm and
global_clipnorm, alternating in one process.

    python profiles/tools/clip_step.py [--steps 30] [--warmup 10] [--rounds 3] [--out file.jsonl]

Step: the shapes of bench.py (26 tables, 102 M rows, D = 16, B = 65536, 429-256-128-1, Adam; tables up to 131072 rows
dense-updated), ONE engine built with a clip so that its FM buffer exists; the modes are swapped by setting `engine.clip` (None:
exactly the unclipped step).  >= 10 warm-up steps cycle through every mode (past the backward autotune trials in steps 3-6), then
`--rounds` x (30 steps per mode) timed with CUDA events over a rotating pool of 4 batches.  Launches per step are read from
hrb_launch_count around one more step of each mode (library kernels only; the torch memset of the norm sums is not counted).
Prints one JSON line per measurement with the GPU name, power limit and max SM clock read by nvidia-smi in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bench  # noqa: E402
from optimizer_step import NB, batches, gpu_info  # noqa: E402

from handyrec_b200 import kernels as K  # noqa: E402
from handyrec_b200.clip import GradClip  # noqa: E402
from handyrec_b200.engine import DeepFMEngine, launch_count  # noqa: E402

MODES = {"none": None, "clipvalue": (1e-5, None, None), "clipnorm": (None, 1e-2, None), "global_clipnorm": (None, None, 1e-2)}


def time_steps(eng, pool, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        eng.train_step_on_device(*pool[s % NB])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clip_step.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    vocabs, D, B = bench.CRITEO_VOCABS, bench.EMB_DIM, bench.BATCH
    tables = []
    for f, v in enumerate(vocabs):
        t = torch.empty(v, D, device=dev)
        K.init_uniform(t, seed=7 + f)
        tables.append(t)
    eng = DeepFMEngine(tables, [(f, 1, "none") for f in range(len(vocabs))], bench.N_DENSE, bench.DNN_HIDDEN, "relu", batch_size=B,
                       optimizer="adam", lr=1e-3, dense_table_max_rows=131072, clipnorm=1.0)
    del tables
    clips = {m: (None if a is None else GradClip(a, eng.clip.n_vars, len(eng.tables), dev)) for m, a in MODES.items()}
    pool = batches(dev, vocabs, B, "uniform")
    for s in range(max(args.warmup, 10)):
        eng.clip = clips[list(MODES)[s % len(MODES)]]
        eng.train_step_on_device(*pool[s % NB])
    torch.cuda.synchronize()
    recs = []
    for mode, c in clips.items():
        eng.clip = c
        n0 = launch_count()
        eng.train_step_on_device(*pool[0])
        torch.cuda.synchronize()
        rec = {"what": "launches_per_step", "mode": mode, "launches": launch_count() - n0, **info}
        print(json.dumps(rec), flush=True)
        recs.append(rec)
    for r in range(args.rounds):
        for mode, c in clips.items():
            eng.clip = c
            rec = {"what": "deepfm_step", "mode": mode, "round": r, "batch": B, "steps": args.steps,
                   "step_ms": round(time_steps(eng, pool, args.steps), 4), **info}
            print(json.dumps(rec), flush=True)
            recs.append(rec)
    for mode in ("clipvalue", "global_clipnorm"):
        eng.clip = clips[mode]
        phases = eng.profile_step(*pool[0])
        rec = {"what": "deepfm_step_phases", "mode": mode, "clip_ms": round(phases.get("clip", float("nan")), 4),
               "fm_bwd_ms": round(phases.get("fm_bwd", float("nan")), 4), **info}
        print(json.dumps(rec), flush=True)
        recs.append(rec)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in recs) + "\n")


if __name__ == "__main__":
    main()
