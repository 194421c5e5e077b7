"""Cost of a Keras learning-rate schedule in `fit`: the Criteo-shape DeepFM fitted end to end with a float rate, an
ExponentialDecay and a CosineDecayRestarts, alternating in one process.

    python profiles/tools/lr_schedule_step.py [--steps 30] [--rounds 3] [--out file.jsonl]

Model: bench.py's reference-shaped construction (26 tables, 102 M rows, D = 16, 429-256-128-1, tables up to 131072 rows
dense-updated), three copies built from the same seed, each compiled with Adam at one of the three rates.  Each model's engine
takes 8 warm-up steps (past the backward autotune trials in steps 3-6) and one warm-up fit.  Then `--rounds` x (one
`fit(dict of 39 host arrays, batch_size=65536)` of `--steps` batches per model), host clock around fit + a device synchronise:
host packing, H2D copies and the loss read-back are inside the timed region, as in bench.py's e2e figure.  Prints one JSON line
per measurement with the GPU name, power limit and max SM clock read by nvidia-smi in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bench  # noqa: E402
from optimizer_step import NB, batches, gpu_info  # noqa: E402

from handyrec_b200 import keras_lite as KL  # noqa: E402
from handyrec_b200.schedules import CosineDecayRestarts, ExponentialDecay  # noqa: E402

RATES = {"float": lambda: 1e-3, "ExponentialDecay": lambda: ExponentialDecay(1e-3, 1000, 0.96),
         "CosineDecayRestarts": lambda: CosineDecayRestarts(1e-3, 100, t_mul=2.0, m_mul=0.9, alpha=0.01)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lr_schedule_step.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    B, vocabs = bench.BATCH, bench.CRITEO_VOCABS
    pool = batches(dev, vocabs, B, "uniform")
    n = args.steps * B
    reps = (args.steps + NB - 1) // NB
    ids = np.concatenate([p[0].cpu().numpy() for p in pool] * reps)[:n]
    dense = np.concatenate([p[1].cpu().numpy() for p in pool] * reps)[:n]
    y = np.concatenate([p[2].cpu().numpy() for p in pool] * reps)[:n]
    x = {f"C{f + 1}": np.ascontiguousarray(ids[:, f : f + 1]) for f in range(len(vocabs))}
    x.update({f"I{j + 1}": np.ascontiguousarray(dense[:, j : j + 1]) for j in range(bench.N_DENSE)})
    models = {}
    for name, rate in RATES.items():
        torch.manual_seed(2022)
        m, _ = bench.build_deepfm_model(vocabs)
        m.dense_table_max_rows = 131072
        m.compile(optimizer=KL.Adam(learning_rate=rate()), loss=KL.binary_crossentropy)
        m._fused.build(B, m.optimizer)
        eng = m._fused.engine
        for s in range(8):
            eng.train_step_on_device(*pool[s % NB])
        m.fit({k: v[: 3 * B] for k, v in x.items()}, y[: 3 * B], batch_size=B)
        models[name] = m
    torch.cuda.synchronize()
    recs = []
    for r in range(args.rounds):
        for name, m in models.items():
            t0 = time.perf_counter()
            m.fit(x, y, batch_size=B)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            eng = m._fused.engine
            rec = {"what": "deepfm_fit", "rate": name, "round": r, "batch": B, "steps": args.steps, "samples_per_s": round(n / dt),
                   "ms_per_step": round(dt * 1e3 / args.steps, 4), "iterations": m.optimizer.iterations, "last_lr": eng.lr, **info}
            print(json.dumps(rec), flush=True)
            recs.append(rec)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in recs) + "\n")


if __name__ == "__main__":
    main()
