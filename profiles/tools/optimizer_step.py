"""One-GPU step time of the Criteo-shape DeepFM engine under Adam, Adagrad, Ftrl and SGD, uniform and Zipf ids.

    python profiles/tools/optimizer_step.py [--steps 30] [--warmup 10] [--rounds 2]

The shapes come from bench.py (26 tables, 102 M rows, D = 16, B = 65536, 429-256-128-1; tables up to 131072 rows dense-updated).
For every (optimiser, ids) pair: >= 10 warm-up steps (past the engine's backward autotune trials in steps 3-6), 30 steps timed with
CUDA events over a rotating pool of 4 batches (6.5 GB of tables >> the 126 MB L2), then one profile_step phase breakdown.  The
optimisers alternate, `--rounds` times, in this one process; each engine is freed before the next is built.  Prints one JSON line
per measurement, each with the GPU name and power limit read by nvidia-smi in the same run.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from handyrec_b200 import kernels as K  # noqa: E402
from handyrec_b200.engine import DeepFMEngine  # noqa: E402

NB = 4


def gpu_info():
    idx = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]
    q = subprocess.run(["nvidia-smi", "-i", idx, "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, sm = [s.strip() for s in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "sm_max_clock": sm}


def batches(dev, vocabs, B, ids, seed=1234):
    g = torch.Generator(device=dev).manual_seed(seed)
    out = []
    for _ in range(NB):
        cols = []
        for v in vocabs:
            if ids == "uniform":
                cols.append(torch.randint(0, v, (B,), device=dev, generator=g, dtype=torch.int64))
            else:  # Zipf(1.05) over [1, V), as bench.py --ids zipf
                u = torch.rand(B, device=dev, generator=g, dtype=torch.float64)
                a = 1.05
                cols.append((((v ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))).long().clamp_(1, v - 1))
        out.append((torch.stack(cols, 1).to(torch.int32).contiguous(),
                    torch.log1p(torch.empty(B, bench.N_DENSE, device=dev).exponential_(1.0, generator=g)),
                    (torch.rand(B, device=dev, generator=g) < 0.25).float()))
    return out


def measure(dev, opt, ids, steps, warmup):
    vocabs, D, B = bench.CRITEO_VOCABS, bench.EMB_DIM, bench.BATCH
    tables = []
    for f, v in enumerate(vocabs):
        t = torch.empty(v, D, device=dev)
        K.init_uniform(t, seed=7 + f)
        tables.append(t)
    eng = DeepFMEngine(tables, [(f, 1, "none") for f in range(len(vocabs))], bench.N_DENSE, bench.DNN_HIDDEN, "relu", batch_size=B,
                       optimizer=opt, lr=1e-3, dense_table_max_rows=131072)
    del tables
    pool = batches(dev, vocabs, B, ids)
    for s in range(max(warmup, 10)):
        eng.train_step_on_device(*pool[s % NB])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        eng.train_step_on_device(*pool[s % NB])
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    phases = eng.profile_step(*pool[0])
    rec = {"optimizer": opt, "ids": ids, "batch": B, "steps": steps, "step_ms": round(step_ms, 4),
           "samples_per_s": round(B / step_ms * 1e3), "embedding_bwd_ms": round(phases.get("embedding_bwd_update", float("nan")), 4),
           "dense_optimizer_ms": round(phases.get("dense_optimizer", float("nan")), 4), "bwd_algo": eng.bwd_algo,
           "bwd_algo_trial_ms": getattr(eng, "bwd_algo_ms", None), "profile_step_ms": {k: round(v, 4) for k, v in phases.items()}}
    del eng, pool
    gc.collect()
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("optimizer_step.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    lines = []
    for rnd in range(args.rounds):
        for ids in ("uniform", "zipf"):
            for opt in ("adam", "adagrad", "ftrl", "sgd"):
                rec = dict(measure(dev, opt, ids, args.steps, args.warmup), round=rnd, **info)
                line = json.dumps(rec)
                print(line, flush=True)
                lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
