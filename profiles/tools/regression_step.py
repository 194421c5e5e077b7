"""Cost of the regression head on the GPU: the bench-shape DeepFM step with the sigmoid / BCE head next to the same step with the
linear head and mean_squared_error, and the two head kernels alone.

    python profiles/tools/regression_step.py [--steps 30] [--warmup 10] [--rounds 3] [--out file.jsonl]

Step: the shapes of bench.py (26 tables, 102 M rows, D = 16, B = 65536, 429-256-128-1, Adam; tables up to 131072 rows
dense-updated), two engines over the same large tables (task="binary" and task="regression", loss="mean_squared_error"); >= 10
warm-up steps each (past the backward autotune trials in steps 3-6), then `--rounds` x (30 binary steps, 30 regression steps) timed
with CUDA events over a rotating pool of 4 batches, alternating in this one process.  Kernel: hrb_sigmoid_bce and
hrb_regression_loss (MSE) at B = 65536, 200 back-to-back calls between two CUDA events after 20 warm-up calls.  Prints one JSON line
per measurement, each with the GPU name and power limit read by nvidia-smi in the same run.
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
from handyrec_b200._lib import call  # noqa: E402
from handyrec_b200.engine import DeepFMEngine, launch_count  # noqa: E402


def time_steps(eng, pool, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        eng.train_step_on_device(*pool[s % NB])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def step_cost(dev, steps, warmup, rounds, info):
    vocabs, D, B = bench.CRITEO_VOCABS, bench.EMB_DIM, bench.BATCH
    tables = []
    for f, v in enumerate(vocabs):
        t = torch.empty(v, D, device=dev)
        K.init_uniform(t, seed=7 + f)
        tables.append(t)
    fields = [(f, 1, "none") for f in range(len(vocabs))]
    common = dict(batch_size=B, optimizer="adam", lr=1e-3, dense_table_max_rows=131072)
    engines = {"binary_bce": DeepFMEngine(tables, fields, bench.N_DENSE, bench.DNN_HIDDEN, "relu", **common),
               "regression_mse": DeepFMEngine(tables, fields, bench.N_DENSE, bench.DNN_HIDDEN, "relu", task="regression",
                                              loss="mean_squared_error", **common)}
    del tables
    pool = batches(dev, vocabs, B, "uniform")
    launches = {}
    for name, eng in engines.items():
        for s in range(max(warmup, 10)):
            eng.train_step_on_device(*pool[s % NB])
        torch.cuda.synchronize()
        c0 = launch_count()
        eng.train_step_on_device(*pool[0])
        torch.cuda.synchronize()
        launches[name] = launch_count() - c0
    out = []
    for r in range(rounds):
        for name, eng in engines.items():
            ms = time_steps(eng, pool, steps)
            rec = {"what": "deepfm_step", "variant": name, "round": r, "batch": B, "steps": steps, "step_ms": round(ms, 4),
                   "samples_per_s_M": round(B / ms / 1e3, 2), "launches_per_step": launches[name], **info}
            print(json.dumps(rec), flush=True)
            out.append(rec)
    del engines, pool
    torch.cuda.empty_cache()
    return out


def kernel_cost(dev, info, reps=200):
    B = bench.BATCH
    g = torch.Generator(device=dev).manual_seed(3)
    dnn, fm = torch.randn(B, device=dev, generator=g), torch.randn(B, device=dev, generator=g)
    label = torch.randn(B, device=dev, generator=g)
    prob, dlogit, ls = torch.empty(B, device=dev), torch.empty(B, device=dev), torch.zeros(1, device=dev)
    ws = K.regression_loss_workspace(B, dev)
    calls = (("hrb_sigmoid_bce", lambda: call("hrb_sigmoid_bce", K._p(dnn), K._p(fm), K._p(label), B, 1.0 / B, K._p(prob), K._p(dlogit),
                                                  K._p(ls), K._stream())),
             ("hrb_regression_loss", lambda: K.regression_loss("mean_squared_error", 1.0, dnn, fm, label, B, 1, 1.0 / B, prob, dlogit, ls,
                                                               workspace=ws)))
    out = []
    for name, fn in calls:
        for _ in range(20):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        rec = {"what": name, "batch": B, "us_per_call": round(e0.elapsed_time(e1) / reps * 1e3, 2), **info}
        print(json.dumps(rec), flush=True)
        out.append(rec)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("regression_step.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    recs = kernel_cost(dev, info) + step_cost(dev, args.steps, args.warmup, args.rounds, info)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in recs) + "\n")


if __name__ == "__main__":
    main()
