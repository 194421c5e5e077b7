"""Cost of Keras sample weights on the GPU: the bench-shape DeepFM step without weights, with sample weights, and with sample weights
plus a weighted AUC; and hrb_metric_update_weighted alone next to hrb_metric_update.

    python profiles/tools/sample_weight_step.py [--steps 30] [--warmup 10] [--rounds 3] [--out file.jsonl]

Step: the shapes of bench.py (26 tables, 102 M rows, D = 16, B = 65536, 429-256-128-1, Adam; tables up to 131072 rows
dense-updated), ONE engine; >= 10 warm-up steps (past the backward autotune trials in steps 3-6, every variant warmed), then
`--rounds` x (30 unweighted steps, 30 steps with per-sample weights, 30 steps with weights and a weighted AUC(200 thresholds))
timed with CUDA events over a rotating pool of 4 batches, alternating in this one process.  Kernel: hrb_metric_update and
hrb_metric_update_weighted over n = 65 536 and 10^7 samples with 200 and 8192 thresholds (an AUC's 4 variables per threshold), 200
back-to-back calls between two CUDA events after 20 warm-up calls, each issued straight through the bound C entry with prebuilt
arguments.  Prints one JSON line per measurement, each with the GPU name and power limit read by nvidia-smi in the same run.
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

from handyrec_b200 import _lib  # noqa: E402
from handyrec_b200 import kernels as K  # noqa: E402
from handyrec_b200.engine import DeepFMEngine  # noqa: E402
from handyrec_b200.metrics import AUC, MetricSet  # noqa: E402


def time_steps(eng, pool, weights, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        eng.train_step_on_device(*pool[s % NB], weights[s % NB] if weights is not None else None)
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
    eng = DeepFMEngine(tables, [(f, 1, "none") for f in range(len(vocabs))], bench.N_DENSE, bench.DNN_HIDDEN, "relu", batch_size=B,
                       optimizer="adam", lr=1e-3, dense_table_max_rows=131072)
    del tables
    pool = batches(dev, vocabs, B, "uniform")
    g = torch.Generator(device=dev).manual_seed(5)
    weights = [torch.rand(B, device=dev, generator=g) * 2 for _ in range(NB)]
    auc = AUC()
    wms = MetricSet([auc], weighted=[auc])
    variants = (("unweighted", None, None), ("sample_weight", weights, None), ("sample_weight_weighted_auc", weights, wms))
    for s in range(max(warmup, 10)):
        _, w, m = variants[s % 3]
        eng.metrics = m
        eng.train_step_on_device(*pool[s % NB], w[s % NB] if w is not None else None)
    torch.cuda.synchronize()
    out = []
    for r in range(rounds):
        for label, w, m in variants:
            eng.metrics = m
            rec = {"what": "deepfm_step", "variant": label, "round": r, "batch": B, "steps": steps,
                   "step_ms": round(time_steps(eng, pool, w, steps), 4), **info}
            print(json.dumps(rec), flush=True)
            out.append(rec)
    del eng, pool
    torch.cuda.empty_cache()
    return out


def kernel_cost(dev, info, reps=200):
    out = []
    g = torch.Generator(device=dev).manual_seed(3)
    for n in (65_536, 10_000_000):
        prob = torch.rand(n, device=dev, generator=g)
        label = (torch.rand(n, device=dev, generator=g) < 0.25).float()
        weight = torch.rand(n, device=dev, generator=g) * 2
        for T in (200, 8192):
            auc = AUC(num_thresholds=T)
            ms = MetricSet([auc], weighted=[auc])
            ms.update(prob, label, weight)  # allocates the set's buffers, both scratches
            ms.update(prob, label)
            b = ms._buffers()
            common = (K._p(b["thresholds"]), T)
            tail = (K._p(b["thr_index"]), len(ms.kinds), K._p(b["vars"]))
            calls = (("hrb_metric_update", _lib.lib().hrb_metric_update,
                      (K._p(prob), K._p(label), n, *common, K._p(b["kinds"]), *tail, K._p(b["scratch"]), K._p(b["flags"]), K._stream())),
                     ("hrb_metric_update_weighted", _lib.lib().hrb_metric_update_weighted,
                      (K._p(prob), K._p(label), K._p(weight), n, *common, K._p(b["weighted_kinds"]), *tail, K._p(b["wscratch"]),
                       K._p(b["flags"]), K._stream())))
            for name, fn, args in calls:
                for _ in range(20):
                    assert fn(*args) == 0
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn(*args)
                e1.record()
                torch.cuda.synchronize()
                us = e0.elapsed_time(e1) / reps * 1e3
                rec = {"what": name, "n": n, "thresholds": T, "variables": 4 * T, "us_per_call": round(us, 2), **info}
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
        raise SystemExit("sample_weight_step.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    recs = kernel_cost(dev, info) + step_cost(dev, args.steps, args.warmup, args.rounds, info)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in recs) + "\n")


if __name__ == "__main__":
    main()
