"""Cost of Keras metrics on the GPU: the Criteo-shape DeepFM step with and without metrics=["AUC"], and hrb_metric_update alone.

    python profiles/tools/metrics_step.py [--steps 30] [--warmup 10] [--rounds 3] [--out file.jsonl]

Step: the shapes of bench.py (26 tables, 102 M rows, D = 16, B = 65536, 429-256-128-1, Adam; tables up to 131072 rows
dense-updated), ONE engine; >= 10 warm-up steps (past the backward autotune trials in steps 3-6), then `--rounds` x (30 steps
without metrics, 30 steps with an AUC(200 thresholds) MetricSet attached) timed with CUDA events over a rotating pool of 4
batches, alternating in this one process.  Kernel: hrb_metric_update over n = 65 536 and 10^7 samples with 200 and 8192
thresholds (an AUC's 4 variables per threshold), 200 back-to-back launches between two CUDA events after 20 warm-up launches, each
issued straight through the bound C entry with prebuilt arguments (MetricSet.update's Python checks would make the host the
bound of such a loop);
reported as time per launch and as bytes/s against the 8 bytes per sample the kernel must read (prob + label).  Prints one JSON
line per measurement, each with the GPU name and power limit read by nvidia-smi in the same run.
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
    eng = DeepFMEngine(tables, [(f, 1, "none") for f in range(len(vocabs))], bench.N_DENSE, bench.DNN_HIDDEN, "relu", batch_size=B,
                       optimizer="adam", lr=1e-3, dense_table_max_rows=131072)
    del tables
    pool = batches(dev, vocabs, B, "uniform")
    ms = MetricSet([AUC()])
    for s in range(max(warmup, 10)):
        eng.metrics = ms if s % 2 else None
        eng.train_step_on_device(*pool[s % NB])
    torch.cuda.synchronize()
    out = []
    for r in range(rounds):
        for label, m in (("without_metrics", None), ("with_auc", ms)):
            eng.metrics = m
            rec = {"what": "deepfm_step", "metrics": label, "round": r, "batch": B, "steps": steps,
                   "step_ms": round(time_steps(eng, pool, steps), 4), **info}
            print(json.dumps(rec), flush=True)
            out.append(rec)
    eng.metrics = ms
    phases = eng.profile_step(*pool[0])
    rec = {"what": "deepfm_step_phases", "metrics": "with_auc", "metric_update_ms": round(phases.get("metric_update", float("nan")), 4),
           "profile_step_ms": {k: round(v, 4) for k, v in phases.items()}, **info}
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
        for T in (200, 8192):
            ms = MetricSet([AUC(num_thresholds=T)])
            ms.update(prob, label)  # allocates the set's buffers
            b = ms._buffers()
            fn = _lib.lib().hrb_metric_update
            args = (K._p(prob), K._p(label), n, K._p(b["thresholds"]), T, K._p(b["kinds"]), K._p(b["thr_index"]), len(ms.kinds),
                    K._p(b["vars"]), K._p(b["scratch"]), K._p(b["flags"]), K._stream())
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
            rec = {"what": "hrb_metric_update", "n": n, "thresholds": T, "variables": 4 * T, "us_per_launch": round(us, 2),
                   "bytes_per_s": round(8 * n / (us * 1e-6)), "l2_resident": 8 * n < 126e6, **info}
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
        raise SystemExit("metrics_step.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    recs = kernel_cost(dev, info) + step_cost(dev, args.steps, args.warmup, args.rounds, info)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in recs) + "\n")


if __name__ == "__main__":
    main()
