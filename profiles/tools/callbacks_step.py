"""Cost of Keras callbacks in `fit`: the Criteo-shape DeepFM fitted end to end with no callbacks, with the epoch-level set
[EarlyStopping, ModelCheckpoint(save_best_only=True), ReduceLROnPlateau, CSVLogger] and with TerminateOnNaN (a batch hook: one
host sync per step), alternating in one process.

    python profiles/tools/callbacks_step.py [--steps 30] [--rounds 6] [--out file.jsonl]

Model: bench.py's reference-shaped construction (26 tables, 102 M rows, D = 16, 429-256-128-1, Adam, tables up to 131072 rows
dense-updated), three copies built from the same seed.  Each model's engine takes 8 warm-up steps (past the backward autotune
trials in steps 3-6) and one warm-up fit with its callbacks.  Then `--rounds` x (one `fit(dict of 39 host arrays,
batch_size=65536)` of `--steps` batches per model, in an order that rotates from round to round), host clock around fit + a
device synchronise, as in bench.py's e2e figure; launches per step from `handyrec_b200.engine.launch_count()`.  The epoch-level callbacks monitor `loss` with patience far
beyond the run, so the rate is never cut and training never stops; ModelCheckpoint compares and skips (its best is set to a
value no loss beats), so no 6.5 GB table save falls inside a timed fit -- the timed work is the per-epoch callback logic.
Prints one JSON line per measurement with the GPU name, power limit and max SM clock read by nvidia-smi in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bench  # noqa: E402
from optimizer_step import NB, batches, gpu_info  # noqa: E402

from handyrec_b200 import callbacks as C  # noqa: E402
from handyrec_b200 import keras_lite as KL  # noqa: E402
from handyrec_b200.engine import launch_count  # noqa: E402


def _configs(tmp: str):
    mc = C.ModelCheckpoint(os.path.join(tmp, "ck"), monitor="loss", save_best_only=True, save_weights_only=True)
    mc.best = -np.inf  # mode "min": no loss is below -inf, so the callback compares and never writes
    return {
        "none": None,
        "epoch_level": [C.EarlyStopping(monitor="loss", patience=10**6), mc, C.ReduceLROnPlateau(monitor="loss", patience=10**6),
                        C.CSVLogger(os.path.join(tmp, "log.csv"), append=True)],
        "TerminateOnNaN": [C.TerminateOnNaN()],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("callbacks_step.py measures on a CUDA device; none is visible")
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
    with tempfile.TemporaryDirectory() as tmp:
        configs = _configs(tmp)
        models = {}
        for name, cbs in configs.items():
            torch.manual_seed(2022)
            m, _ = bench.build_deepfm_model(vocabs)
            m.dense_table_max_rows = 131072
            m.compile(optimizer=KL.Adam(learning_rate=1e-3), loss=KL.binary_crossentropy)
            m._fused.build(B, m.optimizer)
            eng = m._fused.engine
            for s in range(8):
                eng.train_step_on_device(*pool[s % NB])
            m.fit({k: v[: 3 * B] for k, v in x.items()}, y[: 3 * B], batch_size=B, callbacks=cbs)
            models[name] = m
        torch.cuda.synchronize()
        recs = []
        names = list(models)
        for r in range(args.rounds):
            for name in names[r % 3 :] + names[: r % 3]:  # the order rotates from round to round
                m = models[name]
                eng = m._fused.engine
                c0 = launch_count()
                t0 = time.perf_counter()
                h = m.fit(x, y, batch_size=B, callbacks=configs[name])
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                launches = launch_count() - c0
                assert m._fused.engine is eng and len(m.last_losses) == args.steps
                rec = {"what": "deepfm_fit", "callbacks": name, "round": r, "batch": B, "steps": args.steps,
                       "samples_per_s": round(n / dt), "ms_per_step": round(dt * 1e3 / args.steps, 4),
                       "launches_per_step": launches / args.steps, "loss": h.history["loss"][0], **info}
                print(json.dumps(rec), flush=True)
                recs.append(rec)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in recs) + "\n")


if __name__ == "__main__":
    main()
