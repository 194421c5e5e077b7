#!/usr/bin/env python
"""bench.py -- HandyRec hot path on B200: train samples/s on synthetic data of the shapes BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W                 # DeepFM Criteo-shape (configs[2]), this repo's CUDA path
    python bench.py --workload din | retrieval                    # configs[1] (DIN, MovieLens-shaped) / configs[4] (YouTubeDNN, 10 M items)
    python bench.py --impl reference --steps K --warmup W         # the reference restated on CPU (oracle), same workload
    python -m torch.distributed.run ... bench.py --gpus N --verify   # N>1: correctness of the sharded step against a 1-GPU engine
    python bench.py --steps K --warmup W --dump-outputs DIR       # also write the last timed step's outputs as DIR/<name>.npy

One "step" = one full training step on one batch of synthetic samples.  Prints ONE JSON line (contract in the task statement):
`value` = device-resident throughput (CUDA events), `e2e` = through the reference-shaped API -- `handyrec_b200.models.<Model>(...)
.compile(...).fit(dict of host arrays)` -- with host batches packed, copied to the device and the loss read back inside the timed
region, `roofline` for the dominant kernel, `roofline_lookup` / `roofline_embedding_bwd` for the north-star kernels, `cpu_baseline`.
Nothing here reads /root/reference.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Criteo-like vocabulary vector (SURVEY.md 8d), +1 so that id 0 exists everywhere
CRITEO_VOCABS = [40_000_000, 40_000_000, 10_000_000, 5_000_000, 3_000_000, 2_000_000, 1_000_000, 500_000, 300_000, 100_000,
                 50_000, 20_000, 12_000, 10_000, 7_000, 5_000, 2_000, 1_500, 1_000, 600, 300, 100, 30, 20, 10, 4]
CRITEO_VOCABS = [v + 1 for v in CRITEO_VOCABS]
N_DENSE, EMB_DIM, BATCH = 13, 16, 65536
DNN_HIDDEN = (256, 128, 1)
LOOKUP_BYTES_PER_SAMPLE = len(CRITEO_VOCABS) * (4 + EMB_DIM * 4 + EMB_DIM * 4)  # ids + rows + output = 3432 (SURVEY 8d)
CPU_VOCAB_CAP = 2_000_000  # rows per table on the CPU arm (dense Keras Adam over all 102 M rows would take minutes per step)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]), "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def load_traffic(kernel_key: str):
    """DRAM bytes per launch of a kernel as parsed from this round's `ncu --set full` capture (profiles/summarize.py writes
    profiles/r02_ncu_full.json); None when no capture is committed -- never a hand-typed number."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_full.json")
    if not os.path.exists(p):
        return None, None
    rows = [r for r in json.load(open(p)).get("kernels", []) if kernel_key in r.get("name", "")]
    if not rows:
        return None, None
    tot = sum(r["dram_read_bytes"] + r["dram_write_bytes"] for r in rows) / len(rows)
    return tot, f"mean dram read+write per launch over {len(rows)} launches of {kernel_key} in profiles/r02_ncu_full.json"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms; samples count from mark() (start of the timed steps) to stop()."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        """index: one GPU index or a list of them (rank 0 of a multi-GPU run samples every GPU of the job from ONE nvidia-smi process:
        eight of them starting up beside the timed region -- NVML initialisation walks all GPUs -- perturbed the launches)."""
        self.index = ",".join(str(i) for i in index) if isinstance(index, (list, tuple, range)) else str(index)
        self.proc, self.lines, self.first = None, [], 0

    def mark(self):
        """Samples from here on count (call at the start of the timed region; the process was started earlier)."""
        self.first = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.index, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines[self.first:]:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "gpus": self.index,
                "window": "from the start of the timed steps to the end of the end-to-end runs (GPU under load throughout)"}


# -------------------------------------------------------------------------------------------------
# CPU restatement of one training step (oracle) -- used by cpu_baseline and by --impl reference
# -------------------------------------------------------------------------------------------------
def cpu_deepfm_arm(batch: int, vocab_cap: int, steps: int, warmup: int, seed: int = 1234):
    """Time the op-for-op CPU restatement (oracle/) of the same DeepFM step: 26 tables D=16, 13 dense, DNN [429,256,128,1], FM,
    BCE, dense Adam on every table like Keras; embeddings looked up once per feature group exactly like the reference
    (DeepFM.py:62-63).  Vocabularies are capped at `vocab_cap` rows so that the dense Adam state fits and a step stays bounded."""
    import torch

    import oracle

    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(seed)
    vocabs = [min(v, vocab_cap) for v in CRITEO_VOCABS]
    tables = [((torch.rand(v, EMB_DIM, generator=g) - 0.5) * 0.1).requires_grad_(True) for v in vocabs]
    p = oracle.dnn_init(N_DENSE + len(vocabs) * EMB_DIM, DNN_HIDDEN, seed=seed)
    for t in p.W + p.b:
        t.requires_grad_(True)
    fm_w = (torch.rand(EMB_DIM, 1, generator=g) - 0.5).requires_grad_(True)
    fm_w0 = torch.zeros(1, requires_grad=True)
    params = tables + p.W + p.b + [fm_w, fm_w0]
    opt = torch.optim.Adam(params, lr=1e-3, eps=1e-7)
    ids = torch.stack([torch.randint(0, v, (batch,), generator=g) for v in vocabs], 1)
    dense = torch.log1p(torch.empty(batch, N_DENSE).exponential_(1.0, generator=g))
    label = (torch.rand(batch, generator=g) < 0.25).float()
    from collections import OrderedDict

    def step():
        opt.zero_grad(set_to_none=True)
        sparse = OrderedDict((f"C{f}", (tables[f], ids[:, f : f + 1], False)) for f in range(len(vocabs)))
        fm_embds = oracle.group_embedding_lookup(sparse, OrderedDict(), "mean")   # fm_feature_group.embedding_lookup
        dnn_embds = oracle.group_embedding_lookup(sparse, OrderedDict(), "mean")  # dnn_feature_group.embedding_lookup
        logit = oracle.deepfm_forward([dense], fm_embds, dnn_embds, p, fm_w, fm_w0, return_logit=True)
        loss = oracle.bce_from_logits(logit[:, 0], label)
        loss.backward()
        opt.step()
        return float(loss.detach())

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"samples_per_s": batch * steps / dt, "ms_per_step": dt / steps * 1e3, "cores": torch.get_num_threads(),
            "sample": f"{steps} steps of batch {batch}, every vocabulary capped at {vocab_cap} rows (dense Keras-style Adam over all rows of all tables), "
                      "torch-CPU op-for-op restatement of the reference layers (TensorFlow is not in the image)"}


WORKLOADS = {
    "deepfm": f"DeepFM Criteo-shape: 26 sparse + 13 dense, emb dim 16, DNN 429-256-128-1, batch 65536/GPU (BASELINE.json configs[2]); the CPU arm caps every vocabulary at {CPU_VOCAB_CAP} rows",
    "din": "DIN MovieLens-1M-shaped: history seq len 50, emb dim 32, batch 4096, LAU (32,1) dice, DNN (64,32,1) dice (BASELINE.json configs[1])",
    "retrieval": "YouTubeMatchDNN retrieval: 10 M-item catalogue, history L=50 mean-pooled, emb dim 32, genres L=6 D=8, batch 4096, 100 sampled (BASELINE.json configs[4])",
}
METRICS = {"deepfm": "DeepFM train samples/s", "din": "DIN train samples/s", "retrieval": "YouTubeMatchDNN train samples/s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "deepfm":
        r = cpu_deepfm_arm(batch=args.batch or BATCH, vocab_cap=CPU_VOCAB_CAP, steps=args.steps, warmup=args.warmup)
        gb = args.batch or BATCH
    else:
        import bench_models

        r = bench_models.cpu_arm(args.workload, steps=args.steps, warmup=args.warmup)
        gb = r["batch"]
    line = {
        "impl": "reference", "metric": METRICS[args.workload], "value": r["samples_per_s"], "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload], "global_batch": gb,
                   "reference_sample": "CPU restatement of the reference (oracle/) on a bounded sample of the workload: " + r["sample"]},
        "cpu_baseline": {"value": r["samples_per_s"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["samples_per_s"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------
def build_deepfm_model(vocabs):
    """The reference-shaped construction: feature definitions -> feature groups -> DeepFM(...) -> compile (DeepFM.py / README)."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
    from handyrec_b200.models import DeepFM

    sparse = [SparseFeature(f"C{i + 1}", v, EMB_DIM) for i, v in enumerate(vocabs)]
    dense = [DenseFeature(f"I{i + 1}") for i in range(N_DENSE)]
    pool = FeaturePool()
    fm_group = FeatureGroup("fm", sparse, pool, l2_embd=0.0)
    dnn_group = FeatureGroup("dnn", dense + sparse, pool, l2_embd=0.0)
    model = DeepFM(fm_group, dnn_group, dnn_hidden_units=DNN_HIDDEN, dnn_activation="relu")
    return model, KL


def deepfm_outputs(eng, ids):
    """What a caller of `train_step_on_device(ids, ...)` holds after the step: the mean loss and the click probabilities of the
    batch, the DNN and FM weights after the update, and, per field, the table rows of a fixed sample of the batch's ids after the
    update (the tables hold 6.5 GB)."""
    import torch

    import bench_models

    B = ids.shape[0]
    pos = torch.from_numpy(bench_models.sample_rows(B)).to(ids.device)
    out = {"loss": eng.loss_sum.double().cpu() / B, "prob": eng.prob[:B].cpu(), "fm_w": eng.fm_w.cpu(), "fm_w0": eng.fm_w0.cpu()}
    for i in range(len(eng.units)):
        out[f"dnn_W{i}"], out[f"dnn_b{i}"] = eng.get_dense_weights(i)
    out["table_rows"] = torch.stack([eng.tables[t][ids[pos, col].long()] for t, _, _, col, _ in eng.plan_fields]).cpu()
    return {k: v.numpy() for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="deepfm", choices=list(WORKLOADS))
    ap.add_argument("--optimizer", default="adam", choices=["adam", "sgd"])
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"])
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-peer-lookup", action="store_true", help="N>1: forward through the all-to-all row exchange instead of NVLink peer loads")
    ap.add_argument("--no-p2p-grads", action="store_true", help="N>1: move gradient rows with NCCL all-to-alls instead of the fused gather + NVLink store kernel")
    ap.add_argument("--small-table-rows", type=int, default=131072,
                    help="tables up to this many rows take the dense (Keras-exact) optimiser step; at N>1 they are replicated instead of sharded (0 = off)")
    ap.add_argument("--large-table-rows", type=int, default=0, help="C4: give every table above --small-table-rows this many rows (e.g. 100000000 at --gpus 8)")
    ap.add_argument("--scale-vocab", type=float, default=1.0, help="shrink every vocabulary (debug only; reported in config)")
    ap.add_argument("--bwd-algo", default="auto", choices=["auto", "units", "sort"],
                    help="embedding backward: auto = the engine times both implementations in its first steps and keeps the faster one; "
                         "units / sort pin one (profiling under ncu distorts the trial timings)")
    ap.add_argument("--verify", action="store_true", help="N>1: 3 sharded steps at a small batch compared with a single-GPU engine on the concatenated batch")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="one GPU: after the timed steps, write what the last of them computed as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB; large embedding tables as a fixed sample of rows), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.verify or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the outputs of the CUDA path's timed steps on one GPU (--impl ours, no --verify, one process)")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload != "deepfm":
        import bench_models

        return bench_models.run(args, load_peaks, ClockSampler, WORKLOADS, METRICS)

    import torch

    from handyrec_b200 import kernels as K
    from handyrec_b200.engine import launch_count

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    if args.verify:
        import bench_models

        return bench_models.verify_sharded(args, CRITEO_VOCABS, N_DENSE, EMB_DIM)
    peaks = load_peaks()
    # ONE nvidia-smi process (rank 0) samples every GPU of the job; it is started here, seconds before the timed region, so that its
    # start-up (NVML walks all GPUs) is over when the timing begins -- samples count from ClockSampler.mark() on
    vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
    gpu_ids = vis[:world] if len(vis) >= world else list(range(world))  # nvidia-smi counts physical GPUs: follow CUDA_VISIBLE_DEVICES if it is set
    clocks = ClockSampler(gpu_ids) if rank == 0 else None
    if clocks is not None:
        clocks.start()

    # ---- workload -------------------------------------------------------------------------------
    B = args.batch or BATCH
    vocabs = [max(4, int(v * args.scale_vocab)) for v in CRITEO_VOCABS]
    if args.large_table_rows:
        vocabs = [args.large_table_rows if v > args.small_table_rows else v for v in vocabs]
    fields = [(f, 1, "none") for f in range(len(vocabs))]
    # the reference-shaped call chain: feature groups -> DeepFM(...) -> compile; compile() lowers the graph onto the fused engine.
    # N > 1: the same calls inside `ShardedTables()` -- tables above --small-table-rows are CREATED row-sharded (this rank allocates
    # rows r % N == rank only, in symmetric memory that peers read over NVLink), the rest replicated; every rank fits its own data
    import contextlib

    from handyrec_b200 import keras_lite as KL_

    torch.manual_seed(2022)
    with (KL_.ShardedTables(min_rows=args.small_table_rows) if world > 1 else contextlib.nullcontext()):
        model, KL = build_deepfm_model(vocabs)
        model.dense_table_max_rows = args.small_table_rows
        model.peer_lookup = not args.no_peer_lookup
        model.p2p_grad_exchange = not args.no_p2p_grads
        model.compile(optimizer=KL.Adam(learning_rate=1e-3) if args.optimizer == "adam" else KL.SGD(learning_rate=1e-3), loss=KL.binary_crossentropy)
    assert model._fused is not None, "the DeepFM graph was not lowered onto the fused engine"
    model._fused.build(B, model.optimizer)
    eng = model._fused.engine
    if args.bwd_algo != "auto":
        from handyrec_b200 import _lib
        from handyrec_b200._lib import call

        eng.autotune_embedding_bwd = False
        eng.bwd_algo = args.bwd_algo
        for pl in [eng.plan] + [p for p in (getattr(eng, "plan_rep", None),) if p is not None]:
            call("hrb_plan_set_bwd_algo", pl._h, _lib.BWD_UNITS if args.bwd_algo == "units" else _lib.BWD_SORT)
    NB = 4  # rotating pool of distinct batches (tables are 6.5 GB >> 126 MB L2: every step touches fresh rows)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    ids_pool, dense_pool, label_pool = [], [], []
    for _ in range(NB):
        cols = []
        for v in vocabs:
            if args.ids == "uniform":
                cols.append(torch.randint(0, v, (B,), device=dev, generator=g, dtype=torch.int64))
            else:  # Zipf(1.05) over [1, V): inverse-CDF of the continuous approximation
                u = torch.rand(B, device=dev, generator=g, dtype=torch.float64)
                a = 1.05
                x = ((v ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))
                cols.append(x.long().clamp_(1, v - 1))
        ids_pool.append(torch.stack(cols, 1).to(torch.int32).contiguous())
        dense_pool.append(torch.log1p(torch.empty(B, N_DENSE, device=dev).exponential_(1.0, generator=g)))
        label_pool.append((torch.rand(B, device=dev, generator=g) < 0.25).float())
    host = [(i.cpu().pin_memory(), d.cpu().pin_memory(), l.cpu().pin_memory()) for i, d, l in zip(ids_pool, dense_pool, label_pool)]

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timed region -----------------------------------------------------------
    for s in range(max(args.warmup, 8 if eng.autotune_embedding_bwd else 0)):  # the engine picks its backward algorithm in steps 3-6
        eng.train_step_on_device(ids_pool[s % NB], dense_pool[s % NB], label_pool[s % NB])
    barrier()
    l0 = launch_count()
    if clocks is not None:
        clocks.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for s in range(args.steps):
        eng.train_step_on_device(ids_pool[s % NB], dense_pool[s % NB], label_pool[s % NB])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = launch_count() - l0
    if args.dump_outputs:
        import bench_models

        bench_models.write_outputs(args.dump_outputs, deepfm_outputs(eng, ids_pool[(args.steps - 1) % NB]))

    # ---- end-to-end through the reference-shaped API ----------------------------------------------
    if True:
        # (a) Model.fit on a dict of per-feature host arrays (what Keras takes): steps x B samples; per step the host packs the
        # batch (hrb_host_pack_*, background thread), copies it to the device on a copy stream and reads the loss back
        import numpy as np

        n_fit = args.steps * B
        x_host, reps = {}, (args.steps + NB - 1) // NB
        ids_np = np.concatenate([h[0].numpy() for h in host] * reps)[:n_fit]
        dense_np = np.concatenate([h[1].numpy() for h in host] * reps)[:n_fit]
        y_host = np.concatenate([h[2].numpy() for h in host] * reps)[:n_fit]
        for f in range(len(vocabs)):
            x_host[f"C{f + 1}"] = np.ascontiguousarray(ids_np[:, f : f + 1])
        for j in range(N_DENSE):
            x_host[f"I{j + 1}"] = np.ascontiguousarray(dense_np[:, j : j + 1])
        small = {k: v[: 3 * B] for k, v in x_host.items()}
        model.fit(small, y_host[: 3 * B], batch_size=B, epochs=1)  # warm-up of the fit path (pinned slots, copy stream)
        barrier()
        t0 = time.perf_counter()
        hist = model.fit(x_host, y_host, batch_size=B, epochs=1)
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        loss = float(model.last_losses[-1])
        e2e_api = "handyrec_b200.models.DeepFM(...).compile(Adam, binary_crossentropy).fit(dict of 39 per-feature host arrays, batch_size=65536): host packing, H2D and loss D2H every step inside the timed region"
        # (b) one blocking train_on_batch call per step through the same Model, for comparison
        xb = {k: v[:B] for k, v in x_host.items()}
        model.train_on_batch(xb, y_host[:B])
        barrier()
        t0 = time.perf_counter()
        for s in range(args.steps):
            model.train_on_batch(xb, y_host[:B])
        torch.cuda.synchronize()
        e2e_sync_ms = (time.perf_counter() - t0) * 1e3
    clk = clocks.stop() if clocks is not None else None

    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([ms, e2e_ms, e2e_sync_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, e2e_sync_ms = float(t[0]), float(t[1]), float(t[2])

    # ---- per-kernel timing (CUDA events on the launching stream, same steps) ----------------------
    phases = {}
    reps = max(5, min(args.steps, 20))
    for s in range(reps):
        for k, v in eng.profile_step(ids_pool[s % NB], dense_pool[s % NB], label_pool[s % NB]).items():
            phases[k] = phases.get(k, 0.0) + v / reps
    # lookup kernel alone, back to back (burst), for the roofline of the north-star kernel
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for s in range(reps):
        if world == 1 or eng.peer_lookup:
            eng.plan.forward(ids_pool[s % NB], out=eng.X0, fm=(eng.fm_w, eng.fm_w0), want_fm_sum=False)
        else:
            eng.exchange.forward(ids_pool[s % NB], eng.X0)
    b.record()
    torch.cuda.synchronize()
    lookup_alone_ms = a.elapsed_time(b) / reps

    timeline = None
    if world > 1:  # completion time of every phase of a production step (side streams running), ms since the step started
        barrier()
        timeline = eng.timeline_step(ids_pool[0], dense_pool[0], label_pool[0])
        barrier()
    if rank != 0:
        return
    step_ms = ms / args.steps
    total_phase = sum(phases.values())
    flops = {}
    units = eng.units
    Ks = [eng.K0] + units[:-1]
    for i, (kk, n) in enumerate(zip(Ks, units)):
        f = 2.0 * B * kk * n
        flops[f"dense_fwd_{i}"] = f
        flops[f"dense_bwd_w_{i}"] = f
        flops[f"dense_bwd_x_{i}"] = f
    lookup_bytes = LOOKUP_BYTES_PER_SAMPLE * B

    # dominant kernel = the tcgen05 GEMM kernel (one kernel, 9 launches per step: 3 fwd, 3 bwd_x, 3 split-K bwd_w)
    gemm_names = [k for k in phases if k in flops and not k.endswith("_3")]
    gemm_ms = sum(phases[k] for k in gemm_names)
    gemm_flops = sum(flops[k] for k in gemm_names)
    ach = gemm_flops / (gemm_ms * 1e-3) / 1e12
    full_batch = B == BATCH and args.scale_vocab == 1.0
    g_traffic, g_note = load_traffic("gemm_tc_kernel") if full_batch else (None, None)
    roofline = {"kernel": "tc::gemm_tc_kernel (tcgen05 3xTF32, %d launches/step; bwd_w phases include their split-reduce kernels)" % len(gemm_names),
                "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops_sustained"],
                "traffic": g_traffic, "traffic_note": g_note,
                "share_of_step": gemm_ms / total_phase, "flops_per_step": gemm_flops,
                "peak_source": f"{peaks['source']} bf16 sustained (kernel timed inside a long step)",
                "note": "fp32 parity needs 3 TF32 MMAs per product at half the bf16 rate: ceiling of this scheme = 1/6 = 0.167 of the bf16 peak (DESIGN.md 3)"}
    lk = "lookup_fm_fwd" if (world == 1 or eng.peer_lookup) else "sharded_lookup_fwd"
    lk_ach = lookup_bytes / (phases[lk] * 1e-3) / 1e9
    peer = world > 1 and eng.peer_lookup
    n_small = sum(1 for v in vocabs if v <= args.small_table_rows)
    n_sharded = len(vocabs) - n_small
    l_traffic, l_note = load_traffic("lookup_tile_kernel") if (full_batch and world == 1) else (None, None)
    rl_lookup = {"kernel": "hrb::lookup_tile_kernel (fused lookup + FM)" if world == 1 else
                 ("hrb::lookup_tile_kernel reading row-sharded tables over NVLink peer mappings" if peer else "row exchange (route + all-to-all + gather + scatter)"),
                 "bound": "hbm", "achieved": lk_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": lk_ach / peaks["hbm_gbs"],
                 "traffic": l_traffic, "traffic_note": l_note,
                 "nvlink_bytes_per_step_algorithmic": None if world == 1 else B * n_sharded * EMB_DIM * 4 * (world - 1) / world,
                 "peak_source": f"{peaks['source']} copy bandwidth", "bytes_per_sample": LOOKUP_BYTES_PER_SAMPLE, "in_step_ms": phases[lk],
                 "alone_ms": lookup_alone_ms, "alone_achieved": lookup_bytes / (lookup_alone_ms * 1e-3) / 1e9,
                 "alone_frac": lookup_bytes / (lookup_alone_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
    eb = "embedding_bwd_update" if world == 1 else "sharded_embedding_bwd_update"
    uniq = int(sum(torch.unique(ids_pool[0][:, f]).numel() for f in range(len(vocabs))))
    S = 3 if eng.emb_opt == "adam_lazy" else 1
    eb_bytes = B * len(vocabs) * (4 + EMB_DIM * 4) + uniq * EMB_DIM * 4 * 2 * S
    eb_ms = phases.get(eb, 0.0) + phases.get("replicated_embedding_bwd", 0.0)
    eb_ach = eb_bytes / (eb_ms * 1e-3) / 1e9
    b_traffic, b_note = load_traffic("bwd_unit_kernel") if (full_batch and world == 1) else (None, None)
    rl_emb = {"kernel": "a13: bwd_prep + split_count/scan/scatter + bwd_unit_kernel (two-level radix partition fused with the row update)"
              if getattr(eng, "bwd_algo", "auto") != "sort" else "a13: bwd_keys + radix sort + bwd_chunk/hot/merge",
              "algo": getattr(eng, "bwd_algo", "auto"), "algo_trial_ms": getattr(eng, "bwd_algo_ms", None),
              "bound": "hbm", "achieved": eb_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
              "frac": eb_ach / peaks["hbm_gbs"], "unique_rows": uniq, "bytes_per_step": eb_bytes, "in_step_ms": eb_ms,
              "traffic": b_traffic, "traffic_note": b_note}

    cpu = None
    if not args.no_cpu_baseline and world == 1:  # the CPU arm is timed at N=1 only (the N>1 lines carry cpu_baseline: null)
        r = cpu_deepfm_arm(batch=B, vocab_cap=CPU_VOCAB_CAP, steps=3, warmup=1)
        cpu = {"value": r["samples_per_s"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}

    line = {
        "metric": METRICS["deepfm"], "value": B * world * args.steps / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS["deepfm"],
                   "global_batch": B * world, "tables_rows": sum(vocabs), "tables_gb": sum(vocabs) * EMB_DIM * 4 / 1e9, "ids": args.ids,
                   "optimizer": f"{args.optimizer} (dense params and the {n_small} tables of <= {args.small_table_rows} rows, Keras-exact dense step) + {eng.emb_opt} (touched rows of the {n_sharded} large tables)", "l2_embd": 0.0,
                   "l2_flush": "inputs larger than L2 (%.1f GB of tables, rotating pool of 4 batches)" % (sum(vocabs) * EMB_DIM * 4 / 1e9), "scale_vocab": args.scale_vocab,
                   "parallelism": "single GPU" if world == 1 else f"dp{world}: batch split, {n_sharded} large tables row-sharded (row % {world}), {n_small} small tables replicated (gradients all-reduced with the dense ones), forward = fused lookup+FM reading peer shards over NVLink (symmetric memory), backward = " + ("one kernel gathers the gradient rows and stores them into the owners' receive buffers over NVLink (symmetric memory)" if getattr(getattr(eng, "exchange", None), "rx", None) is not None else "NCCL all-to-all of gradient rows to the owners") + ", all-reduce for dense grads"},
        "e2e": {"value": B * world * args.steps / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": eng.h2d_bytes_per_step(B), "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps, "last_loss": loss, "api": e2e_api,
                "blocking_train_on_batch_samples_per_s": B * world * args.steps / (e2e_sync_ms * 1e-3)},
        "gpu_launches": launches, "gpu_launches_per_step": launches / max(args.steps, 1),
        "clocks": clk, "roofline": roofline, "roofline_lookup": rl_lookup, "roofline_embedding_bwd": rl_emb, "cpu_baseline": cpu,
        "kernel_ms": {k: round(v, 4) for k, v in phases.items()},
    }
    if timeline is not None:
        line["timeline_ms"] = timeline
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
