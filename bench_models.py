"""bench.py workloads besides DeepFM: DIN (BASELINE.json configs[1]), YouTubeMatchDNN retrieval (configs[4]), their CPU arms
(oracle/), the multi-GPU --verify mode, and the writer of --dump-outputs.  Imported by bench.py only."""
from __future__ import annotations

import json
import os
import time
from collections import OrderedDict

import numpy as np

# MovieLens-1M shaped vocabularies (examples/DIN/DIN_cfg.yaml, examples/YouTubeDNN/YouTubeMatchDNN_cfg.yaml; vocab = max id + 1)
ML = {"user_id": (6041, 32), "gender": (3, 4), "occupation": (22, 16), "zip": (3440, 32), "age": (8, 16), "movie_id": (3953, 32), "year": (83, 16),
      "genre_id": (19, 8)}
DIN_B, DIN_T, GENRES_L = 4096, 50, 6
RET_B, RET_ITEMS, RET_SAMPLED, RET_EMBD = 4096, 10_000_000, 100, 64
RET_CPU_ITEMS = 1_000_000  # catalogue rows on the CPU arm (the reference recomputes EVERY catalogue row every step)
DUMP_ROWS = 4096  # --dump-outputs: rows kept of a table too large to write whole
DUMP_MAX_BYTES = 64 << 20


def sample_rows(n, seed=0):
    """--dump-outputs: a fixed, seeded, sorted choice of min(n, DUMP_ROWS) distinct indices below n."""
    return np.sort(np.random.RandomState(seed).choice(n, min(n, DUMP_ROWS), replace=False))


def write_outputs(directory, arrays):
    """--dump-outputs: DIR/<name>.npy for every array, float32 kept as it is and anything else as float64."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs, more than {DUMP_MAX_BYTES}")
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, f"{k}.npy"), v)


def model_outputs(model, loss):
    """What a caller of `Model.train_on_batch` holds after the step: the loss it returned and the model's weights, tables of
    more than 2^20 entries as a fixed sample of their rows."""
    import torch

    from handyrec_b200.checkpoint import _named_weights

    out = {"loss": np.array([loss], dtype=np.float64)}
    for name, _, p in _named_weights(model):
        w = p.detach()
        if w.numel() > (1 << 20):
            w = w[torch.from_numpy(sample_rows(w.shape[0])).to(w.device)]
        out[name] = w.cpu().numpy()
    return out


def _hist(rng, n, T, vocab):
    """History-like ids: Zipf(1.05) items, random length U{0..T}, zero padding in FRONT (data/utils.py:46-49)."""
    u = rng.random_sample((n, T))
    a = 1.05
    ids = (((vocab ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))).astype(np.int64).clip(1, vocab - 1).astype(np.int32)
    lens = rng.randint(0, T + 1, n)
    keep = np.arange(T)[None, :] >= (T - lens)[:, None]
    return np.where(keep, ids, 0).astype(np.int32)


def din_data(n, seed=2022, item_vocab=ML["movie_id"][0]):
    rng = np.random.RandomState(seed)
    x = {k: rng.randint(1, ML[k][0], (n, 1)).astype(np.int32) for k in ("user_id", "gender", "occupation", "zip", "age", "year")}
    x["movie_id"] = rng.randint(1, item_vocab, (n, 1)).astype(np.int32)
    x["hist_movie"] = _hist(rng, n, DIN_T, item_vocab)
    x["genres"] = _hist(rng, n, GENRES_L, ML["genre_id"][0])
    y = (rng.random_sample(n) < 0.25).astype(np.float32)
    return x, y


def build_din(item_vocab=ML["movie_id"][0]):
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.features import FeatureGroup, FeaturePool, SparseFeature, SparseSeqFeature
    from handyrec_b200.models import DIN

    movie = SparseFeature("movie_id", item_vocab, 32)
    pool = FeaturePool()
    seq_group = FeatureGroup("item_seq", [SparseSeqFeature(movie, "hist_movie", DIN_T)], pool, l2_embd=0.0)
    other = [SparseFeature(k, ML[k][0], ML[k][1]) for k in ("user_id", "gender", "occupation", "zip", "age")] + [movie, SparseFeature("year", *ML["year"])]
    other.append(SparseSeqFeature(SparseFeature("genre_id", *ML["genre_id"]), "genres", GENRES_L))
    other_group = FeatureGroup("other_feats", other, pool, l2_embd=0.0)
    model = DIN(seq_group, other_group, dnn_hidden_units=(64, 32), dnn_activation="dice", lau_dnn_hidden_units=(32, 1), lau_dnn_activation="dice")
    model.compile(optimizer=KL.Adam(learning_rate=1e-3), loss=KL.binary_crossentropy)
    return model


def retrieval_data(n, n_items, seed=2022):
    rng = np.random.RandomState(seed)
    x = {k: rng.randint(1, ML[k][0], (n, 1)).astype(np.int32) for k in ("user_id", "gender", "occupation")}
    x["hist_movie"] = _hist(rng, n, DIN_T, n_items)
    x["movie_id"] = _hist(rng, n, 1, n_items).clip(1, None).astype(np.int32)
    return x, np.zeros(n, dtype=np.float32)


def build_retrieval(n_items=RET_ITEMS, seed=0):
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.features import EmbdFeatureGroup, FeatureGroup, FeaturePool, SparseFeature, SparseSeqFeature
    from handyrec_b200.layers.utils import sampledsoftmaxloss
    from handyrec_b200.models import YouTubeMatchDNN

    rng = np.random.RandomState(seed)
    movie, genre = SparseFeature("movie_id", n_items, 32), SparseFeature("genre_id", *ML["genre_id"])
    values = {"movie_id": np.arange(n_items, dtype=np.int32), "genres": _hist(rng, n_items, GENRES_L, ML["genre_id"][0])}
    pool = FeaturePool()
    item_group = EmbdFeatureGroup("item", "movie_id", [movie, SparseSeqFeature(genre, "genres", GENRES_L)], pool, values, embd_dim=RET_EMBD, l2_embd=0.0)
    user = [SparseFeature(k, *ML[k]) for k in ("user_id", "gender", "occupation")] + [SparseSeqFeature(movie, "hist_movie", DIN_T)]
    user_group = FeatureGroup("user", user, pool, l2_embd=0.0)
    model = YouTubeMatchDNN(user_group, item_group, dnn_hidden_units=(128, RET_EMBD), num_sampled=RET_SAMPLED)
    model.compile(optimizer=KL.Adam(learning_rate=1e-3), loss=sampledsoftmaxloss)
    return model


# -------------------------------------------------------------------------------------------------
# CPU arms: the reference restated op for op (oracle/), dense Adam like Keras
# -------------------------------------------------------------------------------------------------
def cpu_arm(workload: str, steps: int, warmup: int):
    import torch

    import oracle

    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(0)

    def table(v, d):
        return ((torch.rand(v, d, generator=g) - 0.5) * 0.1).requires_grad_(True)

    if workload == "din":
        B = DIN_B
        x, y = din_data(B)
        T = {k: table(*ML[k]) for k in ML}
        width = sum(ML[k][1] for k in ("user_id", "gender", "occupation", "zip", "age", "movie_id", "year")) + ML["genre_id"][1] + 32
        lau = oracle.dnn_init(4 * 32, (32, 1), seed=1)
        dnn = oracle.dnn_init(width, (64, 32, 1), seed=2)
        params = list(T.values()) + [t.requires_grad_(True) for t in lau.tensors() + dnn.tensors()]
        xt = {k: torch.from_numpy(v) for k, v in x.items()}
        yt = torch.from_numpy(y)

        def fwd():
            sparse = OrderedDict((k, (T[k], xt[k], k == "movie_id")) for k in ("user_id", "gender", "occupation", "zip", "age", "movie_id", "year"))
            seqs = OrderedDict(genres=(T["genre_id"], xt["genres"]))
            embds = oracle.group_embedding_lookup(sparse, seqs, "mean")
            keys, mask = oracle.custom_embedding(T["movie_id"], xt["hist_movie"], True)
            keys, kmask = oracle.squeeze_mask(keys, mask)
            q, _ = oracle.custom_embedding(T["movie_id"], xt["movie_id"], True)
            att = oracle.local_activation_unit(q, keys, kmask, lau, act="dice", training=True)
            pooled = oracle.din_attention_pool(att, keys)
            h = oracle.concat([], embds + [pooled])
            p = oracle.dnn(h, dnn, act="dice", output_activation="sigmoid", training=True)
            return torch.nn.functional.binary_cross_entropy(p[:, 0].clamp(1e-7, 1 - 1e-7), yt)

        sample = f"batch {B}, full MovieLens-1M-shaped model, torch-CPU op-for-op restatement (materialised (B,T,4D) attention input, dense Adam)"
    else:
        B, n_items = RET_B, RET_CPU_ITEMS
        x, _ = retrieval_data(B, n_items)
        rng = np.random.RandomState(0)
        genres = torch.from_numpy(_hist(rng, n_items, GENRES_L, ML["genre_id"][0]))
        T = {"movie_id": table(n_items, 32), "genre_id": table(*ML["genre_id"]), "user_id": table(*ML["user_id"]), "gender": table(*ML["gender"]),
             "occupation": table(*ML["occupation"])}
        red_W = ((torch.rand(40, RET_EMBD, generator=g) - 0.5) * 0.3).requires_grad_(True)
        red_b = torch.zeros(RET_EMBD, requires_grad=True)
        user = oracle.dnn_init(32 + 4 + 16 + 32, (128, RET_EMBD), seed=3)
        params = list(T.values()) + [red_W, red_b] + [t.requires_grad_(True) for t in user.tensors()]
        xt = {k: torch.from_numpy(v) for k, v in x.items()}
        all_ids = torch.arange(n_items, dtype=torch.int32)

        def fwd():
            # EmbdFeatureGroup.get_embd: EVERY catalogue row, every step (group.py:464-483)
            e_id, _ = oracle.custom_embedding(T["movie_id"], all_ids, False)
            e_g = oracle.sequence_pooling(*oracle.custom_embedding(T["genre_id"], genres, True), "mean")[:, 0]
            items = torch.cat([e_id, e_g], 1) @ red_W + red_b
            sparse = OrderedDict((k, (T[k], xt[k], False)) for k in ("user_id", "gender", "occupation"))
            seqs = OrderedDict(hist_movie=(T["movie_id"], xt["hist_movie"]))
            u = oracle.dnn(oracle.concat([], oracle.group_embedding_lookup(sparse, seqs, "mean")), user, act="relu", output_activation="linear")
            sampled, tries = oracle.log_uniform_sample(RET_SAMPLED, n_items, rng)
            te = oracle.unique_expected_count(oracle.log_uniform_prob(x["movie_id"].reshape(-1), n_items), tries)
            se = oracle.unique_expected_count(oracle.log_uniform_prob(sampled, n_items), tries)
            return oracle.sampled_softmax_loss(items, torch.zeros(n_items), xt["movie_id"], u, torch.from_numpy(sampled), torch.from_numpy(te),
                                               torch.from_numpy(se)).mean()

        sample = (f"batch {B}, catalogue capped at {n_items} items (the reference evaluates the whole catalogue every step), torch-CPU op-for-op "
                  "restatement, dense Adam")
    opt = torch.optim.Adam(params, lr=1e-3, eps=1e-7)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = fwd()
        loss.backward()
        opt.step()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"samples_per_s": B * steps / dt, "ms_per_step": dt / steps * 1e3, "cores": torch.get_num_threads(), "batch": B,
            "sample": f"{steps} steps of " + sample}


# -------------------------------------------------------------------------------------------------
def run(args, load_peaks, ClockSampler, WORKLOADS, METRICS):
    """DIN / retrieval on one GPU through the reference-shaped API (constructor -> compile -> train_on_batch / fit)."""
    import torch

    from handyrec_b200.engine import launch_count

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    peaks = load_peaks()
    vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
    clocks = ClockSampler(vis[0] if vis else 0)  # started before the model is built: its start-up is over when the timing begins; samples count from mark()
    clocks.start()
    wl = args.workload
    if wl == "din":
        B = args.batch or DIN_B
        model = build_din()
        x, y = din_data(B * 4)
        flops_fwd = B * DIN_T * 2.0 * (128 * 128 + 128 * 32 + 32 * 1)  # LAU MLP: 41 024 flop per (sample, position) (SURVEY 8d)
        tensor_note = "LocalActivationUnit MLP [128,128,32,1] over B*T = 204 800 rows; forward+backward = 3 x forward flops"
    else:
        B = args.batch or RET_B
        model = build_retrieval()
        x, y = retrieval_data(B * 4, RET_ITEMS)
        flops_fwd = B * 2.0 * (84 * 84 + 84 * 128 + 128 * 64 + 64 * RET_SAMPLED) + (B + RET_SAMPLED) * 2.0 * 40 * RET_EMBD
        tensor_note = "user tower [84,84,128,64] + sampled logits (B x 100 x 64) + item rows (B+100) x 40 x 64; forward+backward = 3 x forward flops"
    NB = 4
    pool_dev = [({k: torch.from_numpy(v[i * B : (i + 1) * B]).to(dev) for k, v in x.items()}, torch.from_numpy(y[i * B : (i + 1) * B]).to(dev)) for i in range(NB)]
    for s in range(max(args.warmup, 3)):
        model.train_on_batch(*pool_dev[s % NB])
    torch.cuda.synchronize()
    clocks.mark()
    l0 = launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        loss = model.train_on_batch(*pool_dev[s % NB])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = launch_count() - l0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, model_outputs(model, loss))
    # end to end: Model.fit on host dict-of-arrays (numpy), one epoch of `steps` batches
    reps = (args.steps + NB - 1) // NB
    xh = {k: np.concatenate([v] * reps)[: args.steps * B] for k, v in x.items()}
    yh = np.concatenate([y] * reps)[: args.steps * B]
    model.fit({k: v[: 2 * B] for k, v in xh.items()}, yh[: 2 * B], batch_size=B, epochs=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    hist = model.fit(xh, yh, batch_size=B, epochs=1)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    clk = clocks.stop()
    h2d = sum(int(np.prod(v.shape[1:])) * 4 for v in x.values()) * B + 4 * B
    ach = 3 * flops_fwd / (ms / args.steps * 1e-3) / 1e12
    cpu = None
    if not args.no_cpu_baseline:
        r = cpu_arm(wl, steps=3, warmup=1)
        cpu = {"value": r["samples_per_s"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    line = {
        "metric": METRICS[wl], "value": B * args.steps / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[wl], "global_batch": B, "ids": "zipf(1.05) histories, random lengths, front padding",
                   "optimizer": "adam (dense Keras-exact step on tables < 131072 rows, touched-rows update on larger ones)",
                   "l2_flush": "rotating pool of 4 batches; tables of the DIN config are L2-resident (0.5 MB), the 10 M-item table (1.28 GB) is not",
                   "parallelism": "single GPU", "path": "layer-by-layer ops of libhrb200 driven by the Keras-like Model (no fused engine for this graph yet)"},
        "e2e": {"value": B * args.steps / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps, "last_loss": float(hist.history["loss"][-1]),
                "api": f"handyrec_b200.models.{'DIN' if wl == 'din' else 'YouTubeMatchDNN'}(...).compile(...).fit(dict of host arrays)"},
        "gpu_launches": launches, "gpu_launches_per_step": launches / max(args.steps, 1), "clocks": clk,
        "roofline": {"kernel": tensor_note, "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": ach / peaks["bf16_tflops_sustained"], "traffic": None,
                     "note": "whole-step time against the dense flops of the step: the step is launch- and latency-bound at this batch (see gpu_launches_per_step)"},
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------
def verify_model_api(CRITEO_VOCABS, N_DENSE, EMB_DIM, b, small_rows):
    """The same comparison through the reference-shaped API: `with ShardedTables(): DeepFM(...).compile(...)` + per-rank `fit(dict)`
    on N GPUs against ONE single-GPU `DeepFM(...).fit` on the concatenated batches, then a save_weights / load_weights round trip of
    the sharded model (every rank writes the rows it owns)."""
    import shutil
    import tempfile

    import numpy as np
    import torch
    import torch.distributed as dist

    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
    from handyrec_b200.layers import CustomEmbedding
    from handyrec_b200.models import DeepFM

    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device())
    vocabs = [max(4, min(v, 300_000)) for v in CRITEO_VOCABS]
    steps = 3

    def make():
        sparse = [SparseFeature(f"C{i + 1}", v, EMB_DIM) for i, v in enumerate(vocabs)]
        dense = [DenseFeature(f"I{i + 1}") for i in range(N_DENSE)]
        pool = FeaturePool()
        return DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", dense + sparse, pool, l2_embd=0.0),
                      dnn_hidden_units=(64, 32, 1), dnn_activation="relu")

    def data(r):
        g = np.random.default_rng(1000 + r)
        x = {f"C{i + 1}": g.integers(0, v, size=(steps * b, 1)).astype(np.int32) for i, v in enumerate(vocabs)}
        for j in range(N_DENSE):
            x[f"I{j + 1}"] = g.random((steps * b, 1), dtype=np.float32)
        return x, (g.random(steps * b) < 0.25).astype(np.float32)

    out = {}
    for opt in ("sgd", "adam_eps1e-3"):
        def optimizer():
            return KL.SGD(learning_rate=0.05) if opt == "sgd" else KL.Adam(learning_rate=1e-3, epsilon=1e-3)

        torch.manual_seed(4321)  # replicated tables / dense weights are broadcast from rank 0 anyway
        with KL.ShardedTables(min_rows=small_rows, seed=99):
            model = make()
            model.compile(optimizer=optimizer(), loss=KL.binary_crossentropy)
        model._fused.build(b, model.optimizer)
        model._fused.engine.autotune_embedding_bwd = False
        emb_layers = [l for l in model._all_layers() if isinstance(l, CustomEmbedding)]
        # the single-GPU twin on rank 0: same graph, tables assembled from the shards, dense weights copied
        full = {}
        for l in emb_layers:
            w = l.embeddings.data
            if l._sharded is None:
                full[l.name] = w.clone()
                continue
            rows0 = (l.input_dim + world - 1) // world
            pad = torch.zeros(rows0, EMB_DIM, device=dev)
            pad[: w.shape[0]] = w
            parts = [torch.empty_like(pad) for _ in range(world)]
            dist.all_gather(parts, pad)
            t = torch.empty(l.input_dim, EMB_DIM, device=dev)
            for r in range(world):
                t[r::world] = parts[r][: t[r::world].shape[0]]
            full[l.name] = t
        ref = None
        if rank == 0:
            ref = make()
            for l in ref._all_layers():
                if isinstance(l, CustomEmbedding):
                    l.embeddings.data = full[l.name].clone()
            src = {n: p for n, _, p in _named(model)}
            for n, lay, p in _named(ref):
                if not isinstance(lay, CustomEmbedding):
                    p.data.copy_(src[n].data)
            ref.dense_table_max_rows = small_rows
            ref.compile(optimizer=optimizer(), loss=KL.binary_crossentropy)
            ref._fused.build(b * world, ref.optimizer)
            ref._fused.engine.autotune_embedding_bwd = False
        x, y = data(rank)
        model.fit(x, y, batch_size=b, epochs=1)
        ls = torch.tensor(model.last_losses, device=dev, dtype=torch.float64)
        dist.all_reduce(ls)
        losses_s = (ls / world).tolist()
        err = {"dense": 0.0, "replicated": 0.0, "sharded": 0.0, "loss": 0.0, "checkpoint": 0.0}
        if rank == 0:
            xs, ys = zip(*[data(r) for r in range(world)])
            xc = {k: np.concatenate([np.concatenate([xr[k][s * b : (s + 1) * b] for xr in xs]) for s in range(steps)]) for k in x}
            yc = np.concatenate([np.concatenate([yr[s * b : (s + 1) * b] for yr in ys]) for s in range(steps)])
            ref.fit(xc, yc, batch_size=b * world, epochs=1)
            err["loss"] = max(abs(a - c) / max(abs(c), 1e-12) for a, c in zip(losses_s, ref.last_losses))
            ref.sync()
        model.sync()
        refw = {n: (lay, p) for n, lay, p in _named(ref)} if rank == 0 else {}
        for n, lay, p in _named(model):
            w = p.data
            if isinstance(lay, CustomEmbedding) and lay._sharded is not None:
                rows0 = (lay.input_dim + world - 1) // world
                pad = torch.zeros(rows0, EMB_DIM, device=dev)
                pad[: w.shape[0]] = w
                parts = [torch.empty_like(pad) for _ in range(world)]
                dist.all_gather(parts, pad)
                if rank == 0:
                    want_full = refw[n][1].data
                    for r in range(world):
                        want = want_full[r::world]
                        err["sharded"] = max(err["sharded"], float((parts[r][: want.shape[0]] - want).abs().max()) / float(want_full.abs().max()))
            elif rank == 0:
                want = refw[n][1].data
                key = "replicated" if isinstance(lay, CustomEmbedding) else "dense"
                err[key] = max(err[key], float((w - want).abs().max()) / max(float(want.abs().max()), 1e-12))
        # checkpoint round trip of the sharded model
        d = [tempfile.mkdtemp(prefix="hrb_ckpt_") if rank == 0 else None]
        dist.broadcast_object_list(d, src=0)
        model.save_weights(d[0])
        dist.barrier()
        before = {n: p.data.clone() for n, _, p in _named(model)}
        for n, _, p in _named(model):
            p.data.add_(1.0)
        model.load_weights(d[0])
        ck = torch.tensor(max(float((p.data - before[n]).abs().max()) for n, _, p in _named(model)), device=dev)
        dist.all_reduce(ck, op=dist.ReduceOp.MAX)
        err["checkpoint"] = float(ck)
        dist.barrier()
        if rank == 0:
            shutil.rmtree(d[0], ignore_errors=True)
            out[f"model_api/{opt}/b{b}"] = {"err": {k: float(f"{v:.3g}") for k, v in err.items()}, "loss_sharded": losses_s,
                                           "loss_single_gpu": [float(v) for v in ref.last_losses]}
        del model, ref, full
        torch.cuda.empty_cache()
        dist.barrier()
    return out


def _named(model):
    from handyrec_b200.checkpoint import _named_weights

    return list(_named_weights(model)) if model is not None else []


def verify_sharded(args, CRITEO_VOCABS, N_DENSE, EMB_DIM):
    """N>1 correctness on real hardware: 3 steps of the row-sharded engine (symmetric-memory peer lookup, NCCL all-to-all of
    gradient rows, all-reduce of the dense + replicated-table gradients) on per-rank batches == 3 steps of ONE single-GPU engine on
    the concatenated batch (rank 0 holds it).  Compares dense parameters, replicated tables and every shard, and reports the
    global-batch loss of both so that the `last_loss` growing with N in the scaling records is shown to be the larger global batch
    (same weights -> same loss), not lost updates."""
    import torch
    import torch.distributed as dist

    from handyrec_b200 import kernels as K
    from handyrec_b200.engine import DeepFMEngine
    from handyrec_b200.sharded import ShardedDeepFMEngine, TorchDistComm

    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device())
    b = args.batch or 4096
    hidden = (64, 32, 1)
    small_rows = 2048
    vocabs = [max(4, min(v, 300_000)) for v in CRITEO_VOCABS]
    fields = [(f, 1, "none") for f in range(len(vocabs))]
    results = {}
    b_full = b
    # the last case runs a batch below the tensor-core threshold: the FFMA step takes the non-overlapped backward, whose reads of
    # the side-stream routing results are ordered by an event (round-1 advisor finding)
    # Adam divides by sqrt(v) + eps with eps = 1e-7 (Keras): where |g| is of the order of eps -- most entries at these 1/(B*N)-scaled
    # gradients -- rounding-level differences between the two summation orders are magnified by up to 0.1/eps in the step.  The
    # "adam_eps1e-3" cases repeat Adam with a benign eps to separate that conditioning from lost or misplaced updates; SGD is exact.
    for opt, peer, b in (("sgd", True, b_full), ("sgd", False, b_full), ("adam", True, b_full), ("adam", False, b_full), ("adam_eps1e-3", True, b_full),
                         ("sgd", True, 256), ("adam", True, 256), ("adam_eps1e-3", True, 256)):
        eps = 1e-3 if opt.endswith("eps1e-3") else 1e-7
        label_opt, opt = opt, opt.split("_")[0]
        if True:
            comm = TorchDistComm()
            tables, peer_ptrs = comm.alloc_tables(vocabs, EMB_DIM, dev, replicate_max_rows=small_rows)
            for f, t in enumerate(tables):
                if vocabs[f] <= small_rows:
                    K.init_uniform(t, seed=7 + f)
                else:
                    K.init_uniform(t, seed=7 + f, row_start=rank, row_step=world)
            eng = ShardedDeepFMEngine(tables, vocabs, fields, N_DENSE, comm, peer_ptrs=peer_ptrs if peer else None, dnn_hidden_units=hidden,
                                      dnn_activation="relu", batch_size=b, optimizer=opt, lr=0.05 if opt == "sgd" else 1e-3, l2_embd=0.0, seed=2022,
                                      replicate_max_rows=small_rows)
            eng.autotune_embedding_bwd = False
            eng.eps = eps
            ref = None
            if rank == 0:
                full = []
                for f, v in enumerate(vocabs):
                    t = torch.empty(v, EMB_DIM, device=dev)
                    K.init_uniform(t, seed=7 + f)
                    full.append(t)
                ref = DeepFMEngine(full, fields, N_DENSE, hidden, "relu", batch_size=b * world, optimizer=opt, lr=0.05 if opt == "sgd" else 1e-3, l2_embd=0.0,
                                   seed=2022, dense_table_max_rows=small_rows)
                ref.autotune_embedding_bwd = False
                ref.eps = eps
            losses_s, losses_r = [], []
            for step in range(3):
                g = torch.Generator(device=dev).manual_seed(100 * step + rank)
                ids = torch.stack([torch.randint(0, v, (b,), device=dev, generator=g) for v in vocabs], 1).to(torch.int32).contiguous()
                dense = torch.rand(b, N_DENSE, device=dev, generator=g)
                label = (torch.rand(b, device=dev, generator=g) < 0.25).float()
                gi = [torch.empty_like(ids) for _ in range(world)]
                gd = [torch.empty_like(dense) for _ in range(world)]
                gl = [torch.empty_like(label) for _ in range(world)]
                dist.all_gather(gi, ids)
                dist.all_gather(gd, dense)
                dist.all_gather(gl, label)
                eng.train_step_on_device(ids, dense, label)
                ls = eng.loss_sum.clone()
                dist.all_reduce(ls)
                losses_s.append(float(ls) / (b * world))
                if ref is not None:
                    ref.train_step_on_device(torch.cat(gi), torch.cat(gd), torch.cat(gl))
                    losses_r.append(float(ref.loss_sum) / (b * world))
            torch.cuda.synchronize()
            # gather every shard on rank 0 and compare
            err = {"dense": 0.0, "replicated": 0.0, "sharded": 0.0, "loss": 0.0}
            n_dense_params = eng.n_dense_params
            pd = [torch.empty_like(eng.params[:n_dense_params]) for _ in range(world)]
            dist.all_gather(pd, eng.params[:n_dense_params].contiguous())
            for f, v in enumerate(vocabs):
                if v <= small_rows:
                    tl = [torch.empty_like(eng.tables[f]) for _ in range(world)]
                    dist.all_gather(tl, eng.tables[f].contiguous())
                    if rank == 0:
                        scale = float(ref.tables[f].abs().max())
                        err["replicated"] = max(err["replicated"], max(float((t - ref.tables[f]).abs().max()) / scale for t in tl))
                else:
                    rows0 = (v + world - 1) // world
                    pad = torch.zeros(rows0, EMB_DIM, device=dev)
                    pad[: eng.tables[f].shape[0]] = eng.tables[f]
                    tl = [torch.empty_like(pad) for _ in range(world)]
                    dist.all_gather(tl, pad)
                    if rank == 0:
                        scale = float(ref.tables[f].abs().max())
                        for r in range(world):
                            want = ref.tables[f][r::world]
                            err["sharded"] = max(err["sharded"], float((tl[r][: want.shape[0]] - want).abs().max()) / scale)
            if rank == 0:
                rp = ref.params[:n_dense_params]
                err["dense"] = max(float((p - rp).abs().max()) for p in pd) / float(rp.abs().max())
                err["loss"] = max(abs(a - c) / max(abs(c), 1e-12) for a, c in zip(losses_s, losses_r))
                results[f"{label_opt}/{'peer' if peer else 'all_to_all'}/b{b}"] = {"err": {k: float(f"{v:.3g}") for k, v in err.items()}, "loss_sharded": losses_s, "loss_single_gpu": losses_r}
            del eng, ref, tables
            torch.cuda.empty_cache()
            dist.barrier()
    api = verify_model_api(CRITEO_VOCABS, N_DENSE, EMB_DIM, b_full, small_rows)
    if rank == 0:
        results.update(api)
        tol = 2e-4
        # pass / fail on the well-conditioned cases; default-eps Adam is reported next to them
        ok = all(max(r["err"].values()) <= tol for k, r in results.items() if not k.startswith("adam/"))
        print(json.dumps({"verify": "ok" if ok else "FAILED", "n_gpus": world, "batch_per_gpu": b_full, "tolerance": tol, "cases": results,
                          "note": "errors are max |sharded - single GPU| / max |single GPU| after 3 steps; loss_* is the mean BCE over the GLOBAL batch: equal on "
                                  "both sides, i.e. a larger N changes the loss only through the larger global batch it trains on"}), flush=True)
    dist.barrier()
