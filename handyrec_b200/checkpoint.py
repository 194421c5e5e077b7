"""Table / dense checkpoint I/O (SURVEY 8f3).

The reference moves weights in and out through Keras: `weights=[ndarray]` on the embedding layers (features/group.py:283-291,
fed by `FeaturePool(pre_embd)`) and `model.save_weights / load_weights` (docs/source/Quickstart.md:250-262).  Here:

    save_weights(model, dir)      one `.npy` per weight; tables with more than `shard_rows` rows are written as row shards
                                  streamed from the device chunk by chunk (a 40 M x 16 table never exists on the host in one piece)
    load_weights(model, dir)      the inverse, shape-checked, streamed back to the device the same way
    save_sharded_tables(engine, dir) / load_sharded_tables(engine, dir)
                                  the row-sharded engine: rank r writes the rows it owns (row % N == r) of every sharded table as
                                  `<table>.rank<r>of<N>.npy`, rank 0 the replicated tables and the dense parameters; loading accepts
                                  the same N only (re-sharding = load on one GPU, save, shard again)
    export_pre_embd(model)        {feature name: ndarray} in the form `FeaturePool(pre_embd=...)` takes (group.py:283-284)

Weights are keyed by the position of their layer in the model's execution order + the layer class + the weight name, which is
stable for the same constructor call; `manifest.json` also records the layer names for humans.
"""
from __future__ import annotations

import json
import os
from typing import Dict, Iterator, Tuple

import numpy as np
import torch

SHARD_ROWS = 1 << 22


def _named_weights(model) -> Iterator[Tuple[str, str, torch.nn.Parameter]]:
    seen = set()
    for i, layer in enumerate(model._all_layers()):
        for key, p in layer._weights.items():
            if id(p) in seen:
                continue
            seen.add(id(p))
            yield f"{i:03d}_{type(layer).__name__}.{key}", layer, p


def _save_tensor(t: torch.Tensor, base: str, shard_rows: int):
    files = []
    if t.dim() == 2 and t.shape[0] > shard_rows:
        for r0 in range(0, t.shape[0], shard_rows):
            r1 = min(t.shape[0], r0 + shard_rows)
            f = f"{base}.rows{r0:012d}-{r1:012d}.npy"
            np.save(f, t[r0:r1].detach().cpu().numpy())
            files.append(os.path.basename(f))
    else:
        np.save(base + ".npy", t.detach().cpu().numpy())
        files.append(os.path.basename(base) + ".npy")
    return files


def _shard_file_names(t: torch.Tensor, base: str, shard_rows: int):
    if t.dim() == 2 and t.shape[0] > shard_rows:
        return [os.path.basename(f"{base}.rows{r0:012d}-{min(t.shape[0], r0 + shard_rows):012d}.npy") for r0 in range(0, t.shape[0], shard_rows)]
    return [os.path.basename(base) + ".npy"]


def _load_tensor(dst: torch.Tensor, directory: str, files) -> None:
    if len(files) == 1 and ".rows" not in files[0]:
        a = np.load(os.path.join(directory, files[0]))
        if tuple(a.shape) != tuple(dst.shape):
            raise ValueError(f"{files[0]}: shape {a.shape} does not match the model's {tuple(dst.shape)}")
        dst.copy_(torch.from_numpy(a).to(dst.dtype))
        return
    done = 0
    for f in files:
        span = f.split(".rows")[1].split(".npy")[0]
        r0, r1 = (int(x) for x in span.split("-"))
        a = np.load(os.path.join(directory, f))
        if a.shape[0] != r1 - r0 or tuple(a.shape[1:]) != tuple(dst.shape[1:]) or r1 > dst.shape[0]:
            raise ValueError(f"{f}: shard does not fit a table of shape {tuple(dst.shape)}")
        dst[r0:r1].copy_(torch.from_numpy(a).to(dst.dtype))
        done += r1 - r0
    if done != dst.shape[0]:
        raise ValueError(f"row shards cover {done} of {dst.shape[0]} rows")


def _world(model) -> Tuple[int, int]:
    comm = getattr(model, "_comm", None)
    return (comm.rank, comm.N) if comm is not None and comm.N > 1 else (0, 1)


def _manifest_name(rank: int, world: int) -> str:
    return "manifest.json" if world == 1 else f"manifest.rank{rank}of{world}.json"


def save_weights(model, directory: str, shard_rows: int = SHARD_ROWS) -> Dict:
    """Multi-GPU models (keras_lite.ShardedTables): every rank calls this; a row-sharded table is written by each rank as
    `<key>.rank<r>of<N>...npy` (the rows r % N == rank it owns), replicated weights by rank 0 only, and every rank writes its
    own manifest.  Loading takes the same N (re-sharding = load on one GPU, save, shard again)."""
    model.sync()  # fused training keeps dense weights in the engine's flat buffer
    rank, world = _world(model)
    os.makedirs(directory, exist_ok=True)
    manifest = {"format": "handyrec_b200.weights.v1", "world": world, "weights": {}}
    for key, layer, p in _named_weights(model):
        sharded = getattr(layer, "_sharded", None) is not None and p is getattr(layer, "embeddings", None)
        base = os.path.join(directory, key + (f".rank{rank}of{world}" if sharded else ""))
        if sharded or rank == 0:
            files = _save_tensor(p.data, base, shard_rows)
        else:  # rank 0 writes the replicated weights; the names are a pure function of shape and shard_rows
            files = _shard_file_names(p.data, base, shard_rows)
        manifest["weights"][key] = {"layer": layer.name, "shape": list(p.shape), "files": files, "row_sharded": bool(sharded)}
    with open(os.path.join(directory, _manifest_name(rank, world)), "w") as f:
        json.dump(manifest, f, indent=1)
    return manifest


def load_weights(model, directory: str) -> None:
    rank, world = _world(model)
    path = os.path.join(directory, _manifest_name(rank, world))
    if not os.path.exists(path):
        raise FileNotFoundError(f"{path}: no checkpoint for rank {rank} of {world} (saved with another world size?)")
    manifest = json.load(open(path))
    have = manifest["weights"]
    for key, _, p in _named_weights(model):
        if key not in have:
            raise KeyError(f"{directory}: no weight {key!r} (was the model built by the same constructor call?)")
        _load_tensor(p.data, directory, have[key]["files"])
    fused = getattr(model, "_fused", None)
    if fused is not None:  # dense / FM weights also live in the engine: push the loaded values there
        fused.push_to_engine()


def export_pre_embd(model) -> Dict[str, np.ndarray]:
    """{feature name: table} for `FeaturePool(pre_embd=...)`: embedding layers are named "embd_" + feature (group.py:286)."""
    from .layers import CustomEmbedding

    model.sync()
    return {l.name[len("embd_"):]: l.embeddings.data.detach().cpu().numpy() for l in model._all_layers()
            if isinstance(l, CustomEmbedding) and l.name.startswith("embd_")}


# ---- row-sharded engine -------------------------------------------------------------------------
def save_sharded_tables(engine, directory: str) -> None:
    rank, world = engine.comm.rank, engine.world
    os.makedirs(directory, exist_ok=True)
    for t, w in enumerate(engine.tables):
        if t in engine.replicated:
            if rank == 0:
                np.save(os.path.join(directory, f"table{t:03d}.replicated.npy"), w.detach().cpu().numpy())
        else:
            np.save(os.path.join(directory, f"table{t:03d}.rank{rank}of{world}.npy"), w.detach().cpu().numpy())
    if rank == 0:
        np.save(os.path.join(directory, "dense_params.npy"), engine.params[: engine.n_dense_params].detach().cpu().numpy())


def load_sharded_tables(engine, directory: str) -> None:
    rank, world = engine.comm.rank, engine.world
    for t, w in enumerate(engine.tables):
        f = f"table{t:03d}.replicated.npy" if t in engine.replicated else f"table{t:03d}.rank{rank}of{world}.npy"
        a = np.load(os.path.join(directory, f))
        if tuple(a.shape) != tuple(w.shape):
            raise ValueError(f"{f}: shape {a.shape} does not match this rank's {tuple(w.shape)} (saved with another world size?)")
        w.copy_(torch.from_numpy(a))
    engine.params[: engine.n_dense_params].copy_(torch.from_numpy(np.load(os.path.join(directory, "dense_params.npy"))))
    engine._refresh_wt()
