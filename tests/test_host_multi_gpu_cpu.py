"""Host logic of checkpoints and of the multi-GPU creation scope without a GPU: file layout of single- and multi-GPU (row-sharded)
models (SURVEY 8f3), `ShardedTables`, `compile(distribute=...)`.  The weights of a keras_lite model built on a machine without
CUDA are CPU tensors; no kernel runs here."""


import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from handyrec_b200 import checkpoint
from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
from handyrec_b200.layers import CustomEmbedding
from handyrec_b200.models import DeepFM


@pytest.fixture(autouse=True)
def _weights_on_the_host(monkeypatch):
    """keras_lite creates weights on the GPU when there is one; these tests check host logic, so they see no GPU anywhere."""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)


def _model(vocabs=(50, 7000, 11)):
    torch.manual_seed(3)
    sparse = [SparseFeature(f"C{i}", v, 8) for i, v in enumerate(vocabs)]
    dense = [DenseFeature("I0")]
    pool = FeaturePool()
    return DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", dense + sparse, pool, l2_embd=0.0), dnn_hidden_units=(8, 1))


def _weights(model):
    return {k: p.data.clone() for k, _, p in checkpoint._named_weights(model)}


def test_round_trip_with_row_shards(tmp_path):
    m = _model()
    before = _weights(m)
    man = checkpoint.save_weights(m, str(tmp_path), shard_rows=2048)  # the 7000-row table is written as 4 row shards
    big = next(v for v in man["weights"].values() if v["shape"] == [7000, 8])
    assert len(big["files"]) == 4 and all(".rows" in f for f in big["files"])
    assert os.path.exists(tmp_path / "manifest.json")
    for _, _, p in checkpoint._named_weights(m):
        p.data.add_(1.0)
    checkpoint.load_weights(m, str(tmp_path))
    after = _weights(m)
    assert all(torch.equal(before[k], after[k]) for k in before)


def test_sharded_model_layout(tmp_path):
    """Two ranks of a row-sharded model write into one directory: each its own rows of the sharded table (+ its own manifest),
    rank 0 the replicated weights; each rank reads back exactly what it wrote, and another world size is refused."""
    world = 2
    models, shards = [], []
    full = _model()
    for rank in range(world):
        m = _model()  # same seed on every rank: identical replicated weights
        lay = next(l for l in m._all_layers() if isinstance(l, CustomEmbedding) and l.input_dim == 7000)
        lay.embeddings.data = lay.embeddings.data[rank::world].clone()  # this rank's rows r % N == rank
        lay._sharded = (rank, world, 7000)
        m._comm = SimpleNamespace(rank=rank, N=world)
        checkpoint.save_weights(m, str(tmp_path))
        models.append(m)
        shards.append(lay)
    names = sorted(os.listdir(tmp_path))
    assert "manifest.rank0of2.json" in names and "manifest.rank1of2.json" in names and "manifest.json" not in names
    assert sum(".rank0of2" in n and n.endswith(".npy") for n in names) == 1 and sum(".rank1of2" in n and n.endswith(".npy") for n in names) == 1
    man1 = json.load(open(tmp_path / "manifest.rank1of2.json"))
    assert sum(v["row_sharded"] for v in man1["weights"].values()) == 1
    for v in man1["weights"].values():  # every file a manifest names exists (rank 1 points at rank 0's files for replicated weights)
        assert all(os.path.exists(tmp_path / f) for f in v["files"])
    # the two shards interleave to the table a single GPU would hold
    full_lay = next(l for l in full._all_layers() if isinstance(l, CustomEmbedding) and l.input_dim == 7000)
    got = torch.empty_like(full_lay.embeddings.data)
    for rank in range(world):
        got[rank::world] = torch.from_numpy(np.load(tmp_path / next(n for n in names if f".rank{rank}of2" in n and n.endswith(".npy"))))
    assert torch.equal(got, full_lay.embeddings.data)
    for rank, m in enumerate(models):
        want = _weights(m)
        for _, _, p in checkpoint._named_weights(m):
            p.data.mul_(0.0)
        checkpoint.load_weights(m, str(tmp_path))
        got_w = _weights(m)
        assert all(torch.equal(want[k], got_w[k]) for k in want)
    models[0]._comm = SimpleNamespace(rank=0, N=4)
    with pytest.raises(FileNotFoundError):
        checkpoint.load_weights(models[0], str(tmp_path))


def test_sharded_table_refuses_the_layer_path():
    m = _model()
    lay = next(l for l in m._all_layers() if isinstance(l, CustomEmbedding) and l.input_dim == 7000)
    lay._sharded = (0, 2, 7000)
    with pytest.raises(RuntimeError, match="row-sharded"):
        lay.call(torch.zeros(4, 1, dtype=torch.int32))


class _FakeComm:
    def __init__(self, rank, n):
        self.rank, self.N = rank, n


def test_sharded_tables_scope_creates_row_shards_from_given_weights():
    """Under `ShardedTables` a table above `min_rows` is CREATED as this rank's rows r % N == rank (here from pre-trained weights,
    features/group.py:283-291, so that no kernel is needed); smaller tables stay whole."""
    from handyrec_b200 import keras_lite as KL

    big = np.arange(7000 * 8, dtype=np.float32).reshape(7000, 8)
    small = np.arange(50 * 8, dtype=np.float32).reshape(50, 8)
    for rank in range(3):
        with KL.ShardedTables(_FakeComm(rank, 3), min_rows=1000):
            pool = FeaturePool(pre_embd={"C0": small, "C1": big})
            sparse = [SparseFeature("C0", 50, 8), SparseFeature("C1", 7000, 8)]
            m = DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", [DenseFeature("I0")] + sparse, pool, l2_embd=0.0),
                       dnn_hidden_units=(8, 1))
        assert KL.ShardedTables.active is None
        lays = {l.input_dim: l for l in m._all_layers() if isinstance(l, CustomEmbedding)}
        assert lays[50]._sharded is None and tuple(lays[50].embeddings.shape) == (50, 8)
        assert lays[7000]._sharded == (rank, 3, 7000)
        assert np.array_equal(lays[7000].embeddings.data.cpu().numpy(), big[rank::3])


def test_distribute_refuses_graphs_the_engine_does_not_cover():
    """A multi-GPU compile of a graph that does not lower onto the fused engine raises instead of training the layer path on a shard."""
    from handyrec_b200 import keras_lite as KL

    m = _model()
    m.fuse = False  # stands for any graph `lowering.lower` declines (BatchNorm, Dropout, DIN, ...)
    with pytest.raises(ValueError, match="multi-GPU"):
        m.compile(optimizer=KL.Adam(1e-3), loss=KL.binary_crossentropy, distribute=_FakeComm(0, 2))
    m.compile(optimizer=KL.Adam(1e-3), loss=KL.binary_crossentropy, distribute=_FakeComm(0, 1))  # one rank: nothing to shard
