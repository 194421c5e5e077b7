"""CPU: the reference's OWN model files, imported unchanged through handyrec_b200.compat, build the same graphs as this package's
constructors -- layer for layer -- and DeepFM-shaped graphs are recognised by the lowering.

The graphs the reference's files build (input names, then layer kind, configuration, input and output shapes per node) are stored in
tests/golden/compat_graphs.json, so the comparison runs without a checkout of the reference.  With a checkout
(REFERENCE_ROOT=/path/to/HandyRec) the reference's files are also built through the compat shim and held to the stored graphs, and
`python -m tests.test_compat_cpu /path/to/HandyRec` rewrites the file from them.  The stored file was recorded from
`handyrec_b200.models` at a commit whose graphs this test had found equal to those of the reference's files."""
import importlib
import json
import os
import sys

import numpy as np
import pytest

REF = os.environ.get("REFERENCE_ROOT")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "compat_graphs.json")


def _is_checkout(root):
    return root is not None and os.path.isdir(os.path.join(root, "handyrec", "models"))


@pytest.fixture(scope="module")
def ref_models():
    """The reference's `handyrec.models` over the compat shim; None without a checkout, or when a real TensorFlow is importable
    (the shim is not needed then)."""
    if not _is_checkout(REF):
        yield None
        return
    try:
        import tensorflow  # noqa: F401

        if not getattr(tensorflow, "__handyrec_b200_shim__", False):
            yield None
            return
    except ImportError:
        pass
    from handyrec_b200 import compat

    pkg = compat.install(REF)
    yield pkg.models
    compat.uninstall()


def _features():
    from handyrec_b200.features import DenseFeature, SparseFeature, SparseSeqFeature

    movie = SparseFeature("movie_id", 50, 8)
    genre = SparseFeature("genre_id", 19, 8)
    user = [SparseFeature("user_id", 40, 8), SparseFeature("gender", 3, 8), DenseFeature("age"),
            SparseSeqFeature(SparseFeature("movie_id", 50, 8), "hist_movie", 4)]
    item = [movie, SparseSeqFeature(genre, "genres", 3)]
    return user, item


def _signature(model):
    """(layer kind, input shapes, output shapes) per node in execution order; Lambdas are named by what they compute."""
    alias = {"AttentionPooling": "matmul", "item_embedding": "embedding_lookup"}
    sig = []
    for node in model._order:
        lay = node.layer
        kind = type(lay).__name__
        if kind == "Lambda":
            kind = lay.name.rstrip("0123456789_")
        kind = alias.get(kind, kind)
        cfg = {k: v for k, v in lay.get_config().items() if k not in ("name", "trainable")} if hasattr(lay, "get_config") else {}
        ins = [tuple(t.shape) for t in (node.inputs if isinstance(node.inputs, (list, tuple)) else [node.inputs])]
        sig.append((kind, tuple(sorted((k, str(v)) for k, v in cfg.items())), tuple(ins), tuple(tuple(o.shape) for o in node.outputs)))
    return sig


def _graph(model, family):
    """What the comparison covers, in the form the golden file stores it (JSON: tuples read back as lists)."""
    g = {"inputs": [t.name for t in model.inputs], "nodes": _signature(model)}
    if family == "retrieval":
        for attr in ("user_input", "user_embedding", "item_input", "item_embedding"):
            assert hasattr(model, attr)
        g["item_embedding_shape"] = tuple(model.item_embedding.shape)
    return json.loads(json.dumps(g))


def _groups(kind):
    from handyrec_b200.features import EmbdFeatureGroup, FeatureGroup, FeaturePool

    user, item = _features()
    pool = FeaturePool()
    if kind == "deepfm":
        feats = [f for f in user if type(f).__name__ != "DenseFeature"] + item[:1]
        dnn_feats = user + item[:1]
        return FeatureGroup("fm", feats, pool), FeatureGroup("dnn", dnn_feats, pool)
    if kind == "din":
        seq = [f for f in user if type(f).__name__ == "SparseSeqFeature"]
        other = [f for f in user if type(f).__name__ != "SparseSeqFeature"]
        return FeatureGroup("seq", seq, pool), FeatureGroup("other", other, pool)
    if kind == "rank":
        return FeatureGroup("user", user, pool), FeatureGroup("item", item, pool)
    values = {"movie_id": np.arange(50), "genres": np.random.RandomState(0).randint(0, 19, (50, 3))}
    item_group = EmbdFeatureGroup("item", "movie_id", item, pool, values, embd_dim=8)
    return FeatureGroup("user", user, pool), item_group


CASES = [
    ("deepfm", "ranking", "DeepFM", dict(dnn_hidden_units=(16, 8, 1)), {}),
    ("din", "ranking", "DIN", dict(dnn_hidden_units=(16, 8), lau_dnn_hidden_units=(8, 1)), {}),
    ("rank", "ranking", "YouTubeRankDNN", dict(dnn_hidden_units=(16, 8)), {}),
    ("retrieval", "retrieval", "DSSM", dict(user_dnn_hidden_units=(16, 8), item_dnn_hidden_units=(16, 8), num_sampled=3), dict(lazy_catalogue=False)),
    ("retrieval", "retrieval", "DSSM", dict(user_dnn_hidden_units=(16, 8), item_dnn_hidden_units=(16, 8), num_sampled=3, cos_sim=True), {}),
    ("retrieval", "retrieval", "YouTubeMatchDNN", dict(dnn_hidden_units=(16, 8), num_sampled=3), dict(lazy_catalogue=False)),
]


def _key(name, kw):
    return name + json.dumps(kw, sort_keys=True)


def _reference_graph(family, name, kw, kind):
    ref_ctor = getattr(importlib.import_module("handyrec.models." + family), name)  # the reference's package __init__ imports nothing
    assert ref_ctor.__code__.co_filename.startswith(REF)  # really the reference's file
    return _graph(ref_ctor(*_groups(kind), **kw), family)


@pytest.mark.parametrize("kind,family,name,kw,ours_kw", CASES)
def test_reference_model_files_build_the_same_graph(ref_models, kind, family, name, kw, ours_kw):
    import handyrec_b200.models as ours

    with open(GOLDEN) as f:
        want = json.load(f)[_key(name, kw)]
    if ref_models is not None:
        assert _reference_graph(family, name, kw, kind) == want
    assert _graph(getattr(ours, name)(*_groups(kind), **kw, **ours_kw), family) == want


def test_reference_deepfm_is_lowered_onto_the_fused_engine(ref_models):
    """`compile()` recognises the graph the reference's DeepFM.py builds (shared FM / DNN features) and binds the fused engine;
    a DNN with BatchNorm keeps the layer-by-layer path.  Without a checkout the graph comes from this package's DeepFM, which the
    test above holds to the reference's."""
    from handyrec_b200.features import FeatureGroup, FeaturePool
    from handyrec_b200.lowering import match_deepfm
    from handyrec_b200.models import DeepFM

    user, item = _features()
    feats = [f for f in user if type(f).__name__ != "DenseFeature"] + item[:1]
    pool = FeaturePool()
    fm, dnn = FeatureGroup("fm", feats, pool), FeatureGroup("dnn", user + item[:1], pool)
    if ref_models is not None:
        DeepFM = importlib.import_module("handyrec.models.ranking").DeepFM
    m = DeepFM(fm, dnn, dnn_hidden_units=(16, 1))
    spec = match_deepfm(m)
    assert spec is not None and len(spec.fields) == len(feats) and [t.name for t in spec.dense_inputs] == ["age"]
    assert [f.pool for f in spec.fields] == ["none", "none", "none", "mean"] and spec.fields[3].seq_len == 4  # sparse first, then sequences
    pool2 = FeaturePool()
    m_bn = DeepFM(FeatureGroup("fm", feats, pool2), FeatureGroup("dnn", user + item[:1], pool2), dnn_hidden_units=(16, 1), dnn_bn=True)
    assert match_deepfm(m_bn) is None
    pool3 = FeaturePool()  # different feature lists in the two groups: two lookups are needed, no fusion
    m_diff = DeepFM(FeatureGroup("fm", feats[:2], pool3), FeatureGroup("dnn", user + item[:1], pool3), dnn_hidden_units=(16, 1))
    assert match_deepfm(m_diff) is None


if __name__ == "__main__":
    REF = sys.argv[1] if len(sys.argv) > 1 else REF
    if not _is_checkout(REF):
        raise SystemExit("usage: python -m tests.test_compat_cpu /path/to/HandyRec  (a checkout of the reference)")
    from handyrec_b200 import compat

    compat.install(REF)
    graphs = {_key(name, kw): _reference_graph(family, name, kw, kind) for kind, family, name, kw, _ in CASES}
    with open(GOLDEN, "w") as f:  # one graph per line
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(g)}" for k, g in graphs.items()) + "\n}\n")
    print(f"wrote {GOLDEN}: {len(graphs)} graphs from {REF}")
