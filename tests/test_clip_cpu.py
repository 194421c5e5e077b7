"""CPU: Keras gradient clipping -- the optimizers' arguments, the compile-time refusals, the float64 oracle on hand-worked cases and
the C ABI declarations (no GPU)."""
import math

import numpy as np
import pytest
import torch

from oracle.clip_ref import IndexedSlices, clip_gradients, concat_slices, densify


@pytest.fixture(autouse=True)
def _weights_on_the_host(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # graph construction and lowering only


def _optimizers():
    from handyrec_b200 import keras_lite as KL

    return [KL.SGD, KL.Adam, KL.Adagrad, KL.Ftrl]


# ---- arguments (OptimizerV2.__init__) -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("i", range(4))
def test_clip_arguments_default_to_none_and_are_exposed(i):
    cls = _optimizers()[i]
    o = cls()
    assert (o.clipnorm, o.clipvalue, o.global_clipnorm) == (None, None, None)
    o = cls(0.1, clipnorm=1.0, clipvalue=0.5)
    assert (o.clipnorm, o.clipvalue, o.global_clipnorm) == (1.0, 0.5, None)
    o = cls(0.1, global_clipnorm=2.0, clipvalue=0.0)
    assert (o.clipnorm, o.clipvalue, o.global_clipnorm) == (None, 0.0, 2.0)


@pytest.mark.parametrize("i", range(4))
def test_clip_argument_errors(i):
    cls = _optimizers()[i]
    for name in ("clipnorm", "clipvalue", "global_clipnorm"):
        with pytest.raises(ValueError, match=f"Expected {name} >= 0"):
            cls(**{name: -1.0})
    with pytest.raises(ValueError, match="both `clipnorm` and `global_clipnorm`"):
        cls(clipnorm=1.0, global_clipnorm=1.0)
    with pytest.raises(TypeError):
        cls(clip_norm=1.0)


def test_clip_args_summary():
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.clip import clip_args

    assert clip_args(KL.Adam()) is None
    assert clip_args(KL.SGD(clipvalue=1)) == (1.0, None, None)
    assert clip_args(KL.Ftrl(global_clipnorm=3)) == (None, None, 3.0)


# ---- compile refusals ---------------------------------------------------------------------------------------------------------
class _FakeComm:
    def __init__(self, rank, n):
        self.rank, self.N = rank, n


def _deepfm(vocabs=(50, 7000, 11), l2=0.0):
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
    from handyrec_b200.models import DeepFM

    torch.manual_seed(3)
    sparse = [SparseFeature(f"C{i}", v, 8) for i, v in enumerate(vocabs)]
    pool = FeaturePool()
    return DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=l2), FeatureGroup("dnn", [DenseFeature("I0")] + sparse, pool, l2_embd=l2),
                  dnn_hidden_units=(8, 1))


@pytest.mark.parametrize("fuse", [True, False])
def test_multi_gpu_compile_with_clipping_is_refused(fuse):
    from handyrec_b200 import keras_lite as KL

    for kw in (dict(clipnorm=1.0), dict(clipvalue=0.1), dict(global_clipnorm=1.0)):
        m = _deepfm()
        m.fuse = fuse
        with pytest.raises(ValueError, match="multi-GPU"):
            m.compile(optimizer=KL.Adam(1e-3, **kw), loss=KL.binary_crossentropy, distribute=_FakeComm(0, 2))
        m.compile(optimizer=KL.Adam(1e-3, **kw), loss=KL.binary_crossentropy, distribute=_FakeComm(0, 1))  # one rank: fine
    m = _deepfm()
    with KL.ShardedTables(_FakeComm(0, 2), min_rows=1000):
        with pytest.raises(ValueError, match="multi-GPU"):
            m.compile(optimizer=KL.SGD(0.1, clipnorm=1.0), loss=KL.binary_crossentropy)
    m.compile(optimizer=KL.Adam(1e-3), loss=KL.binary_crossentropy, distribute=_FakeComm(0, 2))  # no clip argument: as before


def test_clipping_with_l2_on_a_touched_rows_table_is_refused():
    from handyrec_b200 import keras_lite as KL

    # fused path: tables above dense_table_max_rows take the touched-rows update
    m = _deepfm(l2=1e-4)
    m.dense_table_max_rows = 1000
    with pytest.raises(ValueError, match="touched-rows update"):
        m.compile(optimizer=KL.Adagrad(0.1, clipnorm=1.0), loss=KL.binary_crossentropy)
    m.compile(optimizer=KL.Adagrad(0.1), loss=KL.binary_crossentropy)  # without a clip argument it compiles as before
    m = _deepfm(l2=1e-4)
    m.dense_table_max_rows = 10_000  # every table dense-updated: clipping is exact
    m.compile(optimizer=KL.Adagrad(0.1, clipnorm=1.0), loss=KL.binary_crossentropy)
    assert m._fused is not None
    # layer path: tables of at least SPARSE_UPDATE_MIN_ROWS rows
    from handyrec_b200.layers import CustomEmbedding

    m = _deepfm(l2=1e-4)
    m.fuse = False
    m.compile(optimizer=KL.SGD(0.1, clipvalue=1.0), loss=KL.binary_crossentropy)
    big = next(l for l in m._all_layers() if isinstance(l, CustomEmbedding) and l.input_dim == 7000)
    big.SPARSE_UPDATE_MIN_ROWS = 5000
    with pytest.raises(ValueError, match="touched-rows update"):
        m.compile(optimizer=KL.SGD(0.1, clipvalue=1.0), loss=KL.binary_crossentropy)
    m = _deepfm(l2=0.0)  # no regulariser: the touched-rows update clips exactly
    m.fuse = False
    next(l for l in m._all_layers() if isinstance(l, CustomEmbedding) and l.input_dim == 7000).SPARSE_UPDATE_MIN_ROWS = 5000
    m.compile(optimizer=KL.SGD(0.1, global_clipnorm=1.0), loss=KL.binary_crossentropy)


# ---- the oracle ----------------------------------------------------------------------------------------------------------------
def test_oracle_clipnorm_of_two_lookups_with_a_duplicate_is_not_the_merged_norm():
    """One table looked up twice (FM and DNN group), id 2 in both lookups and twice in the first.  Keras' norm covers the five
    concatenated value rows; the merged (deduplicated) gradient has a different norm and so a different clipped result."""
    a = IndexedSlices(np.array([2, 2, 0]), np.array([[3.0, 0.0], [0.0, 4.0], [1.0, 0.0]]))
    b = IndexedSlices(np.array([2, 1]), np.array([[-3.0, 0.0], [0.0, 2.0]]))
    g = concat_slices(a, b)
    assert list(g.indices) == [2, 2, 0, 2, 1]
    norm = math.sqrt(9 + 16 + 1 + 9 + 4)  # sqrt(39)
    (out,) = clip_gradients([g], clipnorm=1.0)
    np.testing.assert_allclose(densify(out, 3), densify(g, 3) / norm, rtol=1e-15)
    merged = densify(g, 3)  # row 2 = [0, 4]: norm sqrt(16 + 1 + 4) = sqrt(21)
    (out_m,) = clip_gradients([merged], clipnorm=1.0)
    np.testing.assert_allclose(out_m, merged / math.sqrt(21), rtol=1e-15)
    assert not np.allclose(densify(out, 3), out_m)


def test_oracle_clipvalue_is_per_position_before_duplicates_are_summed():
    g = IndexedSlices(np.array([0, 0]), np.array([[2.0], [2.0]]))
    (out,) = clip_gradients([g], clipvalue=1.0)
    assert densify(out, 1)[0, 0] == 2.0  # each position clamped to 1, then summed
    (dense,) = clip_gradients([densify(g, 1)], clipvalue=1.0)
    assert dense[0, 0] == 1.0


def test_oracle_clipvalue_runs_before_clipnorm():
    g = np.array([3.0, 4.0])
    (out,) = clip_gradients([g], clipvalue=1.0, clipnorm=1.0)  # [1, 1] first, norm sqrt(2)
    np.testing.assert_allclose(out, [1 / math.sqrt(2)] * 2, rtol=1e-15)
    (norm_first,) = clip_gradients([np.clip(g / 5.0, -1, 1)])  # the other order would give [0.6, 0.8]
    assert not np.allclose(out, norm_first)


def test_oracle_norm_modes():
    g1, g2 = np.array([3.0, 4.0]), np.array([[12.0]])
    o1, o2 = clip_gradients([g1, g2], clipnorm=5.0)  # per variable: g1 at the bound (s = 1 exactly), g2 scaled to 5
    assert np.array_equal(o1, g1) and o2[0, 0] == 5.0
    o1, o2 = clip_gradients([g1, g2], global_clipnorm=6.5)  # global norm 13
    np.testing.assert_allclose(o1, g1 / 2, rtol=1e-15)
    np.testing.assert_allclose(o2, g2 / 2, rtol=1e-15)
    o1, none = clip_gradients([g1, None], global_clipnorm=100.0)
    assert np.array_equal(o1, g1) and none is None


def test_oracle_global_norm_with_inf_makes_every_gradient_nan():
    o1, o2 = clip_gradients([np.array([1.0, np.inf]), np.array([2.0])], global_clipnorm=1.0)
    assert np.isnan(o1).all() and np.isnan(o2).all()


def test_oracle_zero_clip():
    (z,) = clip_gradients([np.zeros(3)], clipnorm=0.0)  # 0 / max(0, 0): NaN, as TF
    assert np.isnan(z).all()
    (z,) = clip_gradients([np.array([1.0, -2.0])], clipnorm=0.0)  # 0 / 2
    assert np.array_equal(z, [0.0, -0.0])
    (z,) = clip_gradients([np.array([1.0, -2.0])], clipvalue=0.0)
    assert np.array_equal(z, [0.0, 0.0])


# ---- ABI ------------------------------------------------------------------------------------------------------------------------
def test_header_declares_the_clip_entries_and_the_build_compiles_them():
    from handyrec_b200 import _lib, build

    protos = _lib.parse_header()
    for name, n in (("hrb_clip_workspace_bytes", 2), ("hrb_clip_prepare_multi", 11), ("hrb_plan_clip_grads", 13), ("hrb_clip_scales", 6),
                    ("hrb_clip_apply_multi", 6), ("hrb_plan_clip_apply", 6)):
        assert name in protos and len(protos[name][1]) == n, name
    assert "clip.cu" in build.SOURCES
