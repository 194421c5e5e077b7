"""CPU: Keras Ftrl -- the oracle against hand-computed steps, the optimiser object, the C ABI declarations, the lowering and the
compat shim (no GPU)."""
import math
import re

import pytest
import torch

from oracle.ftrl_ref import ftrl_dense, ftrl_sparse, kernel_l2


def _one(g, w=1.0, acc=0.1, lin=0.0, lr=0.1, **kw):
    v, a, l = ftrl_dense([w], [acc], [lin], [g], lr, **kw)
    return float(v[0]), float(a[0]), float(l[0])


def test_oracle_lr_power_minus_half():
    """w 1, acc 0.1, g 0.5, lr 0.1: acc' = 0.35; linear = 0.5 - (sqrt(0.35) - sqrt(0.1)) / 0.1; w = -linear / (sqrt(0.35) / 0.1)."""
    w, a, l = _one(0.5)
    lin = 0.5 - (math.sqrt(0.35) - math.sqrt(0.1)) / 0.1
    assert math.isclose(a, 0.35, rel_tol=1e-15) and math.isclose(l, lin, rel_tol=1e-13)
    assert math.isclose(w, -lin / (math.sqrt(0.35) / 0.1), rel_tol=1e-13)


def test_oracle_lr_power_zero_and_minus_one():
    # lr_power 0: p(a) = 1, so linear = g and y = 1 / lr
    w, a, l = _one(0.5, lr_power=0.0)
    assert (l, a) == (0.5, 0.35) and math.isclose(w, -0.05, rel_tol=1e-15)
    # lr_power -1: p(a) = a; linear = 0.5 - (0.35 - 0.1) / 0.1 = -2; y = 0.35 / 0.1 = 3.5
    w, a, l = _one(0.5, lr_power=-1.0)
    assert math.isclose(l, -2.0, rel_tol=1e-14) and math.isclose(w, 2.0 / 3.5, rel_tol=1e-14)


def test_oracle_l1_zeroes_small_linear():
    w, _, l = _one(0.5, lr_power=0.0, l1=0.6)  # |linear| = 0.5 <= l1
    assert l == 0.5 and w == 0.0
    w, _, _ = _one(0.5, lr_power=0.0, l1=0.2)  # (l1 - 0.5) / 10
    assert math.isclose(w, -0.03, rel_tol=1e-14)


def test_oracle_l2_shrinkage_enters_linear_not_the_accumulator():
    """g_s = 0.5 + 2 * 0.25 * 1 = 1 goes into linear; the accumulator takes the un-shrunk g."""
    w, a, l = _one(0.5, lr_power=0.0, l2_shrinkage=0.25)
    assert a == 0.35 and l == 1.0 and math.isclose(w, -0.1, rel_tol=1e-15)


def test_oracle_beta_is_folded_into_l2():
    l2 = kernel_l2(lr=0.1, l2=0.5, beta=0.2)  # 0.5 + 0.2 / (2 * 0.1)
    assert math.isclose(l2, 1.5, rel_tol=1e-15)
    w, _, _ = _one(0.5, lr_power=0.0, l2=l2)  # y = 1 / 0.1 + 2 * 1.5 = 13
    assert math.isclose(w, -0.5 / 13.0, rel_tol=1e-14)


def test_oracle_zero_accumulator_and_zero_gradient_gives_zero_not_nan():
    w, a, l = _one(0.0, w=1.0, acc=0.0)  # y = 0 and linear = 0: the select gives 0
    assert (w, a, l) == (0.0, 0.0, 0.0)


def test_oracle_sparse_steps_listed_rows_once_even_with_zero_gradient():
    var = torch.tensor([[1.0, -1.0], [0.5, 0.25], [2.0, 3.0]])
    acc, lin = torch.full((3, 2), 0.1), torch.zeros(3, 2)
    vals = torch.tensor([[0.0, 0.0], [0.25, -0.5], [0.25, 0.5]])
    v, a, l = ftrl_sparse(var, acc, lin, [0, 2, 2], vals, lr=0.1)
    assert torch.equal(v[1], var[1].double())  # not listed: untouched
    assert bool((v[0] == 0).all())  # listed with g = 0: w recomputed from linear = 0
    vd, ad, ld = ftrl_dense(var[2:], acc[2:], lin[2:], vals[1:2] + vals[2:3], 0.1)
    assert torch.equal(v[2:], vd) and torch.equal(a[2:], ad) and torch.equal(l[2:], ld)


def test_ftrl_defaults_and_value_errors():
    from handyrec_b200 import keras_lite as KL

    o = KL.Ftrl()
    assert (o.lr, o.learning_rate_power, o.initial_accumulator_value, o.l1, o.l2, o.l2_shrinkage, o.beta) == (0.001, -0.5, 0.1, 0, 0, 0, 0)
    assert o.name == "Ftrl" and o.hyper() == dict(l1=0.0, l2=0.0, lr_power=-0.5, l2_shrinkage=0.0)
    assert KL.Ftrl(0.2).lr == 0.2 and KL.Ftrl(lr=0.5).lr == 0.5
    assert math.isclose(KL.Ftrl(0.1, l2_regularization_strength=0.5, beta=0.2).kernel_l2, 1.5)
    for kw in (dict(initial_accumulator_value=-0.1), dict(learning_rate_power=0.5), dict(l1_regularization_strength=-1.0),
               dict(l2_regularization_strength=-1.0), dict(l2_shrinkage_regularization_strength=-1.0)):
        with pytest.raises(ValueError):
            KL.Ftrl(**kw)


def test_compat_shim_exposes_ftrl():
    from handyrec_b200 import compat
    from handyrec_b200 import keras_lite as KL

    assert compat._tf_module().keras.optimizers.Ftrl is KL.Ftrl


def test_header_declares_ftrl_and_the_abi_version_stays():
    from handyrec_b200 import _lib

    protos = _lib.parse_header()
    for name, n in (("hrb_ftrl_step", 14), ("hrb_ftrl_step_multi", 13), ("hrb_plan_mark_rows", 6), ("hrb_plan_pad_flags", 6),
                    ("hrb_plan_ftrl_pad_step", 4)):
        assert name in protos and len(protos[name][1]) == n, name
    text = open(_lib.HEADER).read()
    assert re.search(r"HRB_OPT_FTRL\s*=\s*3\b", text) and _lib.OPT_FTRL == 3
    assert re.search(r"#define\s+HRB_ABI_VERSION\s+1\b", text)
    # the Ftrl fields are appended: the v1 prefix of hrb_opt_params keeps its layout
    names = [f for f, _ in _lib.OptParams._fields_]
    assert names[:8] == ["opt", "lr", "beta1", "beta2", "eps", "l2_scale", "bias_corr1", "bias_corr2"]
    assert names[8:] == ["l1", "l2", "lr_power", "l2_shrinkage"]


def test_deepfm_compiled_with_ftrl_gets_the_fused_binding(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # graph construction and lowering only
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
    from handyrec_b200.layers import CustomEmbedding
    from handyrec_b200.models import DeepFM

    torch.manual_seed(3)
    sparse = [SparseFeature(f"C{i}", v, 8) for i, v in enumerate((50, 7000, 11))]
    pool = FeaturePool()
    m = DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", [DenseFeature("I0")] + sparse, pool, l2_embd=0.0),
               dnn_hidden_units=(8, 1))
    m.compile(optimizer=KL.Ftrl(0.05, l1_regularization_strength=0.01), loss=KL.binary_crossentropy)
    assert m._fused is not None
    embs = [l for l in m._all_layers() if isinstance(l, CustomEmbedding)]
    assert embs and all(l._ftrl for l in embs)  # compile told the tables which optimiser runs
