"""CPU: Keras Adagrad -- the oracle against hand-computed steps, the optimiser object, the C ABI declarations and the lowering
(no GPU)."""
import math
import re

import numpy as np
import pytest
import torch

from oracle.optim_ref import adagrad_dense, adagrad_sparse


def test_oracle_known_answer_over_two_steps():
    """var (1, -2), accum 0.1, lr 0.1: step 1 g = (0.5, 0), step 2 g = (-1, 2).
    step 1: acc = (0.35, 0.1); var0 = 1 - 0.1*0.5/sqrt(0.35); var1 unchanged (g = 0).
    step 2: acc = (1.35, 4.1); var0 += 0.1/sqrt(1.35); var1 = -2 - 0.2/sqrt(4.1)."""
    var, acc = torch.tensor([1.0, -2.0], dtype=torch.float64), torch.full((2,), 0.1, dtype=torch.float64)
    var, acc = adagrad_dense(var, acc, [0.5, 0.0], lr=0.1, eps=1e-7)
    np.testing.assert_allclose(acc.numpy(), [0.35, 0.1], rtol=1e-15)
    np.testing.assert_allclose(var.numpy(), [0.9154845888128602, -2.0], rtol=1e-13)
    var, acc = adagrad_dense(var, acc, [-1.0, 2.0], lr=0.1, eps=1e-7)
    np.testing.assert_allclose(acc.numpy(), [1.35, 4.1], rtol=1e-15)
    np.testing.assert_allclose(var.numpy(), [1.0015508779878406, -2.0987729547869103], rtol=1e-13)
    # eps sits outside the square root: with acc = 0 and g = 1 the step is lr / (1 + eps), not lr / sqrt(1 + eps)
    v, _ = adagrad_dense([0.0], [0.0], [1.0], lr=1.0, eps=0.5)
    assert float(v[0]) == -1.0 / 1.5
    # l2: g' = g + l2_scale * var
    v, a = adagrad_dense([2.0], [0.0], [0.0], lr=1.0, eps=0.0, l2_scale=0.25)
    assert float(a[0]) == 0.25 and float(v[0]) == 1.0


def test_oracle_sparse_sums_duplicates_then_steps_the_listed_rows():
    var = torch.arange(8.0).reshape(4, 2)
    acc = torch.full((4, 2), 0.1)
    vals = torch.tensor([[1.0, 2.0], [3.0, -1.0], [0.5, 0.5]])
    v, a = adagrad_sparse(var, acc, [2, 2, 0], vals, lr=0.1)
    dense_g = torch.zeros(4, 2)
    dense_g[2] = vals[0] + vals[1]
    dense_g[0] = vals[2]
    vd, ad = adagrad_dense(var, acc, dense_g, lr=0.1)
    assert torch.equal(v, vd) and torch.equal(a, ad)  # untouched rows: g = 0 leaves var and accum alone, so sparse == dense
    assert torch.equal(v[[1, 3]], var[[1, 3]].double()) and torch.equal(a[[1, 3]], acc[[1, 3]].double())
    assert math.isclose(float(a[2, 0]), 0.1 + 16.0)


def test_adagrad_defaults_and_negative_initial_value():
    from handyrec_b200 import keras_lite as KL

    opt = KL.Adagrad()
    assert opt.lr == 0.001 and opt.initial_accumulator_value == 0.1 and opt.eps == 1e-7
    assert KL.Adagrad(lr=0.5).lr == 0.5 and KL.Adagrad(0.2).lr == 0.2
    assert KL.Adagrad(initial_accumulator_value=0.0).initial_accumulator_value == 0.0
    with pytest.raises(ValueError):
        KL.Adagrad(initial_accumulator_value=-0.1)


def test_compat_shim_exposes_adagrad():
    from handyrec_b200 import compat
    from handyrec_b200 import keras_lite as KL

    tf = compat._tf_module()  # the module install() places in sys.modules as `tensorflow`
    assert tf.keras.optimizers.Adagrad is KL.Adagrad


def test_header_declares_adagrad():
    from handyrec_b200 import _lib

    protos = _lib.parse_header()
    assert "hrb_adagrad_step" in protos and "hrb_adagrad_step_multi" in protos
    assert len(protos["hrb_adagrad_step"][1]) == 8 and len(protos["hrb_adagrad_step_multi"][1]) == 9
    text = open(_lib.HEADER).read()
    assert re.search(r"HRB_OPT_ADAGRAD\s*=\s*2\b", text)
    assert _lib.OPT_ADAGRAD == 2


def test_deepfm_compiled_with_adagrad_gets_the_fused_binding(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # graph construction and lowering only
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
    from handyrec_b200.models import DeepFM

    torch.manual_seed(3)
    sparse = [SparseFeature(f"C{i}", v, 8) for i, v in enumerate((50, 7000, 11))]
    pool = FeaturePool()
    m = DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", [DenseFeature("I0")] + sparse, pool, l2_embd=0.0),
               dnn_hidden_units=(8, 1))
    m.compile(optimizer=KL.Adagrad(0.05), loss=KL.binary_crossentropy)
    assert m._fused is not None
