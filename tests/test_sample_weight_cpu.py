"""CPU: the sample-weight oracle against hand-worked answers, the host-side rules of sample_weight / class_weight (keys, labels,
shapes, the float64-then-float32 product), `compile(weighted_metrics=...)` naming and order, the shim, and the header entries."""
import numpy as np
import pytest

from oracle import weights_ref as W


# ---- the oracle by hand ----------------------------------------------------------------------------------------------------------
def test_weighted_loss_counts_zero_weights_in_the_batch_size():
    # logits 0: l = ln 2 for every sample, p = 1/2
    loss, d = W.weighted_bce_from_logits([0.0, 0.0, 0.0, 0.0], [1.0, 0.0, 1.0, 0.0], [2.0, 0.0, -1.0, 1.0])
    assert loss == pytest.approx((2.0 + 0.0 - 1.0 + 1.0) * np.log(2.0) / 4)  # B = 4, not sum(w) = 2
    assert d.tolist() == pytest.approx([2.0 * -0.5 / 4, 0.0, -1.0 * -0.5 / 4, 1.0 * 0.5 / 4])
    _, d2 = W.weighted_bce_from_logits([0.0, 0.0], [1.0, 0.0], [1.0, 1.0], ranks=2)
    assert d2.tolist() == pytest.approx([-0.5 / 4, 0.5 / 4])
    loss, d = W.weighted_bce_from_probs([0.5, 0.0, 0.25], [1.0, 0.0, 0.0], [3.0, 5.0, 0.0])
    assert loss == pytest.approx((3.0 * np.log(2.0) + 5.0 * -np.log(1.0 - 1e-7)) / 3)
    assert d[1] == 0.0 and d[2] == 0.0 and d[0] == pytest.approx(3.0 * -2.0 / 3)


def test_class_weight_gathers_by_truncated_label():
    assert W.class_weights([0.0, 1.0, 0.7, 1.99, -0.5], {0: 1.0, 1: 4.0}).tolist() == [1.0, 4.0, 1.0, 4.0, 1.0]
    for bad in (2.0, -1.0, np.nan):
        with pytest.raises(ValueError):
            W.class_weights([0.0, bad], {0: 1.0, 1: 4.0})
    with pytest.raises(ValueError, match="keys from 0"):
        W.class_weights([0.0], {1: 1.0, 2: 2.0})


def test_product_is_formed_in_float64_and_rounded_once():
    sw = np.array([0.1, 1.0 / 3.0], dtype=np.float64)
    cw = {0: 0.3, 1: 0.7}
    got = W.sample_weights([0.0, 1.0], sw, cw)
    want = (sw * np.array([np.float32(0.3), np.float32(0.7)], dtype=np.float64)).astype(np.float32)
    assert got.dtype == np.float32 and np.array_equal(got, want)
    # float32 sample weights: the float64 product of two float32 is exact, so this equals one float32 multiply (Keras on float32)
    sw32 = sw.astype(np.float32)
    assert np.array_equal(W.sample_weights([0.0, 1.0], sw32, cw), sw32 * np.array([0.3, 0.7], np.float32))


def test_weighted_confusion_and_accuracy_by_hand():
    p = [0.9, 0.6, 0.3, 0.8, 0.1]
    y = [1.0, 1.0, 1.0, 0.0, 0.0]
    w = [2.0, -1.0, 0.5, 3.0, 0.0]
    c = W.weighted_confusion(p, y, w, [0.5])
    assert (c["tp"][0], c["fp"][0], c["tn"][0], c["fn"][0]) == (1.0, 3.0, 0.0, 0.5)
    # correct: 0.9/1 yes, 0.6/1 yes, 0.3/1 no, 0.8/0 no, 0.1/0 yes -> 2 - 1 + 0 = 1; count 4.5
    assert W.weighted_binary_accuracy(p, y, w) == (1.0, 4.5)


# ---- the host rules ----------------------------------------------------------------------------------------------------------------
def test_host_weights_follow_the_oracle():
    from handyrec_b200.keras_lite import sample_weights

    rng = np.random.RandomState(0)
    y = (rng.rand(100) < 0.3).astype(np.float32)
    sw = rng.rand(100)
    cw = {0: 0.25, 1: 3.1}
    assert sample_weights(y) is None
    for args in ((sw, None), (None, cw), (sw, cw), (sw.reshape(-1, 1), cw), (sw.astype(np.float32), cw)):
        got = sample_weights(y, *args)
        assert got.dtype == np.float32 and got.shape == (100,)
        assert np.array_equal(got, W.sample_weights(y, None if args[0] is None else args[0].reshape(-1), args[1]))
    # negative, zero and NaN weights are taken as given
    odd = np.array([-2.0, 0.0, np.nan], np.float32)
    assert np.array_equal(sample_weights(np.zeros(3), odd), odd, equal_nan=True)


def test_host_class_weight_checks():
    from handyrec_b200.keras_lite import sample_weights

    for cw in ({1: 1.0, 2: 2.0}, {0: 1.0, 2: 2.0}, {0: 1.0, 1: 1.0, 3: 1.0}):
        with pytest.raises(ValueError, match=r"Expected `class_weight` to be a dict with keys from 0 to one less than the number of classes"):
            sample_weights(np.zeros(2), class_weight=cw)
    assert sample_weights(np.array([0.7, 1.2, -0.9]), class_weight={0: 1.0, 1: 2.0}).tolist() == [1.0, 2.0, 1.0]
    for bad in (2.0, -1.0, np.nan, np.inf):
        with pytest.raises(ValueError, match="class_weight"):
            sample_weights(np.array([0.0, bad]), class_weight={0: 1.0, 1: 2.0})
    with pytest.raises(NotImplementedError):
        sample_weights(np.eye(2), class_weight={0: 1.0, 1: 2.0})


@pytest.mark.parametrize("shape", [(5,), (5, 1), (1, 5), (5, 2), (4,), (6, 1), ()])
def test_host_sample_weight_shape(shape):
    from handyrec_b200.keras_lite import sample_weights

    sw = np.ones(shape, np.float32)
    if shape in ((5,), (5, 1)):
        assert sample_weights(np.zeros(5), sw).shape == (5,)
    else:
        with pytest.raises(ValueError, match="sample_weight"):
            sample_weights(np.zeros(5), sw)


def _tiny_model():
    from handyrec_b200 import keras_lite as K

    x = K.Input((1,), name="x")
    return K.Model(x, K.Activation("sigmoid")(x))


def test_weights_need_binary_crossentropy():
    from handyrec_b200 import keras_lite as K

    m = _tiny_model()
    m.compile(optimizer=K.SGD(0.1), loss=lambda y, p: p.mean())
    with pytest.raises(NotImplementedError, match="binary_crossentropy"):
        m.train_on_batch({"x": np.zeros((2, 1), np.float32)}, np.zeros(2), sample_weight=np.ones(2))
    with pytest.raises(NotImplementedError, match="binary_crossentropy"):
        m.fit({"x": np.zeros((2, 1), np.float32)}, np.zeros(2), class_weight={0: 1.0, 1: 1.0})
    with pytest.raises(NotImplementedError, match="temporal"):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, sample_weight_mode="temporal")


def test_refused_spellings_and_outputs():
    """Weights need one probability per sample; evaluate's sample_weight keyword and a metric's own update_state(sample_weight=)
    stay refused (evaluate takes the weights with the data)."""
    from handyrec_b200 import keras_lite as K

    x = K.Input((3,), name="x")
    wide = K.Model(x, K.Activation("sigmoid")(x))  # (batch, 3): three probabilities per sample
    with pytest.raises(NotImplementedError, match=r"\(batch, 1\)"):
        wide.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, weighted_metrics=["AUC"])
    wide.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["AUC"])
    with pytest.raises(NotImplementedError, match=r"\(batch, 1\)"):
        wide.train_on_batch({"x": np.zeros((2, 3), np.float32)}, np.zeros(2), sample_weight=np.ones(2))
    m = _tiny_model()
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy)
    with pytest.raises(NotImplementedError, match=r"evaluate\(\(x, y, sample_weight\)\)"):
        m.evaluate({"x": np.zeros((2, 1), np.float32)}, np.zeros(2), sample_weight=np.ones(2))
    with pytest.raises(NotImplementedError, match="weighted_metrics"):
        K.BinaryAccuracy().update_state([1.0, 0.0], [0.5, 0.2], sample_weight=[1.0, 2.0])


# ---- compile(weighted_metrics=...) ------------------------------------------------------------------------------------------------
def test_weighted_metric_names_and_order():
    from handyrec_b200 import keras_lite as K

    m = _tiny_model()
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["AUC", "accuracy"],
              weighted_metrics=["AUC", K.Precision(), "accuracy", K.AUC(name="roc")])
    assert m.metrics_names == ["loss", "auc", "accuracy", "weighted_auc", "precision", "weighted_accuracy", "roc"]
    ms = m._metric_set
    assert ms.weighted == [False, False, True, True, True, True]
    from handyrec_b200.metrics import WEIGHTED

    for sl, w in zip(ms.slices, ms.weighted):
        assert np.array_equal(ms.weighted_kinds[sl], ms.kinds[sl] + (WEIGHTED if w else 0))
    assert ms.kinds.max() <= 5
    # weighted metrics alone keep their names
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, weighted_metrics=["AUC", "AUC"])
    assert m.metrics_names == ["loss", "auc", "auc_1"]


def test_weighted_metric_errors():
    from handyrec_b200 import keras_lite as K

    m = _tiny_model()
    a = K.AUC()
    with pytest.raises(ValueError, match="both"):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=[a], weighted_metrics=[a])
    with pytest.raises(ValueError, match="same name"):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["AUC", K.AUC(name="weighted_auc")], weighted_metrics=["AUC"])


def test_history_keys_follow_metrics_names():
    """fit's history is keyed by metrics_names (then val_ + each): checked here through the key order fit builds."""
    from handyrec_b200 import keras_lite as K

    m = _tiny_model()
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["AUC"], weighted_metrics=["AUC"])
    assert [k for k in m._metric_set.names] == ["auc", "weighted_auc"]


def test_shim_compile_takes_weighted_metrics():
    from handyrec_b200 import compat

    compat.install(force=True)
    try:
        import tensorflow as tf

        x = tf.keras.layers.Input((1,), name="x")
        m = tf.keras.Model(x, tf.keras.layers.Activation("sigmoid")(x))
        m.compile(optimizer=tf.keras.optimizers.Adam(1e-3), loss=tf.keras.losses.binary_crossentropy, metrics=["AUC"],
                  weighted_metrics=[tf.keras.metrics.AUC()])
        assert m.metrics_names == ["loss", "auc", "weighted_auc"]
    finally:
        compat.uninstall()


def test_header_declares_the_weighted_entries():
    import ctypes

    from handyrec_b200 import _lib

    protos = _lib.parse_header()
    P, I64, I32, F = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float
    assert protos["hrb_sigmoid_bce_weighted"][1] == [P, P, P, P, I64, F, P, P, P, P]
    assert protos["hrb_clipped_bce_weighted"][1] == [P, P, P, I64, F, F, P, P, P]
    assert protos["hrb_metric_update_weighted"][1] == [P, P, P, I64, P, I32, P, P, I32, P, P, P, P]
    assert protos["hrb_metric_weighted_scratch_bytes"][1] == [I32, P]
