"""CPU: the Keras regression losses -- the float64 oracle against hand-worked values, the string identifiers of `compile`, which
(head, loss) pairs lower onto the fused engine, the loss objects' refusals, the shim and the header entries."""
import numpy as np
import pytest

from handyrec_b200 import keras_lite as K
from handyrec_b200.features import FeatureGroup, FeaturePool, SparseFeature
from oracle import losses_ref as R


# ---- 1. the oracle ------------------------------------------------------------------------------------------------------------
def test_oracle_hand_worked_values():
    y = np.array([0.0, 0.0, 0.0, 0.0, 0.0])
    p = np.array([0.5, -2.0, 1.0, -1.0, 0.0])  # inside, outside, both ties |e| == delta, zero
    assert R.per_sample("mean_squared_error", y, p[:, None]).tolist() == [0.25, 4.0, 1.0, 1.0, 0.0]
    assert R.per_sample("mean_absolute_error", y, p[:, None]).tolist() == [0.5, 2.0, 1.0, 1.0, 0.0]
    # huber, delta = 1: 0.5*0.25; 0.5*1 + 1*(2-1); the tie on both formulas = 0.5
    assert R.per_sample("huber", y, p[:, None]).tolist() == [0.125, 1.5, 0.5, 0.5, 0.0]
    # delta = 2: e = -2 sits on the tie, quadratic branch: 0.5 * 4
    assert R.per_sample("huber", y, p[:, None], delta=2.0).tolist() == [0.125, 2.0, 0.5, 0.5, 0.0]
    # MSE gradient: 2e / B
    _, g = R.compiled_loss("mean_squared_error", y, p[:, None])
    assert g[:, 0].tolist() == [2 * 0.5 / 5, -4.0 / 5, 2.0 / 5, -2.0 / 5, 0.0]


def test_oracle_gradients_at_the_kinks():
    e = np.array([0.0, 1.0, -1.0, 1.5, -0.25])
    _, d = R.elementwise("mean_absolute_error", e)
    assert d.tolist() == [0.0, 1.0, -1.0, 1.0, -1.0]  # d|e|/de = 0 at e = 0
    _, d = R.elementwise("huber", e, 1.0)
    assert d.tolist() == [0.0, 1.0, -1.0, 1.0, -0.25]  # the tie takes the quadratic branch: dl/de = e
    _, d = R.elementwise("huber", e, 0.0)
    assert d.tolist() == [0.0, 0.0, 0.0, 0.0, 0.0]


def test_oracle_label_rank_rule():
    y = np.array([1.0, 2.0, 3.0])
    p = np.array([[1.5], [2.0], [1.0]])
    yy, pp = R.match_label(y, p)
    assert yy.shape == (3, 1)
    loss, g = R.compiled_loss("mean_squared_error", y, p)
    assert loss == pytest.approx((0.25 + 0.0 + 4.0) / 3)  # a (B, B) broadcast would give a different mean
    assert g.shape == (3, 1)
    with pytest.raises(ValueError):
        R.match_label(np.zeros(3), np.zeros((3, 2)))
    # the mean over the last axis of a wider output
    assert R.per_sample("mean_absolute_error", np.zeros((2, 2)), np.array([[1.0, 3.0], [0.0, -2.0]])).tolist() == [2.0, 1.0]


def test_oracle_weighted_reduction_divides_by_the_batch_size():
    y = np.zeros(4)
    p = np.array([[1.0], [2.0], [3.0], [4.0]])
    w = np.array([1.0, 0.0, 2.0, 0.5])
    loss, g = R.compiled_loss("mean_absolute_error", y, p, w)
    assert loss == (1.0 + 0.0 + 6.0 + 2.0) / 4  # not / sum(w) = 3.5
    assert g[:, 0].tolist() == [0.25, 0.0, 0.5, 0.125]
    _, g2 = R.compiled_loss("mean_absolute_error", y, p, w, ranks=2)
    assert np.array_equal(g2, g / 2)


# ---- 2. identifiers ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,fn", [("mse", "mean_squared_error"), ("MSE", "mean_squared_error"), ("mean_squared_error", "mean_squared_error"),
                                     ("mae", "mean_absolute_error"), ("MAE", "mean_absolute_error"),
                                     ("mean_absolute_error", "mean_absolute_error"), ("binary_crossentropy", "binary_crossentropy")])
def test_loss_strings_resolve(name, fn):
    assert K.get_loss(name) is getattr(K, fn)


def test_loss_objects_pass_through_and_unknown_strings_raise():
    h = K.Huber(0.5)
    f = lambda y, p: p.mean()  # noqa: E731
    assert K.get_loss(h) is h and K.get_loss(f) is f and K.get_loss(K.mse) is K.mean_squared_error
    for bad in ("log_cosh", "msle", "poisson", "categorical_crossentropy", "Mse", "huber"):
        with pytest.raises(ValueError, match=bad):
            K.get_loss(bad)


@pytest.mark.parametrize("name,cls", [("adam", "Adam"), ("Adam", "Adam"), ("SGD", "SGD"), ("sgd", "SGD"), ("adagrad", "Adagrad"),
                                      ("AdaGrad", "Adagrad"), ("ftrl", "Ftrl"), ("FTRL", "Ftrl")])
def test_optimizer_strings_resolve_case_insensitively_with_keras_defaults(name, cls):
    opt = K.get_optimizer(name)
    assert type(opt) is getattr(K, cls)
    assert opt.lr == {"Adam": 1e-3, "SGD": 0.01, "Adagrad": 1e-3, "Ftrl": 1e-3}[cls]


def test_unknown_optimizer_string_raises():
    with pytest.raises(ValueError, match="rmsprop"):
        K.get_optimizer("rmsprop")


def test_loss_objects_refuse_what_they_do_not_implement():
    with pytest.raises(NotImplementedError):
        K.BinaryCrossentropy(from_logits=True)
    with pytest.raises(NotImplementedError):
        K.BinaryCrossentropy(label_smoothing=0.1)
    for cls in (K.BinaryCrossentropy, K.MeanSquaredError, K.MeanAbsoluteError, K.Huber):
        with pytest.raises(NotImplementedError):
            cls(reduction="sum")
        cls(reduction="auto")
        cls(reduction="sum_over_batch_size")
    assert K.builtin_loss(K.BinaryCrossentropy()) == ("binary_crossentropy", 0.0)
    assert K.builtin_loss(K.Huber(2.5)) == ("huber", 2.5)
    assert K.builtin_loss(lambda y, p: p) is None


def test_compile_resolves_strings_and_refuses_loss_weights():
    x = K.Input((1,), name="x")
    m = K.Model(x, K.Activation("sigmoid")(x))
    m.compile("Adagrad", "mae")
    assert isinstance(m.optimizer, K.Adagrad) and m.loss is K.mean_absolute_error
    with pytest.raises(ValueError, match="hinge"):
        m.compile("adam", "hinge")
    with pytest.raises(NotImplementedError, match="loss_weights"):
        m.compile("adam", "mse", loss_weights=[1.0])
    with pytest.raises(NotImplementedError, match="per-output"):
        m.compile("adam", ["mse"])


# ---- 3. lowering decisions -------------------------------------------------------------------------------------------------------
def _deepfm(task):
    from handyrec_b200.models import DeepFM

    sparse = [SparseFeature("a", 50, 8), SparseFeature("b", 7, 8)]
    pool = FeaturePool()
    return DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", sparse, pool, l2_embd=0.0), dnn_hidden_units=(8, 1),
                  task=task)


@pytest.mark.parametrize("loss", ["mse", K.MeanSquaredError(), "mae", K.MeanAbsoluteError(), K.Huber(0.3)])
def test_regression_deepfm_with_a_regression_loss_lowers(loss):
    m = _deepfm("regression")
    m.compile(K.Adam(), loss)
    assert m._fused is not None and m._fused.spec.head == "linear"
    assert m._fused.spec.loss == K.builtin_loss(K.get_loss(loss))


@pytest.mark.parametrize("task,loss", [("regression", "binary_crossentropy"), ("regression", K.BinaryCrossentropy()), ("binary", "mse"),
                                       ("binary", K.Huber()), ("regression", lambda y, p: (p - y).abs().mean())])
def test_mismatched_pairs_keep_the_layer_path(task, loss):
    m = _deepfm(task)
    m.compile(K.Adam(), loss)
    assert m._fused is None


def test_string_bce_lowers_like_the_function():
    for opt, loss in (("adam", "binary_crossentropy"), (K.Adam(), K.binary_crossentropy), ("sgd", K.BinaryCrossentropy())):
        m = _deepfm("binary")
        m.compile(opt, loss)
        assert m._fused is not None and m._fused.spec.head == "sigmoid" and m._fused.spec.loss == ("binary_crossentropy", 0.0)


def test_weights_with_a_user_loss_still_name_binary_crossentropy():
    m = _deepfm("regression")
    m.compile(K.SGD(0.1), lambda y, p: p.mean())
    with pytest.raises(NotImplementedError, match="binary_crossentropy"):
        m._weights(np.zeros(2), np.ones(2))
    m.compile(K.SGD(0.1), "mse")
    assert m._weights(np.zeros(2), np.ones(2)).tolist() == [1.0, 1.0]


def test_host_loss_matches_the_oracle():
    rng = np.random.RandomState(0)
    p, y = rng.randn(50).astype(np.float32), rng.randn(50).astype(np.float32)
    for kind in (("mean_squared_error", 0.0), ("mean_absolute_error", 0.0), ("huber", 0.7)):
        want = R.per_sample(kind[0], y, p.reshape(-1, 1), delta=kind[1])
        assert np.allclose(K.host_loss(kind, p.reshape(-1, 1), y), want, rtol=0, atol=0)


# ---- 4. shim and header --------------------------------------------------------------------------------------------------------
def test_shim_exposes_the_losses():
    from handyrec_b200 import compat

    compat.install(force=True)
    try:
        import tensorflow as tf

        L = tf.keras.losses
        assert L.mse is L.MSE is L.mean_squared_error is K.mean_squared_error
        assert L.mae is L.MAE is L.mean_absolute_error is K.mean_absolute_error
        assert L.Huber is K.Huber and L.MeanSquaredError is K.MeanSquaredError and L.MeanAbsoluteError is K.MeanAbsoluteError
        assert L.BinaryCrossentropy is K.BinaryCrossentropy and L.binary_crossentropy is K.binary_crossentropy
        assert L.get("mse") is K.mean_squared_error and isinstance(tf.keras.optimizers.get("Ftrl"), K.Ftrl)
    finally:
        compat.uninstall()


def test_header_declares_the_regression_entries():
    import ctypes

    from handyrec_b200 import _lib

    protos = _lib.parse_header()
    P, I64, I32, F, SZ = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_size_t
    assert protos["hrb_regression_loss"][1] == [I32, F, P, P, P, I64, I32, F, P, P, P, P, SZ, P]
    assert protos["hrb_regression_loss_weighted"][1] == [I32, F, P, P, P, P, I64, I32, F, P, P, P, P, SZ, P]
    assert protos["hrb_regression_loss_workspace"][1] == [I64, P]
