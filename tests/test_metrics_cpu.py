"""CPU: the Keras metrics oracle against hand-worked cases and the exact Mann-Whitney AUC, the float32 accumulation rule, the metric
objects' defaults and errors, `compile(metrics=...)`, the shim's tensorflow.keras.metrics and the header entries."""
import numpy as np
import pytest
from scipy.stats import rankdata

from oracle import metrics_ref as R

# six samples worked by hand: labels and predictions, thresholds [-eps, 0.25, 0.5, 0.75, 1+eps] (num_thresholds=5)
Y6 = np.array([1, 0, 1, 1, 0, 0], dtype=np.float32)
P6 = np.array([0.9, 0.8, 0.6, 0.3, 0.2, 0.1], dtype=np.float32)
# counts per threshold:  -eps   0.25  0.5  0.75  1+eps
TP6, FP6 = [3, 3, 2, 1, 0], [3, 1, 1, 1, 0]
TN6, FN6 = [0, 2, 2, 2, 3], [0, 0, 1, 2, 3]


def test_oracle_counts_six_samples_by_hand():
    c = R.confusion_counts(P6, Y6, R.auc_thresholds(5))
    assert c["tp"].tolist() == TP6 and c["fp"].tolist() == FP6 and c["tn"].tolist() == TN6 and c["fn"].tolist() == FN6


def test_oracle_auc_six_samples_by_hand():
    # ROC points (fpr, tpr): (1,1) (1/3,1) (1/3,2/3) (1/3,1/3) (0,0)
    # interpolation: (2/3)(1) + (1/3)(1/6) = 13/18; minoring: (2/3)(1) + (1/3)(0) = 2/3; majoring: (2/3)(1) + (1/3)(1/3) = 7/9
    args = (TP6, FP6, TN6, FN6)
    assert R.auc_result(*args, "ROC", "interpolation") == pytest.approx(13 / 18)
    assert R.auc_result(*args, "ROC", "minoring") == pytest.approx(2 / 3)
    assert R.auc_result(*args, "ROC", "majoring") == pytest.approx(7 / 9)
    # PR points (recall, precision): (1, 1/2) (1, 3/4) (2/3, 2/3) (1/3, 1/2) (0, 0 by div_no_nan)
    # minoring (1/3)(2/3) + (1/3)(1/2) + (1/3)(0) = 7/18; majoring (1/3)(3/4) + (1/3)(2/3) + (1/3)(1/2) = 23/36
    assert R.auc_result(*args, "PR", "minoring") == pytest.approx(7 / 18)
    assert R.auc_result(*args, "PR", "majoring") == pytest.approx(23 / 36)
    # interpolate_pr_auc, interval by interval (p = tp + fp = [6, 4, 3, 2, 0], tp + fn = 3):
    #   [0]: dtp = 0 -> 0
    #   [1]: dtp = 1, dp = 1, slope 1, intercept 2 - 3 = -1, ratio 4/3 -> (1 - ln 4/3) / 3
    #   [2]: dtp = 1, dp = 1, slope 1, intercept 1 - 2 = -1, ratio 3/2 -> (1 - ln 3/2) / 3
    #   [3]: p[4] = 0 -> ratio 1; slope 1/2, intercept 0 -> (1/2)(1) / 3
    want = (1 - np.log(4 / 3)) / 3 + (1 - np.log(1.5)) / 3 + 0.5 / 3
    assert R.auc_result(*args, "PR", "interpolation") == pytest.approx(want)
    assert R.interpolate_pr_auc(TP6, FP6, FN6) == pytest.approx(want)


@pytest.mark.parametrize("kind,want", [("perfect", 1.0), ("reversed", 0.0), ("equal", 0.5)])
def test_oracle_roc_auc_known_answers(kind, want):
    y = np.array([0, 0, 0, 1, 1, 1, 1], dtype=np.float32)
    p = {"perfect": np.linspace(0.1, 0.9, 7), "reversed": np.linspace(0.9, 0.1, 7), "equal": np.full(7, 0.4)}[kind].astype(np.float32)
    c = R.confusion_counts(p, y, R.auc_thresholds(200))
    assert R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"]) == pytest.approx(want, abs=1e-12)


def test_oracle_roc_auc_converges_to_mann_whitney():
    """10 001 thresholds, 1e5 samples: the trapezoid over the thresholds is the exact AUC up to the pairs that share a bucket."""
    rng = np.random.RandomState(0)
    n = 100_000
    y = (rng.rand(n) < 0.3).astype(np.float32)
    p = np.clip(rng.beta(2, 5, n) + 0.15 * y, 0, 1).astype(np.float32)
    c = R.confusion_counts(p, y, R.auc_thresholds(10_001))
    got = R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"])
    r = rankdata(p)
    npos, nneg = int(y.sum()), int(n - y.sum())
    exact = (r[y == 1].sum() - npos * (npos + 1) / 2) / (npos * nneg)
    # pairs inside one bucket are counted as half-right by the trapezoid: the error is at most their share
    bucket = np.searchsorted(R.auc_thresholds(10_001), p, side="left")
    pos_b = np.bincount(bucket[y == 1], minlength=10_003).astype(np.float64)
    neg_b = np.bincount(bucket[y == 0], minlength=10_003).astype(np.float64)
    bound = 0.5 * float((pos_b * neg_b).sum()) / (npos * nneg)
    assert abs(got - exact) <= bound + 1e-12
    assert abs(got - exact) < 1e-3


def test_float32_accumulation_rounds_past_2_24():
    v = np.float32(2**24)
    assert R.accumulate_f32(v, 1) == np.float32(2**24)  # 2^24 + 1 is not a float32: ties to even
    assert R.accumulate_f32(v, 3) == np.float32(2**24 + 4)
    assert R.accumulate_f32(np.float32(2**24 - 1), 1) == np.float32(2**24)
    acc = np.float32(0)
    for _ in range(300):
        acc = R.accumulate_f32(acc, 65_536 - 7)
    exact = 300 * (65_536 - 7)
    assert exact > 2**24 and float(acc) != exact  # the running sum has rounded


def test_labels_are_cast_to_bool_and_accuracy_needs_exact_labels():
    p = np.array([0.7, 0.7, 0.7, 0.2], dtype=np.float32)
    y = np.array([0.3, np.nan, 1.0, 0.0], dtype=np.float32)
    c = R.confusion_counts(p, y, [0.5])
    assert c["tp"].tolist() == [3] and c["fp"].tolist() == [0] and c["tn"].tolist() == [1] and c["fn"].tolist() == [0]
    assert R.binary_accuracy_counts(p, y) == (2, 4)  # 0.3 and NaN are never correct


# ---- the metric objects ----------------------------------------------------------------------------------------------------------
def test_auc_defaults_and_thresholds():
    from handyrec_b200.metrics import AUC

    m = AUC()
    assert m.name == "auc" and m.num_thresholds == 200 and m.curve == "ROC" and m.summation_method == "interpolation"
    assert np.array_equal(m._thresholds, R.auc_thresholds(200))
    assert m._thresholds[0] == np.float32(-1e-7) and m._thresholds[-1] == np.float32(1 + 1e-7) > 1.0
    e = AUC(thresholds=[0.7, 0.2, 0.4], curve="pr", summation_method="Majoring", name="x")
    assert e.num_thresholds == 5 and e.curve == "PR" and e.summation_method == "majoring" and e.name == "x"
    assert np.array_equal(e._thresholds, R.auc_thresholds(thresholds=[0.7, 0.2, 0.4]))


def test_auc_errors():
    from handyrec_b200.metrics import AUC

    with pytest.raises(ValueError, match=r"^`num_thresholds` must be > 1\.$"):
        AUC(num_thresholds=1)
    with pytest.raises(ValueError, match=r'^Invalid AUC curve value "ROCX"\.$'):
        AUC(curve="ROCX")
    with pytest.raises(ValueError, match=r'^Invalid AUC summation method value "trapezoid"\.$'):
        AUC(summation_method="trapezoid")
    for curve in ("Roc", "pR"):  # AUCCurve.from_str takes "roc" / "ROC" / "pr" / "PR" only
        with pytest.raises(ValueError, match="Invalid AUC curve value"):
            AUC(curve=curve)
    for method in ("MAJORING", "minOring"):  # the lower-case or capitalised spellings only
        with pytest.raises(ValueError, match="Invalid AUC summation method value"):
            AUC(summation_method=method)
    assert AUC(curve="PR", summation_method="Interpolation").summation_method == "interpolation"
    for kw in (dict(multi_label=True), dict(num_labels=3), dict(label_weights=[1.0]), dict(from_logits=True)):
        with pytest.raises(NotImplementedError):
            AUC(**kw)


def test_precision_recall_accuracy_defaults_and_errors():
    from handyrec_b200.metrics import BinaryAccuracy, Precision, Recall

    assert Precision().thresholds == [0.5] and Precision().name == "precision" and Recall().name == "recall"
    assert Recall(thresholds=0.3).thresholds == [0.3] and Precision(thresholds=[0.3, 0.7]).thresholds == [0.3, 0.7]
    with pytest.raises(ValueError, match=r"^Threshold values must be in \[0, 1\]\. Invalid values: \[1\.5\]$"):
        Precision(thresholds=[0.2, 1.5])
    with pytest.raises(ValueError, match=r"Threshold values must be in \[0, 1\]"):
        Recall(thresholds=-0.1)
    for cls in (Precision, Recall):
        with pytest.raises(NotImplementedError):
            cls(top_k=2)
        with pytest.raises(NotImplementedError):
            cls(class_id=0)
    a = BinaryAccuracy()
    assert a.name == "binary_accuracy" and a.threshold == 0.5
    with pytest.raises(NotImplementedError):
        a.update_state([1.0], [0.5], sample_weight=[1.0])


def test_results_from_variables_follow_keras():
    """result() on given variables (no device involved): the float32 formulas against the float64 oracle."""
    from handyrec_b200.metrics import AUC, BinaryAccuracy, Precision, Recall

    for curve in ("ROC", "PR"):
        for s in ("interpolation", "minoring", "majoring"):
            m = AUC(num_thresholds=5, curve=curve, summation_method=s)
            v = np.array(TP6 + FP6 + TN6 + FN6, dtype=np.float32)
            assert m._result(v) == pytest.approx(R.auc_result(TP6, FP6, TN6, FN6, curve, s), rel=1e-6)
    assert Precision()._result(np.array([2, 1], np.float32)) == pytest.approx(2 / 3)
    assert Recall()._result(np.array([0, 0], np.float32)) == 0.0  # div_no_nan
    r = Recall(thresholds=[0.3, 0.7])._result(np.array([2, 1, 1, 2], np.float32))
    assert r.shape == (2,) and r.tolist() == pytest.approx([2 / 3, 1 / 3])
    assert BinaryAccuracy()._result(np.array([3, 4], np.float32)) == pytest.approx(0.75)


def test_metric_set_union_and_descriptors():
    from handyrec_b200.metrics import AUC, COUNT, CORRECT, FN, TP, BinaryAccuracy, MetricSet, Recall

    a, r, b = AUC(num_thresholds=3), Recall(thresholds=[0.5, 0.7]), BinaryAccuracy()
    s = MetricSet([a, r, b])
    assert s.thresholds.tolist() == [np.float32(-1e-7), 0.5, np.float32(0.7), np.float32(1 + 1e-7)]
    assert s.slices[1] == slice(12, 16) and s.kinds[12:16].tolist() == [TP, TP, FN, FN] and s.thr_index[12:16].tolist() == [1, 2, 1, 2]
    assert s.kinds[16:].tolist() == [CORRECT, COUNT] and s.thr_index[16] == 1
    with pytest.raises(ValueError, match="8192"):
        MetricSet([AUC(num_thresholds=8000), AUC(num_thresholds=300)])
    MetricSet([AUC(num_thresholds=8192)])


# ---- compile --------------------------------------------------------------------------------------------------------------------
def _tiny_model():
    from handyrec_b200 import keras_lite as K

    x = K.Input((3,), name="x")
    return K.Model(x, K.Activation("sigmoid")(x))


def test_compile_maps_strings_and_dedupes_names():
    from handyrec_b200 import keras_lite as K

    m = _tiny_model()
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["AUC", "accuracy", "acc", "binary_accuracy", K.AUC(),
                                                                          K.Precision(), "Precision", "Recall", K.Recall(thresholds=[0.3, 0.7])])
    assert m.metrics_names == ["loss", "auc", "accuracy", "acc", "binary_accuracy", "auc_1", "precision", "precision_1", "recall",
                               "recall_1"]
    assert [type(x).__name__ for x in m.metrics] == ["AUC", "BinaryAccuracy", "BinaryAccuracy", "BinaryAccuracy", "AUC", "Precision",
                                                     "Precision", "Recall", "Recall"]
    assert m._metric_set is not None and len(m._metric_set) == 9
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy)
    assert m.metrics == [] and m.metrics_names == ["loss"] and m._metric_set is None


def test_compile_errors():
    from handyrec_b200 import keras_lite as K

    m = _tiny_model()
    with pytest.raises(ValueError, match="Unknown metric"):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["mse"])
    with pytest.raises(ValueError, match="8192"):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=[K.AUC(num_thresholds=9000)])
    with pytest.raises(NotImplementedError):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, weighted_metrics=["AUC"])
    a = K.AUC()
    with pytest.raises(ValueError, match="twice"):
        m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=[a, a])


def test_shim_exposes_keras_metrics():
    from handyrec_b200 import compat
    from handyrec_b200 import keras_lite as K

    compat.install(force=True)
    try:
        import tensorflow as tf
        from tensorflow.keras.metrics import AUC, BinaryAccuracy, Precision, Recall

        assert (AUC, BinaryAccuracy, Precision, Recall) == (K.AUC, K.BinaryAccuracy, K.Precision, K.Recall)
        assert tf.keras.metrics.AUC is K.AUC
    finally:
        compat.uninstall()


def test_header_declares_the_metric_entries():
    import ctypes

    from handyrec_b200 import _lib

    protos = _lib.parse_header()
    assert protos["hrb_metric_update"][1] == [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int32,
                                              ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                              ctypes.c_void_p, ctypes.c_void_p]
    assert protos["hrb_metric_scratch_bytes"][1] == [ctypes.c_int32, ctypes.c_void_p]
    from handyrec_b200 import build

    assert "metrics.cu" in build.SOURCES
