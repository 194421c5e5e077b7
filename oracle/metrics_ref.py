"""Keras 2.6 metrics AUC / Precision / Recall / BinaryAccuracy restated with numpy (TEST INFRASTRUCTURE ONLY, like the rest of
``oracle``).  Every function cites the Keras rule it implements.

Confusion variables (keras/utils/metrics_utils.py ``update_confusion_matrix_variables``):

* ``y_true`` is cast to bool: every label ``!= 0`` is a positive (NaN included);
* a prediction is "above" threshold ``t`` iff ``y_pred > t``, compared in float32 against the thresholds converted to float32;
* each batch adds its ``tp, fp, tn, fn`` per threshold into float32 variables (``assign_add``): a batch's counts are exact
  integers, the running sum rounds in float32 once it passes 2^24 (``accumulate_f32``).

``result()`` formulas (keras/metrics.py ``AUC.result``, ``AUC.interpolate_pr_auc``, ``Precision.result``, ``Recall.result``,
``MeanMetricWrapper`` over ``binary_accuracy``) are given in float64 and, with ``dtype=np.float32``, op by op in float32.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import numpy as np

EPSILON = 1e-7  # keras.backend.epsilon()


def auc_thresholds(num_thresholds: int = 200, thresholds: Optional[Sequence[float]] = None) -> np.ndarray:
    """AUC.__init__: explicit thresholds are sorted (num_thresholds = len + 2); otherwise [(i + 1) / (num_thresholds - 1) for i in
    range(num_thresholds - 2)] in Python doubles.  Either way [-epsilon] goes in front and [1 + epsilon] at the end, then float32."""
    if thresholds is not None:
        inner = sorted(float(t) for t in thresholds)
    else:
        inner = [(i + 1) * 1.0 / (num_thresholds - 1) for i in range(num_thresholds - 2)]
    return np.array([0.0 - EPSILON] + inner + [1.0 + EPSILON], dtype=np.float64).astype(np.float32)


def confusion_counts(y_pred, y_true, thresholds) -> Dict[str, np.ndarray]:
    """One batch's exact integer counts per threshold (update_confusion_matrix_variables): pred_is_pos = y_pred > t in float32,
    label_is_pos = bool(y_true)."""
    p = np.asarray(y_pred, dtype=np.float32).reshape(-1)
    y = np.asarray(y_true, dtype=np.float32).reshape(-1)
    t = np.asarray(thresholds, dtype=np.float32).reshape(-1)
    pos = y != 0  # NaN != 0 is True
    above = p[None, :] > t[:, None]  # (T, n)
    tp = (above & pos[None]).sum(1).astype(np.int64)
    fp = (above & ~pos[None]).sum(1).astype(np.int64)
    return {"tp": tp, "fp": fp, "tn": int((~pos).sum()) - fp, "fn": int(pos.sum()) - tp}


def binary_accuracy_counts(y_pred, y_true, threshold: float = 0.5):
    """keras.metrics.binary_accuracy: values = (y_true == float(y_pred > threshold)); MeanMetricWrapper adds sum(values) to
    `total` and the number of values to `count`.  A label outside {0, 1} is never correct."""
    p = np.asarray(y_pred, dtype=np.float32).reshape(-1)
    y = np.asarray(y_true, dtype=np.float32).reshape(-1)
    pred = (p > np.float32(threshold)).astype(np.float32)
    return int((y == pred).sum()), int(p.size)


def accumulate_f32(var, inc) -> np.ndarray:
    """assign_add on a float32 variable: fl32(var + fl32(inc))."""
    return (np.asarray(var, dtype=np.float32) + np.asarray(inc, dtype=np.float64).astype(np.float32)).astype(np.float32)


def div_no_nan(a, b):
    a, b = np.asarray(a), np.asarray(b)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(b == 0, np.zeros_like(a), a / np.where(b == 0, np.ones_like(b), b))


def interpolate_pr_auc(tp, fp, fn, dtype=np.float64):
    """AUC.interpolate_pr_auc (Davis & Goadrich 2006): precision interpolated linearly in the number of positives between
    thresholds."""
    tp, fp, fn = (np.asarray(v, dtype=dtype) for v in (tp, fp, fn))
    dtp = tp[:-1] - tp[1:]
    p = tp + fp
    dp = p[:-1] - p[1:]
    slope = div_no_nan(dtp, np.maximum(dp, 0))
    intercept = tp[1:] - slope * p[1:]
    both = (p[:-1] > 0) & (p[1:] > 0)
    ratio = np.where(both, div_no_nan(p[:-1], np.maximum(p[1:], 0)), np.ones_like(p[1:]))
    with np.errstate(divide="ignore", invalid="ignore"):
        inc = div_no_nan(slope * (dtp + intercept * np.log(ratio)), np.maximum(tp[1:] + fn[1:], 0))
    return dtype(np.sum(inc, dtype=dtype))


def auc_result(tp, fp, tn, fn, curve: str = "ROC", summation_method: str = "interpolation", dtype=np.float64):
    """AUC.result: recall = tp/(tp+fn); ROC: x = fp/(fp+tn), y = recall; PR: x = recall, y = tp/(tp+fp); heights by interpolation
    (mean), minoring (min) or majoring (max); sum((x[:-1]-x[1:]) * heights).  PR + interpolation: interpolate_pr_auc."""
    curve, summation_method = curve.upper(), summation_method.lower()
    if curve == "PR" and summation_method == "interpolation":
        return interpolate_pr_auc(tp, fp, fn, dtype)
    tp, fp, tn, fn = (np.asarray(v, dtype=dtype) for v in (tp, fp, tn, fn))
    recall = div_no_nan(tp, tp + fn)
    if curve == "ROC":
        x, y = div_no_nan(fp, fp + tn), recall
    else:
        x, y = recall, div_no_nan(tp, tp + fp)
    if summation_method == "interpolation":
        h = (y[:-1] + y[1:]) / dtype(2)
    elif summation_method == "minoring":
        h = np.minimum(y[:-1], y[1:])
    else:
        h = np.maximum(y[:-1], y[1:])
    return dtype(np.sum((x[:-1] - x[1:]) * h, dtype=dtype))


def precision_result(tp, fp, dtype=np.float64):
    return div_no_nan(np.asarray(tp, dtype=dtype), np.asarray(tp, dtype=dtype) + np.asarray(fp, dtype=dtype))


def recall_result(tp, fn, dtype=np.float64):
    return div_no_nan(np.asarray(tp, dtype=dtype), np.asarray(tp, dtype=dtype) + np.asarray(fn, dtype=dtype))
