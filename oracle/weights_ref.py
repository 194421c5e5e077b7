"""Keras 2.6 sample weights restated in float64 (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).  Every function cites the
Keras rule it implements.

* Loss (keras/utils/losses_utils.py ``compute_weighted_loss``, reduction ``SUM_OVER_BATCH_SIZE``): the batch loss is
  ``sum_i w_i * l_i / B`` with ``B`` the batch size (not ``sum w``: a zero weight still counts in the denominator); the gradient of
  logit ``i`` is ``w_i * (p_i - y_i) / B`` (``/ (B * N)`` under N data-parallel ranks, each averaging its own slice).
* class_weight (keras/engine/data_adapter.py ``_make_class_weight_map_fn``): keys exactly ``0..k-1``; the label is cast to int64
  by truncation and gathers the weight (converted to float32 first); with a sample_weight too, the product.
* Metrics (keras/utils/metrics_utils.py ``update_confusion_matrix_variables`` with ``sample_weight``; ``Mean.update_state``):
  every confusion variable adds ``sum_i w_i * [class_i, p_i > t]``; BinaryAccuracy adds ``sum w * correct`` to total and
  ``sum w`` to count.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np

EPSILON = 1e-7  # keras.backend.epsilon()


def weighted_bce_from_logits(logit, y, w, ranks: int = 1):
    """(loss, dlogit) of binary_crossentropy on a sigmoid output (sigmoid_cross_entropy_with_logits), weighted per sample."""
    z, y, w = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (logit, y, w))
    B = z.size
    l = np.maximum(z, 0) - z * y + np.log1p(np.exp(-np.abs(z)))
    p = 1.0 / (1.0 + np.exp(-z))
    return float((w * l).sum() / B), w * (p - y) / (B * ranks)


def weighted_bce_from_probs(prob, y, w):
    """(loss, dprob) of binary_crossentropy on probabilities clipped to [eps, 1 - eps] (Keras' path without logits); the clip's
    gradient is 0 outside."""
    p0, y, w = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (prob, y, w))
    B = p0.size
    p = np.clip(p0, EPSILON, 1.0 - EPSILON)
    l = -(y * np.log(p) + (1.0 - y) * np.log(1.0 - p))
    inside = (p0 >= EPSILON) & (p0 <= 1.0 - EPSILON)
    return float((w * l).sum() / B), np.where(inside, w * ((1.0 - y) / (1.0 - p) - y / p) / B, 0.0)


def class_weights(y, class_weight: Dict[int, float]) -> np.ndarray:
    """_make_class_weight_map_fn: the weight of each label, labels truncated to int64; ValueError for a key set other than 0..k-1
    or a label outside the classes after truncation (NaN included), as Keras raises on the CPU."""
    class_ids = sorted(class_weight.keys())
    if class_ids != list(range(len(class_ids))):
        raise ValueError("Expected `class_weight` to be a dict with keys from 0 to one less than the number of classes, "
                         f"found {class_weight}")
    table = np.array([class_weight[int(c)] for c in class_ids], dtype=np.float32)
    yf = np.asarray(y, dtype=np.float64).reshape(-1)
    with np.errstate(invalid="ignore"):
        ok = np.isfinite(yf) & (np.trunc(yf) >= 0) & (np.trunc(yf) < len(class_ids))
    if not ok.all():
        raise ValueError(f"label {yf[~ok][0]} is outside the classes 0..{len(class_ids) - 1}")
    return table[np.trunc(yf).astype(np.int64)].astype(np.float64)


def sample_weights(y, sample_weight=None, class_weight: Optional[Dict[int, float]] = None) -> Optional[np.ndarray]:
    """The float32 weight of every sample: sample_weight times the class weight, the product formed in float64 (Keras multiplies
    in the sample weight's dtype: float32 x float32 is exact in float64, float64 rounds once) and rounded once to float32."""
    if sample_weight is None and class_weight is None:
        return None
    w = np.ones(len(np.asarray(y)), np.float64)
    if sample_weight is not None:
        w = np.asarray(sample_weight, dtype=np.float64).reshape(-1)
    if class_weight is not None:
        w = w * class_weights(y, class_weight)
    return w.astype(np.float32)


def weighted_confusion(y_pred, y_true, w, thresholds) -> Dict[str, np.ndarray]:
    """update_confusion_matrix_variables with sample_weight: per threshold t, the float64 sums of w over the samples of each cell
    (p > t compared in float32, label_is_pos = bool(y_true))."""
    p = np.asarray(y_pred, dtype=np.float32).reshape(-1)
    y = np.asarray(y_true, dtype=np.float32).reshape(-1)
    w = np.asarray(w, dtype=np.float64).reshape(-1)
    t = np.asarray(thresholds, dtype=np.float32).reshape(-1)
    pos = y != 0
    above = p[None, :] > t[:, None]
    cell = lambda m: (m * w[None, :]).sum(1)  # noqa: E731
    return {"tp": cell(above & pos[None]), "fp": cell(above & ~pos[None]), "tn": cell(~above & ~pos[None]),
            "fn": cell(~above & pos[None])}


def weighted_binary_accuracy(y_pred, y_true, w, threshold: float = 0.5):
    """MeanMetricWrapper(binary_accuracy) with sample_weight: (sum w * correct, sum w) in float64."""
    p = np.asarray(y_pred, dtype=np.float32).reshape(-1)
    y = np.asarray(y_true, dtype=np.float32).reshape(-1)
    w = np.asarray(w, dtype=np.float64).reshape(-1)
    correct = y == (p > np.float32(threshold)).astype(np.float32)
    return float((w * correct).sum()), float(w.sum())
