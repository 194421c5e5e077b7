"""Keras 2.6 regression losses restated in float64 (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).  Every function cites
the Keras rule it implements.

* Per-sample loss (keras/losses.py ``mean_squared_error``, ``mean_absolute_error``, ``huber``), ``e = y_pred - y_true``, the mean
  over the last axis: MSE ``e^2``, MAE ``|e|``, Huber ``0.5*q^2 + delta*(|e| - q)`` with ``q = min(|e|, delta)``.
* Gradients as TF's autodiff forms them: ``d|e|/de = sign(e)``, 0 at ``e = 0``; ``tf.minimum`` passes the gradient of a tie to its
  first argument, so at ``|e| == delta`` the quadratic branch takes it (``dl/de = e``).
* Shapes (keras/engine/compile_utils.py ``match_dtype_and_rank``): a ``(B,)`` label meets a ``(B, 1)`` prediction as ``(B, 1)``;
  it is never broadcast into a ``(B, B)`` matrix.
* Reduction (keras/utils/losses_utils.py ``compute_weighted_loss``, ``SUM_OVER_BATCH_SIZE``): ``sum_b w_b * l_b / B`` with ``B``
  the batch size, not ``sum w``; the gradient of prediction element ``(b, j)`` is ``w_b * dl/de / (cols * B * ranks)``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np


def match_label(y_true, y_pred) -> Tuple[np.ndarray, np.ndarray]:
    """(label, prediction) as float64 arrays of one shape: a label one rank short of a prediction whose last axis is 1 is expanded."""
    y, p = np.asarray(y_true, dtype=np.float64), np.asarray(y_pred, dtype=np.float64)
    if y.ndim == p.ndim - 1 and p.shape[-1] == 1:
        y = y[..., None]
    if y.shape != p.shape:
        raise ValueError(f"labels of shape {y.shape} for predictions of shape {p.shape}")
    return y, p


def elementwise(loss: str, e, delta: float = 1.0) -> Tuple[np.ndarray, np.ndarray]:
    """(l, dl/de) of one error array for loss "mean_squared_error", "mean_absolute_error" or "huber"."""
    e = np.asarray(e, dtype=np.float64)
    a, s = np.abs(e), np.sign(e)  # np.sign(0) = 0: TF's gradient of |e| at 0
    if loss == "mean_squared_error":
        return e * e, 2.0 * e
    if loss == "mean_absolute_error":
        return a, s
    if loss == "huber":
        q = np.minimum(a, delta)
        return 0.5 * q * q + delta * (a - q), np.where(a <= delta, e, delta * s)
    raise ValueError(f"unknown loss {loss!r}")


def per_sample(loss: str, y_true, y_pred, delta: float = 1.0) -> np.ndarray:
    """The per-sample loss: the elementwise loss averaged over the last axis of the (matched) prediction."""
    y, p = match_label(y_true, y_pred)
    l, _ = elementwise(loss, p - y, delta)
    return l.reshape(l.shape[0], -1).mean(axis=1)


def compiled_loss(loss: str, y_true, y_pred, w: Optional[np.ndarray] = None, delta: float = 1.0, ranks: int = 1):
    """(batch loss, dL/dy_pred) of Keras' compiled loss: sum(w * l) / B and its gradient (shaped as y_pred)."""
    y, p = match_label(y_true, y_pred)
    B = p.shape[0]
    cols = p.size // max(B, 1)
    wv = np.ones(B) if w is None else np.asarray(w, dtype=np.float64).reshape(-1)
    l, dl = elementwise(loss, p - y, delta)
    ls = l.reshape(B, -1).mean(axis=1)
    grad = dl.reshape(B, -1) * wv[:, None] / (cols * B * ranks)
    return float((wv * ls).sum() / B), grad.reshape(p.shape)
