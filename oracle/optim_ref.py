"""Keras 2.6 Adagrad restated in float64 (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).

``tf.keras.optimizers.Adagrad(learning_rate=0.001, initial_accumulator_value=0.1, epsilon=1e-7)`` (keras/optimizer_v2/adagrad.py)
applies one of two TF kernels per variable:

* a dense gradient: ``_resource_apply_dense`` -> ``ResourceApplyAdagradV2``
  (tensorflow/core/kernels/training_ops.cc, functor ``ApplyAdagradV2``);
* an ``IndexedSlices`` gradient (an embedding table): ``_resource_apply_sparse_duplicate_indices`` first sums the values of
  duplicate indices (optimizer_v2.py ``_deduplicate_indexed_slices``), then ``_resource_apply_sparse`` ->
  ``ResourceSparseApplyAdagradV2`` (training_ops.cc, ``SparseApplyAdagradV2Op``) updates the listed rows only.

Both compute, with ``update_slots = True``::

    accum += grad * grad
    var   -= lr * grad / (sqrt(accum) + epsilon)      # epsilon OUTSIDE the square root

There is no step counter and no bias correction.  A Keras l2 regulariser adds ``2 * l2 * var`` to ``grad`` first (and makes an
embedding table's gradient dense: every row steps).

``adam_lazy_sparse`` restates the lazy Adam row update of the embedding backward (Keras Adam's formula on the listed rows only).
"""
from __future__ import annotations

import numpy as np
import torch

__all__ = ["adagrad_dense", "adagrad_sparse", "adam_lazy_sparse"]


def _f64(x) -> torch.Tensor:
    return torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x).to(torch.float64)


def adagrad_dense(var, accum, grad, lr: float, eps: float = 1e-7, l2_scale: float = 0.0):
    """ResourceApplyAdagradV2 on a whole variable -> (new var, new accum) in float64.  l2_scale = 2*l2."""
    var, accum, grad = _f64(var), _f64(accum), _f64(grad)
    g = grad + l2_scale * var
    accum = accum + g * g
    return var - lr * g / (torch.sqrt(accum) + eps), accum


def adagrad_sparse(var, accum, indices, values, lr: float, eps: float = 1e-7):
    """_deduplicate_indexed_slices + ResourceSparseApplyAdagradV2: values (N, D) of rows indices (N,) are summed per row, then
    only those rows step -> (new var, new accum) in float64."""
    var, accum, values = _f64(var).clone(), _f64(accum).clone(), _f64(values)
    idx = torch.as_tensor(np.asarray(indices) if not isinstance(indices, torch.Tensor) else indices).long().reshape(-1)
    uniq, inv = torch.unique(idx, return_inverse=True)
    summed = torch.zeros(len(uniq), values.shape[-1], dtype=torch.float64).index_add_(0, inv, values.reshape(len(idx), -1))
    a = accum[uniq] + summed * summed
    accum[uniq] = a
    var[uniq] = var[uniq] - lr * summed / (torch.sqrt(a) + eps)
    return var, accum


def adam_lazy_sparse(var, m, v, indices, values, lr: float, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-7,
                     step: int = 1, l2_scale: float = 0.0):
    """Lazy Adam (tf.keras Adam's update restricted to the rows an IndexedSlices gradient lists, as in TF-Addons LazyAdam):
    values (N, D) of rows indices (N,) are summed per row, then only those rows step -> (var, m, v) in float64::

        g  = summed + l2_scale * var
        m  = beta1 * m + (1 - beta1) * g
        v  = beta2 * v + (1 - beta2) * g * g
        var -= lr * sqrt(1 - beta2^step) / (1 - beta1^step) * m / (sqrt(v) + eps)

    Rows not listed keep var, m and v (their moments do not decay)."""
    var, m, v, values = _f64(var).clone(), _f64(m).clone(), _f64(v).clone(), _f64(values)
    idx = torch.as_tensor(np.asarray(indices) if not isinstance(indices, torch.Tensor) else indices).long().reshape(-1)
    if idx.numel() == 0:
        return var, m, v
    uniq, inv = torch.unique(idx, return_inverse=True)
    summed = torch.zeros(len(uniq), var.shape[-1], dtype=torch.float64).index_add_(0, inv, values.reshape(len(idx), -1))
    g = summed + l2_scale * var[uniq]
    mu = beta1 * m[uniq] + (1.0 - beta1) * g
    vu = beta2 * v[uniq] + (1.0 - beta2) * g * g
    lr_t = lr * np.sqrt(1.0 - beta2 ** step) / (1.0 - beta1 ** step)
    var[uniq] = var[uniq] - lr_t * mu / (torch.sqrt(vu) + eps)
    m[uniq], v[uniq] = mu, vu
    return var, m, v
