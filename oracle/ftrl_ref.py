"""Keras 2.6 Ftrl restated in float64 (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).

``tf.keras.optimizers.Ftrl(learning_rate=0.001, learning_rate_power=-0.5, initial_accumulator_value=0.1,
l1_regularization_strength=0.0, l2_regularization_strength=0.0, l2_shrinkage_regularization_strength=0.0, beta=0.0)``
(keras/optimizer_v2/ftrl.py) keeps two slots per variable, ``accumulator`` (starting at ``initial_accumulator_value``) and
``linear`` (starting at 0), and hands its kernels ``l2 = l2_regularization_strength + beta / (2 * lr)``:

* a dense gradient: ``ResourceApplyFtrl`` (``ResourceApplyFtrlV2`` when ``l2_shrinkage > 0``; training_ops.cc, ``ApplyFtrl`` /
  ``ApplyFtrlV2`` functors);
* an ``IndexedSlices`` gradient (an embedding table): ``_resource_apply_sparse_duplicate_indices`` sums the values of duplicate
  indices, then ``ResourceSparseApplyFtrl(V2)`` steps the listed rows only.

Per element, with ``g`` the gradient (a Keras l2 regulariser's ``2 * l2_reg * w`` already added)::

    g_s     = g + 2 * l2_shrinkage * w
    acc_new = acc + g * g
    p(a)    = sqrt(a) if lr_power == -0.5 else a ** (-lr_power)
    linear += g_s - (p(acc_new) - p(acc)) / lr * w
    y       = p(acc_new) / lr + 2 * l2
    w       = (sign(linear) * l1 - linear) / y  where |linear| > l1, else 0
    acc     = acc_new

A step with a zero gradient is not a no-op: it recomputes ``w`` from the slots.  So which rows an IndexedSlices step lists
matters; Keras lists every gathered position, the padding id 0 of a pooled sequence field included (with a zero gradient).
"""
from __future__ import annotations

import numpy as np
import torch

__all__ = ["ftrl_dense", "ftrl_sparse", "kernel_l2"]


def _f64(x) -> torch.Tensor:
    return torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x).to(torch.float64)


def kernel_l2(lr: float, l2: float = 0.0, beta: float = 0.0) -> float:
    """The l2 Keras' Ftrl hands its kernels."""
    return l2 + beta / (2.0 * lr)


def _step(w, acc, lin, g, lr, l1, l2, lr_power, l2_shrinkage):
    gs = g + 2.0 * l2_shrinkage * w
    acc_new = acc + g * g
    p = (lambda a: torch.sqrt(a)) if lr_power == -0.5 else (lambda a: a ** (-lr_power))
    lin = lin + gs - (p(acc_new) - p(acc)) / lr * w
    y = p(acc_new) / lr + 2.0 * l2
    big = lin.abs() > l1
    w = torch.where(big, (torch.sign(lin) * l1 - lin) / torch.where(big, y, torch.ones_like(y)), torch.zeros_like(lin))
    return w, acc_new, lin


def ftrl_dense(var, accum, linear, grad, lr: float, l1: float = 0.0, l2: float = 0.0, lr_power: float = -0.5,
               l2_shrinkage: float = 0.0, l2_scale: float = 0.0):
    """ResourceApplyFtrl(V2) on a whole variable -> (var, accum, linear) in float64.  l2 is the kernel's (beta folded in);
    l2_scale = 2 * l2 of a Keras regulariser, added to the gradient first."""
    var, accum, linear, grad = _f64(var), _f64(accum), _f64(linear), _f64(grad)
    return _step(var, accum, linear, grad + l2_scale * var, lr, l1, l2, lr_power, l2_shrinkage)


def ftrl_sparse(var, accum, linear, indices, values, lr: float, l1: float = 0.0, l2: float = 0.0, lr_power: float = -0.5,
                l2_shrinkage: float = 0.0):
    """_deduplicate_indexed_slices + ResourceSparseApplyFtrl(V2): values (N, D) of rows indices (N,) are summed per row, then only
    those rows step -> (var, accum, linear) in float64.  A row listed with zero values still steps."""
    var, accum, linear, values = _f64(var).clone(), _f64(accum).clone(), _f64(linear).clone(), _f64(values)
    idx = torch.as_tensor(np.asarray(indices) if not isinstance(indices, torch.Tensor) else indices).long().reshape(-1)
    if idx.numel() == 0:
        return var, accum, linear
    uniq, inv = torch.unique(idx, return_inverse=True)
    summed = torch.zeros(len(uniq), var.shape[-1], dtype=torch.float64).index_add_(0, inv, values.reshape(len(idx), -1))
    w, a, l = _step(var[uniq], accum[uniq], linear[uniq], summed, lr, l1, l2, lr_power, l2_shrinkage)
    var[uniq], accum[uniq], linear[uniq] = w, a, l
    return var, accum, linear
