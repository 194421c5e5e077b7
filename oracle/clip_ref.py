"""Keras 2.6 gradient clipping restated in float64 (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).

``OptimizerV2(clipnorm=None, clipvalue=None, global_clipnorm=None)`` (keras/optimizer_v2/optimizer_v2.py) transforms the
gradients of ``tape.gradient(loss + regularisation losses, trainable_variables)`` in ``_transform_gradients`` before any
variable steps, in this order:

* ``clipvalue`` v: ``tf.clip_by_value(g, -v, v)``; on an ``IndexedSlices`` the values are clamped, one row per gathered
  position, before duplicate indices are summed;
* ``clipnorm`` c: ``tf.clip_by_norm(g, c)`` per variable, ``g * c / max(||g||, c)``; the norm of an ``IndexedSlices`` covers
  its un-deduplicated values;
* ``global_clipnorm`` c: ``tf.clip_by_global_norm(grads, c)`` with the norm over every gradient; a non-finite global norm makes
  every gradient NaN (TF's ``scale + (norm - norm)``).

Both norm modes are written here as ``g * s`` with ``s = c / max(norm, c)``: the same value as TF's expressions up to rounding,
exactly 1 when the norm is <= c, and NaN for a zero norm with c = 0 (0 / 0, as in TF).

An embedding table looked up by several layers (DeepFM's FM and DNN groups, DIN's query / keys / history) has one
``IndexedSlices`` gradient whose values are the lookups' values concatenated (``backprop_util.AggregateIndexedSlicesGradients``);
a mean-pooled position carries ``dout / n_valid``, a padding position a zero row.  A table with an l2 regulariser has a dense
gradient instead (the positions summed per row plus ``2 * l2 * w`` on every row).
"""
from __future__ import annotations

from typing import List, NamedTuple, Optional, Sequence, Union

import numpy as np

__all__ = ["IndexedSlices", "concat_slices", "densify", "clip_gradients"]


class IndexedSlices(NamedTuple):
    indices: np.ndarray  # (N,) rows of the variable
    values: np.ndarray   # (N, D) one value row per position, duplicates not summed


Grad = Union[np.ndarray, IndexedSlices]


def concat_slices(*parts: IndexedSlices) -> IndexedSlices:
    """AggregateIndexedSlicesGradients: the lookups' (indices, values) concatenated."""
    return IndexedSlices(np.concatenate([np.asarray(p.indices).reshape(-1) for p in parts]),
                         np.concatenate([np.asarray(p.values, dtype=np.float64) for p in parts]))


def densify(g: Grad, rows: int) -> np.ndarray:
    """The dense gradient an IndexedSlices stands for (duplicates summed)."""
    if not isinstance(g, IndexedSlices):
        return np.asarray(g, dtype=np.float64)
    out = np.zeros((rows, g.values.shape[1]), dtype=np.float64)
    np.add.at(out, np.asarray(g.indices).reshape(-1), g.values)
    return out


def _vals(g: Grad) -> np.ndarray:
    return g.values if isinstance(g, IndexedSlices) else g


def _with(g: Grad, v: np.ndarray) -> Grad:
    return IndexedSlices(g.indices, v) if isinstance(g, IndexedSlices) else v


def _scale(norm: float, c: float) -> float:
    with np.errstate(invalid="ignore", divide="ignore"):
        return float(np.float64(c) / max(norm, c)) if not np.isnan(norm) else float("nan")


def clip_gradients(grads: Sequence[Optional[Grad]], clipvalue: Optional[float] = None, clipnorm: Optional[float] = None,
                   global_clipnorm: Optional[float] = None) -> List[Optional[Grad]]:
    """OptimizerV2._transform_gradients on float64 gradients (None entries: variables without a gradient)."""
    if clipnorm is not None and global_clipnorm is not None:
        raise ValueError("Cannot accept both `clipnorm` and `global_clipnorm`")
    out = [None if g is None else _with(g, np.asarray(_vals(g), dtype=np.float64)) for g in grads]
    if clipvalue is not None:
        out = [None if g is None else _with(g, np.clip(_vals(g), -clipvalue, clipvalue)) for g in out]
    if clipnorm is not None:
        out = [None if g is None else _with(g, _vals(g) * _scale(float(np.sqrt((_vals(g) ** 2).sum())), clipnorm)) for g in out]
    if global_clipnorm is not None:
        norm = float(np.sqrt(sum(float((_vals(g) ** 2).sum()) for g in out if g is not None)))
        s = _scale(norm, global_clipnorm) if np.isfinite(norm) else float("nan")
        out = [None if g is None else _with(g, _vals(g) * s) for g in out]
    return out
