"""The embedding backward of a lookup plan restated on the CPU (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).

* ``plan_grad_sums``: the per-table gradient sums TF autodiff forms for a feature group (layers/tools.py CustomEmbedding,
  layers/sequence.py SequencePoolingLayer), deduplicated like Keras' IndexedSlices, in float64.  A plain field names every id; a
  pooled field drops the padding id 0; mean pooling scales by ``1 / n_valid`` (0 for an all-padding row); negative and
  out-of-range ids are dropped (the forward reports them when asked, the backward writes them nowhere).
* ``table_units`` / ``unit_path_taken``: ``build_units`` and ``unit_path_supported`` of csrc/embedding_bwd.cu -- how the
  sort-free backward cuts each table into power-of-two row ranges ("units"), which rows it splits over list slices, and when
  ``hrb_lookup_bwd_update`` takes the sorted path instead.  Tests use them to build ids that land exactly on a boundary.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

__all__ = ["plan_grad_sums", "table_units", "unit_path_taken", "unit_counts", "UB_CAP", "UB_MAX_BINS", "UB_MAX_COLS",
           "UB_MAX_SLICES"]

UB_CAP = 4096          # positions one pass of bwd_unit_kernel sorts in shared memory
UB_EXPECT_MAX = 3686   # 0.9 * UB_CAP: the most positions a unit should expect under uniform ids
UB_MAX_BINS = 256      # units per table
UB_MAX_COLS = 256      # position columns per table
UB_SLICE_TARGET = 4096  # positions per slice of a row the host knows to be hot
UB_MAX_SLICES = 64


def plan_grad_sums(shapes: Sequence[Tuple[int, int]], fields, ids, dout) -> List[Dict[str, torch.Tensor]]:
    """Per table t: {"rows": the distinct rows that take a gradient (sorted, int64), "grad": their summed gradient rows (float64),
    "pad": True when a pooled field of t holds padding}.  fields: (table, seq_len, pool, ids_col, out_col) as LookupPlan takes
    them; ids (B, >= ids_cols) int; dout (B, >= out_cols)."""
    ids = torch.as_tensor(ids).long()
    dout = torch.as_tensor(dout).to(torch.float64)
    idx: List[List[torch.Tensor]] = [[] for _ in shapes]
    val: List[List[torch.Tensor]] = [[] for _ in shapes]
    pad = [False] * len(shapes)
    for ti, L, pool, ids_col, out_col in fields:
        rows, dim = shapes[ti]
        cols = ids[:, ids_col: ids_col + L]
        g = dout[:, out_col: out_col + dim]
        in_range = (cols >= 0) & (cols < rows)
        valid = in_range if pool == "none" else in_range & (cols != 0)
        if pool != "none":
            pad[ti] |= bool((cols == 0).any())
        scale = torch.ones(cols.shape[0], 1, dtype=torch.float64)
        if pool == "mean":
            n = valid.sum(1, keepdim=True).to(torch.float64)
            scale = torch.where(n > 0, 1.0 / n.clamp(min=1), torch.zeros_like(n))
        for l in range(L):
            keep = valid[:, l]
            idx[ti].append(cols[keep, l])
            val[ti].append(g[keep] * scale[keep])
    out = []
    for t, (rows, dim) in enumerate(shapes):
        i = torch.cat(idx[t]) if idx[t] else torch.zeros(0, dtype=torch.long)
        v = torch.cat(val[t]) if val[t] else torch.zeros(0, dim, dtype=torch.float64)
        uniq, inv = torch.unique(i, return_inverse=True)
        summed = torch.zeros(len(uniq), dim, dtype=torch.float64).index_add_(0, inv, v)
        out.append({"rows": uniq, "grad": summed, "pad": pad[t]})
    return out


def table_units(rows: int, n_cols: int, batch: int) -> Optional[List[Dict[str, int]]]:
    """build_units for one table of `rows` rows read by `n_cols` position columns at `batch` samples: the units in row order,
    each {"lo", "hi", "shift", "slices", "expect"}; None when the table needs more than UB_MAX_BINS units (the sorted path)."""
    if n_cols == 0:
        return []
    n_t = batch * n_cols
    shift = 0
    while shift < 31 and (2 << shift) * n_t <= UB_EXPECT_MAX * rows:
        shift += 1
    rng = 1 << shift
    n_bins = (rows + rng - 1) // rng
    if n_bins > UB_MAX_BINS:
        return None
    units = []
    for b in range(n_bins):
        lo, hi = b * rng, min(rows, (b + 1) * rng)
        expect = n_t * (hi - lo) // rows
        slices = 1
        if hi - lo == 1 and expect > 2 * UB_SLICE_TARGET:
            slices = min(UB_MAX_SLICES, (expect + UB_SLICE_TARGET - 1) // UB_SLICE_TARGET)
        units.append({"lo": lo, "hi": hi, "shift": shift, "slices": slices, "expect": expect})
    return units


def unit_path_taken(shapes: Sequence[Tuple[int, int]], fields, batch: int) -> bool:
    """unit_path_supported: does hrb_lookup_bwd_update under hrb_plan_set_bwd_algo(UNITS) (or AUTO) take the sort-free path?
    Every table needs dim/4 a power of two <= 32, at most UB_MAX_COLS position columns and at most UB_MAX_BINS units; no field
    may be max-pooled; 0 < batch < 2^24."""
    if not (0 < batch < (1 << 24)) or any(f[2] == "max" for f in fields):
        return False
    for t, (rows, dim) in enumerate(shapes):
        g = dim // 4
        n_cols = sum(f[1] for f in fields if f[0] == t)
        if g & (g - 1) or g > 32 or n_cols > UB_MAX_COLS:
            return False
        if table_units(rows, n_cols, batch) is None:
            return False
    return True


def unit_counts(units: List[Dict[str, int]], ids) -> np.ndarray:
    """Positions each unit's list receives from the valid ids `ids` (any shape) of its table."""
    ids = np.asarray(ids).reshape(-1)
    if not units:
        return np.zeros(0, np.int64)
    return np.bincount(ids >> units[0]["shift"], minlength=len(units))[: len(units)]
