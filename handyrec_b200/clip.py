"""Keras gradient clipping (OptimizerV2 `clipvalue`, `clipnorm`, `global_clipnorm`) for the layer path and the fused engine.

Keras 2.6 transforms the gradients before any variable steps (optimizer_v2.py `_transform_gradients`): first `clipvalue`
(tf.clip_by_value), then `clipnorm` (tf.clip_by_norm per variable), then `global_clipnorm` (tf.clip_by_global_norm over all
trainable variables).  The gradient is that of the loss plus the regularisation losses, so the `2 * l2 * w` of a regularised
variable is inside it; the prepare pass folds it in and the optimiser then steps that variable with l2 = 0.  An embedding
table without a regulariser has an IndexedSlices gradient: one value row per gathered position, duplicates not summed,
clamped and counted per position (csrc/clip.cu).  The norm modes are applied as g * s with s = c / max(norm, c), exactly 1
while the norm is <= c, so an inactive clip changes no bit.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple

import torch

from . import kernels as K


def init_clip(opt, clipnorm=None, clipvalue=None, global_clipnorm=None) -> None:
    """OptimizerV2.__init__'s checks and attributes."""
    for name, v in (("clipnorm", clipnorm), ("clipvalue", clipvalue), ("global_clipnorm", global_clipnorm)):
        if v is not None and v < 0:
            raise ValueError(f"Expected {name} >= 0, received: {v}")
    if clipnorm is not None and global_clipnorm is not None:
        raise ValueError(f"Cannot accept both `clipnorm` and `global_clipnorm`, passed `clipnorm` {clipnorm}, "
                         f"`global_clipnorm` {global_clipnorm}")
    opt.clipnorm, opt.clipvalue, opt.global_clipnorm = clipnorm, clipvalue, global_clipnorm


def clip_args(opt) -> Optional[Tuple[Optional[float], Optional[float], Optional[float]]]:
    """(clipvalue, clipnorm, global_clipnorm) of an optimizer, or None when it clips nothing."""
    a = (getattr(opt, "clipvalue", None), getattr(opt, "clipnorm", None), getattr(opt, "global_clipnorm", None))
    return None if all(v is None for v in a) else tuple(None if v is None else float(v) for v in a)


class GradClip:
    """Device buffers of one model's clipping: sumsq / scale per Keras variable (index `var`), a reduction workspace."""

    def __init__(self, args, n_vars: int, n_tables: int, device):
        clipvalue, clipnorm, global_clipnorm = args
        self.value = math.inf if clipvalue is None else clipvalue
        self.norm = clipnorm if clipnorm is not None else global_clipnorm
        self.global_norm = global_clipnorm is not None
        self.n_vars = n_vars
        self.sumsq = torch.zeros(max(n_vars, 1), device=device, dtype=torch.float32)
        self.scale = torch.ones(max(n_vars, 1), device=device, dtype=torch.float32)
        self.ws = K.clip_workspace(n_tables, device)

    @property
    def scales(self) -> bool:
        return self.norm is not None

    def begin(self) -> None:
        if self.scales:
            self.sumsq.zero_()

    def prepare(self, grads: Sequence[torch.Tensor], weights, l2s, var: Sequence[int]) -> None:
        K.clip_prepare_multi(grads, weights, l2s, var, self.value, self.sumsq if self.scales else None, self.ws)

    def finish(self) -> None:
        if self.scales:
            K.clip_scales(self.sumsq[: self.n_vars], self.norm, self.global_norm, self.scale)

    def apply(self, grads: Sequence[torch.Tensor], var: Sequence[int]) -> None:
        if self.scales:
            K.clip_apply_multi(grads, var, self.scale)
