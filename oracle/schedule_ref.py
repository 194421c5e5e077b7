"""Keras 2.6 learning-rate schedules and ``_decayed_lr`` restated in float64 (TEST INFRASTRUCTURE ONLY, like the rest of ``oracle``).

From keras/optimizer_v2/learning_rate_schedule.py (``__call__`` of each class; ``step`` is the optimizer's ``iterations``):

* ``ExponentialDecay``: ``lr0 * decay_rate ** p``, ``p = step / decay_steps``, ``floor(p)`` when ``staircase``;
* ``InverseTimeDecay``: ``lr0 / (1 + decay_rate * p)``, same ``p``;
* ``PiecewiseConstantDecay``: ``values[0]`` for ``step <= boundaries[0]``, ``values[i]`` for
  ``boundaries[i-1] < step <= boundaries[i]``, ``values[-1]`` for ``step > boundaries[-1]``;
* ``PolynomialDecay``: without ``cycle`` ``step = min(step, decay_steps)``; with ``cycle``
  ``decay_steps *= (1 if step == 0 else ceil(step / decay_steps))``; then ``(lr0 - end) * (1 - step / decay_steps) ** power + end``;
* ``CosineDecay`` (``tf.keras.experimental`` in 2.6): ``f = min(step, decay_steps) / decay_steps``,
  ``lr0 * ((1 - alpha) * 0.5 * (1 + cos(pi * f)) + alpha)``;
* ``CosineDecayRestarts``: ``f = step / first_decay_steps``; with ``t_mul == 1`` ``i = floor(f)``, ``f -= i``; otherwise
  ``i = floor(log(1 - f * (1 - t_mul)) / log(t_mul))``, ``f = (f - (1 - t_mul ** i) / (1 - t_mul)) / t_mul ** i``; then
  ``lr0 * ((1 - alpha) * 0.5 * m_mul ** i * (1 + cos(pi * f)) + alpha)``.

keras/optimizer_v2/optimizer_v2.py ``_decayed_lr``: the schedule at ``iterations`` (a float rate as it is), then, when the
optimizer's ``decay > 0``, ``lr_t / (1 + decay * iterations)``.  ``iterations`` counts the steps applied, so the first step
takes the rate at 0.  Keras evaluates this in float32; this module is the exact-arithmetic reference.
"""
from __future__ import annotations

import math
from typing import Callable, Sequence, Union

__all__ = ["exponential_decay", "inverse_time_decay", "piecewise_constant_decay", "polynomial_decay", "cosine_decay",
           "cosine_decay_restarts", "decayed_lr"]


def exponential_decay(step, initial_learning_rate, decay_steps, decay_rate, staircase=False) -> float:
    p = step / decay_steps
    if staircase:
        p = math.floor(p)
    return initial_learning_rate * decay_rate ** p


def inverse_time_decay(step, initial_learning_rate, decay_steps, decay_rate, staircase=False) -> float:
    p = step / decay_steps
    if staircase:
        p = math.floor(p)
    return initial_learning_rate / (1.0 + decay_rate * p)


def piecewise_constant_decay(step, boundaries: Sequence, values: Sequence) -> float:
    if len(boundaries) != len(values) - 1:
        raise ValueError("The length of boundaries should be 1 less than the length of values")
    if step <= boundaries[0]:
        return float(values[0])
    if step > boundaries[-1]:
        return float(values[-1])
    for low, high, v in zip(boundaries[:-1], boundaries[1:], values[1:-1]):
        if low < step <= high:
            return float(v)
    raise AssertionError("unreachable")


def polynomial_decay(step, initial_learning_rate, decay_steps, end_learning_rate=0.0001, power=1.0, cycle=False) -> float:
    if cycle:
        decay_steps = decay_steps * (1.0 if step == 0 else math.ceil(step / decay_steps))
    else:
        step = min(step, decay_steps)
    return (initial_learning_rate - end_learning_rate) * (1.0 - step / decay_steps) ** power + end_learning_rate


def cosine_decay(step, initial_learning_rate, decay_steps, alpha=0.0) -> float:
    f = min(step, decay_steps) / decay_steps
    return initial_learning_rate * ((1.0 - alpha) * 0.5 * (1.0 + math.cos(math.pi * f)) + alpha)


def cosine_decay_restarts(step, initial_learning_rate, first_decay_steps, t_mul=2.0, m_mul=1.0, alpha=0.0) -> float:
    f = step / first_decay_steps
    if t_mul == 1.0:
        i = math.floor(f)
        f -= i
    else:
        i = math.floor(math.log(1.0 - f * (1.0 - t_mul)) / math.log(t_mul))
        f = (f - (1.0 - t_mul ** i) / (1.0 - t_mul)) / t_mul ** i
    return initial_learning_rate * ((1.0 - alpha) * 0.5 * m_mul ** i * (1.0 + math.cos(math.pi * f)) + alpha)


def decayed_lr(lr: Union[float, Callable[[int], float]], iterations: int, decay: float = 0.0) -> float:
    """OptimizerV2._decayed_lr: `lr` a float or a function of the step (one of the above with its arguments bound)."""
    lr_t = lr(iterations) if callable(lr) else float(lr)
    if decay > 0.0:
        lr_t = lr_t / (1.0 + decay * iterations)
    return lr_t
