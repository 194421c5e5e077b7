"""Keras 2.6 learning-rate schedules and the legacy time-based `decay` of every optimizer.

`tf.keras.optimizers.schedules` (keras/optimizer_v2/learning_rate_schedule.py): `ExponentialDecay`, `InverseTimeDecay`,
`PiecewiseConstantDecay`, `PolynomialDecay`, and `CosineDecay` / `CosineDecayRestarts` (in Keras 2.6 under
`tf.keras.experimental`).  Each takes Keras' arguments and defaults and computes in float32 as TF does: the step and every
constant are cast to float32 and each operation rounds to float32.

`decayed_lr(opt)` is `OptimizerV2._decayed_lr`: the schedule at `opt.iterations` (0 for the first step), then
`lr_t / (1 + decay * iterations)`.  The optimizers evaluate it once per training step, on either training path, and then count
the step in `iterations`.
"""
from __future__ import annotations

import math
from typing import Sequence

import numpy as np

__all__ = ["LearningRateSchedule", "ExponentialDecay", "InverseTimeDecay", "PiecewiseConstantDecay", "PolynomialDecay",
           "CosineDecay", "CosineDecayRestarts", "decayed_lr", "init_lr", "ftrl_kernel_l2"]

_f32 = np.float32


class LearningRateSchedule:
    """tf.keras.optimizers.schedules.LearningRateSchedule: `__call__(step)` gives the learning rate of the step with that index
    (the optimizer's `iterations` before the step)."""

    def __call__(self, step) -> float:
        raise NotImplementedError(f"{type(self).__name__} must implement __call__(step)")


class ExponentialDecay(LearningRateSchedule):
    """lr0 * decay_rate ** (step / decay_steps), the exponent floored when `staircase`."""

    def __init__(self, initial_learning_rate, decay_steps, decay_rate, staircase=False, name=None):
        self.initial_learning_rate, self.decay_steps, self.decay_rate = initial_learning_rate, decay_steps, decay_rate
        self.staircase, self.name = staircase, name

    def __call__(self, step) -> float:
        p = _f32(step) / _f32(self.decay_steps)
        if self.staircase:
            p = np.floor(p)
        return float(_f32(self.initial_learning_rate) * np.power(_f32(self.decay_rate), p))


class InverseTimeDecay(LearningRateSchedule):
    """lr0 / (1 + decay_rate * step / decay_steps), the quotient floored when `staircase`."""

    def __init__(self, initial_learning_rate, decay_steps, decay_rate, staircase=False, name=None):
        self.initial_learning_rate, self.decay_steps, self.decay_rate = initial_learning_rate, decay_steps, decay_rate
        self.staircase, self.name = staircase, name

    def __call__(self, step) -> float:
        p = _f32(step) / _f32(self.decay_steps)
        if self.staircase:
            p = np.floor(p)
        return float(_f32(self.initial_learning_rate) / (_f32(1.0) + _f32(self.decay_rate) * p))


class PiecewiseConstantDecay(LearningRateSchedule):
    """values[0] while step <= boundaries[0], values[i] for boundaries[i-1] < step <= boundaries[i], values[-1] after the last."""

    def __init__(self, boundaries: Sequence, values: Sequence, name=None):
        if len(boundaries) != len(values) - 1:
            raise ValueError("The length of boundaries should be 1 less than the length of values")
        self.boundaries, self.values, self.name = list(boundaries), list(values), name

    def __call__(self, step) -> float:
        for b, v in zip(self.boundaries, self.values):
            if step <= b:
                return float(_f32(v))
        return float(_f32(self.values[-1]))


class PolynomialDecay(LearningRateSchedule):
    """(lr0 - end) * (1 - step / decay_steps) ** power + end, the step held at decay_steps; with `cycle`, decay_steps is
    stretched to the first multiple of itself that is >= step (multiplier 1 at step 0)."""

    def __init__(self, initial_learning_rate, decay_steps, end_learning_rate=0.0001, power=1.0, cycle=False, name=None):
        self.initial_learning_rate, self.decay_steps, self.end_learning_rate = initial_learning_rate, decay_steps, end_learning_rate
        self.power, self.cycle, self.name = power, cycle, name

    def __call__(self, step) -> float:
        lr0, end = _f32(self.initial_learning_rate), _f32(self.end_learning_rate)
        s, ds = _f32(step), _f32(self.decay_steps)
        if self.cycle:
            ds = ds * (_f32(1.0) if s == 0 else np.ceil(s / ds))
        else:
            s = min(s, ds)
        p = s / ds
        return float((lr0 - end) * np.power(_f32(1.0) - p, _f32(self.power)) + end)


class CosineDecay(LearningRateSchedule):
    """tf.keras.experimental.CosineDecay: lr0 * ((1 - alpha) * 0.5 * (1 + cos(pi * min(step, decay_steps) / decay_steps)) + alpha)."""

    def __init__(self, initial_learning_rate, decay_steps, alpha=0.0, name=None):
        self.initial_learning_rate, self.decay_steps, self.alpha, self.name = initial_learning_rate, decay_steps, alpha, name

    def __call__(self, step) -> float:
        ds = _f32(self.decay_steps)
        frac = min(_f32(step), ds) / ds
        cosine = _f32(0.5) * (_f32(1.0) + np.cos(_f32(math.pi) * frac))
        # Keras forms (1 - alpha) from the Python float here (CosineDecayRestarts casts alpha first)
        return float(_f32(self.initial_learning_rate) * (_f32(1.0 - self.alpha) * cosine + _f32(self.alpha)))


class CosineDecayRestarts(LearningRateSchedule):
    """tf.keras.experimental.CosineDecayRestarts (SGDR): cosine decay over periods of first_decay_steps * t_mul**i, the i-th
    starting from lr0 * m_mul**i.  The restart index is geometric when t_mul != 1, as in Keras."""

    def __init__(self, initial_learning_rate, first_decay_steps, t_mul=2.0, m_mul=1.0, alpha=0.0, name=None):
        self.initial_learning_rate, self.first_decay_steps = initial_learning_rate, first_decay_steps
        self._t_mul, self._m_mul, self.alpha, self.name = t_mul, m_mul, alpha, name

    def __call__(self, step) -> float:
        one = _f32(1.0)
        t_mul, m_mul, alpha = _f32(self._t_mul), _f32(self._m_mul), _f32(self.alpha)
        frac = _f32(step) / _f32(self.first_decay_steps)
        if t_mul == one:
            i_restart = np.floor(frac)
            frac = frac - i_restart
        else:
            i_restart = np.floor(np.log(one - frac * (one - t_mul)) / np.log(t_mul))
            sum_r = (one - np.power(t_mul, i_restart)) / (one - t_mul)
            frac = (frac - sum_r) / np.power(t_mul, i_restart)
        m_fac = np.power(m_mul, i_restart)
        cosine = _f32(0.5) * m_fac * (one + np.cos(_f32(math.pi) * frac))
        return float(_f32(self.initial_learning_rate) * ((one - alpha) * cosine + alpha))


def init_lr(opt, learning_rate, decay=0.0) -> None:
    """The learning-rate attributes of an optimizer: `lr` (a float, or the schedule object as in Keras), `decay`, `iterations`
    (steps applied) and `lr_t`, the rate of the step being applied (None before the first step of a schedule)."""
    if decay < 0.0:
        raise ValueError(f"decay cannot be less than 0: {decay}")
    opt.lr = learning_rate if isinstance(learning_rate, LearningRateSchedule) else float(learning_rate)
    opt.decay = float(decay)
    opt.iterations = 0
    opt.lr_t = None if isinstance(opt.lr, LearningRateSchedule) else decayed_lr(opt)


def decayed_lr(opt) -> float:
    """OptimizerV2._decayed_lr at opt.iterations, in float32.  A float rate without decay is returned as it is."""
    lr, decay = opt.lr, opt.decay
    schedule = isinstance(lr, LearningRateSchedule)
    if not schedule and not decay:
        return lr
    it = opt.iterations
    lr_t = _f32(lr(it) if schedule else lr)
    if decay > 0.0:
        lr_t = lr_t / (_f32(1.0) + _f32(decay) * _f32(it))
    return float(lr_t)


def ftrl_kernel_l2(l2: float, beta: float, lr: float) -> float:
    """l2 + beta / (2 * lr), the l2 Keras' Ftrl hands its kernels; a rate that a schedule took to 0 divides as in TF (inf, or nan
    for 0 / 0) instead of raising."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return l2 + float(np.float64(beta) / (2.0 * lr))
