"""CPU: Keras learning-rate schedules and time-based decay -- every schedule against the float64 restatement of Keras' formulas
(oracle/schedule_ref.py), the argument errors, the optimizers' `lr` / `decay` / `iterations`, the fused engine's per-step rate, and
the compat shim's names."""
import math

import numpy as np
import pytest

from oracle import schedule_ref as R


def _S():
    from handyrec_b200 import schedules

    return schedules


def _optimizers():
    from handyrec_b200 import keras_lite as KL

    return [KL.SGD, KL.Adam, KL.Adagrad, KL.Ftrl]


# (name, class kwargs, oracle function, decay_steps the steps are counted in).  Parameters keep the rates away from values
# formed by cancellation (alpha > 0, end_learning_rate well above the float32 rounding of lr0), where float32 keeps 1e-6.
CASES = [
    ("ExponentialDecay", dict(initial_learning_rate=0.1, decay_steps=7, decay_rate=0.5), R.exponential_decay, 7),
    ("ExponentialDecay", dict(initial_learning_rate=0.1, decay_steps=7, decay_rate=0.5, staircase=True), R.exponential_decay, 7),
    ("ExponentialDecay", dict(initial_learning_rate=3e-3, decay_steps=100, decay_rate=0.96), R.exponential_decay, 100),
    ("InverseTimeDecay", dict(initial_learning_rate=0.1, decay_steps=5, decay_rate=0.5), R.inverse_time_decay, 5),
    ("InverseTimeDecay", dict(initial_learning_rate=0.1, decay_steps=5, decay_rate=0.5, staircase=True), R.inverse_time_decay, 5),
    ("PiecewiseConstantDecay", dict(boundaries=[3, 10, 11], values=[0.1, 0.05, 0.01, 1e-3]), R.piecewise_constant_decay, 5),
    ("PiecewiseConstantDecay", dict(boundaries=[0], values=[1.0, 0.5]), R.piecewise_constant_decay, 2),
    ("PolynomialDecay", dict(initial_learning_rate=0.1, decay_steps=9, end_learning_rate=0.01), R.polynomial_decay, 9),
    ("PolynomialDecay", dict(initial_learning_rate=0.1, decay_steps=9, end_learning_rate=0.01, power=2.0), R.polynomial_decay, 9),
    ("PolynomialDecay", dict(initial_learning_rate=0.1, decay_steps=9, end_learning_rate=0.01, power=0.5, cycle=True),
     R.polynomial_decay, 9),
    ("PolynomialDecay", dict(initial_learning_rate=0.1, decay_steps=8), R.polynomial_decay, 8),  # Keras' default end 1e-4
    ("CosineDecay", dict(initial_learning_rate=0.1, decay_steps=11, alpha=0.1), R.cosine_decay, 11),
    ("CosineDecayRestarts", dict(initial_learning_rate=0.1, first_decay_steps=6, t_mul=1.0, m_mul=0.7, alpha=0.2),
     R.cosine_decay_restarts, 6),
    ("CosineDecayRestarts", dict(initial_learning_rate=0.1, first_decay_steps=5, alpha=0.1), R.cosine_decay_restarts, 5),
    ("CosineDecayRestarts", dict(initial_learning_rate=0.1, first_decay_steps=4, t_mul=1.5, m_mul=0.8, alpha=0.3),
     R.cosine_decay_restarts, 4),
]


@pytest.mark.parametrize("i", range(len(CASES)))
def test_schedule_matches_the_float64_formula(i):
    name, kw, ref, ds = CASES[i]
    s = getattr(_S(), name)(**kw)
    for step in range(3 * ds + 1):
        got, want = s(step), ref(step, **kw)
        assert isinstance(got, float)
        assert got == np.float32(got)  # computed in float32
        assert abs(got - want) <= 1e-6 * abs(want), (name, kw, step, got, want)


def test_boundary_steps_of_the_stepwise_schedules():
    S = _S()
    staircase = S.ExponentialDecay(0.1, 10, 0.5, staircase=True)
    assert [staircase(s) for s in (9, 10, 19, 20)] == [np.float32(0.1), np.float32(0.05), np.float32(0.05), np.float32(0.025)]
    inv = S.InverseTimeDecay(1.0, 4, 1.0, staircase=True)
    assert [inv(s) for s in (3, 4, 8)] == [1.0, 0.5, np.float32(1 / 3)]
    pw = S.PiecewiseConstantDecay([3, 10], [0.1, 0.05, 0.01])  # a step ON a boundary takes the value before it
    assert [pw(s) for s in (0, 3, 4, 10, 11)] == [np.float32(v) for v in (0.1, 0.1, 0.05, 0.05, 0.01)]
    cyc = S.PolynomialDecay(1.0, 4, end_learning_rate=0.0, cycle=True)
    assert [cyc(s) for s in (0, 4, 5, 8)] == [1.0, 0.0, np.float32(1 - 5 / 8), 0.0]  # step 0: multiplier 1, not 0
    assert S.PolynomialDecay(1.0, 4, end_learning_rate=0.25)(100) == 0.25  # held at decay_steps
    r = S.CosineDecayRestarts(1.0, 4, t_mul=2.0)  # periods of 4, 8, 16 steps: restarts at 4 and 12
    assert r(4) == 1.0 and r(12) == 1.0 and r(3) < r(4) and r(11) < r(12)
    r1 = S.CosineDecayRestarts(1.0, 4, t_mul=1.0, m_mul=0.5)
    assert r1(4) == 0.5 and r1(8) == 0.25


def test_cosine_decay_to_zero():
    """alpha = 0 ends at exactly 0; just before, 1 + cos(pi * f) is a cancellation, which float32 keeps to ~1e-7 of lr0."""
    s = _S().CosineDecay(0.1, 16)
    for step in range(3 * 16 + 1):
        assert abs(s(step) - R.cosine_decay(step, 0.1, 16)) <= 1e-7 * 0.1
    assert s(16) == 0.0 and s(40) == 0.0


def test_schedule_and_optimizer_errors():
    S = _S()
    with pytest.raises(ValueError, match="1 less than"):
        S.PiecewiseConstantDecay([1, 2], [0.1, 0.2])
    with pytest.raises(ValueError, match="1 less than"):
        R.piecewise_constant_decay(0, [1, 2], [0.1, 0.2])
    for cls in _optimizers():
        with pytest.raises(ValueError, match="decay cannot be less than 0"):
            cls(0.1, decay=-1e-6)
    with pytest.raises(NotImplementedError):
        S.LearningRateSchedule()(0)


def test_optimizer_lr_decay_and_iterations_attributes():
    from handyrec_b200 import keras_lite as KL

    S = _S()
    for cls in _optimizers():
        o = cls(0.2)
        assert o.lr == 0.2 and o.decay == 0.0 and o.iterations == 0 and o.lr_t == 0.2
        assert cls(learning_rate=0.3, lr=0.25).lr == 0.25  # the legacy `lr` wins, as before
        sched = S.ExponentialDecay(0.1, 10, 0.9)
        o = cls(learning_rate=sched)
        assert o.lr is sched and o.lr_t is None  # Keras: a schedule stays the optimizer's learning rate
    assert KL.Ftrl(0.2).lr == 0.2 and KL.Ftrl(0.2).kernel_l2 == 0.0 and KL.Adam(0.1).t == 0
    assert KL.Ftrl(0.1, l2_regularization_strength=0.5, beta=0.2).hyper()["l2"] == 0.5 + 0.2 / (2 * 0.1)


@pytest.mark.parametrize("i", range(4))
def test_step_rate_and_iterations_on_the_layer_path(i):
    """`step` (no trainable variables: no kernel launch) takes _decayed_lr at `iterations`, keeps it in lr_t, then counts."""
    S = _S()
    cls = _optimizers()[i]
    sched = S.PolynomialDecay(0.1, 4, end_learning_rate=0.02)
    o = cls(sched, decay=0.5)
    for it in range(6):
        o.step([])
        want = R.decayed_lr(lambda s: R.polynomial_decay(s, 0.1, 4, end_learning_rate=0.02), it, 0.5)
        assert abs(o.lr_t - want) <= 1e-6 * want
        assert o.iterations == it + 1
    if cls.__name__ == "Adam":
        assert o.t == 6
    if cls.__name__ == "Ftrl":  # beta / (2 * lr_t) at the step's rate
        f = cls(S.ExponentialDecay(0.2, 1, 0.5), beta=0.4)
        for _ in range(3):  # iterations 0, 1, 2
            f.step([])
        assert f.lr_t == np.float32(0.05) and f.kernel_l2 == 0.4 / (2 * f.lr_t)


def test_float_rate_without_decay_is_the_float_itself():
    from handyrec_b200.schedules import decayed_lr

    for cls in _optimizers():
        o = cls(0.1)
        for _ in range(3):
            o.step([])
            assert o.lr_t == 0.1 and type(o.lr_t) is float  # not float32(0.1): exactly the value steps took before
        assert decayed_lr(o) == 0.1 and o.iterations == 3


def test_time_based_decay_is_float32_keras():
    from handyrec_b200.schedules import decayed_lr

    o = _optimizers()[0](0.1, decay=1e-2)
    rates = []
    for _ in range(5):
        o.step([])
        rates.append(o.lr_t)
    want = [np.float32(0.1) / (np.float32(1) + np.float32(1e-2) * np.float32(it)) for it in range(5)]
    assert rates == [float(w) for w in want]
    o.iterations = 1000
    assert abs(decayed_lr(o) - R.decayed_lr(0.1, 1000, 1e-2)) <= 1e-6 * R.decayed_lr(0.1, 1000, 1e-2)


def test_user_schedule_is_called_once_per_step():
    S = _S()
    calls = []

    class Halve(S.LearningRateSchedule):
        def __call__(self, step):
            calls.append(step)
            return 0.5 ** step

    o = _optimizers()[1](Halve())
    for _ in range(4):
        o.step([])
    assert calls == [0, 1, 2, 3] and o.lr_t == 0.125


def test_engine_rate_hook_counts_every_step_once():
    """lowering._lr_step: what the fused engine calls once per training step."""
    from handyrec_b200.lowering import _lr_step

    S = _S()
    for cls in _optimizers():
        o = cls(S.InverseTimeDecay(0.1, 2, 1.0), decay=0.1)
        o.iterations = 3  # e.g. three layer-path steps before the engine was built
        hook = _lr_step(o)
        got = [hook() for _ in range(4)]
        want = [R.decayed_lr(lambda s: R.inverse_time_decay(s, 0.1, 2, 1.0), it, 0.1) for it in range(3, 7)]
        assert all(abs(g - w) <= 1e-6 * w for g, w in zip(got, want))
        assert o.iterations == 7 and o.lr_t == got[-1]
        f = cls(0.05)
        assert [_lr_step(f)() for _ in range(2)] == [0.05, 0.05] and f.iterations == 2


def test_engine_set_lr_recomputes_the_ftrl_kernel_l2():
    """DeepFMEngine.set_lr without a device: the Ftrl l2 follows the rate (beta / (2 * lr)), a zero rate divides as in TF."""
    from handyrec_b200.engine import DeepFMEngine

    eng = DeepFMEngine.__new__(DeepFMEngine)
    eng.ftrl_l2_reg, eng.beta = 0.01, 0.2
    eng.set_lr(0.1)
    assert eng.lr == 0.1 and eng.ftrl_l2 == 0.01 + 0.2 / (2 * 0.1)
    eng.set_lr(0.0)
    assert eng.ftrl_l2 == math.inf
    eng.beta = 0.0
    eng.set_lr(0.5)
    assert eng.ftrl_l2 == 0.01


def test_compat_shim_exposes_the_schedules():
    from handyrec_b200 import compat, schedules

    try:
        compat.install(force=True)
        import tensorflow as tf
        from tensorflow.keras.experimental import CosineDecay, CosineDecayRestarts
        from tensorflow.keras.optimizers.schedules import (ExponentialDecay, InverseTimeDecay, LearningRateSchedule,
                                                           PiecewiseConstantDecay, PolynomialDecay)

        assert tf.keras.optimizers.schedules.ExponentialDecay is schedules.ExponentialDecay is ExponentialDecay
        assert (InverseTimeDecay, PiecewiseConstantDecay, PolynomialDecay, LearningRateSchedule) == (
            schedules.InverseTimeDecay, schedules.PiecewiseConstantDecay, schedules.PolynomialDecay, schedules.LearningRateSchedule)
        assert (CosineDecay, CosineDecayRestarts) == (schedules.CosineDecay, schedules.CosineDecayRestarts)
        assert tf.keras.experimental.CosineDecay is CosineDecay
        opt = tf.keras.optimizers.Adam(learning_rate=ExponentialDecay(1e-3, 1000, 0.96), decay=1e-6)
        assert isinstance(opt.lr, LearningRateSchedule) and opt.decay == 1e-6
    finally:
        compat.uninstall()
