"""CPU: Keras callbacks (handyrec_b200.callbacks) driven with a stub model and scripted logs -- EarlyStopping, ReduceLROnPlateau,
LearningRateScheduler, ModelCheckpoint, CSVLogger, TerminateOnNaN, LambdaCallback, the batch-hook detection, the compat shim's
names, and the refusal of batch-hook callbacks on a multi-GPU compile."""
import csv

import numpy as np
import pytest
import torch

from handyrec_b200 import callbacks as C
from handyrec_b200 import keras_lite as KL


class _Stub:
    """What the callbacks touch on a model: optimizer, stop_training, get/set_weights, save_weights, the rate setter."""

    _fused = None
    _set_learning_rate = KL.Model._set_learning_rate

    def __init__(self, optimizer=None):
        self.optimizer = optimizer if optimizer is not None else KL.Adam(0.01)
        self.stop_training = False
        self.version = 0  # the "weights": the epoch they come from
        self.calls = []
        self.saved = []

    def get_weights(self):
        self.calls.append(("get", self.version))
        return [np.array([self.version], dtype=np.float32)]

    def set_weights(self, w):
        self.calls.append(("set", int(w[0][0])))
        self.version = int(w[0][0])

    def save_weights(self, path, **kw):
        self.saved.append(path)


def _drive(cb, model, values, key="val_loss"):
    """fit's epoch loop over scripted monitor values; returns the epoch after which training stopped (or None)."""
    cb.set_model(model)
    model.stop_training = False
    cb.on_train_begin()
    for e, v in enumerate(values):
        model.version = e
        cb.on_epoch_begin(e)
        cb.on_epoch_end(e, {key: v} if v is not None else {"loss": 1.0})
        if model.stop_training:
            return e
    cb.on_train_end()
    return None


# ---- EarlyStopping --------------------------------------------------------------------------------------------------------------
def test_early_stopping_modes():
    assert _drive(C.EarlyStopping(patience=1), _Stub(), [1.0, 0.9, 0.95, 0.8]) == 2  # val_loss: min
    assert _drive(C.EarlyStopping(monitor="val_acc", patience=1), _Stub(), [0.5, 0.6, 0.55], key="val_acc") == 2  # "acc": max
    # val_auc minimises in auto mode, as in Keras 2.6 (only "acc" in the name means max)
    assert _drive(C.EarlyStopping(monitor="val_auc", patience=0), _Stub(), [0.7, 0.8], key="val_auc") == 1
    assert _drive(C.EarlyStopping(monitor="val_auc", mode="max", patience=0), _Stub(), [0.7, 0.8, 0.75], key="val_auc") == 2
    assert C.EarlyStopping(mode="bogus").monitor_op is np.less  # unknown mode -> auto


def test_early_stopping_min_delta_takes_the_sign_of_the_mode():
    es = C.EarlyStopping(min_delta=-0.1)
    assert es.min_delta == -0.1
    assert _drive(C.EarlyStopping(min_delta=0.1, patience=0), _Stub(), [1.0, 0.95]) == 1  # 0.05 better: not enough
    assert _drive(C.EarlyStopping(min_delta=0.1, patience=0), _Stub(), [1.0, 0.85, 0.7]) is None
    es = C.EarlyStopping(monitor="acc", min_delta=0.1)
    assert es.min_delta == 0.1
    assert _drive(C.EarlyStopping(monitor="acc", min_delta=0.1, patience=0), _Stub(), [0.5, 0.55], key="acc") == 1


def test_early_stopping_patience_and_baseline():
    assert _drive(C.EarlyStopping(patience=2), _Stub(), [1.0, 1.1, 1.2, 0.5]) == 2
    assert _drive(C.EarlyStopping(patience=2), _Stub(), [1.0, 1.1, 0.9, 1.0, 1.0]) == 4
    # the baseline is the best to beat from the start
    assert _drive(C.EarlyStopping(patience=1, baseline=0.5), _Stub(), [0.9, 0.8]) == 0
    assert _drive(C.EarlyStopping(patience=1, baseline=0.5), _Stub(), [0.4, 0.45, 0.3]) == 1
    es = C.EarlyStopping(patience=1)
    m = _Stub()
    _drive(es, m, [1.0, 2.0])
    assert es.stopped_epoch == 1
    _drive(es, m, [1.0, 0.5])  # re-used: on_train_begin resets it
    assert es.wait == 0 and es.stopped_epoch == 0


def test_early_stopping_missing_monitor_does_nothing(caplog):
    m = _Stub()
    with caplog.at_level("WARNING"):
        assert _drive(C.EarlyStopping(patience=0, restore_best_weights=True), m, [None, None, None]) is None
    assert "not available" in caplog.text
    assert m.calls == []


def test_early_stopping_restores_the_best_weights():
    m = _Stub()
    assert _drive(C.EarlyStopping(patience=2, restore_best_weights=True), m, [1.0, 0.7, 0.9, 0.8]) == 3
    # snapshot at the first epoch end, again at the improvement (epoch 1); restored once, when it stops
    assert m.calls == [("get", 0), ("get", 0), ("get", 1), ("set", 1)]
    m = _Stub()
    assert _drive(C.EarlyStopping(patience=1, restore_best_weights=True, baseline=0.5), m, [0.9, 0.8]) == 0
    assert m.calls == [("get", 0), ("set", 0)]  # nothing improved on the baseline: the first epoch's weights come back
    m = _Stub()
    assert _drive(C.EarlyStopping(patience=5, restore_best_weights=True), m, [1.0, 0.9, 1.2]) is None
    assert ("set", 1) not in m.calls and all(c[0] == "get" for c in m.calls)  # never stopped: never restored


# ---- ReduceLROnPlateau ----------------------------------------------------------------------------------------------------------
def _plateau(cb, m, values):
    cb.set_model(m)
    cb.on_train_begin()
    lrs, logged = [], []
    for e, v in enumerate(values):
        logs = {"val_loss": v}
        cb.on_epoch_end(e, logs)
        logged.append(logs["lr"])
        lrs.append(m.optimizer.lr)
    return lrs, logged


def test_reduce_lr_on_plateau_rates_are_float32():
    m = _Stub(KL.Adam(0.01))
    lrs, logged = _plateau(C.ReduceLROnPlateau(factor=0.3, patience=1), m, [1.0, 1.0, 1.0, 1.0])
    want1 = float(np.float32(float(np.float32(0.01)) * 0.3))
    want2 = float(np.float32(want1 * 0.3))
    want3 = float(np.float32(want2 * 0.3))
    assert lrs == [0.01, want1, want2, want3]  # no cooldown: every epoch without improvement after the first cuts the rate
    assert logged == [float(np.float32(0.01)), float(np.float32(0.01)), want1, want2]  # the rate in use during the epoch
    assert all(isinstance(x, float) and x == np.float32(x) for x in lrs[1:])


def test_reduce_lr_on_plateau_cooldown_and_min_lr():
    m = _Stub(KL.SGD(1.0))
    lrs, _ = _plateau(C.ReduceLROnPlateau(factor=0.5, patience=1, cooldown=2, min_lr=0.2), m, [1.0] * 9)
    # Keras' counters: a cut at epoch 1 sets cooldown 2; epoch 2 counts it down to 1 (no cut), epoch 3 to 0 and, out of cooldown,
    # waits 1 = patience: cut.  Epoch 5 would cut to 0.125 and takes min_lr; at min_lr nothing is cut any more.
    lo = float(np.float32(0.2))
    assert lrs == [1.0, 0.5, 0.5, 0.25, 0.25, lo, lo, lo, lo]
    m = _Stub(KL.SGD(1.0))
    lrs, _ = _plateau(C.ReduceLROnPlateau(factor=0.5, patience=2, min_delta=0.1), m, [1.0, 0.95, 0.85, 0.84, 0.83])
    assert lrs == [1.0, 1.0, 1.0, 1.0, 0.5]  # 0.85 beats 1.0 - 0.1; 0.84 / 0.83 do not beat 0.85 - 0.1
    with pytest.raises(ValueError, match="factor >= 1.0"):
        C.ReduceLROnPlateau(factor=1.0)
    assert C.ReduceLROnPlateau(epsilon=0.5).min_delta == 0.5


def test_lr_callbacks_refuse_a_schedule_optimizer():
    from handyrec_b200.schedules import ExponentialDecay

    for cb in (C.ReduceLROnPlateau(), C.LearningRateScheduler(lambda e: 0.1)):
        m = _Stub(KL.Adam(ExponentialDecay(0.1, 10, 0.5)))
        cb.set_model(m)
        with pytest.raises(ValueError, match="ExponentialDecay"):
            cb.on_train_begin()


# ---- LearningRateScheduler -----------------------------------------------------------------------------------------------------
def test_learning_rate_scheduler_one_and_two_arguments():
    m = _Stub(KL.SGD(0.1))
    seen = []

    def two(epoch, lr):
        seen.append((epoch, lr))
        return lr * 0.5

    cb = C.LearningRateScheduler(two)
    cb.set_model(m)
    cb.on_train_begin()
    for e in range(3):
        cb.on_epoch_begin(e)
        logs = {}
        cb.on_epoch_end(e, logs)
        assert logs["lr"] == m.optimizer.lr
    assert seen[0] == (0, float(np.float32(0.1)))
    assert m.optimizer.lr == float(np.float32(seen[2][1] * 0.5))
    cb = C.LearningRateScheduler(lambda epoch: 0.01 * (epoch + 1))  # one argument: the TypeError of the first call falls back
    cb.set_model(m)
    cb.on_epoch_begin(2)
    assert m.optimizer.lr == float(np.float32(0.03))
    cb = C.LearningRateScheduler(lambda epoch, lr: np.float64(0.25))
    cb.set_model(m)
    cb.on_epoch_begin(0)
    assert m.optimizer.lr == 0.25


def test_learning_rate_scheduler_refuses_a_non_float():
    m = _Stub(KL.SGD(0.1))
    for bad in (lambda e, lr: 1, lambda e, lr: "0.1", lambda e, lr: None):
        cb = C.LearningRateScheduler(bad)
        cb.set_model(m)
        with pytest.raises(ValueError, match="should be float"):
            cb.on_epoch_begin(0)


def test_rate_setter_keeps_iterations_and_decay():
    opt = KL.Adam(0.01, decay=0.5)
    opt.iterations = 4
    m = _Stub(opt)
    m._set_learning_rate(0.1)
    assert opt.iterations == 4 and opt.lr == float(np.float32(0.1))
    assert opt.lr_t == float(np.float32(np.float32(0.1) / (np.float32(1.0) + np.float32(0.5) * np.float32(4))))


# ---- ModelCheckpoint ------------------------------------------------------------------------------------------------------------
def test_model_checkpoint_filepath_and_save_best_only(tmp_path):
    m = _Stub()
    cb = C.ModelCheckpoint(str(tmp_path / "w.{epoch:02d}-{val_loss:.2f}"), save_weights_only=True)
    _drive(cb, m, [0.5, 0.25])
    assert m.saved == [str(tmp_path / "w.01-0.50"), str(tmp_path / "w.02-0.25")]
    m = _Stub()
    cb = C.ModelCheckpoint("ck{epoch}", save_best_only=True, save_weights_only=True)
    _drive(cb, m, [1.0, 0.8, 0.9, 0.7])
    assert m.saved == ["ck1", "ck2", "ck4"]
    m = _Stub()
    cb = C.ModelCheckpoint("ck{epoch}", monitor="val_acc", save_best_only=True, save_weights_only=True)
    _drive(cb, m, [0.5, 0.4, 0.6], key="val_acc")
    assert m.saved == ["ck1", "ck3"]
    m = _Stub()
    _drive(C.ModelCheckpoint("ck{epoch}", save_best_only=True, save_weights_only=True), m, [None, None])
    assert m.saved == []  # monitor missing: skipped


def test_model_checkpoint_integer_save_freq():
    m = _Stub()
    cb = C.ModelCheckpoint("ck{epoch}-{loss:.1f}", save_freq=3, save_weights_only=True)
    assert cb._implements_train_batch_hooks()
    assert not C.ModelCheckpoint("x", save_weights_only=True)._implements_train_batch_hooks()
    cb.set_model(m)
    cb.on_train_begin()
    for e in range(2):
        cb.on_epoch_begin(e)
        for b in range(4):  # 4 batches an epoch: saves after batches 3 and 6 (epoch 1, batch 1)
            cb.on_train_batch_end(b, {"loss": float(b)})
        cb.on_epoch_end(e, {"loss": 1.0})
    assert m.saved == ["ck1-2.0", "ck2-1.0"]
    with pytest.raises(ValueError, match="save_freq"):
        C.ModelCheckpoint("x", save_weights_only=True, save_freq="batch")


def test_model_checkpoint_refuses_whole_model_saves():
    with pytest.raises(NotImplementedError, match="save_weights_only"):
        C.ModelCheckpoint("x")


# ---- CSVLogger, TerminateOnNaN, LambdaCallback -----------------------------------------------------------------------------------
def test_csv_logger(tmp_path):
    f = tmp_path / "log.csv"
    cb = C.CSVLogger(str(f))
    cb.set_model(_Stub())
    cb.on_train_begin()
    cb.on_epoch_end(0, {"val_loss": 0.5, "loss": 0.75, "auc": 0.625})
    cb.on_epoch_end(1, {"loss": 0.5, "auc": 0.75})
    cb.on_train_end()
    rows = list(csv.reader(open(f)))
    assert rows == [["epoch", "auc", "loss", "val_loss"], ["0", "0.625", "0.75", "0.5"], ["1", "0.75", "0.5", "NA"]]
    cb = C.CSVLogger(str(f), separator=";", append=True)
    cb.on_train_begin()
    cb.on_epoch_end(0, {"loss": 0.25})
    cb.on_train_end()
    assert open(f).read().splitlines()[-1] == "0;0.25"  # appended, no second header
    assert len(open(f).read().splitlines()) == 4


def test_terminate_on_nan():
    m = _Stub()
    cb = C.TerminateOnNaN()
    cb.set_model(m)
    cb.on_train_batch_end(0, {"loss": 0.5})
    assert not m.stop_training
    cb.on_train_batch_end(1, {"loss": float("inf")})
    assert m.stop_training
    m.stop_training = False
    cb.on_train_batch_end(2, {"loss": float("nan")})
    assert m.stop_training


def test_batch_hook_detection():
    class EpochOnly(C.Callback):
        def on_epoch_end(self, epoch, logs=None):
            pass

    class BatchAlias(C.Callback):
        def on_batch_end(self, batch, logs=None):
            pass

    class TrainBatch(C.Callback):
        def on_train_batch_begin(self, batch, logs=None):
            pass

    class TestBatch(C.Callback):
        def on_test_batch_end(self, batch, logs=None):
            pass

    epoch_level = [C.EarlyStopping(), C.ModelCheckpoint("x", save_best_only=True, save_weights_only=True), C.ReduceLROnPlateau(),
                   C.CSVLogger("x"), C.LearningRateScheduler(lambda e: 0.1), C.History(), EpochOnly(), TestBatch(),
                   C.LambdaCallback(on_epoch_end=lambda e, l: None)]
    assert not C.CallbackList(epoch_level).should_call_train_batch_hooks
    assert C.CallbackList([TestBatch()]).should_call_test_batch_hooks
    for cb in (C.TerminateOnNaN(), BatchAlias(), TrainBatch(), C.ModelCheckpoint("x", save_freq=5, save_weights_only=True),
               C.LambdaCallback(on_batch_end=lambda b, l: None), C.LambdaCallback(on_train_batch_begin=lambda b, l: None)):
        cl = C.CallbackList(epoch_level + [cb])
        assert cl.should_call_train_batch_hooks, cb
        assert cl.train_batch_hook_names() == [type(cb).__name__]
    with pytest.raises(TypeError):
        C.CallbackList([object()])
    with pytest.raises(TypeError, match="unknown hook"):
        C.LambdaCallback(on_something=lambda: None)


def test_callback_list_calls_in_order_and_skips_batch_hooks_nobody_implements():
    seen = []

    class Rec(C.Callback):
        def __init__(self, tag):
            super().__init__()
            self.tag = tag

        def on_epoch_end(self, epoch, logs=None):
            seen.append((self.tag, epoch, dict(logs)))

    m = _Stub()
    cl = C.CallbackList([Rec("a"), Rec("b")], model=m, epochs=3, verbose=0, steps=None)
    assert cl.callbacks[0].model is m and cl.callbacks[1].params == {"epochs": 3, "verbose": 0, "steps": None}
    cl.on_epoch_end(0, {"loss": 1.0})
    cl.on_train_batch_end(0, {"loss": 1.0})
    assert seen == [("a", 0, {"loss": 1.0}), ("b", 0, {"loss": 1.0})]
    h = C.History()
    h.set_model(m)
    h.on_train_begin()
    h.on_epoch_end(0, {"loss": 1.0, "lr": 0.5})
    h.on_epoch_end(1, {"loss": 0.5, "lr": 0.5})
    assert h.history == {"loss": [1.0, 0.5], "lr": [0.5, 0.5]} and h.epoch == [0, 1] and m.history is h


# ---- the shim -------------------------------------------------------------------------------------------------------------------
def test_shim_callbacks_module():
    from handyrec_b200 import compat

    compat.install(force=True)
    try:
        import tensorflow as tf
        from tensorflow.keras import callbacks as tkc
        from tensorflow.keras.callbacks import EarlyStopping, ModelCheckpoint

        assert tf.keras.callbacks is tkc
        assert EarlyStopping is C.EarlyStopping and ModelCheckpoint is C.ModelCheckpoint
        for n in C.__all__:
            assert getattr(tkc, n) is getattr(C, n)
        for n in ("TensorBoard", "ProgbarLogger", "BackupAndRestore", "RemoteMonitor"):
            with pytest.raises(NotImplementedError, match=n):
                getattr(tkc, n)()
            assert issubclass(getattr(tkc, n), C.Callback)
    finally:
        compat.uninstall()
    for n in C.__all__:
        assert getattr(KL, n) is getattr(C, n)


# ---- a multi-GPU compile ---------------------------------------------------------------------------------------------------------
class _FakeComm:
    def __init__(self, rank, n):
        self.rank, self.N = rank, n


def test_multi_gpu_fit_refuses_batch_hook_callbacks(monkeypatch):
    """Batch hooks on several GPUs raise at the start of fit, before any step, naming the callback; epoch-level ones are let
    through to training (which needs the GPU, so it is not run here)."""
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature
    from handyrec_b200.models import DeepFM

    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    torch.manual_seed(3)
    sparse = [SparseFeature(f"C{i}", v, 8) for i, v in enumerate((50, 7000))]
    pool = FeaturePool()
    m = DeepFM(FeatureGroup("fm", sparse, pool, l2_embd=0.0), FeatureGroup("dnn", [DenseFeature("I0")] + sparse, pool, l2_embd=0.0),
               dnn_hidden_units=(8, 1))
    m.compile(optimizer=KL.Adam(1e-3), loss=KL.binary_crossentropy, distribute=_FakeComm(0, 2))
    assert m._fused is not None
    x = {"C0": np.zeros((8, 1), np.int32), "C1": np.zeros((8, 1), np.int32), "I0": np.zeros((8, 1), np.float32)}
    y = np.zeros(8, np.float32)
    built = []
    monkeypatch.setattr(type(m._fused), "build", lambda *a, **k: built.append(1))
    for cb in (C.TerminateOnNaN(), C.ModelCheckpoint("x", save_freq=2, save_weights_only=True)):
        with pytest.raises(ValueError, match=type(cb).__name__):
            m.fit(x, y, batch_size=4, callbacks=[C.EarlyStopping(), cb])
    assert built == []
    m._comm = _FakeComm(0, 1)  # one rank: batch hooks are fine (they get as far as building the engine)
    with pytest.raises(Exception) as e:
        m.fit(x, y, batch_size=4, callbacks=[C.TerminateOnNaN()])
    assert "batch hooks" not in str(e.value) and built == [1]
