"""Keras 2.6 training callbacks (`tf.keras.callbacks`) for `keras_lite.Model.fit / evaluate / predict`.

Every hook runs on the host, at an epoch or batch boundary; no callback launches anything on the GPU.  The classes take Keras'
argument names and defaults, and each docstring states the rules it follows, as Keras 2.6 applies them.

How `fit` drives them (keras_lite.Model.fit):

    on_train_begin -> per epoch: on_epoch_begin -> per batch: on_train_batch_begin(b) / on_train_batch_end(b, logs)
    -> [validation: on_test_begin -> on_test_batch_begin / _end -> on_test_end] -> on_epoch_end(e, logs) -> on_train_end

`model.stop_training` is reset at `on_train_begin`; it is checked after every batch end and every epoch end.  Epoch logs are the
values `fit` records in `history`: `loss`, the compiled metrics, `val_loss` and `val_<metric>`.  Batch logs carry the epoch's
running sample-count-weighted mean loss and the running metric results.  Batch hooks run only when some callback overrides one
(`CallbackList.should_call_train_batch_hooks`, Keras' `_implements_train_batch_hooks`): on the fused engine they cost one host
sync per step, and without them the engine runs its usual one-step-ahead pipeline.
"""
from __future__ import annotations

import csv
import logging
import os
from collections import OrderedDict
from typing import Callable, Dict, Iterable, List, Optional

import numpy as np

__all__ = ["Callback", "CallbackList", "History", "EarlyStopping", "ModelCheckpoint", "ReduceLROnPlateau", "LearningRateScheduler",
           "TerminateOnNaN", "CSVLogger", "LambdaCallback"]

_log = logging.getLogger(__name__)


def _default(fn):
    """Marks a base-class hook that does nothing; a subclass or an instance attribute that replaces it implements the hook."""
    fn._is_default = True
    return fn


class Callback:
    """tf.keras.callbacks.Callback: `model` and `params` are set by `fit` / `evaluate` / `predict` before the first hook runs."""

    def __init__(self):
        self.model = None
        self.params: Dict = {}

    def set_params(self, params) -> None:
        self.params = params

    def set_model(self, model) -> None:
        self.model = model

    @_default
    def on_batch_begin(self, batch, logs=None):
        """Alias of on_train_batch_begin."""

    @_default
    def on_batch_end(self, batch, logs=None):
        """Alias of on_train_batch_end."""

    @_default
    def on_epoch_begin(self, epoch, logs=None):
        pass

    @_default
    def on_epoch_end(self, epoch, logs=None):
        pass

    @_default
    def on_train_batch_begin(self, batch, logs=None):
        self.on_batch_begin(batch, logs=logs)

    @_default
    def on_train_batch_end(self, batch, logs=None):
        self.on_batch_end(batch, logs=logs)

    @_default
    def on_test_batch_begin(self, batch, logs=None):
        pass

    @_default
    def on_test_batch_end(self, batch, logs=None):
        pass

    @_default
    def on_predict_batch_begin(self, batch, logs=None):
        pass

    @_default
    def on_predict_batch_end(self, batch, logs=None):
        pass

    @_default
    def on_train_begin(self, logs=None):
        pass

    @_default
    def on_train_end(self, logs=None):
        pass

    @_default
    def on_test_begin(self, logs=None):
        pass

    @_default
    def on_test_end(self, logs=None):
        pass

    @_default
    def on_predict_begin(self, logs=None):
        pass

    @_default
    def on_predict_end(self, logs=None):
        pass

    def _implements_hook(self, *names: str) -> bool:
        return any(not getattr(getattr(self, n), "_is_default", False) for n in names)

    def _implements_train_batch_hooks(self) -> bool:
        return self._implements_hook("on_batch_begin", "on_batch_end", "on_train_batch_begin", "on_train_batch_end")

    def _implements_test_batch_hooks(self) -> bool:
        return self._implements_hook("on_test_batch_begin", "on_test_batch_end")

    def _implements_predict_batch_hooks(self) -> bool:
        return self._implements_hook("on_predict_batch_begin", "on_predict_batch_end")


class CallbackList:
    """The callbacks of one `fit` / `evaluate` / `predict` call, called in list order.  `should_call_train_batch_hooks` (and the test /
    predict ones) say whether any callback implements a batch hook of that kind; when none does, the batch hooks are skipped and
    the caller need not form batch logs."""

    def __init__(self, callbacks: Optional[Iterable[Callback]] = None, model=None, **params):
        self.callbacks: List[Callback] = list(callbacks or [])
        for cb in self.callbacks:
            if not isinstance(cb, Callback):
                raise TypeError(f"callbacks must be tf.keras.callbacks.Callback instances, got {cb!r}")
            if model is not None:
                cb.set_model(model)
            cb.set_params(dict(params))
        self.should_call_train_batch_hooks = any(cb._implements_train_batch_hooks() for cb in self.callbacks)
        self.should_call_test_batch_hooks = any(cb._implements_test_batch_hooks() for cb in self.callbacks)
        self.should_call_predict_batch_hooks = any(cb._implements_predict_batch_hooks() for cb in self.callbacks)

    def train_batch_hook_names(self) -> List[str]:
        return [type(cb).__name__ for cb in self.callbacks if cb._implements_train_batch_hooks()]

    def _call(self, hook: str, *args) -> None:
        for cb in self.callbacks:
            getattr(cb, hook)(*args)

    def on_train_begin(self, logs=None):
        self._call("on_train_begin", logs)

    def on_train_end(self, logs=None):
        self._call("on_train_end", logs)

    def on_epoch_begin(self, epoch, logs=None):
        self._call("on_epoch_begin", epoch, logs)

    def on_epoch_end(self, epoch, logs=None):
        self._call("on_epoch_end", epoch, logs)

    def on_train_batch_begin(self, batch, logs=None):
        if self.should_call_train_batch_hooks:
            self._call("on_train_batch_begin", batch, logs)

    def on_train_batch_end(self, batch, logs=None):
        if self.should_call_train_batch_hooks:
            self._call("on_train_batch_end", batch, logs)

    def on_test_begin(self, logs=None):
        self._call("on_test_begin", logs)

    def on_test_end(self, logs=None):
        self._call("on_test_end", logs)

    def on_test_batch_begin(self, batch, logs=None):
        if self.should_call_test_batch_hooks:
            self._call("on_test_batch_begin", batch, logs)

    def on_test_batch_end(self, batch, logs=None):
        if self.should_call_test_batch_hooks:
            self._call("on_test_batch_end", batch, logs)

    def on_predict_begin(self, logs=None):
        self._call("on_predict_begin", logs)

    def on_predict_end(self, logs=None):
        self._call("on_predict_end", logs)

    def on_predict_batch_begin(self, batch, logs=None):
        if self.should_call_predict_batch_hooks:
            self._call("on_predict_batch_begin", batch, logs)

    def on_predict_batch_end(self, batch, logs=None):
        if self.should_call_predict_batch_hooks:
            self._call("on_predict_batch_end", batch, logs)


class History(Callback):
    """What `fit` returns.  `history`: {log key: [value per epoch]}; `epoch`: the epoch indices; `params`: {"verbose", "epochs",
    "steps"}.  It runs after every callback given to `fit`, so it records the `lr` key the learning-rate callbacks add."""

    def __init__(self):
        super().__init__()
        self.history: Dict[str, list] = {}
        self.epoch: List[int] = []

    def on_train_begin(self, logs=None):
        self.epoch = []

    def on_epoch_end(self, epoch, logs=None):
        self.epoch.append(epoch)
        for k, v in (logs or {}).items():
            self.history.setdefault(k, []).append(v)
        self.model.history = self


def _monitor_op(monitor: str, mode: str, cls: str):
    """(np.less or np.greater) for `mode`; "auto" maximises exactly when "acc" is in the monitor's name (Keras 2.6), so val_auc
    minimises in auto mode.  An unknown mode warns and falls back to "auto"."""
    if mode not in ("auto", "min", "max"):
        _log.warning("%s mode %s is unknown, fallback to auto mode.", cls, mode)
        mode = "auto"
    if mode == "min" or (mode == "auto" and "acc" not in monitor):
        return np.less
    return np.greater


class EarlyStopping(Callback):
    """Stop training when `monitor` has stopped improving (Keras 2.6).

    - `mode`: "min", "max" or "auto" ("max" iff "acc" is in the monitor name).  `min_delta` takes the sign of the mode: a value
      improves on the best when `current < best - |min_delta|` ("min") or `current > best + |min_delta|` ("max").
    - At `on_train_begin` the best is `baseline`, or +-inf without one; the wait counter and `stopped_epoch` are 0.
    - At every epoch end with the monitor in the logs: an improvement sets best and resets the wait; otherwise the wait grows by
      one, and once it reaches `patience` the callback sets `model.stop_training` and records `stopped_epoch`.
    - A monitor missing from the logs logs a warning and does nothing.
    - `restore_best_weights`: the first epoch end snapshots `model.get_weights()`, so those weights are restored if no later epoch
      improves; every improvement snapshots again.  The snapshot is restored (`model.set_weights`) only when this callback stops
      training."""

    def __init__(self, monitor="val_loss", min_delta=0, patience=0, verbose=0, mode="auto", baseline=None, restore_best_weights=False):
        super().__init__()
        self.monitor, self.patience, self.verbose, self.baseline = monitor, patience, verbose, baseline
        self.restore_best_weights = restore_best_weights
        self.monitor_op = _monitor_op(monitor, mode, "EarlyStopping")
        self.min_delta = abs(min_delta) * (1 if self.monitor_op == np.greater else -1)
        self.wait = self.stopped_epoch = 0
        self.best_weights = None

    def on_train_begin(self, logs=None):
        self.wait = 0
        self.stopped_epoch = 0
        if self.baseline is not None:
            self.best = self.baseline
        else:
            self.best = np.inf if self.monitor_op == np.less else -np.inf
        self.best_weights = None

    def on_epoch_end(self, epoch, logs=None):
        current = (logs or {}).get(self.monitor)
        if current is None:
            _log.warning("Early stopping conditioned on metric `%s` which is not available. Available metrics are: %s",
                         self.monitor, ",".join((logs or {}).keys()))
            return
        if self.restore_best_weights and self.best_weights is None:
            self.best_weights = self.model.get_weights()
        if self.monitor_op(current - self.min_delta, self.best):
            self.best = current
            self.wait = 0
            if self.restore_best_weights:
                self.best_weights = self.model.get_weights()
        else:
            self.wait += 1
            if self.wait >= self.patience:
                self.stopped_epoch = epoch
                self.model.stop_training = True
                if self.restore_best_weights and self.best_weights is not None:
                    if self.verbose > 0:
                        print("Restoring model weights from the end of the best epoch.")
                    self.model.set_weights(self.best_weights)

    def on_train_end(self, logs=None):
        if self.stopped_epoch > 0 and self.verbose > 0:
            print("Epoch %05d: early stopping" % (self.stopped_epoch + 1))


class ModelCheckpoint(Callback):
    """Save the model's weights with `Model.save_weights` (handyrec_b200.checkpoint: a directory of `.npy` files; a row-sharded
    model writes its per-rank layout, every rank saving its own rows) (Keras 2.6).

    - The path is `filepath.format(epoch=epoch + 1, **logs)`.
    - `save_freq="epoch"` saves at every epoch end; an integer saves after every `save_freq` training batches, counted across
      epochs (a batch index at or below the last one seen starts a new epoch and counts batch + 1), with the batch logs.  An
      integer makes this a batch-hook callback.
    - `save_best_only`: saves only when the monitor improves on the best seen so far (`mode` as EarlyStopping, no min_delta; best
      starts at +-inf); a monitor missing from the logs logs a warning and skips the save.
    - `save_weights_only=False` raises NotImplementedError: there is no `Model.save` (whole-model serialisation)."""

    def __init__(self, filepath, monitor="val_loss", verbose=0, save_best_only=False, save_weights_only=False, mode="auto",
                 save_freq="epoch"):
        super().__init__()
        if not save_weights_only:
            raise NotImplementedError("ModelCheckpoint(save_weights_only=False): there is no Model.save here; pass "
                                      "save_weights_only=True (the checkpoint is Model.save_weights' directory)")
        if save_freq != "epoch" and not (isinstance(save_freq, int) and save_freq > 0):
            raise ValueError(f"Unrecognized save_freq: {save_freq}")
        self.filepath, self.monitor, self.verbose = os.fspath(filepath), monitor, verbose
        self.save_best_only, self.save_weights_only, self.save_freq = save_best_only, save_weights_only, save_freq
        self.monitor_op = _monitor_op(monitor, mode, "ModelCheckpoint")
        self.best = np.inf if self.monitor_op == np.less else -np.inf
        self._current_epoch = 0
        self._batches_seen_since_last_saving = 0
        self._last_batch_seen = 0

    def _implements_train_batch_hooks(self) -> bool:
        return self.save_freq != "epoch"

    def on_epoch_begin(self, epoch, logs=None):
        self._current_epoch = epoch

    def on_train_batch_end(self, batch, logs=None):
        if self._should_save_on_batch(batch):
            self._save_model(self._current_epoch, logs)

    def on_epoch_end(self, epoch, logs=None):
        if self.save_freq == "epoch":
            self._save_model(epoch, logs)

    def _should_save_on_batch(self, batch) -> bool:
        if self.save_freq == "epoch":
            return False
        add = batch + 1 if batch <= self._last_batch_seen else batch - self._last_batch_seen
        self._batches_seen_since_last_saving += add
        self._last_batch_seen = batch
        if self._batches_seen_since_last_saving >= self.save_freq:
            self._batches_seen_since_last_saving = 0
            return True
        return False

    def _save_model(self, epoch, logs) -> None:
        logs = logs or {}
        path = self.filepath.format(epoch=epoch + 1, **logs)
        if self.save_best_only:
            current = logs.get(self.monitor)
            if current is None:
                _log.warning("Can save best model only with %s available, skipping.", self.monitor)
                return
            if not self.monitor_op(current, self.best):
                if self.verbose > 0:
                    print(f"\nEpoch {epoch + 1:05d}: {self.monitor} did not improve from {self.best:0.5f}")
                return
            if self.verbose > 0:
                print(f"\nEpoch {epoch + 1:05d}: {self.monitor} improved from {self.best:0.5f} to {current:0.5f}, saving model to {path}")
            self.best = current
        elif self.verbose > 0:
            print(f"\nEpoch {epoch + 1:05d}: saving model to {path}")
        self.model.save_weights(path, overwrite=True)


def _float_rate(model, cls: str) -> float:
    from .schedules import LearningRateSchedule

    lr = getattr(model.optimizer, "lr", None)
    if isinstance(lr, LearningRateSchedule):
        raise ValueError(f"{cls}: the optimizer's learning rate is the schedule {type(lr).__name__}, which has no float rate to "
                         "change; compile with a float learning rate or drop the callback")
    if lr is None:
        raise ValueError('Optimizer must have a "lr" attribute.')
    return float(np.float32(lr))


class ReduceLROnPlateau(Callback):
    """Reduce the learning rate when `monitor` has stopped improving (Keras 2.6).

    - `factor >= 1` raises ValueError.  `mode` as EarlyStopping; an improvement is `current < best - min_delta` ("min") or
      `current > best + min_delta` ("max").  At `on_train_begin` best is +-inf and the wait and cooldown counters are 0.
    - At every epoch end: `logs["lr"]` is set to the rate in use (float32).  With the monitor in the logs: while in cooldown, the
      cooldown counter drops by one and the wait is reset; an improvement sets best and resets the wait; otherwise, out of
      cooldown, the wait grows by one and, once it reaches `patience`, a rate above float32(min_lr) becomes
      `max(old * factor, min_lr)` rounded to float32 (Keras' rate is a float32 variable), the cooldown counter is set to
      `cooldown` and the wait reset.  A missing monitor logs a warning.
    - The new rate takes effect at the next training step, on the fused engine without rebuilding it: its optimizer slots and
      the optimizer's `iterations` carry on.
    - An optimizer built on a LearningRateSchedule has no float rate: ValueError at `on_train_begin`."""

    def __init__(self, monitor="val_loss", factor=0.1, patience=10, verbose=0, mode="auto", min_delta=1e-4, cooldown=0, min_lr=0,
                 **kwargs):
        super().__init__()
        if "epsilon" in kwargs:  # Keras' deprecated name of min_delta
            min_delta = kwargs.pop("epsilon")
        if kwargs:
            raise TypeError(f"ReduceLROnPlateau: unexpected arguments {sorted(kwargs)}")
        if factor >= 1.0:
            raise ValueError("ReduceLROnPlateau does not support a factor >= 1.0.")
        self.monitor, self.factor, self.min_lr, self.min_delta = monitor, float(factor), min_lr, min_delta
        self.patience, self.verbose, self.cooldown, self.mode = patience, verbose, cooldown, mode
        self._reset()

    def _reset(self) -> None:
        op = _monitor_op(self.monitor, self.mode, "ReduceLROnPlateau")
        if op == np.less:
            self.monitor_op = lambda a, b: np.less(a, b - self.min_delta)
            self.best = np.inf
        else:
            self.monitor_op = lambda a, b: np.greater(a, b + self.min_delta)
            self.best = -np.inf
        self.cooldown_counter = 0
        self.wait = 0

    def in_cooldown(self) -> bool:
        return self.cooldown_counter > 0

    def on_train_begin(self, logs=None):
        _float_rate(self.model, "ReduceLROnPlateau")
        self._reset()

    def on_epoch_end(self, epoch, logs=None):
        logs = logs if logs is not None else {}
        logs["lr"] = _float_rate(self.model, "ReduceLROnPlateau")
        current = logs.get(self.monitor)
        if current is None:
            _log.warning("Learning rate reduction is conditioned on metric `%s` which is not available. Available metrics are: %s",
                         self.monitor, ",".join(logs.keys()))
            return
        if self.in_cooldown():
            self.cooldown_counter -= 1
            self.wait = 0
        if self.monitor_op(current, self.best):
            self.best = current
            self.wait = 0
        elif not self.in_cooldown():
            self.wait += 1
            if self.wait >= self.patience:
                old = _float_rate(self.model, "ReduceLROnPlateau")
                if old > np.float32(self.min_lr):
                    new = max(old * self.factor, self.min_lr)
                    self.model._set_learning_rate(new)
                    if self.verbose > 0:
                        print(f"\nEpoch {epoch + 1:05d}: ReduceLROnPlateau reducing learning rate to {float(np.float32(new))}.")
                    self.cooldown_counter = self.cooldown
                    self.wait = 0


class LearningRateScheduler(Callback):
    """Set the learning rate at every epoch begin from `schedule` (Keras 2.6).

    - `schedule(epoch, lr)` with the current rate as a float (epoch counted from 0); if that call raises TypeError,
      `schedule(epoch)`.  A result that is not a Python float, np.float32 or np.float64 raises ValueError.  The rate is stored
      rounded to float32, as Keras' rate variable holds it, and takes effect at the next step (on the fused engine without a
      rebuild, as ReduceLROnPlateau).
    - At every epoch end `logs["lr"]` is the rate in use (float32).
    - An optimizer built on a LearningRateSchedule has no float rate: ValueError at `on_train_begin`."""

    def __init__(self, schedule: Callable, verbose=0):
        super().__init__()
        self.schedule, self.verbose = schedule, verbose

    def on_train_begin(self, logs=None):
        _float_rate(self.model, "LearningRateScheduler")

    def on_epoch_begin(self, epoch, logs=None):
        lr = _float_rate(self.model, "LearningRateScheduler")
        try:
            lr = self.schedule(epoch, lr)
        except TypeError:
            lr = self.schedule(epoch)
        if not isinstance(lr, (float, np.float32, np.float64)):
            raise ValueError('The output of the "schedule" function should be float.')
        self.model._set_learning_rate(lr)
        if self.verbose > 0:
            print(f"\nEpoch {epoch + 1:05d}: LearningRateScheduler setting learning rate to {lr}.")

    def on_epoch_end(self, epoch, logs=None):
        if logs is not None:
            logs["lr"] = _float_rate(self.model, "LearningRateScheduler")


class TerminateOnNaN(Callback):
    """Set `model.stop_training` after a training batch whose logged loss (the epoch's running mean) is NaN or +-inf, so no further
    batch runs (Keras 2.6).  A batch-hook callback: on the fused engine every step's loss is then read back before the next step
    is issued."""

    def on_batch_end(self, batch, logs=None):
        loss = (logs or {}).get("loss")
        if loss is not None and (np.isnan(loss) or np.isinf(loss)):
            print("Batch %d: Invalid loss, terminating training" % batch)
            self.model.stop_training = True


class CSVLogger(Callback):
    """Stream the epoch logs to a CSV file (Keras 2.6): columns "epoch" then the log keys in sorted order, fixed by the first epoch
    (a key missing later is written "NA"); `append=True` appends to an existing file without repeating the header.  A value
    that is a sequence is written as its string form in quotes."""

    def __init__(self, filename, separator=",", append=False):
        super().__init__()
        self.filename, self.sep, self.append = os.fspath(filename), separator, append
        self.writer = self.keys = self.csv_file = None
        self.append_header = True

    def on_train_begin(self, logs=None):
        if self.append:
            if os.path.exists(self.filename):
                with open(self.filename) as f:
                    self.append_header = not bool(len(f.readline()))
            mode = "a"
        else:
            mode = "w"
        self.csv_file = open(self.filename, mode, newline="")
        self.writer, self.keys = None, None

    def on_epoch_end(self, epoch, logs=None):
        logs = logs or {}

        def handle(k):
            is_zero_dim = isinstance(k, np.ndarray) and k.ndim == 0
            if isinstance(k, str):
                return k
            if hasattr(k, "__iter__") and not is_zero_dim:
                return '"[%s]"' % (", ".join(map(str, k)))
            return k

        if self.keys is None:
            self.keys = sorted(logs.keys())
        if self.writer is None:
            self.writer = csv.DictWriter(self.csv_file, fieldnames=["epoch"] + self.keys, delimiter=self.sep)
            if self.append_header:
                self.writer.writeheader()
        row = OrderedDict({"epoch": epoch})
        row.update((k, handle(logs[k]) if k in logs else "NA") for k in self.keys)
        self.writer.writerow(row)
        self.csv_file.flush()

    def on_train_end(self, logs=None):
        if self.csv_file is not None:
            self.csv_file.close()
        self.writer = None


class LambdaCallback(Callback):
    """A callback from plain functions (Keras 2.6): `on_epoch_begin(epoch, logs)`, `on_epoch_end(epoch, logs)`,
    `on_batch_begin(batch, logs)`, `on_batch_end(batch, logs)`, `on_train_begin(logs)`, `on_train_end(logs)`, and any other hook
    by its name as a keyword.  Unlike Keras, a LambdaCallback without a batch function is not a batch-hook callback, so it does
    not make the fused engine read back every step's loss."""

    def __init__(self, on_epoch_begin=None, on_epoch_end=None, on_batch_begin=None, on_batch_end=None, on_train_begin=None,
                 on_train_end=None, **kwargs):
        super().__init__()
        given = dict(on_epoch_begin=on_epoch_begin, on_epoch_end=on_epoch_end, on_batch_begin=on_batch_begin, on_batch_end=on_batch_end,
                     on_train_begin=on_train_begin, on_train_end=on_train_end, **kwargs)
        for name, fn in given.items():
            if not name.startswith("on_") or not hasattr(Callback, name):
                raise TypeError(f"LambdaCallback: unknown hook {name!r}")
            if fn is not None:
                setattr(self, name, fn)
