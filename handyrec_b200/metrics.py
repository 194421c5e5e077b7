"""Keras 2.6 metrics for binary single-output models, counted on the GPU: tf.keras.metrics.AUC, Precision, Recall and
BinaryAccuracy.

Every metric is a set of float32 variables that each batch adds integer counts into (Keras `update_confusion_matrix_variables`
and the MeanMetricWrapper of `binary_accuracy`): tp / fp / tn / fn per threshold, or the number of correct predictions and of
predictions.  A `MetricSet` holds the variables of all metrics of one compiled model in one device buffer, next to the union of
their thresholds and one (kind, threshold) descriptor per variable, so that one `hrb_metric_update` launch counts a batch for
every metric at once.  `read()` copies the variables to the host (after a sum over ranks under a communicator) and each metric's
`result()` applies Keras' formula there in float32.

Sample weights (Keras' MetricsContainer): metrics compiled in `weighted_metrics` count every sample as its weight when a step has
weights (tp += sum of w over the true positives, BinaryAccuracy's total += sum of w * correct and count += sum of w); metrics in
`metrics` never do.  A set that holds weighted metrics keeps a second descriptor array in which their variables have the weighted
kinds (hrb200.h: HRB_METRIC_WTP..WCOUNT): a batch with weights is counted by one `hrb_metric_update_weighted` (two launches), the
unweighted metrics of the same set taking their integer counts in it; a batch without weights by `hrb_metric_update` as before.
The weighted sums are accumulated in float64 in a fixed order and rounded once to float32, so they are reproducible bit for bit.

Deviations from Keras (DESIGN.md 3, "Metrics"):
  * Keras asserts 0 <= y_pred <= 1 in the step that sees a bad prediction; here the kernel flags the variables of the confusion
    metrics that counted it, and the ValueError is raised when their results are read (end of epoch, `evaluate`,
    `train_on_batch`, `result()`).  `reset_state()` clears a metric's flags with its variables.
  * at most 8192 distinct thresholds over one model's metrics (ValueError at `compile`).
  * default names are de-duplicated within one `compile` (`auc`, `auc_1`, ...), not by Keras' session-wide counter.
  * a metric's own `update_state` takes no `sample_weight` (NotImplementedError): the weights reach a metric compiled in
    `weighted_metrics` through the model's fit / train_on_batch / evaluate.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

MAX_THRESHOLDS = 8192
TP, FP, TN, FN, CORRECT, COUNT = 0, 1, 2, 3, 4, 5  # hrb200.h: hrb_metric_kind
WEIGHTED = 6  # kind + WEIGHTED: the same variable summing the samples' weights (HRB_METRIC_WTP..WCOUNT)
_EPSILON = 1e-7  # keras.backend.epsilon()


def _div_no_nan(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(b == 0, np.float32(0), a / np.where(b == 0, np.float32(1), b)).astype(np.float32)


def _no_sample_weight(sample_weight) -> None:
    if sample_weight is not None:
        raise NotImplementedError("sample_weight is not supported by a metric's own update_state: compile the metric in "
                                  "weighted_metrics and pass the weights to fit / train_on_batch / evaluate")


def _parse_thresholds(thresholds, default: float) -> List[float]:
    """metrics_utils.parse_init_thresholds: None -> [default]; a float or a list; every value in [0, 1]."""
    ts = [default] if thresholds is None else (list(thresholds) if isinstance(thresholds, (list, tuple, np.ndarray)) else [thresholds])
    invalid = [t for t in ts if t is None or t < 0 or t > 1]
    if invalid:
        raise ValueError(f"Threshold values must be in [0, 1]. Invalid values: {invalid}")
    return [float(t) for t in ts]


class Metric:
    """Base of the four metrics: `update_state(y_true, y_pred)`, `result()`, `reset_state()` / `reset_states()`.  The variables
    live in a MetricSet: the model's once compiled, otherwise one of the metric's own."""

    default_name = "metric"

    def __init__(self, name: Optional[str] = None, dtype=None):
        if dtype not in (None, "float32", np.float32, torch.float32):
            raise NotImplementedError("handyrec_b200's metrics keep float32 variables")
        self.name = name or self.default_name
        self._set: Optional["MetricSet"] = None
        self._index = 0

    # (kind, float32 threshold or None) per variable, in the order `_result` reads them
    def _descriptors(self) -> List[tuple]:
        raise NotImplementedError

    def _result(self, v: np.ndarray):
        raise NotImplementedError

    def _owned_set(self) -> "MetricSet":
        if self._set is None:
            MetricSet([self])
        return self._set

    def update_state(self, y_true, y_pred, sample_weight=None) -> None:
        """Count one batch (numpy or torch, host or device; one kernel launch on the current device)."""
        _no_sample_weight(sample_weight)
        self._owned_set().update(y_pred, y_true, only=self)

    def result(self):
        return self._owned_set().results(only=self)[self.name]

    def reset_state(self) -> None:
        if self._set is not None:
            self._set.reset(only=self)

    reset_states = reset_state

    def __repr__(self):
        return f"<{type(self).__name__} name={self.name!r}>"


class AUC(Metric):
    """tf.keras.metrics.AUC (Keras 2.6): tp / fp / tn / fn at num_thresholds thresholds, ROC or PR curve, Riemann sum by
    interpolation / minoring / majoring (PR + interpolation: interpolate_pr_auc)."""

    default_name = "auc"

    def __init__(self, num_thresholds=200, curve="ROC", summation_method="interpolation", name=None, dtype=None, thresholds=None,
                 multi_label=False, num_labels=None, label_weights=None, from_logits=False):
        if multi_label or num_labels is not None or label_weights is not None:
            raise NotImplementedError("AUC: multi_label / num_labels / label_weights are not supported (single-output binary models)")
        if from_logits:
            raise NotImplementedError("AUC: from_logits=True is not supported (the models output probabilities)")
        super().__init__(name, dtype)
        if thresholds is not None:
            self.num_thresholds = len(thresholds) + 2
            inner = sorted(float(t) for t in thresholds)
        else:
            if num_thresholds <= 1:
                raise ValueError("`num_thresholds` must be > 1.")
            self.num_thresholds = int(num_thresholds)
            inner = [(i + 1) * 1.0 / (num_thresholds - 1) for i in range(num_thresholds - 2)]
        # the spellings Keras' AUCCurve.from_str / AUCSummationMethod.from_str accept
        curves = {"roc": "ROC", "ROC": "ROC", "pr": "PR", "PR": "PR"}
        if curve not in curves:
            raise ValueError(f'Invalid AUC curve value "{curve}".')
        methods = {m: m.lower() for m in ("interpolation", "Interpolation", "minoring", "Minoring", "majoring", "Majoring")}
        if summation_method not in methods:
            raise ValueError(f'Invalid AUC summation method value "{summation_method}".')
        self.curve, self.summation_method = curves[curve], methods[summation_method]
        self.multi_label = False
        self._thresholds = np.array([0.0 - _EPSILON] + inner + [1.0 + _EPSILON], dtype=np.float64).astype(np.float32)

    @property
    def thresholds(self) -> List[float]:
        return [float(t) for t in self._thresholds]

    def _descriptors(self):
        return [(k, t) for k in (TP, FP, TN, FN) for t in self._thresholds]

    def _result(self, v):
        T = len(self._thresholds)
        tp, fp, tn, fn = v[:T], v[T : 2 * T], v[2 * T : 3 * T], v[3 * T :]
        if self.curve == "PR" and self.summation_method == "interpolation":
            dtp = tp[:-1] - tp[1:]
            p = tp + fp
            dp = p[:-1] - p[1:]
            slope = _div_no_nan(dtp, np.maximum(dp, np.float32(0)))
            intercept = tp[1:] - slope * p[1:]
            ratio = np.where((p[:-1] > 0) & (p[1:] > 0), _div_no_nan(p[:-1], np.maximum(p[1:], np.float32(0))), np.float32(1))
            with np.errstate(divide="ignore", invalid="ignore"):
                inc = _div_no_nan(slope * (dtp + intercept * np.log(ratio.astype(np.float32))), np.maximum(tp[1:] + fn[1:], np.float32(0)))
            return np.float32(np.sum(inc, dtype=np.float32))
        recall = _div_no_nan(tp, tp + fn)
        if self.curve == "ROC":
            x, y = _div_no_nan(fp, fp + tn), recall
        else:
            x, y = recall, _div_no_nan(tp, tp + fp)
        if self.summation_method == "interpolation":
            h = (y[:-1] + y[1:]) / np.float32(2)
        elif self.summation_method == "minoring":
            h = np.minimum(y[:-1], y[1:])
        else:
            h = np.maximum(y[:-1], y[1:])
        return np.float32(np.sum((x[:-1] - x[1:]) * h, dtype=np.float32))


class _PrecisionRecall(Metric):
    def __init__(self, thresholds=None, top_k=None, class_id=None, name=None, dtype=None):
        if top_k is not None or class_id is not None:
            raise NotImplementedError(f"{type(self).__name__}: top_k / class_id are not supported (single-output binary models)")
        super().__init__(name, dtype)
        self.init_thresholds = thresholds
        self.thresholds = _parse_thresholds(thresholds, 0.5)
        self._thresholds = np.array(self.thresholds, dtype=np.float64).astype(np.float32)

    def _pair(self, a, b):
        r = _div_no_nan(a, a + b)
        return np.float32(r[0]) if len(self._thresholds) == 1 else r


class Precision(_PrecisionRecall):
    """tf.keras.metrics.Precision: tp / (tp + fp) per threshold (default 0.5); a scalar for one threshold."""

    default_name = "precision"

    def _descriptors(self):
        return [(k, t) for k in (TP, FP) for t in self._thresholds]

    def _result(self, v):
        k = len(self._thresholds)
        return self._pair(v[:k], v[k:])


class Recall(_PrecisionRecall):
    """tf.keras.metrics.Recall: tp / (tp + fn) per threshold (default 0.5); a scalar for one threshold."""

    default_name = "recall"

    def _descriptors(self):
        return [(k, t) for k in (TP, FN) for t in self._thresholds]

    def _result(self, v):
        k = len(self._thresholds)
        return self._pair(v[:k], v[k:])


class BinaryAccuracy(Metric):
    """tf.keras.metrics.BinaryAccuracy: total += #(y_true == float(y_pred > threshold)), count += #samples; total / count."""

    default_name = "binary_accuracy"

    def __init__(self, name="binary_accuracy", dtype=None, threshold=0.5):
        super().__init__(name, dtype)
        self.threshold = float(threshold)

    def _descriptors(self):
        return [(CORRECT, np.float32(self.threshold)), (COUNT, None)]

    def _result(self, v):
        return np.float32(_div_no_nan(v[0], v[1]))


_STRINGS = {"AUC": lambda: AUC(), "Precision": lambda: Precision(), "Recall": lambda: Recall(),
            "accuracy": lambda: BinaryAccuracy(name="accuracy"), "acc": lambda: BinaryAccuracy(name="acc"),
            "binary_accuracy": lambda: BinaryAccuracy()}


def get(metric) -> Metric:
    """A compile-time metric identifier -> metric object (keras.metrics.get for the names this package implements)."""
    if isinstance(metric, Metric):
        return metric
    if isinstance(metric, str) and metric in _STRINGS:
        return _STRINGS[metric]()
    raise ValueError(f"Unknown metric {metric!r}: handyrec_b200 implements {sorted(_STRINGS)} and AUC / Precision / Recall / "
                     f"BinaryAccuracy objects")


def from_compile(metrics, weighted_metrics=None) -> Tuple[List[Metric], List[Metric]]:
    """`compile(metrics=..., weighted_metrics=...)`: objects and strings, names made unique within each list (`auc`, `auc_1`, ...);
    then a weighted metric whose name an unweighted one has is renamed `weighted_<name>` (Keras' MetricsContainer).  Returns the
    metrics followed by the weighted metrics, and the weighted metrics."""
    out = _unique(metrics)
    weighted = _unique(weighted_metrics)
    for w in weighted:
        if any(w is m for m in out):
            raise ValueError(f"metric {w.name!r} is listed in both metrics and weighted_metrics")
    names = {m.name for m in out}
    for w in weighted:
        if w.name in names:
            w.name = "weighted_" + w.name
        if w.name in names:
            raise ValueError(f"Found two metrics with the same name: {w.name}")
        names.add(w.name)
    return out + weighted, weighted


def _unique(metrics) -> List[Metric]:
    if metrics is None:
        return []
    items = list(metrics) if isinstance(metrics, (list, tuple)) else [metrics]
    out: List[Metric] = []
    for m in items:
        m = get(m)
        if any(m is o for o in out):
            raise ValueError(f"metric {m.name!r} is listed twice")
        out.append(m)
    seen: Dict[str, int] = {}
    taken = {m.name for m in out}
    for m in out:
        if m.name in seen:
            k = seen[m.name]
            while f"{m.name}_{k}" in taken:
                k += 1
            seen[m.name] = k + 1
            m.name = f"{m.name}_{k}"
            taken.add(m.name)
        else:
            seen[m.name] = 1
    return out


class MetricSet:
    """Device state of the metrics of one model: the union of their float32 thresholds (sorted, distinct, at most 8192), one
    (kind, threshold index) descriptor, one float32 variable and one out-of-range flag per metric variable (each metric owns a
    contiguous slice of them), and the kernel's scratch.  Host-side construction checks everything; device buffers are allocated
    on the current CUDA device at the first update or read."""

    def __init__(self, metrics: Sequence[Metric], weighted: Sequence[Metric] = ()):
        self.metrics = list(metrics)
        self.weighted = [any(m is w for w in weighted) for m in self.metrics]
        thr = sorted({float(t) for m in self.metrics for _, t in m._descriptors() if t is not None})
        if len(thr) > MAX_THRESHOLDS:
            raise ValueError(f"the metrics use {len(thr)} distinct thresholds; at most {MAX_THRESHOLDS} are supported per model")
        self.thresholds = np.array(thr or [0.5], dtype=np.float32)
        index = {float(t): i for i, t in enumerate(self.thresholds)}
        kinds, tidx, self.slices = [], [], []
        for i, m in enumerate(self.metrics):
            off = len(kinds)
            for k, t in m._descriptors():
                kinds.append(k)
                tidx.append(0 if t is None else index[float(t)])
            self.slices.append(slice(off, len(kinds)))
            m._set, m._index = self, i
        self.kinds = np.array(kinds, dtype=np.int32)
        # the descriptors of a batch with weights: the weighted metrics' variables take the weighted kinds
        self.weighted_kinds = self.kinds.copy()
        for sl, w in zip(self.slices, self.weighted):
            if w:
                self.weighted_kinds[sl] += WEIGHTED
        self.thr_index = np.array(tidx, dtype=np.int32)
        self.names = [m.name for m in self.metrics]
        self._dev = None

    def __len__(self):
        return len(self.metrics)

    def _buffers(self):
        if self._dev is None:
            from . import kernels as K

            dev = torch.device("cuda", torch.cuda.current_device())
            nv = len(self.kinds)
            self._dev = dict(
                thresholds=torch.from_numpy(self.thresholds).to(dev), kinds=torch.from_numpy(self.kinds).to(dev),
                thr_index=torch.from_numpy(self.thr_index).to(dev), vars=torch.zeros(nv, device=dev, dtype=torch.float32),
                flags=torch.zeros(nv, device=dev, dtype=torch.int32),
                scratch=torch.zeros(K.metric_scratch_bytes(len(self.thresholds)), device=dev, dtype=torch.uint8))
        return self._dev

    def _weighted_buffers(self):
        """The weighted update's descriptors and scratch, allocated at the first batch with weights."""
        b = self._buffers()
        if "wscratch" not in b:
            from . import kernels as K

            dev = b["vars"].device
            b["weighted_kinds"] = torch.from_numpy(self.weighted_kinds).to(dev)
            b["wscratch"] = torch.zeros(K.metric_weighted_scratch_bytes(len(self.thresholds)), device=dev, dtype=torch.uint8)
        return b

    @property
    def variables(self) -> torch.Tensor:
        """The local float32 variables, one slice per metric (`slices`)."""
        return self._buffers()["vars"]

    def _as_device(self, t, dev) -> torch.Tensor:
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(np.asarray(t, dtype=np.float32))
        return t.detach().to(dev, torch.float32).reshape(-1).contiguous()

    def update(self, y_pred, y_true, weight=None, only: Optional[Metric] = None) -> None:
        """Count one batch into every metric's variables (or `only` one metric's): one hrb_metric_update launch.  With `weight` (one
        float32 per sample) the weighted metrics sum the weights, and the batch takes one hrb_metric_update_weighted instead (two
        launches); when no metric of the update is weighted, the weights are not read."""
        from . import kernels as K

        b = self._buffers()
        dev = b["vars"].device
        p, y = self._as_device(y_pred, dev), self._as_device(y_true, dev)
        if p.numel() != y.numel():
            raise ValueError(f"metrics: {p.numel()} predictions but {y.numel()} labels (single-output binary models)")
        sl = slice(0, len(self.kinds)) if only is None else self.slices[only._index]
        if sl.stop == sl.start:
            return
        if weight is not None and any(self.weighted):
            w = self._as_device(weight, dev)
            if w.numel() != p.numel():
                raise ValueError(f"metrics: {p.numel()} predictions but {w.numel()} sample weights")
            wb = self._weighted_buffers()
            K.metric_update(p, y, b["thresholds"], wb["weighted_kinds"][sl], b["thr_index"][sl], b["vars"][sl], wb["wscratch"], b["flags"][sl],
                            weight=w)
            return
        K.metric_update(p, y, b["thresholds"], b["kinds"][sl], b["thr_index"][sl], b["vars"][sl], b["scratch"], b["flags"][sl])

    def reset(self, only: Optional[Metric] = None) -> None:
        """Zero the variables and out-of-range flags (of `only` one metric)."""
        if self._dev is None:
            return
        sl = slice(None) if only is None else self.slices[only._index]
        self._dev["vars"][sl].zero_()
        self._dev["flags"][sl].zero_()

    def _read(self, comm=None):
        """(variables, flags) on the host in one copy; under a communicator of several ranks a COPY of both is all-reduced (float32
        sum; collective: every rank calls it), so that each rank keeps accumulating its own variables like a Keras replica."""
        b = self._buffers()
        both = torch.cat([b["vars"], b["flags"].to(torch.float32)])
        if comm is not None and comm.N > 1:
            comm.all_reduce_sum(both)
        h = both.cpu().numpy()
        nv = len(self.kinds)
        return h[:nv], h[nv:] != 0

    def read(self, comm=None) -> np.ndarray:
        """The variables on the host (float32), summed over the ranks of `comm` (see `_read`)."""
        return self._read(comm)[0]

    def results(self, comm=None, only: Optional[Metric] = None) -> "OrderedDict[str, object]":
        """name -> Keras result() of every metric (or of `only` one); raises ValueError when a prediction outside [0, 1] was counted
        by a confusion metric (AUC / Precision / Recall) since its last reset."""
        v, bad = self._read(comm)
        out = OrderedDict()
        for m, sl in zip(self.metrics, self.slices):
            if only is not None and m is not only:
                continue
            if bad[sl].any():
                raise ValueError(f"metric {m.name!r}: predictions must be in [0, 1] (Keras asserts 0 <= y_pred <= 1); a prediction "
                                 f"outside that range or NaN was counted since the last reset")
            out[m.name] = m._result(v[sl])
        return out
