"""A very small Keras-functional-API look-alike, just enough for HandyRec's feature groups, layers and model
constructors to be written the way the reference writes them (Input -> layers -> Model -> compile/fit/predict).

* Graph construction is symbolic (`KTensor`s with shapes/dtypes, no GPU needed); execution binds `Input`s to torch
  CUDA tensors and runs each layer's `call`, which launches libhrb200 kernels (handyrec_b200.autograd_ops).
* Masks travel with tensors like in Keras: `compute_mask` of the producing layer, handed to consumers whose `call`
  takes a `mask` argument.
* There is no CPU execution path: building a graph works anywhere, running one needs the CUDA library.
"""
from __future__ import annotations

import inspect
import itertools
import math
from collections import OrderedDict
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .clip import init_clip
from .schedules import decayed_lr, ftrl_kernel_l2, init_lr

_uid = itertools.count()


def device() -> torch.device:
    return torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")


class ShardedTables:
    """Creation scope for multi-GPU models (the role of `tf.distribute.Strategy.scope()`), one process per GPU under torch.distributed:

        with ShardedTables():                      # or ShardedTables(comm, min_rows=..., seed=...)
            model = DeepFM(fm_group, dnn_group, ...)
            model.compile(Adam(1e-3), binary_crossentropy)
        model.fit(x_of_this_rank, y_of_this_rank, batch_size=per_rank_batch)

    Embedding tables with more than `min_rows` rows are created row-sharded: this rank allocates and initialises only rows
    r with r % N == rank (the counter-based initialiser gives every row the value it would have in the full table, so N ranks
    together hold exactly the table one GPU would have built from the same seed).  Such a table is read by the fused engine
    only (`compile` lowers the graph onto `ShardedDeepFMEngine`); a graph that does not lower raises instead of running the
    layer path on a shard.  Smaller tables and dense weights are replicated and broadcast from rank 0 at compile time.

    Collective calls: `fit` / `train_on_batch` / the first `predict` (they build or step the engine) must be made by every rank, with
    the same `batch_size` and the same number of batches -- like any data-parallel training loop.  `predict` after the first `fit`
    and `save_weights` / `load_weights` are rank-local."""

    active: Optional["ShardedTables"] = None

    def __init__(self, comm=None, min_rows: int = 131072, seed: int = 2022):
        if comm is None:
            from .sharded import TorchDistComm

            comm = TorchDistComm()
        self.comm, self.min_rows, self.seed, self.n_built = comm, int(min_rows), int(seed), 0

    def __enter__(self):
        ShardedTables.active = self
        return self

    def __exit__(self, *exc):
        ShardedTables.active = None
        return False

    def next_seed(self) -> int:
        self.n_built += 1
        return self.seed + 7919 * self.n_built


_DTYPES = {"int32": torch.int32, "int64": torch.int64, "float32": torch.float32, "bool": torch.bool, "uint8": torch.uint8}


def _tdtype(d):
    if isinstance(d, torch.dtype):
        return d
    return _DTYPES[getattr(d, "name", d)]


class _DType:
    """Minimal stand-in for tf.DType (`.name`, `.is_integer`)."""

    def __init__(self, name):
        self.name = name

    @property
    def is_integer(self):
        return self.name.startswith("int") or self.name.startswith("uint")

    def __eq__(self, o):
        return self.name == getattr(o, "name", o)

    def __repr__(self):
        return self.name


class KTensor:
    """Symbolic tensor: shape with None for the batch axis, dtype, producing node."""

    def __init__(self, shape, dtype, node=None, index=0, name=None):
        self.shape = tuple(shape)
        self.dtype = _DType(getattr(dtype, "name", dtype) if not isinstance(dtype, torch.dtype) else str(dtype).split(".")[-1])
        self.node, self.index, self.name = node, index, name
        self._keras_mask: Optional["KTensor"] = None

    def __add__(self, other):
        return Lambda(lambda a, b: a + b, lambda sa, sb: sa, name="add")([self, other])

    def __mul__(self, other):
        if isinstance(other, KTensor):
            return Lambda(lambda a, b: a * b, lambda sa, sb: sa, name="multiply")([self, other])
        c = float(other)
        return Lambda(lambda a: a * c, lambda sa: sa, name="scale")(self)

    __rmul__ = __mul__

    def __repr__(self):
        return f"<KTensor {self.name or ''} shape={self.shape} dtype={self.dtype}>"


class Node:
    def __init__(self, layer, inputs, kwargs):
        self.layer, self.inputs, self.kwargs = layer, inputs, kwargs
        self.outputs: List[KTensor] = []
        self.id = next(_uid)


def _flatten(x):
    if isinstance(x, (list, tuple)):
        out = []
        for e in x:
            out += _flatten(e)
        return out
    return [x]


def _map_structure(fn, x):
    if isinstance(x, (list, tuple)):
        return [_map_structure(fn, e) for e in x]
    return fn(x)


class Layer:
    def __init__(self, name: Optional[str] = None, trainable: bool = True, dtype=None, **kwargs):
        self.name = name or f"{type(self).__name__.lower()}_{next(_uid)}"
        self._name = self.name
        self.trainable = trainable
        self.built = False
        self._weights: "OrderedDict[str, torch.nn.Parameter]" = OrderedDict()
        self._weight_l2: Dict[str, float] = {}
        self._sublayers: List["Layer"] = []
        sig = inspect.signature(self.call)
        self._call_takes_mask = "mask" in sig.parameters
        self._call_takes_training = "training" in sig.parameters or any(p.kind == p.VAR_KEYWORD for p in sig.parameters.values())

    # ---- weights -------------------------------------------------------------------------
    def add_weight(self, name=None, shape=None, initializer="glorot_uniform", dtype=None, trainable=True, l2: float = 0.0, value=None):
        shape = tuple(int(s) for s in shape)
        if value is not None:
            t = torch.as_tensor(np.asarray(value), dtype=torch.float32).reshape(shape).clone()
        else:
            t = _init(initializer, shape)
        p = torch.nn.Parameter(t.to(device()), requires_grad=bool(trainable and self.trainable))
        key = name or f"w{len(self._weights)}"
        self._weights[key] = p
        if l2:
            self._weight_l2[key] = float(l2)
        return p

    def _track(self, layer: "Layer") -> "Layer":
        self._sublayers.append(layer)
        return layer

    @property
    def weights(self) -> List[torch.nn.Parameter]:
        out = list(self._weights.values())
        for l in self._sublayers:
            out += l.weights
        return out

    def weights_with_l2(self) -> List[Tuple[torch.nn.Parameter, float]]:
        out = [(p, self._weight_l2.get(k, 0.0)) for k, p in self._weights.items()]
        for l in self._sublayers:
            out += l.weights_with_l2()
        return out

    def get_weights(self):
        return [w.detach().cpu().numpy() for w in self.weights]

    def set_weights(self, values):
        ws = self.weights
        assert len(ws) == len(values), f"{self.name}: expected {len(ws)} arrays, got {len(values)}"
        for w, v in zip(ws, values):
            w.data.copy_(torch.as_tensor(np.asarray(v), dtype=w.dtype).reshape(w.shape))

    # ---- protocol -------------------------------------------------------------------------
    def build(self, input_shape):
        self.built = True

    def call(self, inputs, **kwargs):
        raise NotImplementedError

    def compute_mask(self, inputs, mask=None):
        return None

    def compute_output_shape(self, input_shape):
        return input_shape

    def get_config(self):
        return {"name": self.name, "trainable": self.trainable}

    def output_dtype(self, inputs):
        return "float32"

    def __call__(self, inputs, **kwargs):
        flat = _flatten(inputs)
        symbolic = any(isinstance(t, KTensor) for t in flat)
        shapes = _map_structure(lambda t: tuple(t.shape), inputs)
        if not self.built:
            self.build(shapes)
            self.built = True
        if symbolic:
            node = Node(self, inputs, kwargs)
            out_shape = self.compute_output_shape(shapes)
            multi = isinstance(out_shape, list)
            outs = []
            for i, s in enumerate(out_shape if multi else [out_shape]):
                t = KTensor(s, self.output_dtype(inputs), node, i, name=f"{self.name}:{i}")
                outs.append(t)
            node.outputs = outs
            in_masks = _map_structure(lambda t: t._keras_mask if isinstance(t, KTensor) else None, inputs)
            has_mask = self.symbolic_has_mask(inputs, in_masks)
            for t in outs:
                t._keras_mask = KTensor(t.shape, "bool", node, -1, name=f"{self.name}:mask") if has_mask else None
            return outs if multi else outs[0]
        # eager: inputs are torch tensors; masks ride on the `_keras_mask` attribute
        in_masks = _map_structure(lambda t: getattr(t, "_keras_mask", None), inputs)
        return self._run(inputs, in_masks, kwargs.get("training", False))

    def symbolic_has_mask(self, inputs, in_masks) -> bool:
        """Whether compute_mask will return a mask (decidable at graph-build time for every layer used here)."""
        return False

    def _run(self, inputs, in_masks, training):
        kw = {}
        single_mask = in_masks  # same nesting as `inputs` (a list for multi-input layers)
        if self._call_takes_mask:
            kw["mask"] = single_mask
        if self._call_takes_training:
            kw["training"] = training
        out = self.call(inputs, **kw)
        mask = self.compute_mask(inputs, single_mask)
        if isinstance(out, torch.Tensor):
            out._keras_mask = mask
        return out


def _init(initializer, shape):
    name = initializer if isinstance(initializer, str) else getattr(initializer, "__name__", "zeros")
    name = name.lower()
    if name in ("zeros", "zero"):
        return torch.zeros(shape)
    if name in ("ones", "one"):
        return torch.ones(shape)
    if name in ("uniform", "random_uniform", "randomuniform"):
        n = 1
        for d in shape:
            n *= d
        if n >= (1 << 22) and device().type == "cuda":  # large tables are drawn on the device (no multi-GB host tensor)
            return torch.rand(shape, device=device()).sub_(0.5).mul_(0.1)
        return (torch.rand(shape) - 0.5) * 0.1  # Keras RandomUniform(-0.05, 0.05)
    if name in ("glorot_uniform", "glorotuniform"):
        fan_in, fan_out = (shape[0], shape[-1]) if len(shape) > 1 else (shape[0], shape[0])
        lim = math.sqrt(6.0 / (fan_in + fan_out))
        return (torch.rand(shape) * 2 - 1) * lim
    raise ValueError(f"unknown initializer {initializer!r}")


class Zeros:  # tensorflow.keras.initializers.Zeros look-alike
    __name__ = "zeros"


class InputLayer(Layer):
    def call(self, inputs, **kwargs):
        return inputs


def Input(shape=None, name=None, dtype="float32", **kwargs) -> KTensor:
    t = KTensor((None,) + tuple(shape), dtype, node=None, name=name or f"input_{next(_uid)}")
    t.is_input = True
    return t


class Lambda(Layer):
    """fn over torch tensors + a shape function (used for `dnn_output + fm_output`, squeeze etc.)."""

    def __init__(self, fn: Callable, shape_fn: Callable, dtype_fn: Optional[Callable] = None, **kw):
        super().__init__(**kw)
        self.fn, self.shape_fn, self.dtype_fn = fn, shape_fn, dtype_fn

    def call(self, inputs):
        return self.fn(*inputs) if isinstance(inputs, (list, tuple)) else self.fn(inputs)

    def compute_output_shape(self, input_shape):
        return self.shape_fn(*input_shape) if isinstance(input_shape, list) else self.shape_fn(input_shape)

    def output_dtype(self, inputs):
        return self.dtype_fn(inputs) if self.dtype_fn else "float32"


class Activation(Layer):
    """keras.layers.Activation for the names HandyRec's configs use; sigmoid outputs remember their logits."""

    def __init__(self, activation, **kw):
        super().__init__(**kw)
        self.activation = activation

    def call(self, inputs):
        from .autograd_ops import ActivationFn

        if self.activation in (None, "linear"):
            return inputs
        if self.activation not in ("relu", "sigmoid", "tanh"):
            raise ValueError(f"unsupported activation {self.activation!r}")
        out = ActivationFn.apply(inputs, self.activation)
        if self.activation == "sigmoid":
            out._keras_logits = inputs  # like tf.keras.activations.sigmoid: binary_crossentropy uses the logits
        return out


# ---------------------------------------------------------------------------------------------
# optimisers / losses (Keras formulas, kernels from libhrb200).  Every optimiser takes Keras' clipnorm / clipvalue /
# global_clipnorm (handyrec_b200.clip); the model clips the gradients before it calls `step`.  `learning_rate` is a float or a
# handyrec_b200.schedules schedule, `decay` Keras' time-based decay; `step` takes the rate of `iterations` (decayed_lr, kept in
# `lr_t` for the large tables' row updates that follow it) and then counts itself there.
# ---------------------------------------------------------------------------------------------
class Adam:
    def __init__(self, learning_rate=1e-3, lr=None, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipnorm=None, clipvalue=None,
                 global_clipnorm=None, decay=0.0):
        init_clip(self, clipnorm, clipvalue, global_clipnorm)
        init_lr(self, lr if lr is not None else learning_rate, decay)
        self.b1, self.b2, self.eps, self.t = beta_1, beta_2, epsilon, 0
        self.state: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}

    def step(self, params_l2: Sequence[Tuple[torch.nn.Parameter, float]]):
        from . import kernels as K

        self.t += 1
        lr = self.lr_t = decayed_lr(self)
        ps, gs, ms, vs, l2s = [], [], [], [], []
        for p, l2 in params_l2:
            if p.grad is None or not p.requires_grad:
                continue
            if id(p) not in self.state:
                self.state[id(p)] = (torch.zeros_like(p.data), torch.zeros_like(p.data))
            m, v = self.state[id(p)]
            ps.append(p.data)
            gs.append(p.grad.contiguous())
            ms.append(m)
            vs.append(v)
            l2s.append(2.0 * l2)
        K.adam_step_multi(ps, gs, ms, vs, l2s, lr, self.b1, self.b2, self.eps, self.t)  # all variables in one launch
        self.iterations += 1


class Adagrad:
    """tf.keras.optimizers.Adagrad (Keras 2.6): acc += g^2; w -= lr * g / (sqrt(acc) + eps), acc starting at
    initial_accumulator_value.  Large tables take the same step on the rows a batch touches (CustomEmbedding.apply_sparse)."""

    def __init__(self, learning_rate=0.001, initial_accumulator_value=0.1, epsilon=1e-7, lr=None, clipnorm=None, clipvalue=None,
                 global_clipnorm=None, decay=0.0):
        init_clip(self, clipnorm, clipvalue, global_clipnorm)
        if initial_accumulator_value < 0.0:
            raise ValueError(f"initial_accumulator_value must be non-negative: {initial_accumulator_value}")
        init_lr(self, lr if lr is not None else learning_rate, decay)
        self.initial_accumulator_value, self.eps = float(initial_accumulator_value), float(epsilon)
        self.state: Dict[int, torch.Tensor] = {}

    def step(self, params_l2: Sequence[Tuple[torch.nn.Parameter, float]]):
        from . import kernels as K

        lr = self.lr_t = decayed_lr(self)
        live = [(p, l2) for p, l2 in params_l2 if p.grad is not None and p.requires_grad]
        for p, _ in live:
            if id(p) not in self.state:
                self.state[id(p)] = torch.full_like(p.data, self.initial_accumulator_value)
        K.adagrad_step_multi([p.data for p, _ in live], [p.grad.contiguous() for p, _ in live], [self.state[id(p)] for p, _ in live],
                             [2.0 * l2 for _, l2 in live], lr, self.eps)  # all variables in one launch
        self.iterations += 1


class Ftrl:
    """tf.keras.optimizers.Ftrl (Keras 2.6, FTRL-Proximal): per element, with g the gradient (plus 2*l2*w of a Keras regulariser)
    and p(a) = a^(-learning_rate_power),

        linear += g + 2*l2_shrinkage*w - (p(acc + g^2) - p(acc)) / lr * w;  acc += g^2
        w = |linear| > l1 ? (sign(linear)*l1 - linear) / (p(acc) / lr + 2*l2') : 0,   l2' = l2 + beta / (2*lr)

    acc starting at initial_accumulator_value, linear at 0.  A step with a zero gradient is not a no-op (it recomputes w from the
    slots), so embedding tables step only the rows a batch gathers, as Keras does for their IndexedSlices gradient
    (CustomEmbedding.apply_sparse)."""

    def __init__(self, learning_rate=0.001, learning_rate_power=-0.5, initial_accumulator_value=0.1, l1_regularization_strength=0.0,
                 l2_regularization_strength=0.0, name="Ftrl", l2_shrinkage_regularization_strength=0.0, beta=0.0, lr=None,
                 clipnorm=None, clipvalue=None, global_clipnorm=None, decay=0.0):
        init_clip(self, clipnorm, clipvalue, global_clipnorm)
        if initial_accumulator_value < 0.0:
            raise ValueError(f"initial_accumulator_value {initial_accumulator_value} needs to be positive or zero")
        if learning_rate_power > 0.0:
            raise ValueError(f"learning_rate_power {learning_rate_power} needs to be negative or zero")
        if l1_regularization_strength < 0.0:
            raise ValueError(f"l1_regularization_strength {l1_regularization_strength} needs to be positive or zero")
        if l2_regularization_strength < 0.0:
            raise ValueError(f"l2_regularization_strength {l2_regularization_strength} needs to be positive or zero")
        if l2_shrinkage_regularization_strength < 0.0:
            raise ValueError(f"l2_shrinkage_regularization_strength {l2_shrinkage_regularization_strength} needs to be positive or zero")
        self.name = name
        self.learning_rate_power = float(learning_rate_power)
        self.initial_accumulator_value = float(initial_accumulator_value)
        self.l1 = float(l1_regularization_strength)
        self.l2 = float(l2_regularization_strength)
        self.l2_shrinkage = float(l2_shrinkage_regularization_strength)
        self.beta = float(beta)
        init_lr(self, lr if lr is not None else learning_rate, decay)
        self.state: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}

    @property
    def kernel_l2(self) -> float:
        """The l2 the TF kernel takes: l2_regularization_strength + beta / (2 * learning_rate), at the rate of the current step."""
        return ftrl_kernel_l2(self.l2, self.beta, self.lr_t)

    def hyper(self) -> Dict[str, float]:
        """Keyword arguments of the library's Ftrl entry points."""
        return dict(l1=self.l1, l2=self.kernel_l2, lr_power=self.learning_rate_power, l2_shrinkage=self.l2_shrinkage)

    def step(self, params_l2: Sequence[Tuple[torch.nn.Parameter, float]]):
        from . import kernels as K

        lr = self.lr_t = decayed_lr(self)
        live = [(p, l2) for p, l2 in params_l2 if p.grad is not None and p.requires_grad]
        for p, _ in live:
            if id(p) not in self.state:
                self.state[id(p)] = (torch.full_like(p.data, self.initial_accumulator_value), torch.zeros_like(p.data))
        K.ftrl_step_multi([p.data for p, _ in live], [p.grad.contiguous() for p, _ in live], [self.state[id(p)][0] for p, _ in live],
                          [self.state[id(p)][1] for p, _ in live], [2.0 * l2 for _, l2 in live], lr, **self.hyper())
        self.iterations += 1


class SGD:
    def __init__(self, learning_rate=0.01, lr=None, clipnorm=None, clipvalue=None, global_clipnorm=None, decay=0.0):
        init_clip(self, clipnorm, clipvalue, global_clipnorm)
        init_lr(self, lr if lr is not None else learning_rate, decay)

    def step(self, params_l2):
        from . import kernels as K

        lr = self.lr_t = decayed_lr(self)
        live = [(p, l2) for p, l2 in params_l2 if p.grad is not None and p.requires_grad]
        K.sgd_step_multi([p.data for p, _ in live], [p.grad.contiguous() for p, _ in live], [2.0 * l2 for _, l2 in live], lr)
        self.iterations += 1


_step_weight: Optional[torch.Tensor] = None  # the sample weights of the batch a Model step is computing (device float32), or None


def binary_crossentropy(y_true, y_pred):
    """Keras binary_crossentropy, the mean over the batch.  Inside a Model step with sample weights it is Keras' weighted loss
    sum(w * l) / B: the model hands the batch's weights over in `_step_weight`, as Keras' compiled loss adds them to the call."""
    from .autograd_ops import SigmoidBCEFn

    logits = getattr(y_pred, "_keras_logits", None)
    if logits is None:
        # Keras' fallback when the prediction is not the direct output of a sigmoid (e.g. BatchNormalization / Dropout behind the
        # output activation, layers/core.py:66-73): probabilities clipped to [eps, 1-eps], eps = 1e-7
        from .autograd_ops import ClippedBCEFn

        return ClippedBCEFn.apply(y_pred, y_true, _step_weight)
    return SigmoidBCEFn.apply(logits, y_true, _step_weight)


def _regression(loss: str, y_true, y_pred, delta: float = 1.0):
    """Keras' compiled regression loss `loss` (kernels.REG_LOSS) of one output: the mean over the last axis per sample, then the
    batch mean, or sum(w * l) / B with the step's sample weights.  A (B,) label meets a (B, 1) output as (B, 1), as Keras' compiled
    loss expands it (compile_utils.match_dtype_and_rank) -- a plain broadcast would form a (B, B) matrix."""
    from .autograd_ops import RegressionLossFn

    yt = y_true if isinstance(y_true, torch.Tensor) else torch.as_tensor(np.asarray(y_true))
    yt = yt.to(y_pred.device, torch.float32)
    if yt.dim() == y_pred.dim() - 1 and y_pred.shape[-1] == 1:
        yt = yt.unsqueeze(-1)
    if tuple(yt.shape) != tuple(y_pred.shape):
        raise ValueError(f"{loss}: labels of shape {tuple(yt.shape)} for predictions of shape {tuple(y_pred.shape)}")
    return RegressionLossFn.apply(y_pred, yt, loss, float(delta), _step_weight)


def mean_squared_error(y_true, y_pred):
    """Keras mean_squared_error: mean((y_pred - y_true)^2, axis=-1), averaged over the batch (sample weights as binary_crossentropy)."""
    return _regression("mean_squared_error", y_true, y_pred)


def mean_absolute_error(y_true, y_pred):
    """Keras mean_absolute_error: mean(|y_pred - y_true|, axis=-1), averaged over the batch (sample weights as binary_crossentropy)."""
    return _regression("mean_absolute_error", y_true, y_pred)


mse = MSE = mean_squared_error
mae = MAE = mean_absolute_error


class _Loss:
    """tf.keras.losses.Loss with the default reduction (AUTO, i.e. SUM_OVER_BATCH_SIZE), the only one a compiled model here takes."""

    def __init__(self, reduction="auto", name=None):
        if reduction not in ("auto", "sum_over_batch_size"):
            raise NotImplementedError(f"{type(self).__name__}(reduction={reduction!r}): only AUTO / SUM_OVER_BATCH_SIZE is supported")
        self.reduction, self.name = reduction, name


class MeanSquaredError(_Loss):
    def __init__(self, reduction="auto", name="mean_squared_error"):
        super().__init__(reduction, name)

    def __call__(self, y_true, y_pred):
        return mean_squared_error(y_true, y_pred)


class MeanAbsoluteError(_Loss):
    def __init__(self, reduction="auto", name="mean_absolute_error"):
        super().__init__(reduction, name)

    def __call__(self, y_true, y_pred):
        return mean_absolute_error(y_true, y_pred)


class Huber(_Loss):
    """Keras Huber: 0.5*q^2 + delta*(|e| - q) with q = min(|e|, delta), e = y_pred - y_true, mean over the last axis."""

    def __init__(self, delta=1.0, reduction="auto", name="huber_loss"):
        super().__init__(reduction, name)
        if delta < 0:
            raise ValueError(f"Huber: delta must be non-negative, got {delta}")
        self.delta = float(delta)

    def __call__(self, y_true, y_pred):
        return _regression("huber", y_true, y_pred, self.delta)


class BinaryCrossentropy(_Loss):
    """Keras BinaryCrossentropy with its defaults: binary_crossentropy."""

    def __init__(self, from_logits=False, label_smoothing=0.0, reduction="auto", name="binary_crossentropy"):
        if from_logits:
            raise NotImplementedError("BinaryCrossentropy(from_logits=True): the models here end in a sigmoid; use the default")
        if label_smoothing:
            raise NotImplementedError(f"BinaryCrossentropy(label_smoothing={label_smoothing}): not supported")
        super().__init__(reduction, name)

    def __call__(self, y_true, y_pred):
        return binary_crossentropy(y_true, y_pred)


def builtin_loss(loss) -> Optional[Tuple[str, float]]:
    """(name, huber delta) of a built-in loss function or object, None for anything else (a user callable)."""
    if loss is binary_crossentropy or isinstance(loss, BinaryCrossentropy):
        return ("binary_crossentropy", 0.0)
    if loss is mean_squared_error or isinstance(loss, MeanSquaredError):
        return ("mean_squared_error", 0.0)
    if loss is mean_absolute_error or isinstance(loss, MeanAbsoluteError):
        return ("mean_absolute_error", 0.0)
    if isinstance(loss, Huber):
        return ("huber", loss.delta)
    return None


def host_loss(loss: Tuple[str, float], pred: np.ndarray, y: np.ndarray) -> np.ndarray:
    """Per-sample float64 loss of the built-in `loss` (builtin_loss) on one-column predictions; binary_crossentropy on probabilities
    clipped to [1e-7, 1 - 1e-7], as Keras computes it from probabilities."""
    name, delta = loss
    p, y = np.asarray(pred, np.float64).reshape(-1), np.asarray(y, np.float64).reshape(-1)
    if name == "binary_crossentropy":
        p = np.clip(p, 1e-7, 1.0 - 1e-7)
        return -(y * np.log(p) + (1.0 - y) * np.log1p(-p))
    e = p - y
    if name == "mean_squared_error":
        return e * e
    if name == "mean_absolute_error":
        return np.abs(e)
    q = np.minimum(np.abs(e), delta)
    return 0.5 * q * q + delta * (np.abs(e) - q)


_LOSS_IDS = {"mse": mean_squared_error, "MSE": mean_squared_error, "mean_squared_error": mean_squared_error, "mae": mean_absolute_error,
             "MAE": mean_absolute_error, "mean_absolute_error": mean_absolute_error, "binary_crossentropy": binary_crossentropy}


def get_loss(loss):
    """keras.losses.get for the losses here: a string identifier resolves to its function (ValueError for an unknown one); a loss
    object or function passes through unchanged."""
    if isinstance(loss, str):
        if loss not in _LOSS_IDS:
            raise ValueError(f"Unknown loss function: {loss!r} (supported identifiers: {', '.join(_LOSS_IDS)})")
        return _LOSS_IDS[loss]
    if isinstance(loss, (list, tuple, dict)):
        raise NotImplementedError("per-output losses: the models here have one output and take one loss")
    return loss


def get_optimizer(optimizer):
    """keras.optimizers.get for the optimizers here: "adam", "sgd", "adagrad", "ftrl" in any case resolve to the class with Keras'
    default arguments (ValueError for another name); an optimizer object passes through unchanged."""
    if isinstance(optimizer, str):
        cls = {"adam": Adam, "sgd": SGD, "adagrad": Adagrad, "ftrl": Ftrl}.get(optimizer.lower())
        if cls is None:
            raise ValueError(f"Unknown optimizer: {optimizer!r} (supported identifiers: adam, sgd, adagrad, ftrl)")
        return cls()
    return optimizer


def _as_host(a) -> np.ndarray:
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def sample_weights(y, sample_weight=None, class_weight=None) -> Optional[np.ndarray]:
    """Keras 2.6's per-sample weights of labels `y`: `sample_weight` ((n,) or (n, 1)) times the `class_weight` entry of each label
    (data_adapter._make_class_weight_map_fn: keys exactly 0..k-1, labels truncated to int64), the product formed in float64 and
    rounded once to float32.  None when neither is given.  Raises ValueError on a bad shape, length, key set or label."""
    if sample_weight is None and class_weight is None:
        return None
    yv = _as_host(y)
    n = len(yv)
    w = None
    if sample_weight is not None:
        sw = _as_host(sample_weight)
        if not (sw.ndim == 1 or (sw.ndim == 2 and sw.shape[1] == 1)) or sw.shape[0] != n:
            raise ValueError(f"sample_weight must have shape ({n},) or ({n}, 1) for {n} labels, got {sw.shape}")
        w = sw.reshape(-1).astype(np.float64)
    if class_weight is not None:
        class_ids = sorted(class_weight.keys())
        if class_ids != list(range(len(class_ids))):
            raise ValueError("Expected `class_weight` to be a dict with keys from 0 to one less than the number of classes, "
                             f"found {class_weight}")
        if yv.ndim == 2 and yv.shape[1] > 1:
            raise NotImplementedError("class_weight with one-hot targets: the models here have a single binary output")
        table = np.array([class_weight[int(c)] for c in class_ids], dtype=np.float32).astype(np.float64)
        yf = yv.reshape(-1).astype(np.float64)
        bad = ~((yf > -1.0) & (yf < len(class_ids)))  # int64 truncation lands outside 0..k-1 (NaN included)
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            raise ValueError(f"class_weight: label {yv.reshape(-1)[i]} of sample {i} is not one of the classes 0..{len(class_ids) - 1} "
                             "after truncation to int64")
        cw = table[np.trunc(yf).astype(np.int64)]
        w = cw if w is None else w * cw
    return w.astype(np.float32)


class Model:
    """keras.Model look-alike over the symbolic graph: __call__/predict/compile/fit/train_on_batch."""

    def __init__(self, inputs, outputs, name=None):
        self.inputs = list(inputs) if isinstance(inputs, (list, tuple)) else [inputs]
        self.outputs = outputs
        self.name = name or "model"
        self._order = self._toposort()
        self.optimizer = None
        self.loss = None

    def _toposort(self) -> List[Node]:
        order, seen = [], set()

        def visit(t):
            if not isinstance(t, KTensor) or t.node is None or t.node.id in seen:
                return
            seen.add(t.node.id)
            for i in _flatten(t.node.inputs):
                visit(i)
            order.append(t.node)

        for o in _flatten(self.outputs):
            visit(o)
        return order

    @property
    def layers(self) -> List[Layer]:
        self.sync()
        out, seen = [], set()
        for n in self._order:
            if id(n.layer) not in seen:
                seen.add(id(n.layer))
                out.append(n.layer)
        return out

    def get_layer(self, name):
        for l in self.layers:
            if l.name == name:
                return l
        raise ValueError(f"no layer named {name}")

    def weights_with_l2(self):
        out, seen = [], set()
        for l in self.layers:
            for p, l2 in l.weights_with_l2():
                if id(p) not in seen:
                    seen.add(id(p))
                    out.append((p, l2))
        return out

    @property
    def trainable_weights(self):
        return [p for p, _ in self.weights_with_l2() if p.requires_grad]

    # ---- execution --------------------------------------------------------------------------
    def _bind(self, x) -> Dict[str, torch.Tensor]:
        dev = device()
        if dev.type != "cuda":
            raise RuntimeError("handyrec_b200 executes on CUDA only (no CPU fallback); graph construction alone works on CPU")
        if isinstance(x, dict):
            feed = x
        else:
            xs = x if isinstance(x, (list, tuple)) else [x]
            feed = {t.name: v for t, v in zip(self.inputs, xs)}
        bound = {}
        for t in self.inputs:
            if t.name not in feed:
                raise KeyError(f"missing input {t.name!r}")
            v = feed[t.name]
            v = torch.as_tensor(np.asarray(v)) if not isinstance(v, torch.Tensor) else v
            v = v.to(dev, _tdtype(t.dtype.name))
            if v.dim() == 1:
                v = v.reshape(-1, 1)
            bound[t.name] = v.contiguous()
        return bound

    def __call__(self, x, training=False):
        self.sync()
        feed = self._bind(x)
        vals: Dict[Tuple[int, int], torch.Tensor] = {}

        def get(t):
            if getattr(t, "is_input", False):
                return feed[t.name]
            return vals[(t.node.id, t.index)]

        for n in self._order:
            ins = _map_structure(get, n.inputs)
            masks = _map_structure(lambda v: getattr(v, "_keras_mask", None), ins)
            out = n.layer._run(ins, masks, training)
            for i, o in enumerate(out if isinstance(out, (list, tuple)) else [out]):
                vals[(n.id, i)] = o
        return _map_structure(get, self.outputs)

    # ---- fused execution (handyrec_b200.lowering) ----------------------------------------------------
    _fused = None
    fuse = True  # set to False before compile() to keep the layer-by-layer path (tests compare the two)

    def sync(self) -> None:
        """Make the layers' weights current after fused training steps (train_on_batch leaves them in the engine)."""
        if self._fused is not None:
            self._fused.sync_to_layers()

    def predict(self, x, batch_size=None):
        if (self._fused is not None and self._fused.engine is None and isinstance(x, dict) and self._comm is not None and self._comm.N > 1
                and self.optimizer is not None):
            # a multi-GPU model before its first fit: only the engine can read row-sharded tables, so it is built here (collective:
            # every rank calls predict, as with fit)
            n = len(np.asarray(next(iter(x.values()))))
            self._fused.build(min(batch_size or n, n), self.optimizer)
        if self._fused is not None and self._fused.engine is not None and isinstance(x, dict):
            return self._fused.predict(x, batch_size)
        self.sync()
        n = len(next(iter(x.values()))) if isinstance(x, dict) else len(x[0] if isinstance(x, (list, tuple)) else x)
        bs = batch_size or n
        outs = []
        from .kernels import deferred_id_checks

        with torch.no_grad():
            for s in range(0, n, bs):
                xb = {k: v[s : s + bs] for k, v in x.items()} if isinstance(x, dict) else [v[s : s + bs] for v in x]
                with deferred_id_checks():
                    outs.append(self(xb, training=False).detach().cpu())
        return torch.cat(outs).numpy()

    _comm = None
    _metric_set = None  # handyrec_b200.metrics.MetricSet of the compiled metrics, None without
    _metric_list: Sequence = ()

    def compile(self, optimizer=None, loss=None, distribute=None, metrics=None, weighted_metrics=None, **kwargs):
        """keras.Model.compile.  `distribute` (extra): True under an initialised torch.distributed process group (one process per
        GPU), or a `handyrec_b200.sharded.TorchDistComm` -- a DeepFM-shaped graph then trains on the row-sharded multi-GPU engine.
        `metrics`: AUC / Precision / Recall / BinaryAccuracy objects or the strings "AUC", "Precision", "Recall", "accuracy", "acc",
        "binary_accuracy" (handyrec_b200.metrics; counted on the GPU from each batch's forward output).  `weighted_metrics`: the
        same, counted with the sample weights of fit / train_on_batch / evaluate (a name an unweighted metric has becomes
        `weighted_<name>`).  `optimizer` may be "adam", "sgd", "adagrad" or "ftrl" (any case), `loss` "binary_crossentropy", "mse" /
        "MSE" / "mean_squared_error" or "mae" / "MAE" / "mean_absolute_error" (get_optimizer / get_loss)."""
        from . import metrics as M

        if kwargs.get("loss_weights") is not None:
            raise NotImplementedError("loss_weights: the models here have one output and take one loss")
        if kwargs.get("sample_weight_mode") is not None:
            raise NotImplementedError("sample_weight_mode: only per-sample weights are supported (no temporal weights)")
        if weighted_metrics:
            self._require_one_probability("weighted_metrics")
        self._metric_list, weighted = M.from_compile(metrics, weighted_metrics)
        self._metric_set = M.MetricSet(self._metric_list, weighted) if self._metric_list else None
        self.optimizer = get_optimizer(optimizer) if optimizer is not None else Adam()
        self.loss = get_loss(loss) if loss is not None else binary_crossentropy
        self._fused = None
        if distribute is None and ShardedTables.active is not None:
            distribute = ShardedTables.active.comm
            self.dense_table_max_rows = ShardedTables.active.min_rows
        if distribute:
            from .sharded import TorchDistComm

            self._comm = distribute if not isinstance(distribute, bool) else TorchDistComm()
        from .clip import clip_args

        clip = clip_args(self.optimizer)
        self._clip_state = None
        if clip is not None and self._comm is not None and self._comm.N > 1:
            # Keras clips the global-batch gradient: the per-variable norms would have to ride in the ranks' all-reduce
            raise ValueError("gradient clipping (clipnorm / clipvalue / global_clipnorm) is not supported on a multi-GPU compile: "
                             "Keras clips the global-batch gradient, which the sharded step does not form before it updates")
        for l in self._all_layers():  # under Ftrl a dense step would move the rows a batch does not gather
            if hasattr(l, "SPARSE_UPDATE_MIN_ROWS"):
                l._ftrl = isinstance(self.optimizer, Ftrl)
        kind = builtin_loss(self.loss)
        if self.fuse and kind is not None and isinstance(self.optimizer, (Adam, SGD, Adagrad, Ftrl)):
            from .lowering import lower  # a DeepFM-shaped graph runs on the fused engine (one lookup, tcgen05 towers)

            self._fused = lower(self, kind)
        if self._comm is not None and self._comm.N > 1 and self._fused is None:
            raise ValueError("distribute: only graphs the fused DeepFM engine covers train multi-GPU (lowering.py lists the conditions)")
        if clip is not None:
            for l in self._all_layers():
                if getattr(l, "l2", 0.0) and hasattr(l, "SPARSE_UPDATE_MIN_ROWS") and l.trainable and self._rows_updated(l):
                    raise ValueError(f"{l.name}: gradient clipping with an l2 regulariser on a table that takes the touched-rows update "
                                     f"({l.input_dim} rows): Keras' clipped gradient then covers every row of the table, which that "
                                     "update never forms")

    def _rows_updated(self, emb) -> bool:
        """Whether the table of CustomEmbedding `emb` takes the touched-rows update on the path this compile chose."""
        if self._fused is not None and any(t is emb for t in self._fused.tables):
            return emb.input_dim > getattr(self, "dense_table_max_rows", 131072)
        return emb.input_dim >= emb.SPARSE_UPDATE_MIN_ROWS and emb.output_dim % 4 == 0

    # ---- metrics ---------------------------------------------------------------------------------
    @property
    def metrics(self) -> list:
        """The compiled metric objects (Keras also lists its loss tracker here; this list holds the compiled metrics only)."""
        return list(self._metric_list)

    @property
    def metrics_names(self) -> List[str]:
        return ["loss"] + [m.name for m in self._metric_list]

    def reset_metrics(self) -> None:
        if self._metric_set is not None:
            self._metric_set.reset()

    def _metric_values(self) -> "OrderedDict[str, Any]":
        """Every compiled metric's result (a host read; under a multi-GPU communicator a collective summing the ranks' variables)."""
        comm = self._comm if self._comm is not None and self._comm.N > 1 else None
        res = self._metric_set.results(comm)
        return OrderedDict((k, float(v) if np.ndim(v) == 0 else v) for k, v in res.items())

    def _with_metrics(self, loss: float, res, return_dict: bool):
        if return_dict:
            return OrderedDict([("loss", loss)] + list(res.items()))
        return loss if self._metric_set is None else [loss] + list(res.values())

    def train_on_batch(self, x, y, sample_weight=None, class_weight=None, reset_metrics=True, return_dict=False):
        """keras.Model.train_on_batch: the loss, or [loss, *metric results] when metrics are compiled (a dict with return_dict).
        reset_metrics=False accumulates the metrics over calls.  sample_weight / class_weight: Keras' per-sample weights."""
        w = self._weights(y, sample_weight, class_weight)
        if self._metric_set is None and not return_dict:
            return self._train_step(x, y, w)
        if reset_metrics:
            self.reset_metrics()
        loss = self._train_step(x, y, w)
        return self._with_metrics(loss, self._metric_values() if self._metric_set is not None else {}, return_dict)

    def _weights(self, y, sample_weight=None, class_weight=None) -> Optional[np.ndarray]:
        """sample_weights(), refused for a loss other than the built-in ones and for an output other than one column per sample."""
        w = sample_weights(y, sample_weight, class_weight)
        if w is not None:
            if builtin_loss(self.loss) is None:
                raise NotImplementedError("sample_weight / class_weight are supported with the built-in losses only (binary_crossentropy, "
                                          f"mean_squared_error, mean_absolute_error, Huber), not {self.loss!r}")
            self._require_one_probability("sample_weight / class_weight")
        return w

    def _require_one_probability(self, what: str) -> None:
        """Sample weights are one number per sample: the model must have a single output of shape (batch, 1), the binary models'
        probability (a wider or multi-output model would need Keras' broadcasting of the weights over its columns)."""
        out = self.outputs
        if not isinstance(out, KTensor) or tuple(out.shape[1:]) != (1,):
            shape = out.shape if isinstance(out, KTensor) else [getattr(o, "shape", None) for o in _flatten(out)]
            raise NotImplementedError(f"{what}: supported for a model with one output of shape (batch, 1), not {shape}")

    def _train_step(self, x, y, weight: Optional[np.ndarray] = None) -> float:
        if self._fused is not None and isinstance(x, dict):
            n = len(np.asarray(next(iter(x.values()))))
            self._fused.build(n, self.optimizer)
            return self._fused.train_on_batch(x, y, weight) + self._fused.reg_loss()
        self.sync()
        from .kernels import deferred_id_checks

        with deferred_id_checks():  # the lookups' out-of-range flags are read once, with the loss, instead of one host sync per lookup
            return self._train_on_batch_layers(x, y, weight)

    def _weighted_loss(self, yt: torch.Tensor, out, wt: Optional[torch.Tensor]):
        """self.loss(yt, out), with the batch's sample weights handed to the built-in loss."""
        global _step_weight
        _step_weight = wt
        try:
            return self.loss(yt, out)
        finally:
            _step_weight = None

    def _train_on_batch_layers(self, x, y, weight: Optional[np.ndarray] = None) -> float:
        out = self(x, training=True)
        yt = torch.as_tensor(np.asarray(y), dtype=torch.float32).to(device()) if not isinstance(y, torch.Tensor) else y.to(device())
        wt = torch.from_numpy(weight).to(device()) if weight is not None else None
        loss = self._weighted_loss(yt, out, wt)
        if self._metric_set is not None:  # Keras updates the metrics from the training forward, before the weight update
            self._metric_set.update(out, yt, wt)
        params = self.weights_with_l2()
        for p, _ in params:
            p.grad = None
        clip = self._layer_clip(params)
        if clip is None:
            loss.backward()
        else:
            from . import autograd_ops

            autograd_ops._grad_clip = clip  # EmbeddingFn clamps and counts the position rows of the dense-gradient tables
            try:
                loss.backward()
            finally:
                autograd_ops._grad_clip = None
        sparse = [l for l in self._all_layers() if getattr(l, "_sparse_grads", None)]
        skip = {id(l.embeddings) for l in sparse}
        # Keras adds the regularisation losses to the reported loss; their gradient 2*l2*W is applied inside the update kernels
        # (tables under the sparse row update are left out of the reported term: a full pass over them is what that update avoids)
        reg = sum(float(l2) * float((p.detach() * p.detach()).sum()) for p, l2 in params if l2 and id(p) not in skip)
        if clip is not None:
            params = self._clip_gradients(clip, params, sparse)
        self.optimizer.step(params)
        for l in sparse:  # large tables: IndexedSlices-style gradient -> sorted-segment row update
            l.apply_sparse(self.optimizer)
        self._update_moving_stats()
        return float(loss.detach()) + reg

    _clip_state = None  # handyrec_b200.clip.GradClip of the layer path, built at the first clipped step

    def _layer_clip(self, params):
        """The GradClip of this step (sums zeroed, variables indexed), or None when the optimizer does not clip."""
        from .clip import GradClip, clip_args

        args = clip_args(self.optimizer)
        if args is None:
            return None
        live = [p for p, _ in params if p.requires_grad]
        st = self._clip_state
        if st is None or st.n_vars != len(live):
            st = self._clip_state = GradClip(args, len(live), 0, device())
        st.var = {id(p): i for i, p in enumerate(live)}
        # tables without a regulariser whose gradient is formed densely: their lookups' IndexedSlices values are clipped in
        # EmbeddingFn.backward, position by position
        st.table_vars = {id(l.embeddings): st.var[id(l.embeddings)] for l in self._all_layers()
                         if hasattr(l, "SPARSE_UPDATE_MIN_ROWS") and not l.l2 and id(l.embeddings) in st.var}
        st.begin()
        return st

    def _clip_gradients(self, clip, params, sparse):
        """Keras' _transform_gradients on this step's gradients, in place: the dense gradients with 2*l2*w folded in, the large
        tables' (ids, rows) per position; then the norm scales.  Returns params with l2 = 0 (folded)."""
        var, tv = clip.var, clip.table_vars
        rows = []
        for l in sparse:  # the concatenated lookups of one table: Keras' aggregated IndexedSlices, in a buffer of our own
            ids = torch.cat([i for i, _ in l._sparse_grads])
            r = torch.cat([g for _, g in l._sparse_grads])
            l._sparse_grads[:] = [(ids, r)]
            rows.append((r, var[id(l.embeddings)]))
        dense = [(p, l2) for p, l2 in params if p.grad is not None and p.requires_grad and id(p) not in tv]
        for p, _ in dense:
            p.grad = p.grad.contiguous()
        gs = [p.grad for p, _ in dense] + [r for r, _ in rows]
        vs = [var[id(p)] for p, _ in dense] + [v for _, v in rows]
        clip.prepare(gs, [p.data for p, _ in dense] + [None] * len(rows), [2.0 * l2 for _, l2 in dense] + [0.0] * len(rows), vs)
        clip.finish()
        tabs = [p for p, _ in params if p.grad is not None and id(p) in tv]
        clip.apply(gs + [p.grad for p in tabs], vs + [tv[id(p)] for p in tabs])
        return [(p, 0.0) for p, _ in params]

    def save_weights(self, filepath, **kwargs):
        """keras.Model.save_weights: a directory of `.npy` files (tables row-sharded), see handyrec_b200.checkpoint."""
        from .checkpoint import save_weights

        save_weights(self, filepath)

    def load_weights(self, filepath, **kwargs):
        from .checkpoint import load_weights

        load_weights(self, filepath)

    def _all_layers(self):
        out, seen = [], set()
        for l in self.layers:
            for sub in [l] + _all_sublayers(l):
                if id(sub) not in seen:
                    seen.add(id(sub))
                    out.append(sub)
        return out

    def _update_moving_stats(self):
        for sub in self._all_layers():
            fn = getattr(sub, "_commit_moving_stats", None)
            if fn:
                fn()

    def fit(self, x=None, y=None, batch_size=32, epochs=1, validation_data=None, verbose=0, sample_weight=None, class_weight=None,
            **kwargs):
        """keras.Model.fit over a dict of arrays (+ y), an `(x, y)` / `(x, y, sample_weight)` tuple, or an iterable of such batches.
        sample_weight / class_weight: Keras' per-sample weights of the training data (folded into one float32 weight per sample
        once per fit); validation_data may be `(x, y, sample_weight)`."""
        history = {"loss": []}
        if isinstance(x, tuple) and len(x) in (2, 3) and isinstance(x[0], dict) and y is None:
            x, y, *rest = x
            sample_weight = rest[0] if rest else sample_weight
        weight = self._weights(y, sample_weight, class_weight) if isinstance(x, dict) else None
        if not isinstance(x, dict) and sample_weight is not None:
            raise ValueError("sample_weight with an iterable of batches: yield (x, y, sample_weight) batches instead")
        batches = _batches(x, y, batch_size, weight, class_weight=class_weight, model=self)
        for _ in range(epochs):
            self.reset_metrics()  # Keras resets the metrics at the start of every epoch
            if self._fused is not None and isinstance(x, dict):
                # dict-of-arrays input: batches are packed into pinned memory one step ahead of the GPU and the whole epoch
                # runs on the fused engine with asynchronous loss read-back (lowering.FusedDeepFM.fit_epoch)
                n = len(np.asarray(next(iter(x.values()))))
                self._fused.build(min(batch_size, n), self.optimizer)
                losses = self._fused.fit_epoch(x, y, batch_size, weight)
                sizes = [min(batch_size, n - s) for s in range(0, n, batch_size)]
                history["loss"].append(float(np.average(losses, weights=sizes)) + self._fused.reg_loss())
                self.last_losses = losses
            else:
                tot, cnt = 0.0, 0
                for xb, yb, wb in batches():  # Keras reports the sample-weighted running mean of the batch losses
                    nb = len(yb) if hasattr(yb, "__len__") else 1
                    tot += self._train_step(xb, yb, wb) * nb
                    cnt += nb
                history["loss"].append(tot / max(cnt, 1))
            if self._metric_set is not None:
                for k, v in self._metric_values().items():
                    history.setdefault(k, []).append(v)
            # fused training leaves the dense / FM weights in the engine; they are handed back to the layers lazily, the first time
            # anything reads the layers (`layers`, `get_layer`, `predict` on the layer path, `save_weights`, `sync()`)
            if validation_data is not None:
                vl, vres = self._evaluate_pass(validation_data, batch_size)
                history.setdefault("val_loss", []).append(vl)
                for k, v in vres.items():
                    history.setdefault("val_" + k, []).append(v)

        class H:
            pass

        h = H()
        h.history = history
        return h

    def _evaluate_pass(self, data, batch_size: int):
        """The validation pass of `fit` and the body of `evaluate`: (loss, metric results), the metrics reset first.  `data`: `(x, y)`,
        `(x, y, sample_weight)` or an iterable of such batches."""
        ms = self._metric_set
        self.reset_metrics()
        fused_val = (self._fused is not None and self._fused.engine is not None and isinstance(data, tuple) and len(data) in (2, 3)
                     and isinstance(data[0], dict))
        if fused_val:
            # the fused engine's forward (the only reader a row-sharded table has); the compiled loss of its output on the host
            xv, yv = data[:2]
            w = self._weights(yv, data[2]) if len(data) == 3 else None
            l = host_loss(self._fused.spec.loss, self._fused.predict(xv, batch_size, y=yv, metrics=ms, weight=w), yv)
            loss = float((l if w is None else w.astype(np.float64) * l).mean())
        else:
            vl, vc = 0.0, 0
            with torch.no_grad():
                for xb, yb, wb in _batches(data, None, batch_size, model=self)():
                    out = self(xb, training=False)
                    yt = torch.as_tensor(np.asarray(yb), dtype=torch.float32).to(device())
                    wt = torch.from_numpy(wb).to(device()) if wb is not None else None
                    vl += float(self._weighted_loss(yt, out, wt))
                    if ms is not None:
                        ms.update(out, yt, wt)
                    vc += 1
            loss = vl / max(vc, 1)
        return loss, (self._metric_values() if ms is not None else OrderedDict())

    def evaluate(self, x=None, y=None, batch_size=None, verbose=0, sample_weight=None, steps=None, callbacks=None, return_dict=False,
                 **kwargs):
        """keras.Model.evaluate: the loss, or [loss, *metric results] when metrics are compiled (a dict with return_dict).  The
        loss is what `fit(validation_data=(x, y), batch_size=batch_size)` records as val_loss on the same path.  Sample weights
        come with the data, as `validation_data` takes them: `evaluate((x, y, sample_weight))` or an iterable of
        `(x, y, sample_weight)` batches (the same val_loss as `validation_data=(x, y, sample_weight)`); the `sample_weight`
        keyword is not supported (NotImplementedError)."""
        if sample_weight is not None:
            raise NotImplementedError("evaluate(sample_weight=...): pass the weights with the data, evaluate((x, y, sample_weight)) or "
                                      "an iterable of (x, y, sample_weight) batches")
        bs = batch_size or 32
        data = x if (y is None and not isinstance(x, dict)) else (x, y)
        if (self._fused is not None and self._fused.engine is None and isinstance(data, tuple) and isinstance(data[0], dict)
                and self._comm is not None and self._comm.N > 1 and self.optimizer is not None):
            # a multi-GPU model before its first fit: only the engine reads row-sharded tables (collective, as in predict)
            n = len(np.asarray(next(iter(data[0].values()))))
            self._fused.build(min(bs, n), self.optimizer)
        loss, res = self._evaluate_pass(data, bs)
        return self._with_metrics(loss, res, return_dict)


from .metrics import AUC, BinaryAccuracy, Precision, Recall  # noqa: E402  (tf.keras.metrics look-alikes, re-exported)


def _all_sublayers(l: Layer) -> List[Layer]:
    out = []
    for s in l._sublayers:
        out += [s] + _all_sublayers(s)
    return out


def _batches(x, y, batch_size, weight: Optional[np.ndarray] = None, class_weight=None, model: Optional[Model] = None):
    """x: dict of arrays (+ y, + the float32 sample weights `weight`), an (x, y) or (x, y, sample_weight) tuple, or an iterable of
    (dict, label) or (dict, label, sample_weight) batches (what tf.data yields in the reference tests).  Yields (x, y, weight or
    None) batches; the weights of a tuple or of a batch are checked and class_weight folded in by model._weights."""
    fold = (lambda yy, sw: model._weights(yy, sw, class_weight)) if model is not None else (lambda yy, sw: None)

    def gen():
        if isinstance(x, dict):
            n = len(next(iter(x.values())))
            for s in range(0, n, batch_size):
                yield {k: v[s : s + batch_size] for k, v in x.items()}, y[s : s + batch_size], (weight[s : s + batch_size] if weight is not None else None)
        elif isinstance(x, tuple) and len(x) in (2, 3) and isinstance(x[0], dict):
            xd, yd = x[:2]
            wd = fold(yd, x[2]) if len(x) == 3 else None
            n = len(next(iter(xd.values())))
            for s in range(0, n, batch_size):
                yield {k: v[s : s + batch_size] for k, v in xd.items()}, yd[s : s + batch_size], (wd[s : s + batch_size] if wd is not None else None)
        else:
            for batch in x:
                xb, yb, *swb = batch
                yield xb, yb, fold(yb, swb[0] if swb else None)

    return gen
