"""Run the reference's OWN model files on this package.

`BASELINE.json: north_star` -- "handyrec.models constructs and fits unchanged".  HandyRec's model constructors
(/root/reference/handyrec/models/**) are ~60 lines of graph wiring each: they import `handyrec.features`, `handyrec.layers`,
`tensorflow` / `tensorflow.keras` and call a dozen TF names (`Model`, `Activation`, `tf.matmul`, `tf.nn.l2_normalize`,
`tf.nn.embedding_lookup`, `tf.squeeze`, `tf.int32`).  `install(reference_root)` registers

    tensorflow, tensorflow.keras[.layers|.models|.initializers|.regularizers|.losses|.optimizers[.schedules]|.metrics|.experimental]
                                                                                                    -> thin modules over keras_lite
    handyrec, handyrec.features, handyrec.layers, handyrec.layers.utils, handyrec.features.*        -> this package's drop-in face
    handyrec.models (+ .ranking, .retrieval, ...)                                                   -> the reference's files, loaded
                                                                                                       from `reference_root` UNMODIFIED

in `sys.modules`, so `from handyrec.models.ranking import DeepFM` yields the reference's constructor building a `keras_lite.Model`
whose `compile / fit / predict` run on libhrb200 (and on the fused engine when the graph is DeepFM-shaped).  Nothing is copied:
without a reference checkout only `handyrec.features` / `handyrec.layers` resolve and `handyrec_b200.models` provides the
constructors.  The shim covers what the five in-scope model files use; DIEN / FMLPRec import fine but their recurrent / FFT layers
raise NotImplementedError when called (out of scope, DESIGN.md 7).
"""
from __future__ import annotations

import importlib.machinery
import importlib.util
import os
import sys
import types
from typing import Optional

import torch

from .. import keras_lite as KL


def _unsupported(name):
    class _Stub(KL.Layer):
        def __init__(self, *a, **k):
            raise NotImplementedError(f"{name} is outside the hot path handyrec_b200 implements (DESIGN.md 7)")

    _Stub.__name__ = name
    return _Stub


def _tf_module() -> types.ModuleType:
    from ..autograd_ops import AttPoolFn, EmbeddingFn, L2NormalizeFn
    from ..layers import core as core_layers
    from ..layers.utils import Concatenate, Flatten

    tf = types.ModuleType("tensorflow")
    tf.__version__ = "2.6.0-handyrec_b200-shim"
    for n in ("int32", "int64", "float32", "bool"):
        setattr(tf, n, KL._DType(n))

    def matmul(a, b):  # DIN.py:93: (B,1,T) x (B,T,D) -> (B,1,D)
        return KL.Lambda(lambda s, k: AttPoolFn.apply(s.reshape(s.shape[0], -1), k), lambda sa, sb: (sb[0], 1, sb[2]), name="matmul")([a, b])

    def squeeze(x, axis=None):
        ax = axis if axis is not None else 1
        return KL.Lambda(lambda t: t.squeeze(ax), lambda s: tuple(d for i, d in enumerate(s) if i != ax), name="squeeze")(x)

    nn = types.ModuleType("tensorflow.nn")

    def l2_normalize(x, axis=None, epsilon=1e-12):
        if axis is not None:
            raise NotImplementedError("the shim implements tf.nn.l2_normalize without an axis (DSSM.py:105-106)")
        return KL.Lambda(lambda t: L2NormalizeFn.apply(t, epsilon), lambda s: s, name="l2_normalize")(x)

    def embedding_lookup(params, ids):
        def gather(m, idx):
            out, _ = EmbeddingFn.apply(m, idx.to(m.device).int().contiguous(), False)
            return out

        return KL.Lambda(gather, lambda sm, si: tuple(si) + (sm[-1],), name="embedding_lookup")([params, ids])

    nn.l2_normalize, nn.embedding_lookup = l2_normalize, embedding_lookup
    tf.matmul, tf.squeeze, tf.nn = matmul, squeeze, nn

    keras = types.ModuleType("tensorflow.keras")
    layers = types.ModuleType("tensorflow.keras.layers")
    for n, obj in (("Layer", KL.Layer), ("Input", KL.Input), ("Activation", KL.Activation), ("Dense", core_layers.Dense),
                   ("BatchNormalization", core_layers.BatchNormalization), ("Dropout", core_layers.Dropout), ("Concatenate", Concatenate),
                   ("Flatten", Flatten)):
        setattr(layers, n, obj)
    for n in ("GRU", "RNN", "LayerNormalization", "Embedding"):
        setattr(layers, n, _unsupported(n))
    models = types.ModuleType("tensorflow.keras.models")
    models.Model = keras.Model = KL.Model
    keras.Sequential = _unsupported("Sequential")
    inits = types.ModuleType("tensorflow.keras.initializers")
    inits.Zeros = KL.Zeros
    regs = types.ModuleType("tensorflow.keras.regularizers")
    from ..features.group import _L2

    regs.l2 = _L2
    losses = types.ModuleType("tensorflow.keras.losses")
    opts = types.ModuleType("tensorflow.keras.optimizers")
    opts.Adam, opts.SGD, opts.Adagrad, opts.Ftrl = KL.Adam, KL.SGD, KL.Adagrad, KL.Ftrl
    for n in ("binary_crossentropy", "mean_squared_error", "mse", "MSE", "mean_absolute_error", "mae", "MAE", "MeanSquaredError",
              "MeanAbsoluteError", "Huber", "BinaryCrossentropy"):
        setattr(losses, n, getattr(KL, n))
    losses.get = KL.get_loss
    opts.get = KL.get_optimizer
    from .. import schedules as S

    scheds = types.ModuleType("tensorflow.keras.optimizers.schedules")
    for n in ("LearningRateSchedule", "ExponentialDecay", "InverseTimeDecay", "PiecewiseConstantDecay", "PolynomialDecay"):
        setattr(scheds, n, getattr(S, n))
    opts.schedules = scheds
    experimental = types.ModuleType("tensorflow.keras.experimental")  # Keras 2.6 keeps the cosine schedules here
    experimental.CosineDecay, experimental.CosineDecayRestarts = S.CosineDecay, S.CosineDecayRestarts
    mets = types.ModuleType("tensorflow.keras.metrics")
    mets.AUC, mets.BinaryAccuracy, mets.Precision, mets.Recall = KL.AUC, KL.BinaryAccuracy, KL.Precision, KL.Recall
    keras.layers, keras.models, keras.initializers, keras.regularizers, keras.losses, keras.optimizers = layers, models, inits, regs, losses, opts
    keras.metrics, keras.experimental = mets, experimental
    tf.keras = keras
    tf._submodules = {"tensorflow.nn": nn, "tensorflow.keras": keras, "tensorflow.keras.layers": layers, "tensorflow.keras.models": models,
                      "tensorflow.keras.initializers": inits, "tensorflow.keras.regularizers": regs, "tensorflow.keras.losses": losses,
                      "tensorflow.keras.optimizers": opts, "tensorflow.keras.optimizers.schedules": scheds, "tensorflow.keras.metrics": mets,
                      "tensorflow.keras.experimental": experimental}
    return tf


def install(reference_root: Optional[str] = None, force: bool = False) -> types.ModuleType:
    """Register the shim modules; returns the `handyrec` alias package.  A REAL tensorflow / handyrec that is already imported is
    left alone unless `force`."""
    if not force:
        for name in ("tensorflow", "handyrec"):
            mod = sys.modules.get(name)
            if mod is not None and not getattr(mod, "__handyrec_b200_shim__", False):
                raise RuntimeError(f"a real `{name}` is already imported; pass force=True to shadow it")
    tf = _tf_module()
    tf.__handyrec_b200_shim__ = True
    sys.modules["tensorflow"] = tf
    sys.modules.update(tf._submodules)

    from .. import features as F
    from .. import layers as L
    from ..features import group as Fgroup, type as Ftype, utils as Futils
    from ..layers import activation, core, interaction, sequence, tools, utils as Lutils

    pkg = types.ModuleType("handyrec")
    pkg.__handyrec_b200_shim__ = True
    pkg.__path__ = []
    layers_alias = types.ModuleType("handyrec.layers")
    layers_alias.__dict__.update({k: getattr(L, k) for k in L.__all__})
    layers_alias.AUGRUCell = _unsupported("AUGRUCell")
    layers_alias.PositionEmbedding = _unsupported("PositionEmbedding")
    layers_alias.__path__ = []
    sys.modules.update({
        "handyrec": pkg, "handyrec.features": F, "handyrec.features.group": Fgroup, "handyrec.features.type": Ftype,
        "handyrec.features.utils": Futils, "handyrec.layers": layers_alias, "handyrec.layers.utils": Lutils, "handyrec.layers.core": core,
        "handyrec.layers.tools": tools, "handyrec.layers.sequence": sequence, "handyrec.layers.interaction": interaction,
        "handyrec.layers.activation": activation,
    })
    pkg.features, pkg.layers = F, layers_alias
    if reference_root is not None:
        mdir = os.path.join(reference_root, "handyrec", "models")
        if not os.path.isdir(mdir):
            raise FileNotFoundError(f"{mdir}: no reference checkout there")
        spec = importlib.util.spec_from_file_location("handyrec.models", os.path.join(mdir, "__init__.py"), submodule_search_locations=[mdir])
        models = importlib.util.module_from_spec(spec)
        sys.modules["handyrec.models"] = models
        spec.loader.exec_module(models)  # the reference's file, unmodified; its submodules import through the normal machinery
        pkg.models = models
    return pkg


def uninstall() -> None:
    for name in list(sys.modules):
        if name == "tensorflow" or name.startswith("tensorflow.") or name == "handyrec" or name.startswith("handyrec."):
            mod = sys.modules[name]
            if name.startswith("tensorflow") and not getattr(sys.modules.get("tensorflow"), "__handyrec_b200_shim__", False):
                continue
            del sys.modules[name]
