"""Lowering of a `keras_lite.Model` graph onto the fused engines.

`handyrec.models.DeepFM(...)` (models/ranking/context_aware/DeepFM.py:59-94) wires
    Input -> CustomEmbedding [-> SequencePoolingLayer] -> concat -> {DNN, FM} -> add -> sigmoid   (task="binary")
    ...                                                                              -> add              (task="regression")
out of generic layers.  Executed layer by layer that is two lookups per table, a materialised (B,L,D) tensor + mask, a dense
vocab x D gradient per table and one FFMA GEMM per Dense.  `lower(model)` recognises that graph, checks what the fused
`DeepFMEngine` covers (FM and DNN groups over the same features, one embedding dim, mean / sum pooling, element-wise DNN
activations, no BatchNorm / Dropout) and returns a `FusedDeepFM` binding through which `Model.fit / train_on_batch / predict`
run: ONE plan lookup for both groups, the tcgen05 dense layers, the two-level-partition embedding backward and the flat
optimiser step.  The sigmoid head lowers with binary_crossentropy, the linear head with mean_squared_error, mean_absolute_error
or Huber.  Graphs and pairings the engine does not cover return None and keep the layer-by-layer path -- same results, slower.

Host side of `fit`: the dict-of-arrays batches Keras takes are packed into one int32 id matrix + one fp32 dense matrix in pinned
memory by `hrb_host_pack_*` (a thread pool inside the library) on a background thread, one batch ahead of the GPU.
"""
from __future__ import annotations

import ctypes
import os
import queue
import threading
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import call
from .keras_lite import KTensor, Lambda


def _is_input(t) -> bool:
    return isinstance(t, KTensor) and getattr(t, "is_input", False)


def _producer(t):
    return None if not isinstance(t, KTensor) or t.node is None else t.node.layer


def _elements(t: KTensor, axis_ok: Sequence[int]) -> Optional[List[KTensor]]:
    """Inputs of the Concatenate that made `t` (or [t] when `_concat` passed a single tensor through, layers/utils.py:24-25)."""
    from .layers.utils import Concatenate

    lay = _producer(t)
    if isinstance(lay, Concatenate):
        if lay.axis not in axis_ok:
            return None
        return list(t.node.inputs)
    return [t]


def _through(t: KTensor, cls) -> Optional[KTensor]:
    lay = _producer(t)
    return t.node.inputs if isinstance(lay, cls) else None


class _Field:
    __slots__ = ("emb", "inp", "seq_len", "pool")

    def __init__(self, emb, inp, seq_len, pool):
        self.emb, self.inp, self.seq_len, self.pool = emb, inp, seq_len, pool

    def key(self):
        return (id(self.emb), self.inp.name, self.seq_len, self.pool)


def _field_of(t: KTensor) -> Optional[_Field]:
    """(embedding layer, input, seq_len, pooling) behind one (B,1,D) embedding of FeatureGroup.embedding_lookup (group.py:320-332)."""
    from .layers import CustomEmbedding, SequencePoolingLayer

    lay = _producer(t)
    if isinstance(lay, SequencePoolingLayer):
        src = t.node.inputs
        emb = _producer(src)
        if not isinstance(emb, CustomEmbedding) or not _is_input(src.node.inputs) or lay.method not in ("mean", "sum"):
            return None
        inp = src.node.inputs
        return _Field(emb, inp, int(inp.shape[-1]), lay.method)
    if isinstance(lay, CustomEmbedding):
        inp = t.node.inputs
        if not _is_input(inp) or int(inp.shape[-1]) != 1:
            return None
        return _Field(lay, inp, 1, "none")
    return None


class DeepFMSpec:
    """What `lower` read off the graph.  `head`: "sigmoid" (task="binary") or "linear" (task="regression", the output is the add);
    `loss`: the compiled loss as (name, huber delta), set by `lower`."""

    def __init__(self):
        self.fields: List[_Field] = []
        self.dense_inputs: List[KTensor] = []
        self.dnn = None
        self.fm = None
        self.head = "sigmoid"
        self.loss: Tuple[str, float] = ("binary_crossentropy", 0.0)


def match_deepfm(model) -> Optional[DeepFMSpec]:
    from .keras_lite import Activation
    from .layers import DNN, FM
    from .layers.utils import Cast, Flatten

    out = model.outputs
    if not isinstance(out, KTensor):
        return None
    head = "linear" if isinstance(_producer(out), Lambda) else "sigmoid"
    if head == "sigmoid" and (not isinstance(_producer(out), Activation) or _producer(out).activation != "sigmoid"):
        return None
    summed = out if head == "linear" else out.node.inputs
    add = _producer(summed)
    if not isinstance(add, Lambda) or add.name != "add" and not add.name.startswith("add"):
        return None
    parts = list(summed.node.inputs)
    if len(parts) != 2:
        return None
    dnn_t = next((p for p in parts if isinstance(_producer(p), DNN)), None)
    fm_t = next((p for p in parts if isinstance(_producer(p), FM)), None)
    if dnn_t is None or fm_t is None:
        return None
    dnn, fm = _producer(dnn_t), _producer(fm_t)
    if dnn.use_bn or dnn.dropout_rate or dnn.output_activation not in ("linear", None) or dnn.activation not in ("relu", "sigmoid", "tanh", "linear", None):
        return None
    if not dnn.hidden_units or dnn.hidden_units[-1] != 1:
        return None
    # FM input: concat([], fm_sparse, axis=1, keepdims=True) -> (B, F, D)
    fm_elems = _elements(fm_t.node.inputs, (1,))
    if fm_elems is None:
        return None
    fm_fields = [_field_of(e) for e in fm_elems]
    # DNN input: concat(dense, sparse): Concatenate(-1)[Flatten(dense part), Flatten(sparse part)] or Flatten(sparse part)
    x = dnn_t.node.inputs
    halves = _elements(x, (-1,))
    if halves is None or len(halves) not in (1, 2):
        return None
    flat = [_through(h, Flatten) for h in halves]
    if any(f is None for f in flat):
        return None
    sparse_part = flat[-1]
    dense_inputs: List[KTensor] = []
    if len(flat) == 2:
        dense_elems = _elements(flat[0], (-1,))
        if dense_elems is None:
            return None
        for d in dense_elems:
            src = _through(d, Cast)
            src = d if src is None else src
            if not _is_input(src) or len(src.shape) != 2:
                return None
            dense_inputs.append(src)
    dnn_elems = _elements(sparse_part, (-1,))
    if dnn_elems is None:
        return None
    dnn_fields = [_field_of(e) for e in dnn_elems]
    if any(f is None for f in fm_fields + dnn_fields):
        return None
    if [f.key() for f in fm_fields] != [f.key() for f in dnn_fields]:
        return None  # the engine shares ONE lookup between the FM and the DNN group (DeepFM.py:62-63 with equal feature lists)
    dims = {f.emb.output_dim for f in dnn_fields}
    if len(dims) != 1 or next(iter(dims)) % 4 != 0:
        return None
    if len({f.emb.l2 for f in dnn_fields}) != 1:
        return None
    if any(not f.emb.trainable for f in dnn_fields):
        return None
    spec = DeepFMSpec()
    spec.fields, spec.dense_inputs, spec.dnn, spec.fm, spec.head = dnn_fields, dense_inputs, dnn, fm, head
    return spec


_NP_DTYPE = {np.dtype("int32"): 0, np.dtype("int64"): 1, np.dtype("float32"): 2, np.dtype("float64"): 3}


class _ColumnSet:
    """ctypes descriptors of the per-feature arrays of one `x` dict for hrb_host_pack_*."""

    def __init__(self, arrays: Sequence[np.ndarray]):
        self.keep = []
        n = len(arrays)
        self.ptrs = (ctypes.c_void_p * max(n, 1))()
        self.dtype = (ctypes.c_int32 * max(n, 1))()
        self.width = (ctypes.c_int64 * max(n, 1))()
        self.ld = (ctypes.c_int64 * max(n, 1))()
        self.n = n
        self.total = 0
        for i, a in enumerate(arrays):
            a = np.asarray(a)
            if a.ndim == 1:
                a = a.reshape(-1, 1)
            if a.dtype not in _NP_DTYPE:
                a = a.astype(np.float32 if a.dtype.kind == "f" else np.int64)
            if not a.flags.c_contiguous:
                a = np.ascontiguousarray(a)
            self.keep.append(a)
            self.ptrs[i] = a.ctypes.data
            self.dtype[i] = _NP_DTYPE[a.dtype]
            self.width[i] = a.shape[1]
            self.ld[i] = a.shape[1]
            self.total += a.shape[1]


class HostBatch:
    """One packed batch in pinned memory + the event that says its host->device copies are done (slot reusable).  The sample
    weight column is pinned at the first batch with weights; `weighted` says whether the batch packed now has them."""

    def __init__(self, B: int, ids_cols: int, n_dense: int):
        self.ids = torch.empty(B, max(ids_cols, 1), dtype=torch.int32).pin_memory()
        self.dense = torch.empty(B, max(n_dense, 1), dtype=torch.float32).pin_memory()
        self.label = torch.empty(B, dtype=torch.float32).pin_memory()
        self.weight: Optional[torch.Tensor] = None
        self.weighted = False
        self.copied: Optional[torch.cuda.Event] = None
        self.rows = 0

    def views(self):
        """(ids, dense, label, weight or None) of the packed rows."""
        r = self.rows
        return self.ids[:r], self.dense[:r], self.label[:r], (self.weight[:r] if self.weighted else None)


class FusedDeepFM:
    """A lowered DeepFM: the model's layers keep their weights (shared storage for the tables), the engine runs the steps."""

    def __init__(self, model, spec: DeepFMSpec):
        self.model, self.spec = model, spec
        self.engine = None
        self.tables: List = []  # unique CustomEmbedding layers, in first-use order
        for f in spec.fields:
            if all(f.emb is not t for t in self.tables):
                self.tables.append(f.emb)
        self.n_dense = sum(int(t.shape[-1]) for t in spec.dense_inputs)
        self.ids_cols = sum(f.seq_len for f in spec.fields)
        self._dirty = False
        self._slots: List[HostBatch] = []
        # packing threads: the host's cores are shared by the ranks of this node (torchrun exports LOCAL_WORLD_SIZE)
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
        self._pack_threads = max(1, min(16, cores // ranks - (1 if ranks > 1 else 0)))  # leave a core to the rank's launching thread

    # ---- engine construction ------------------------------------------------------------------
    def _dense_layers(self):
        from .layers.core import Dense

        return [l for l in self.spec.dnn.layers if isinstance(l, Dense)]

    @staticmethod
    def engine_key(optimizer) -> tuple:
        """What an engine is built for: a fit whose optimizer gives another key rebuilds it (fresh optimizer slots).  A schedule is
        keyed by the object, not a value: the engine takes the rate per step and is not rebuilt as it changes."""
        from .clip import clip_args
        from .keras_lite import Adagrad, Adam, Ftrl, SGD

        key = None
        if isinstance(optimizer, Adam):
            opt, lr = "adam", optimizer.lr
        elif isinstance(optimizer, SGD):
            opt, lr = "sgd", optimizer.lr
        elif isinstance(optimizer, Adagrad):
            opt, lr = "adagrad", optimizer.lr
        elif isinstance(optimizer, Ftrl):
            opt, lr = "ftrl", optimizer.lr
            key = (opt, lr, optimizer.learning_rate_power, optimizer.initial_accumulator_value, optimizer.l1, optimizer.l2,
                   optimizer.l2_shrinkage, optimizer.beta)
        else:
            raise ValueError("the fused DeepFM path takes keras_lite.Adam, keras_lite.SGD, keras_lite.Adagrad or keras_lite.Ftrl")
        return (key or (opt, lr), clip_args(optimizer), optimizer.decay)

    def build(self, batch_size: int, optimizer) -> None:
        from .engine import DeepFMEngine
        from .schedules import LearningRateSchedule, decayed_lr

        key = self.engine_key(optimizer)
        opt, lr, clip = key[0][0], optimizer.lr, key[1]
        # every step the engine issues sets its own rate (_lr_step); a schedule is evaluated there only, once per step
        lr = None if isinstance(lr, LearningRateSchedule) else decayed_lr(optimizer)
        if self.engine is not None and self.engine.B >= batch_size and self._opt_key == key:
            self.engine.metrics = getattr(self.model, "_metric_set", None)
            self.engine.lr_step = _lr_step(optimizer)
            return
        self.sync_to_layers()
        dev = torch.device("cuda", torch.cuda.current_device())
        fields = [(next(i for i, t in enumerate(self.tables) if t is f.emb), f.seq_len, f.pool) for f in self.spec.fields]
        dnn = self.spec.dnn
        small = getattr(self.model, "dense_table_max_rows", 131072)
        common = dict(dnn_hidden_units=tuple(dnn.hidden_units), dnn_activation=dnn.activation or "linear", batch_size=batch_size, optimizer=opt,
                      lr=lr, l2_embd=self.spec.fields[0].emb.l2, l2_dnn=float(dnn.l2_reg or 0.0), seed=dnn.seed)
        if self.spec.head == "linear":
            common.update(task="regression", loss=self.spec.loss[0], huber_delta=self.spec.loss[1])
        if opt in ("adagrad", "ftrl"):  # the engine fills its accumulators when it is built
            common["initial_accumulator_value"] = optimizer.initial_accumulator_value
        if opt == "ftrl":
            common.update(l1=optimizer.l1, l2=optimizer.l2, learning_rate_power=optimizer.learning_rate_power,
                          l2_shrinkage=optimizer.l2_shrinkage, beta=optimizer.beta)
        comm = getattr(self.model, "_comm", None)
        if comm is not None and comm.N > 1:
            eng = self._build_sharded(comm, dev, fields, small, common)
        else:
            tabs = [t.embeddings.data.to(dev) for t in self.tables]
            clip_kw = dict(zip(("clipvalue", "clipnorm", "global_clipnorm"), clip)) if clip is not None else {}
            eng = DeepFMEngine(tabs, fields, self.n_dense, dense_table_max_rows=small, **common, **clip_kw)
        if opt == "adam":
            eng.beta1, eng.beta2, eng.eps = optimizer.b1, optimizer.b2, optimizer.eps
        elif opt == "adagrad":
            eng.eps = optimizer.eps
        for i, d in enumerate(self._dense_layers()):
            eng.set_dense_weights(i, d.kernel.data.cpu(), d.bias.data.cpu())
        eng.fm_w.copy_(self.spec.fm.linear.data.reshape(-1).to(dev))
        eng.fm_w0.copy_(self.spec.fm.w_0.data.reshape(-1).to(dev))
        eng.step_count = getattr(optimizer, "t", 0)
        eng.lr_step = _lr_step(optimizer)
        for t, lay in enumerate(self.tables):  # the layer and the engine share ONE copy of every table
            lay.embeddings.data = eng.tables[t]
        eng.metrics = getattr(self.model, "_metric_set", None)  # counted by train_step_on_device right after the loss
        self.engine, self._opt_key = eng, key
        self._slots = []

    def _build_sharded(self, comm, dev, fields, small: int, common: dict):
        """`compile(..., distribute=True)` under torch.distributed (one process per GPU): tables above `dense_table_max_rows` are
        row-sharded (row % N, shards in symmetric memory so that peers read them over NVLink), the others replicated; dense
        parameters are replicated.  Every rank built the model with the SAME seed, so its full-size tables are identical: a
        sharded table keeps this rank's rows of it and the full copy is released; replicated tables and dense weights are
        broadcast from rank 0 anyway.  Each rank then fits its own slice of the data (weak scaling, like DistributedDataParallel)."""
        import torch.distributed as dist

        from .sharded import ShardedDeepFMEngine

        vocabs = [t.input_dim for t in self.tables]
        D = self.tables[0].output_dim
        tabs, peer_ptrs = comm.alloc_tables(vocabs, D, dev, replicate_max_rows=small)
        for t, lay in enumerate(self.tables):
            cur = lay.embeddings.data.to(dev)
            if vocabs[t] <= small:
                if lay._sharded is not None:
                    raise ValueError(f"{lay.name} was created sharded but dense_table_max_rows={small} asks for a replicated copy")
                dist.broadcast(cur, src=0, group=comm.group)
                tabs[t].copy_(cur)
            elif lay._sharded is not None:  # created under ShardedTables (or a rebuild): already this rank's rows
                tabs[t].copy_(cur)
            else:  # a full table built from the same seed on every rank: keep this rank's rows, release the rest
                tabs[t].copy_(cur[comm.rank :: comm.N])
                lay._sharded = (comm.rank, comm.N, vocabs[t])
            lay.embeddings.data = tabs[t]
            del cur
        torch.cuda.empty_cache()
        for d in self._dense_layers():
            dist.broadcast(d.kernel.data, src=0, group=comm.group)
            dist.broadcast(d.bias.data, src=0, group=comm.group)
        dist.broadcast(self.spec.fm.linear.data, src=0, group=comm.group)
        dist.broadcast(self.spec.fm.w_0.data, src=0, group=comm.group)
        peer = getattr(self.model, "peer_lookup", True) and all(f[1] == 1 and f[2] in ("none", None) for f in fields)
        return ShardedDeepFMEngine(tabs, vocabs, fields, self.n_dense, comm, peer_ptrs=peer_ptrs if peer else None, replicate_max_rows=small,
                                   p2p_grad_exchange=getattr(self.model, "p2p_grad_exchange", True), **common)

    def sync_to_layers(self) -> None:
        """Dense / FM weights live in the engine's flat buffer while it trains; hand them back to the layers."""
        eng = self.engine
        if eng is None or not self._dirty:
            return
        for i, d in enumerate(self._dense_layers()):
            w, b = eng.get_dense_weights(i)
            d.kernel.data.copy_(w.to(d.kernel.device))
            d.bias.data.copy_(b.to(d.bias.device))
        self.spec.fm.linear.data.copy_(eng.fm_w.reshape(-1, 1))
        self.spec.fm.w_0.data.copy_(eng.fm_w0.reshape(-1))
        self._dirty = False

    def push_to_engine(self) -> None:
        """The inverse of sync_to_layers, after load_weights / set_weights wrote the layers: the dense / FM weights go into the live
        engine's flat buffer (and its transposed copies).  The engine is not rebuilt and its optimizer slots are kept; the tables
        need nothing, the layers share their storage with the engine."""
        eng = self.engine
        if eng is None:
            return
        for i, d in enumerate(self._dense_layers()):
            eng.set_dense_weights(i, d.kernel.data.cpu(), d.bias.data.cpu())
        eng.fm_w.copy_(self.spec.fm.linear.data.reshape(-1))
        eng.fm_w0.copy_(self.spec.fm.w_0.data.reshape(-1))
        self._dirty = False

    # ---- host input packing ---------------------------------------------------------------------
    def _columns(self, x: Dict[str, np.ndarray]) -> Tuple[_ColumnSet, _ColumnSet, int]:
        for f in self.spec.fields:
            if f.inp.name not in x:
                raise KeyError(f"missing input {f.inp.name!r}")
        id_cols = _ColumnSet([x[f.inp.name] for f in self.spec.fields])
        dense_cols = _ColumnSet([x[t.name] for t in self.spec.dense_inputs])
        if id_cols.total != self.ids_cols or dense_cols.total != self.n_dense:
            raise ValueError("input widths do not match the feature definitions")
        n = len(id_cols.keep[0])
        return id_cols, dense_cols, n

    def _pack(self, slot: HostBatch, id_cols, dense_cols, label_cols, start: int, rows: int, weight_cols=None) -> None:
        if slot.copied is not None:
            slot.copied.synchronize()  # the previous user's host->device copies have left this pinned slot
        slot.weighted = weight_cols is not None
        if slot.weighted:
            if slot.weight is None:
                slot.weight = torch.empty(slot.label.shape[0], dtype=torch.float32).pin_memory()
            call("hrb_host_pack_f32", weight_cols.ptrs, weight_cols.dtype, weight_cols.width, weight_cols.ld, 1, start, rows,
                 ctypes.c_void_p(slot.weight.data_ptr()), 1, 0)
        call("hrb_host_pack_i32", id_cols.ptrs, id_cols.dtype, id_cols.width, id_cols.ld, id_cols.n, start, rows,
             ctypes.c_void_p(slot.ids.data_ptr()), slot.ids.shape[1], self._pack_threads)
        if self.n_dense:
            call("hrb_host_pack_f32", dense_cols.ptrs, dense_cols.dtype, dense_cols.width, dense_cols.ld, dense_cols.n, start, rows,
                 ctypes.c_void_p(slot.dense.data_ptr()), slot.dense.shape[1], self._pack_threads)
        if label_cols is not None:
            call("hrb_host_pack_f32", label_cols.ptrs, label_cols.dtype, label_cols.width, label_cols.ld, 1, start, rows,
                 ctypes.c_void_p(slot.label.data_ptr()), 1, 0)
        slot.rows = rows

    def _get_slots(self, n: int) -> List[HostBatch]:
        while len(self._slots) < n:
            self._slots.append(HostBatch(self.engine.B, self.ids_cols, self.n_dense))
        return self._slots

    def host_batches(self, x, y, batch_size: int, n_slots: int = 4, weight: Optional[np.ndarray] = None):
        """Generator of packed pinned batches; packing runs on a background thread, up to n_slots-2 batches ahead.  `weight`: the
        float32 sample weights of the rows (Keras' sample_weight with class_weight folded in), packed like the label."""
        id_cols, dense_cols, n = self._columns(x)
        label_cols = _ColumnSet([np.asarray(y).reshape(-1, 1)]) if y is not None else None
        weight_cols = _weight_columns(weight)
        slots = self._get_slots(n_slots)
        q: "queue.Queue" = queue.Queue(maxsize=max(1, n_slots - 2))
        dev_index = torch.cuda.current_device()

        stop = threading.Event()

        def producer():
            try:
                torch.cuda.set_device(dev_index)
                k = 1
                for start in range(batch_size, n, batch_size):
                    if stop.is_set():
                        return
                    slot = slots[k % n_slots]
                    self._pack(slot, id_cols, dense_cols, label_cols, start, min(batch_size, n - start), weight_cols)
                    q.put(slot)
                    k += 1
                q.put(None)
            except BaseException as e:  # surface packing errors on the consumer side
                q.put(e)

        if n == 0:
            return
        # The first batch is packed right here: the GPU gets its first step without waiting for a thread to start (0.3-0.8 ms);
        # the producer thread for the remaining batches starts while that step runs.
        self._pack(slots[0], id_cols, dense_cols, label_cols, 0, min(batch_size, n), weight_cols)
        yield slots[0]
        th = threading.Thread(target=producer, daemon=True)
        th.start()
        try:
            while True:
                item = q.get()
                if item is None:
                    break
                if isinstance(item, BaseException):
                    raise item
                yield item
        finally:
            # a consumer that stops early (a callback ended training) closes the generator: the producer stops at its next batch,
            # and whatever it still queues is drained so that it never blocks on the full queue
            stop.set()
            while th.is_alive():
                try:
                    q.get(timeout=0.01)
                except queue.Empty:
                    pass
            th.join()

    # ---- Keras-facing calls -----------------------------------------------------------------------
    def fit_epoch(self, x, y, batch_size: int, weight: Optional[np.ndarray] = None, on_step=None) -> List[float]:
        """One epoch over `x` on the engine; `on_step`: DeepFMEngine.fit_batches' per-step hook (callbacks with batch hooks)."""
        self._dirty = True
        hook = None
        if on_step is not None:

            def hook(t: int, loss: Optional[float]) -> bool:
                stop = on_step(t, loss)
                if loss is None:
                    # step t is issued next: a batch hook may have synced the layers (save_weights, get_weights, layers) or
                    # pushed weights into the engine, and whatever it left in the layers is stale once the step runs
                    self._dirty = True
                return stop

        batches = self.host_batches(x, y, batch_size, weight=weight)
        try:
            return self.engine.fit_batches(batches, on_step=hook)
        finally:
            batches.close()

    def train_on_batch(self, x, y, weight: Optional[np.ndarray] = None) -> float:
        id_cols, dense_cols, n = self._columns(x)
        slot = self._get_slots(1)[0]
        self._pack(slot, id_cols, dense_cols, _ColumnSet([np.asarray(y).reshape(-1, 1)]), 0, n, _weight_columns(weight))
        self._dirty = True
        ids, dense, label, w = slot.views()
        return self.engine.train_on_batch(ids, dense if self.n_dense else None, label, w)

    def predict(self, x, batch_size: Optional[int], y=None, metrics=None, weight: Optional[np.ndarray] = None, on_batch=None) -> np.ndarray:
        """Probabilities (a linear head: predictions) of `x`; with `metrics` (a MetricSet) and labels `y`, every batch is also counted on the device (the
        validation pass of fit / evaluate: no second forward), with the rows' sample weights `weight` when given.  `on_batch(i,
        start, pred)`: called with pred None before batch i runs and with its (rows, 1) predictions after (callbacks' batch hooks)."""
        id_cols, dense_cols, n = self._columns(x)
        bs = min(batch_size or n, self.engine.B)
        slot = self._get_slots(1)[0]
        label_cols = _ColumnSet([np.asarray(y).reshape(-1, 1)]) if metrics is not None else None
        weight_cols = _weight_columns(weight) if metrics is not None else None
        outs = []
        for i, start in enumerate(range(0, n, bs)):
            if on_batch is not None:
                on_batch(i, start, None)
            self._pack(slot, id_cols, dense_cols, label_cols, start, min(bs, n - start), weight_cols)
            ids, dense, label, w = slot.views()
            outs.append(self.engine.predict(ids, dense if self.n_dense else None, label, metrics, w).numpy().copy())
            slot.copied = None
            if on_batch is not None:
                on_batch(i, start, outs[-1])
        return np.concatenate(outs, 0)

    def reg_loss(self) -> float:
        """Keras adds the regularisation losses to the reported loss: l2_dnn * sum(W^2) over the Dense kernels + l2_embd * sum over
        the dense-updated tables (tables under the touched-rows update are left out -- a full pass over them every step is
        exactly the cost the lazy update avoids, DESIGN.md 3)."""
        eng = self.engine
        tot = 0.0
        if eng.l2_dnn:
            tot += eng.l2_dnn * float(sum((w * w).sum() for w in eng.W))
        if eng.l2_embd and eng.dense_tables:
            tot += eng.l2_embd * float(sum((eng.tables[t] ** 2).sum() for t in eng.dense_tables))
        return tot


def _weight_columns(weight: Optional[np.ndarray]) -> Optional[_ColumnSet]:
    return _ColumnSet([np.asarray(weight, dtype=np.float32).reshape(-1, 1)]) if weight is not None else None


def _lr_step(optimizer):
    """The engine's per-step rate: Keras' _decayed_lr at the optimizer's `iterations`, which then counts the step.  Called once per
    step the engine issues, so a later fit, rebuild or layer-path step continues the schedule; every rank of a multi-GPU model
    issues the same steps and counts alike."""
    from .schedules import decayed_lr

    def step() -> float:
        lr = optimizer.lr_t = decayed_lr(optimizer)
        optimizer.iterations += 1
        return lr

    return step


def lower(model, loss: Tuple[str, float] = ("binary_crossentropy", 0.0)) -> Optional[FusedDeepFM]:
    """The fused binding of a DeepFM-shaped `model` compiled with `loss` ((name, huber delta) of a built-in loss), or None: a sigmoid
    head trains binary_crossentropy only and a linear head the regression losses only; any other pairing keeps the layer path."""
    spec = match_deepfm(model)
    if spec is None or (spec.head == "sigmoid") != (loss[0] == "binary_crossentropy"):
        return None
    spec.loss = loss
    return FusedDeepFM(model, spec)
