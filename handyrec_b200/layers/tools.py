"""Tool layers (mirror of /root/reference/handyrec/layers/tools.py)."""
from __future__ import annotations

from typing import List

import numpy as np
import torch

from ..autograd_ops import AttPoolFn, EmbeddingFn, MatmulNTFn, RowDotFn, SampledSoftmaxFn
from ..keras_lite import KTensor, Layer, device


class ValueTable(Layer):
    """Output the full list of values of a feature (tools.py:10-29): `call` ignores its input."""

    def __init__(self, value_list: List, dtype: str = "int32", **kwargs):
        self._np = np.asarray(value_list)
        self._dtype = dtype
        self.value = None
        super().__init__(**kwargs)

    def call(self, *args, **kwargs):
        if self.value is None:
            from ..keras_lite import _tdtype

            self.value = torch.as_tensor(self._np).to(device(), _tdtype(self._dtype))
        return self.value

    def compute_output_shape(self, input_shape):
        return tuple(self._np.shape)

    def output_dtype(self, inputs):
        return self._dtype


class CustomEmbedding(Layer):
    """Keras Embedding whose mask has the SAME shape as the output (tools.py:87-101).

    Arguments follow keras.layers.Embedding: input_dim, output_dim, embeddings_regularizer (an l2 factor or an object with
    `.l2`), trainable, weights=[ndarray], mask_zero, name.
    """

    def __init__(self, input_dim, output_dim, embeddings_regularizer=None, trainable=True, weights=None, mask_zero=False, **kwargs):
        super().__init__(trainable=trainable, **kwargs)
        self.input_dim, self.output_dim, self.mask_zero = int(input_dim), int(output_dim), bool(mask_zero)
        self.l2 = float(getattr(embeddings_regularizer, "l2", embeddings_regularizer or 0.0))
        self._init_weights = weights
        self.embeddings = None

    def build(self, input_shape):
        from ..keras_lite import ShardedTables

        init = None if self._init_weights is None else np.asarray(self._init_weights[0], dtype=np.float32)
        scope = ShardedTables.active
        if scope is not None and scope.comm.N > 1 and self.input_dim > scope.min_rows and self.trainable:
            # row-sharded creation (keras_lite.ShardedTables): only rows r % N == rank exist on this GPU
            from .. import kernels as K
            from ..keras_lite import device
            from ..sharded import shard_rows

            rank, n = scope.comm.rank, scope.comm.N
            local = torch.empty(shard_rows(self.input_dim, rank, n), self.output_dim, device=device())
            if init is not None:
                local.copy_(torch.from_numpy(np.ascontiguousarray(init[rank::n])))
            else:
                K.init_uniform(local, seed=scope.next_seed(), row_start=rank, row_step=n)
            self.embeddings = torch.nn.Parameter(local, requires_grad=True)
            self._weights["embeddings"] = self.embeddings
            if self.l2:
                self._weight_l2["embeddings"] = self.l2
            self._sharded = (rank, n, self.input_dim)
        else:
            self.embeddings = self.add_weight("embeddings", (self.input_dim, self.output_dim), initializer="uniform", l2=self.l2, value=init)
        self.built = True

    # Tables with at least this many rows keep their gradient sparse (TF: IndexedSlices) and take the touched-rows-only update
    # (lazy Adam: a declared deviation from Keras' dense Adam step, DESIGN.md 3; Adagrad: Keras' own sparse step, exact while
    # l2 = 0); smaller ones get the dense Keras-exact step.  Under Ftrl a table with l2 = 0 takes the touched-rows update at
    # every size: Keras steps only the rows its IndexedSlices gradient lists, and an Ftrl step with a zero gradient is not a
    # no-op, so the dense step would move every other row.
    SPARSE_UPDATE_MIN_ROWS = 131072
    _ftrl = False  # set by Model.compile

    _sharded = None  # (rank, n_ranks, full rows) when `embeddings` is this rank's row shard

    def call(self, inputs):
        if self._sharded is not None:
            raise RuntimeError(f"{self.name}: this table is row-sharded over {self._sharded[1]} GPUs; only the fused engine "
                               "(a DeepFM-shaped model compiled under ShardedTables / distribute=True) reads it")
        ids = inputs.to(torch.int32)
        sink = None
        rows_only = self.input_dim >= self.SPARSE_UPDATE_MIN_ROWS or (self._ftrl and not self.l2)
        if self._ftrl and not self.l2 and self.output_dim % 4 != 0 and self.trainable and torch.is_grad_enabled():
            raise ValueError(f"{self.name}: the touched-rows Ftrl update needs output_dim % 4 == 0, got {self.output_dim}")
        if self.trainable and rows_only and torch.is_grad_enabled() and self.output_dim % 4 == 0:
            if not hasattr(self, "_sparse_grads"):
                self._sparse_grads = []
            sink = self._sparse_grads
        out, mask = EmbeddingFn.apply(self.embeddings, ids, self.mask_zero, sink)
        self._last_mask = mask if self.mask_zero else None
        if not torch.is_grad_enabled():
            out._hrb_src = (self.embeddings.data, ids)  # inference: lets LocalActivationUnit take the fused gather + MLP + pool kernel
        return out

    def apply_sparse(self, optimizer) -> None:
        """One sorted-segment row update for every (ids, gradient rows) pair this step collected (a13: hrb_lookup_bwd_update)."""
        pending = getattr(self, "_sparse_grads", None)
        if not pending:
            return
        from .. import kernels as K
        from ..keras_lite import Adagrad, Adam, Ftrl

        ids = torch.cat([i for i, _ in pending]).reshape(-1, 1).contiguous()
        rows = torch.cat([g for _, g in pending]).contiguous()
        pending.clear()
        adam, adagrad, ftrl = isinstance(optimizer, Adam), isinstance(optimizer, Adagrad), isinstance(optimizer, Ftrl)
        if getattr(self, "_plan", None) is None:
            w = self.embeddings.data
            self._m, self._v = (torch.zeros_like(w), torch.zeros_like(w)) if adam else (None, None)
            self._accum = torch.full_like(w, optimizer.initial_accumulator_value) if (adagrad or ftrl) else None
            self._linear = torch.zeros_like(w) if ftrl else None
            self._plan = K.LookupPlan([w], [(0, 1, "none", 0, 0)], [self._m] if adam else None, [self._v] if adam else None,
                                      accum=[self._accum] if (adagrad or ftrl) else None, linear=[self._linear] if ftrl else None)
        # lr_t: the rate of the step `optimizer.step` just applied (a schedule is evaluated once per step, there)
        if adam:
            self._plan.backward_update(ids, rows, opt="adam", lr=optimizer.lr_t, l2_scale=2.0 * self.l2, beta1=optimizer.b1, beta2=optimizer.b2,
                                       eps=optimizer.eps, step=max(optimizer.t, 1), autotune=True)
        elif adagrad:
            self._plan.backward_update(ids, rows, opt="adagrad", lr=optimizer.lr_t, l2_scale=2.0 * self.l2, eps=optimizer.eps, autotune=True)
        elif ftrl:  # every gathered id is a plain-field position here: row 0 of mask_zero padding steps like any other row
            self._plan.backward_update(ids, rows, opt="ftrl", lr=optimizer.lr_t, l2_scale=2.0 * self.l2, autotune=True, **optimizer.hyper())
        else:
            self._plan.backward_update(ids, rows, opt="sgd", lr=optimizer.lr_t, l2_scale=2.0 * self.l2, autotune=True)

    def compute_mask(self, inputs, mask=None):
        if not self.mask_zero:  # tools.py:94-95
            return None
        return self._last_mask  # tile(expand_dims(inputs != 0), output_dim), produced by the same kernel

    def symbolic_has_mask(self, inputs, in_masks):
        return self.mask_zero

    def compute_output_shape(self, input_shape):
        return tuple(input_shape) + (self.output_dim,)


class SqueezeMask(Layer):
    """tools.py:104-113: pass the values through, keep one mask column."""

    def call(self, inputs, *args, **kwargs):
        if isinstance(inputs, KTensor):
            return inputs
        out = inputs + 0
        if hasattr(inputs, "_hrb_src"):
            out._hrb_src = inputs._hrb_src
        return out

    def compute_mask(self, inputs, mask=None):
        if mask is None:
            return None
        return mask[:, :, 0]

    def symbolic_has_mask(self, inputs, in_masks):
        return in_masks is not None


class AttentionPooling(Layer):
    """`tf.matmul(att_score (B,1,T), embd_seq (B,T,D))` of models/ranking/sequential/DIN.py:93 as a layer."""

    def call(self, inputs):
        att, keys = inputs
        return AttPoolFn.apply(att.reshape(att.shape[0], -1), keys)

    def compute_output_shape(self, input_shape):
        return (input_shape[1][0], 1, input_shape[1][2])


class ValueRows(Layer):
    """Rows of a constant per-item value list picked by an id tensor: the lazy counterpart of `ValueTable` (which always hands
    the WHOLE list on).  `EmbdFeatureGroup.get_embd_rows` uses it to evaluate the item side for the ids a step needs only."""

    def __init__(self, value_list: List, dtype: str = "int32", **kwargs):
        self._np = np.asarray(value_list)
        self._dtype = dtype
        self.value = None
        super().__init__(**kwargs)

    def call(self, inputs, **kwargs):
        if self.value is None:
            from ..keras_lite import _tdtype

            self.value = torch.as_tensor(self._np).to(device(), _tdtype(self._dtype))
        return self.value[inputs.reshape(-1).long()]  # integer plumbing: which feature values belong to the requested items

    def compute_output_shape(self, input_shape):
        return (input_shape[0],) + tuple(self._np.shape[1:])

    def output_dtype(self, inputs):
        return self._dtype


class LogUniformSampler:
    """tf.random.log_uniform_candidate_sampler(unique=True) restated on the host (numpy stream, so draws differ from TF's; the
    distribution is the same): P(k) = log((k+2)/(k+1)) / log(range_max+1), classes drawn until `num_sampled` are distinct."""

    def __init__(self, range_max: int, seed: int = 0):
        self.range_max, self.rng = int(range_max), np.random.RandomState(seed)
        self.log_range = float(np.log(self.range_max + 1.0))

    def sample(self, num_sampled: int):
        want = min(int(num_sampled), self.range_max)
        seen, out, tries = set(), [], 0
        while len(out) < want:
            draws = np.exp(self.rng.random_sample(max(2 * (want - len(out)), 8)) * self.log_range).astype(np.int64) - 1
            for k in draws % self.range_max:
                tries += 1
                k = int(k)
                if k not in seen:
                    seen.add(k)
                    out.append(k)
                    if len(out) == want:
                        break
        return np.asarray(out, dtype=np.int32), tries


class SampledSoftmaxLayer(Layer):
    """Sampled softmax (tools.py:32-84): `tf.nn.sampled_softmax_loss(weights=item embeddings, biases=0, labels=item ids,
    inputs=user embeddings, num_sampled, num_classes)` -> (B, 1) per-sample losses.

    Inputs `[item_embeddings (n, D), user_embeddings (B, D), item_idx (B, 1)]` like the reference.  With `item_rows` (a callable
    ids -> (m, D), see `EmbdFeatureGroup.row_tower`) the inputs are `[user_embeddings, item_idx]` and the item side is evaluated
    for the `B + num_sampled` rows the loss reads instead of the whole catalogue -- the same values and gradients whenever the item
    side has no batch-wide statistics (SURVEY 8f1).
    `sampled_values = (sampled ids (S,), true expected counts (B,), sampled expected counts (S,))` pins the candidates (parity tests).
    """

    def __init__(self, num_sampled=5, item_rows=None, num_classes=None, seed=0, **kwargs):
        self.num_sampled = num_sampled
        self.size = num_classes
        self.zero_bias = None
        self.item_rows = item_rows
        self.sampled_values = None
        self.seed = seed
        self._sampler = None
        super().__init__(**kwargs)
        for sub in getattr(item_rows, "layers", []) or []:
            self._track(sub)

    def build(self, input_shape):
        if self.item_rows is None:
            self.size = input_shape[0][0]
        self.zero_bias = self.add_weight("bias", (int(self.size),), initializer="zeros", trainable=False)
        self.built = True

    def call(self, inputs, **kwargs):
        if self.item_rows is None:
            item_embeddings, user_embeddings, item_idx = inputs
        else:
            (user_embeddings, item_idx), item_embeddings = inputs, None
        dev = user_embeddings.device
        labels = item_idx.reshape(-1).to(torch.int32).contiguous()
        B = labels.numel()
        if self.sampled_values is not None:
            sampled_np, te, se = self.sampled_values
            sampled = torch.as_tensor(np.asarray(sampled_np, dtype=np.int32)).to(dev)
            te = torch.as_tensor(np.asarray(te, dtype=np.float32)).reshape(-1).to(dev)
            se = torch.as_tensor(np.asarray(se, dtype=np.float32)).reshape(-1).to(dev)
            tries = 0.0
        else:
            if self._sampler is None:
                self._sampler = LogUniformSampler(int(self.size), self.seed)
            sampled_np, tries = self._sampler.sample(self.num_sampled)
            sampled = torch.from_numpy(sampled_np).to(dev)
            te = se = None  # the kernel evaluates log Q from (id, tries) itself
        S = sampled.numel()
        if self.item_rows is None:
            true_w, _ = EmbeddingFn.apply(item_embeddings, labels, False)
            sampled_w, _ = EmbeddingFn.apply(item_embeddings, sampled, False)
        else:
            rows = self.item_rows(torch.cat([labels, sampled]).reshape(-1, 1), training=kwargs.get("training", False))
            true_w, sampled_w = rows[:B], rows[B:]
        true_logit = RowDotFn.apply(user_embeddings, true_w)                 # biases are zero (tools.py:45-51)
        sampled_logit = MatmulNTFn.apply(user_embeddings, sampled_w)
        loss = SampledSoftmaxFn.apply(true_logit, sampled_logit, labels, sampled, te, se, float(tries), int(self.size), True)
        return loss.reshape(B, 1)

    def compute_output_shape(self, input_shape):
        return (None, 1)

    def get_config(self):
        return {"num_sampled": self.num_sampled, **super().get_config()}
