"""Op-for-op CPU restatement of the reference layers (torch-CPU, fp32).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  PARITY UNPINNED (no
TensorFlow in this image): every function cites the reference file:line whose
op sequence it follows, and keeps the SAME materialised intermediates as the
reference graph (gathered ``(B,L,D)`` tensor, tiled bool mask, float cast,
``divide_no_nan``, multiply, reduce ...) so that (a) rounding order matches TF's
CPU kernels as closely as a restatement can and (b) timing it is a fair stand-in
for "the reference's CPU path" (BASELINE.md §4).

All functions take/return ``torch.Tensor`` on CPU; everything is differentiable
through torch autograd, which plays the role of TF's ``GradientTape``.

TF semantics assumed (TF 2.6 behaviour; unverifiable here):
  * Keras ``Embedding`` = ``tf.nn.embedding_lookup`` (row gather, no zeroing of
    row 0); out-of-range id raises on CPU.
  * ``Dense`` = ``x @ W + b`` on the last axis.
  * ``l2(lam)`` regulariser = ``lam * sum(w**2)`` (no 1/2).
  * ``BatchNormalization`` defaults momentum=0.99, eps=1e-3; training mode uses
    the biased batch variance over every axis but the last.
  * ``tf.math.divide_no_nan(x, 0) == 0``.
  * ``binary_crossentropy`` on a Keras ``sigmoid`` activation output uses the
    cached logits (``_keras_logits``) -> ``sigmoid_cross_entropy_with_logits``.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

__all__ = [
    "as_t",
    "custom_embedding",
    "sequence_pooling",
    "fm",
    "dense",
    "batch_norm",
    "dice",
    "activation",
    "DNNParams",
    "dnn_init",
    "dnn",
    "squeeze_mask",
    "local_activation_unit",
    "din_attention_pool",
    "concat",
    "group_embedding_lookup",
    "deepfm_forward",
    "bce_from_logits",
    "l2_normalize",
    "hash_uniform_table",
    "hash_uniform_rows",
    "hash_u32",
    "embedding_grad_dense",
    "sharded_lookup_emulated",
    "sampledsoftmaxloss",
    "log_uniform_prob",
    "log_uniform_sample",
    "unique_expected_count",
    "sampled_softmax_loss",
]


def as_t(x, dtype=None) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        t = x
    else:
        t = torch.from_numpy(np.ascontiguousarray(x))
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t


# ----------------------------------------------------------------------------
# a5  CustomEmbedding  (handyrec/layers/tools.py:87-101)
# ----------------------------------------------------------------------------
def custom_embedding(
    table: torch.Tensor, ids: torch.Tensor, mask_zero: bool
) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """``out[..., :] = table[ids[...], :]``; ``mask = tile(ids != 0, D)``.

    Keras ``Embedding.call`` (-> ``tf.nn.embedding_lookup``) then the reference's
    ``compute_mask`` override, tools.py:93-101: not_equal -> expand_dims -> tile
    to the SAME shape as the output.  Row 0 is gathered like any other row.
    """
    ids = as_t(ids).long()
    V = table.shape[0]
    if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= V):
        # TF-CPU GatherV2 raises InvalidArgumentError for out-of-range indices.
        raise IndexError(f"id out of range [0, {V})")
    out = torch.nn.functional.embedding(ids, table)  # gather rows
    if not mask_zero:  # tools.py:94-95
        return out, None
    mask = ids != 0  # tools.py:97
    mask = mask.unsqueeze(-1)  # tools.py:98
    mask = mask.repeat(*([1] * (mask.dim() - 1)), table.shape[1])  # tools.py:99-100
    return out, mask


# ----------------------------------------------------------------------------
# a6  SequencePoolingLayer  (handyrec/layers/sequence.py:26-46)
# ----------------------------------------------------------------------------
def sequence_pooling(x: torch.Tensor, mask: Optional[torch.Tensor], method: str) -> torch.Tensor:
    """Masked mean / sum / max over axis 1, keepdims -> ``(B,1,D)``."""
    assert method in ["mean", "max", "sum"], "Pooling method should be `mean`, `max`, or `sum`"  # sequence.py:19-23
    if mask is None:  # sequence.py:27-28
        raise ValueError("Embedding layer should set `mask_zero` as True")
    mask = mask.to(torch.float32)  # sequence.py:32
    if method == "max":  # sequence.py:34-36
        output = x - (1 - mask) * 1e9
        # amax splits the gradient equally among ties, like TF's reduce_max gradient
        return output.amax(dim=1, keepdim=True)
    elif method == "sum":  # sequence.py:38-40
        output = x * mask
        return output.sum(dim=1, keepdim=True)
    else:  # mean, sequence.py:42-46
        mask_sum = mask.sum(dim=1, keepdim=True)
        # tf.math.divide_no_nan: 0 where the denominator is 0
        mask_weight = torch.where(mask_sum != 0, mask / torch.where(mask_sum != 0, mask_sum, torch.ones_like(mask_sum)), torch.zeros_like(mask))
        output = x * mask_weight
        return output.sum(dim=1, keepdim=True)


# ----------------------------------------------------------------------------
# a9  FM  (handyrec/layers/interaction.py:15-39)
# ----------------------------------------------------------------------------
def fm(x: torch.Tensor, w: torch.Tensor, w0: torch.Tensor) -> torch.Tensor:
    """``x`` (B,F,D), ``w`` (D,1) [Dense(1, use_bias=False)], ``w0`` (1,) -> (B,1)."""
    part2 = (x @ w).sum(dim=1, keepdim=False)  # interaction.py:29  (B,1)
    square_sum = x.sum(dim=1).square()  # interaction.py:33
    sum_square = (x * x).sum(dim=1)  # interaction.py:34
    part3 = square_sum - sum_square  # interaction.py:37
    part3 = 0.5 * part3.sum(dim=1, keepdim=True)  # interaction.py:38
    return part2 + part3 + w0  # interaction.py:39 (bias_add)


# ----------------------------------------------------------------------------
# a11  DNN / Dice / activations  (layers/core.py:53-78, activation.py:27-42,
#      layers/utils.py:117-133)
# ----------------------------------------------------------------------------
def dense(x: torch.Tensor, W: torch.Tensor, b: Optional[torch.Tensor]) -> torch.Tensor:
    y = x @ W
    if b is not None:
        y = y + b
    return y


def batch_norm(
    x: torch.Tensor,
    moving_mean: torch.Tensor,
    moving_var: torch.Tensor,
    gamma: Optional[torch.Tensor],
    beta: Optional[torch.Tensor],
    eps: float,
    training: bool,
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Keras BatchNormalization on the last axis.  Returns (y, batch_mean, batch_var).

    Training: statistics over every axis but the last, biased variance.
    Inference: the moving statistics.  (The moving-average state update,
    ``m = m*0.99 + batch*0.01``, is the caller's business.)
    """
    if training:
        red = tuple(range(x.dim() - 1))
        mean = x.mean(dim=red)
        var = ((x - mean) ** 2).mean(dim=red)
    else:
        mean, var = moving_mean, moving_var
    y = (x - mean) * torch.rsqrt(var + eps)
    if gamma is not None:
        y = y * gamma
    if beta is not None:
        y = y + beta
    return y, mean, var


def dice(
    x: torch.Tensor,
    alpha: torch.Tensor,
    moving_mean: torch.Tensor,
    moving_var: torch.Tensor,
    training: bool = False,
    eps: float = 1e-9,
) -> torch.Tensor:
    """activation.py:27-42: BN(center=False, scale=False, eps=1e-9) -> sigmoid gate."""
    normed, _, _ = batch_norm(x, moving_mean, moving_var, None, None, eps, training)  # activation.py:40
    x_p = torch.sigmoid(normed)  # activation.py:41
    return x_p * x + (1.0 - x_p) * alpha * x  # activation.py:42


def activation(name: Optional[str], x: torch.Tensor) -> torch.Tensor:
    """Keras ``Activation(name)`` for the names the reference's configs use."""
    if name is None or name == "linear":
        return x
    if name == "relu":
        return torch.relu(x)
    if name == "sigmoid":
        return torch.sigmoid(x)
    if name == "tanh":
        return torch.tanh(x)
    raise ValueError(f"unsupported activation {name!r}")


class DNNParams:
    """Weights of one reference ``DNN`` layer: ``hidden = [in] + hidden_units`` (core.py:57)."""

    def __init__(self, in_dim: int, hidden_units: Sequence[int]):
        self.units = [int(in_dim)] + [int(u) for u in hidden_units]
        self.W: List[torch.Tensor] = []
        self.b: List[torch.Tensor] = []
        # per layer optional state
        self.dice_alpha: List[Optional[torch.Tensor]] = []
        self.dice_mean: List[Optional[torch.Tensor]] = []
        self.dice_var: List[Optional[torch.Tensor]] = []
        self.bn_gamma: List[Optional[torch.Tensor]] = []
        self.bn_beta: List[Optional[torch.Tensor]] = []
        self.bn_mean: List[Optional[torch.Tensor]] = []
        self.bn_var: List[Optional[torch.Tensor]] = []

    def tensors(self) -> List[torch.Tensor]:
        out = []
        for lst in (self.W, self.b, self.dice_alpha, self.bn_gamma, self.bn_beta):
            out += [t for t in lst if t is not None]
        return out


def dnn_init(in_dim: int, hidden_units: Sequence[int], seed: int = 0, dtype=torch.float32) -> DNNParams:
    """Glorot-uniform kernels / zero biases like Keras ``Dense`` (random stream is torch's, not TF's)."""
    g = torch.Generator().manual_seed(seed)
    p = DNNParams(in_dim, hidden_units)
    fan_in = in_dim
    for u in p.units:
        lim = float(np.sqrt(6.0 / (fan_in + u)))
        p.W.append(((torch.rand(fan_in, u, generator=g, dtype=torch.float64) * 2 - 1) * lim).to(dtype))
        p.b.append(torch.zeros(u, dtype=dtype))
        p.dice_alpha.append(torch.zeros(u, dtype=dtype))
        p.dice_mean.append(torch.zeros(u, dtype=dtype))
        p.dice_var.append(torch.ones(u, dtype=dtype))
        p.bn_gamma.append(torch.ones(u, dtype=dtype))
        p.bn_beta.append(torch.zeros(u, dtype=dtype))
        p.bn_mean.append(torch.zeros(u, dtype=dtype))
        p.bn_var.append(torch.ones(u, dtype=dtype))
        fan_in = u
    return p


def dnn(
    x: torch.Tensor,
    p: DNNParams,
    act: Optional[str] = "relu",
    use_bn: bool = False,
    output_activation: Optional[str] = None,
    training: bool = False,
    bn_eps: float = 1e-3,
) -> torch.Tensor:
    """core.py:53-78.  Layer i: Dense -> (hidden act | output act) -> [BN] -> Dropout(rate).

    Quirks kept: an extra ``Dense(in)`` heads every DNN (core.py:57); the ``elif``
    at core.py:68 fires for hidden layers too when ``activation`` is falsy; BN
    sits AFTER the activation (core.py:71-72).  Dropout is identity here (parity
    runs use rate 0 / inference).
    """
    n = len(p.units)
    for i in range(n):
        x = dense(x, p.W[i], p.b[i])  # core.py:61-65
        name = None
        if i + 1 != n and act:  # core.py:66-67
            name = act
        elif output_activation:  # core.py:68-69
            name = output_activation
        if name == "dice":  # layers/utils.py:130-131
            x = dice(x, p.dice_alpha[i], p.dice_mean[i], p.dice_var[i], training)
        elif name is not None:
            x = activation(name, x)
        if use_bn:  # core.py:71-72
            x, _, _ = batch_norm(x, p.bn_mean[i], p.bn_var[i], p.bn_gamma[i], p.bn_beta[i], bn_eps, training)
    return x


# ----------------------------------------------------------------------------
# a10  DIN attention  (layers/sequence.py:92-102, tools.py:104-113, DIN.py:87-93)
# ----------------------------------------------------------------------------
def squeeze_mask(x: torch.Tensor, mask: Optional[torch.Tensor]):
    """tools.py:104-113: ``inputs + 0`` and ``mask[:, :, 0]``."""
    return x + 0, (None if mask is None else mask[:, :, 0])


def local_activation_unit(
    query: torch.Tensor,
    keys: torch.Tensor,
    key_mask: torch.Tensor,
    p: DNNParams,
    act: Optional[str] = "sigmoid",
    use_bn: bool = False,
    training: bool = False,
) -> torch.Tensor:
    """``query`` (B,1,D), ``keys`` (B,T,D), ``key_mask`` (B,T) bool -> scores (B,1,T).  No softmax."""
    mask = key_mask.unsqueeze(1)  # sequence.py:94
    queries = query.repeat_interleave(keys.shape[1], dim=1)  # sequence.py:96 (tf.repeat on axis 1)
    att_input = torch.cat([queries, keys, queries - keys, queries * keys], dim=-1)  # sequence.py:97
    att_out = dnn(att_input, p, act=act, use_bn=use_bn, output_activation=None, training=training)  # sequence.py:99
    att_out = att_out.transpose(1, 2)  # sequence.py:100
    att_out = att_out * mask.to(torch.float32)  # sequence.py:101
    return att_out


def din_attention_pool(att_score: torch.Tensor, keys: torch.Tensor) -> torch.Tensor:
    """DIN.py:93: ``tf.matmul(att_score (B,1,T), embd_seq (B,T,D))`` -> (B,1,D)."""
    return att_score @ keys


# ----------------------------------------------------------------------------
# a8  concat glue  (layers/utils.py:9-96)
# ----------------------------------------------------------------------------
def _concat(inputs: List[torch.Tensor], axis: int = -1) -> torch.Tensor:
    if len(inputs) == 1:  # utils.py:24-25
        return inputs[0]
    has_int = any(not t.dtype.is_floating_point for t in inputs)
    has_other = any(t.dtype.is_floating_point for t in inputs)
    if has_int and has_other:  # utils.py:28-36
        inputs = [t.to(torch.float32) for t in inputs]
    return torch.cat(inputs, dim=axis)


def concat(dense_inputs: List[torch.Tensor], embd_inputs: List[torch.Tensor], axis: int = -1, keepdims: bool = False) -> torch.Tensor:
    if len(dense_inputs) + len(embd_inputs) == 0:  # utils.py:67-68
        raise ValueError("Number of inputs should be larger than 0")
    if len(dense_inputs) > 0 and len(embd_inputs) > 0:  # utils.py:70-84
        d = _concat(dense_inputs, axis)
        s = _concat(embd_inputs, axis)
        if not keepdims:
            d = d.flatten(1)
            s = s.flatten(1)
        return _concat([d, s], axis)
    lst = dense_inputs if len(dense_inputs) > 0 else embd_inputs  # utils.py:86-96
    out = _concat(lst, axis)
    if not keepdims:
        out = out.flatten(1)
    return out


# ----------------------------------------------------------------------------
# a7  FeatureGroup.embedding_lookup  (features/group.py:299-336)
# ----------------------------------------------------------------------------
def group_embedding_lookup(
    sparse: "OrderedDict[str, Tuple[torch.Tensor, torch.Tensor, bool]]",
    sparse_seq: "OrderedDict[str, Tuple[torch.Tensor, torch.Tensor]]",
    pool_method: str = "mean",
) -> List[torch.Tensor]:
    """sparse[name] = (table, ids (B,1), mask_zero); sparse_seq[name] = (unit table, ids (B,L)).

    Returns the ``embd_output`` list: sparse features first, then sequence
    features, each ``(B,1,D)`` (group.py:319-334).
    """
    outs = OrderedDict()
    for name, (table, ids, mask_zero) in sparse.items():
        outs[name], _ = custom_embedding(table, ids, mask_zero)  # group.py:320-321
    for name, (table, ids) in sparse_seq.items():
        seq, mask = custom_embedding(table, ids, True)  # group.py:331 (unit tables are mask_zero, :273,292)
        outs[name] = sequence_pooling(seq, mask, pool_method)  # group.py:332
    return list(outs.values())


# ----------------------------------------------------------------------------
# DeepFM head  (models/ranking/context_aware/DeepFM.py:62-88)
# ----------------------------------------------------------------------------
def deepfm_forward(
    dense_inputs: List[torch.Tensor],
    fm_embds: List[torch.Tensor],
    dnn_embds: List[torch.Tensor],
    dnn_p: DNNParams,
    fm_w: torch.Tensor,
    fm_w0: torch.Tensor,
    dnn_activation: str = "relu",
    dnn_bn: bool = False,
    training: bool = False,
    task: str = "binary",
    return_logit: bool = False,
):
    dnn_input = concat(dense_inputs, dnn_embds)  # DeepFM.py:70
    fm_input = concat([], fm_embds, axis=1, keepdims=True)  # DeepFM.py:71
    dnn_out = dnn(dnn_input, dnn_p, act=dnn_activation, use_bn=dnn_bn, output_activation="linear", training=training)  # :73-82
    fm_out = fm(fm_input, fm_w, fm_w0)  # :83
    logit = dnn_out + fm_out  # :86
    if return_logit:
        return logit
    if task == "binary":
        return torch.sigmoid(logit)  # :87-88
    return logit


def bce_from_logits(logit: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """mean over the batch of sigmoid cross-entropy with logits (Keras binary_crossentropy on a sigmoid output)."""
    return torch.nn.functional.binary_cross_entropy_with_logits(logit, y.to(logit.dtype), reduction="mean")


def l2_normalize(x: torch.Tensor, axis=None, eps: float = 1e-12) -> torch.Tensor:
    """tf.nn.l2_normalize: x * rsqrt(max(sum(x^2, axis), eps)).  DSSM.py:105-106 uses axis=None."""
    sq = (x * x).sum() if axis is None else (x * x).sum(dim=axis, keepdim=True)
    return x * torch.rsqrt(torch.clamp(sq, min=eps))


def sampledsoftmaxloss(y_true, y_pred):
    """layers/utils.py:99-114: ``tf.reduce_mean(y_pred)``."""
    return as_t(np.asarray(y_pred, dtype=np.float32)).mean()


# ----------------------------------------------------------------------------
# (f1) tf.nn.sampled_softmax_loss as SampledSoftmaxLayer uses it (layers/tools.py:56-75)
# ----------------------------------------------------------------------------
def log_uniform_prob(ids, range_max: int):
    """P(k) of TF's log-uniform (Zipfian) candidate sampler: log((k+2)/(k+1)) / log(range_max+1)."""
    k = np.asarray(ids, dtype=np.float64)
    return np.log((k + 2.0) / (k + 1.0)) / np.log(range_max + 1.0)


def log_uniform_sample(num_sampled: int, range_max: int, rng: np.random.RandomState):
    """``tf.random.log_uniform_candidate_sampler(unique=True)`` restated: draw ``floor(exp(u*log(range_max+1))) - 1 mod range_max``
    until ``num_sampled`` distinct classes are in hand.  Returns (sampled ids in draw order, number of tries).
    The random stream is numpy's, not TF's: only the DISTRIBUTION matches (statistical parity); numeric parity tests inject the
    sampled values on both sides."""
    seen, out, tries = set(), [], 0
    log_range = np.log(range_max + 1.0)
    while len(out) < num_sampled:
        tries += 1
        k = int(np.exp(rng.random_sample() * log_range)) - 1
        k %= range_max
        if k not in seen:
            seen.add(k)
            out.append(k)
    return np.asarray(out, dtype=np.int32), tries


def unique_expected_count(p, num_tries: int):
    """Expected count of a class under the unique sampler: 1 - (1-p)^num_tries = -expm1(num_tries * log1p(-p))."""
    return -np.expm1(num_tries * np.log1p(-np.asarray(p, dtype=np.float64)))


def sampled_softmax_loss(weights: torch.Tensor, biases: torch.Tensor, labels: torch.Tensor, inputs: torch.Tensor, sampled: torch.Tensor,
                         true_expected: torch.Tensor, sampled_expected: torch.Tensor, remove_accidental_hits: bool = True) -> torch.Tensor:
    """nn_impl._compute_sampled_logits + softmax cross-entropy (TF 2.x defaults: num_true = 1, subtract_log_q = True).

    weights (C, D), biases (C,), labels (B,) or (B,1) int, inputs (B, D), sampled (S,) int; expected counts as the candidate
    sampler returns them.  -> loss (B,).  Op order follows TF: gather both weight sets, true logits as a row-wise product sum,
    sampled logits as a matmul with the transposed sampled weights, accidental hits get -FLOAT_MAX added, log Q subtracted,
    labels one-hot on column 0, softmax_cross_entropy_with_logits."""
    labels = as_t(labels).long().reshape(-1)
    sampled = as_t(sampled).long().reshape(-1)
    true_w = weights[labels]                       # embedding_lookup(weights, labels)
    sampled_w = weights[sampled]
    true_logits = (inputs * true_w).sum(1) + biases[labels]
    sampled_logits = inputs @ sampled_w.t() + biases[sampled]
    if remove_accidental_hits:
        hit = labels[:, None] == sampled[None, :]
        sampled_logits = sampled_logits + hit.to(sampled_logits.dtype) * (-torch.finfo(torch.float32).max)
    true_logits = true_logits - torch.log(as_t(true_expected, torch.float32).reshape(-1))
    sampled_logits = sampled_logits - torch.log(as_t(sampled_expected, torch.float32).reshape(1, -1))
    logits = torch.cat([true_logits[:, None], sampled_logits], 1)
    return torch.logsumexp(logits, 1) - logits[:, 0]


# ----------------------------------------------------------------------------
# a13  Embedding backward as the formula TF autodiff yields
# ----------------------------------------------------------------------------
def embedding_grad_dense(V: int, ids: torch.Tensor, dout: torch.Tensor, table: Optional[torch.Tensor] = None, l2: float = 0.0) -> torch.Tensor:
    """``dW[r] = sum_{(b,l): ids=r} dOut[b,l] (+ 2*l2*W)`` accumulated in float64 then rounded (order-free oracle)."""
    D = dout.shape[-1]
    dW = torch.zeros(V, D, dtype=torch.float64)
    dW.index_add_(0, as_t(ids).long().reshape(-1), dout.reshape(-1, D).to(torch.float64))
    if l2 and table is not None:
        dW += 2.0 * l2 * table.to(torch.float64)
    return dW.to(torch.float32)


# ----------------------------------------------------------------------------
# deterministic synthetic tables shared by oracle and CUDA (bit-identical)
# ----------------------------------------------------------------------------
def hash_u32(x: np.ndarray) -> np.ndarray:
    """32-bit finaliser (lowbias32); mirrored by ``hrb_hash_u32`` in csrc/common.cuh."""
    x = x.astype(np.uint32)
    x ^= x >> np.uint32(16)
    x = (x * np.uint32(0x7FEB352D)).astype(np.uint32)
    x ^= x >> np.uint32(15)
    x = (x * np.uint32(0x846CA68B)).astype(np.uint32)
    x ^= x >> np.uint32(16)
    return x


def hash_uniform_table(V: int, D: int, seed: int, lo: float = -0.05, hi: float = 0.05, row_start: int = 0, row_step: int = 1) -> np.ndarray:
    """U[lo,hi) table, element (r,c) = lo + u*(hi-lo), u = (hash(seed, r*D+c) >> 8) * 2^-24.

    Bit-identical to ``hrb_init_uniform`` (mul and add are separately rounded on
    both sides).  ``row_start/row_step`` give the rows of a ``row % N`` shard.
    """
    return hash_uniform_rows(np.arange(V, dtype=np.uint64) * np.uint64(row_step) + np.uint64(row_start), D, seed, lo, hi)


def hash_uniform_rows(rows, D: int, seed: int, lo: float = -0.05, hi: float = 0.05) -> np.ndarray:
    """Rows ``rows`` (any order, repeats allowed) of ``hash_uniform_table(V, D, seed, lo, hi)`` without forming the table: the
    initial values of the rows a step touches in a table too large to copy to the host."""
    rows = np.asarray(rows).astype(np.uint64).reshape(-1)
    idx = rows[:, None] * np.uint64(D) + np.arange(D, dtype=np.uint64)[None, :]
    lo32 = (idx & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi32 = (idx >> np.uint64(32)).astype(np.uint32)
    with np.errstate(over="ignore"):
        h = hash_u32(lo32 ^ hash_u32(hi32 + np.uint32(seed & 0xFFFFFFFF) * np.uint32(0x9E3779B9) + np.uint32(0x85EBCA6B)))
    u = (h >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)
    scale = np.float32(hi) - np.float32(lo)
    return (u * scale).astype(np.float32) + np.float32(lo)


# ----------------------------------------------------------------------------
# (e) multi-rank emulation of the row-sharded lookup
# ----------------------------------------------------------------------------
def sharded_lookup_emulated(table: torch.Tensor, ids: torch.Tensor, n_ranks: int, method: str) -> torch.Tensor:
    """Row-sharded (``owner = r % N``, local row ``r // N``) gather + partial pooling + combine.

    Emulates SURVEY §8e on one process: every owner gathers its rows and
    partially pools them per sample (sum + valid count, or partial max); the
    requester sums <=N partials and finalises.  ``ids`` (B,L) -> (B,1,D).
    Must equal ``sequence_pooling(custom_embedding(...))`` to <=1e-5.
    """
    ids = as_t(ids).long()
    B, L = ids.shape
    D = table.shape[1]
    shards = [table[r::n_ranks] for r in range(n_ranks)]
    psum = torch.zeros(n_ranks, B, D)
    pcnt = torch.zeros(n_ranks, B)
    pmax = torch.full((n_ranks, B, D), -1e9)
    for r in range(n_ranks):
        mine = (ids % n_ranks == r) & (ids != 0)
        local = torch.where(mine, ids // n_ranks, torch.zeros_like(ids))
        rows = shards[r][local]  # (B,L,D)
        m = mine.unsqueeze(-1).to(torch.float32)
        psum[r] = (rows * m).sum(1)
        pcnt[r] = mine.sum(1).to(torch.float32)
        pmax[r] = torch.where(mine.unsqueeze(-1), rows, torch.full_like(rows, -1e9)).max(1).values
    tot = psum.sum(0)
    cnt = pcnt.sum(0)
    if method == "sum":
        out = tot
    elif method == "mean":
        out = torch.where(cnt.unsqueeze(-1) != 0, tot / torch.clamp(cnt, min=1).unsqueeze(-1), torch.zeros_like(tot))
    else:
        out = pmax.max(0).values
    return out.unsqueeze(1)


# ---------------------------------------------------------------------------------------------
# Scheduling invariant of the sorted embedding backward (handyrec_b200/csrc/lookup.cu, "long runs"): not reference arithmetic,
# but a restatement of the classification every kernel of that path must agree on, so that the tests can check the claim the
# kernels rely on -- the LOCAL test (four sample points around a position) equals the GLOBAL definition.
# ---------------------------------------------------------------------------------------------
def long_run_keys_global(sorted_keys: np.ndarray, step: int, sentinel: int) -> set:
    """Rows whose run of equal keys covers two consecutive sample points (positions 0, step, 2*step, ... < n): what
    bwd_long_detect_kernel lists."""
    k = np.asarray(sorted_keys)
    pts = np.arange(0, len(k), step)
    return {int(k[pts[j]]) for j in range(len(pts) - 1) if k[pts[j]] == k[pts[j + 1]] and k[pts[j]] != sentinel}


def long_run_local_test(sorted_keys: np.ndarray, step: int, sentinel: int, i: int) -> bool:
    """run_is_long() of lookup.cu for the key at sorted position i: only the sample points around i are read."""
    k = np.asarray(sorted_keys)
    n, key = len(k), k[i]
    if key == sentinel:
        return False
    p0 = i // step * step
    s0 = k[p0]
    s1 = k[p0 + step] if p0 + step < n else sentinel
    if s0 == key and s1 == key:
        return True
    if s0 == key:
        return p0 >= step and k[p0 - step] == key
    if s1 == key:
        return p0 + 2 * step < n and k[p0 + 2 * step] == key
    return False
