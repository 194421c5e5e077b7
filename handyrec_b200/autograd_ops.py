"""torch.autograd.Function wrappers of the C-ABI kernels (layer face).

torch's autograd engine only ORDERS the backward calls; every forward and backward computation is a kernel of
libhrb200.so.  These functions are what the Keras-like layers in handyrec_b200.layers call.
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch

from . import _lib
from . import kernels as K
from ._lib import ACT, POOL, call


_grad_clip = None  # handyrec_b200.clip.GradClip while Model._train_on_batch_layers runs a clipped backward


class EmbeddingFn(torch.autograd.Function):
    """layers/tools.py:87-101 forward; TF IndexedSlices gradient as a dense, sorted-segment reduction."""

    @staticmethod
    def forward(ctx, table, ids, mask_zero, sparse_sink=None):
        out, mask = K.embedding_fwd(table, ids.contiguous(), mask_zero)
        ctx.save_for_backward(ids)
        ctx.vocab = table.shape[0]
        ctx.sink = sparse_sink
        ctx.table_id = id(table)
        ctx.mark_non_differentiable(*( [mask] if mask is not None else []))
        return (out, mask) if mask is not None else (out, torch.empty(0, device=table.device, dtype=torch.bool))

    @staticmethod
    def backward(ctx, dout, _dmask):
        (ids,) = ctx.saved_tensors
        D = dout.shape[-1]
        if ctx.sink is not None:
            # a large table: keep the gradient as (ids, rows) -- TF's IndexedSlices -- for the sorted-segment row update
            # (CustomEmbedding.apply_sparse) instead of materialising vocab x D floats per step
            ctx.sink.append((ids.reshape(-1), dout.contiguous().reshape(-1, D)))
            return None, None, None, None
        rows = dout.contiguous().reshape(-1, D)
        var = _grad_clip.table_vars.get(ctx.table_id) if _grad_clip is not None else None
        if var is not None:  # Keras clips this lookup's IndexedSlices values, one row per position, before duplicates are summed
            rows = rows.clone()
            _grad_clip.prepare([rows], None, None, [var])
        return K.embedding_bwd_dense(ids.reshape(-1), rows, ctx.vocab), None, None, None


class SeqPoolFn(torch.autograd.Function):
    """layers/sequence.py:26-46."""

    @staticmethod
    def forward(ctx, x, mask, method):
        x = x.contiguous()
        out = K.seq_pool_fwd(x, mask.contiguous(), method)
        ctx.save_for_backward(x, mask)
        ctx.method = method
        return out

    @staticmethod
    def backward(ctx, dout):
        x, mask = ctx.saved_tensors
        B, L, D = x.shape
        return K.seq_pool_bwd(x, mask.contiguous(), dout.contiguous().reshape(B, D), ctx.method), None, None


class FMFn(torch.autograd.Function):
    """layers/interaction.py:26-39."""

    @staticmethod
    def forward(ctx, x, w, w0):
        x = x.contiguous()
        ctx.save_for_backward(x, w)
        return K.fm_fwd(x, w.contiguous(), w0)

    @staticmethod
    def backward(ctx, dout):
        x, w = ctx.saved_tensors
        dx, dw, dw0 = K.fm_bwd(x, w.contiguous(), dout.contiguous().reshape(-1))
        return dx, dw.reshape(w.shape), dw0


TC_MIN_ROWS = 4096  # layer-face Dense: from this many rows on the GEMMs run on the tcgen05 3xTF32 kernel (DIN's LAU MLP: B*T rows)


def _tc_shape(M: int, Kd: int, N: int) -> bool:
    return M >= TC_MIN_ROWS and Kd >= 16 and N >= 16 and Kd % 4 == 0 and N % 4 == 0


class DenseFn(torch.autograd.Function):
    """Keras Dense on the last axis with a fused element-wise activation (layers/core.py:61-69).

    Tall inputs -- the local-activation MLP of DIN sees B*T = 204 800 rows (sequence.py:99), the towers B -- take the tensor-core
    kernel (error-compensated 3xTF32 with fp32 accumulation, same parity as the FFMA kernel): forward on W^T, backward dx in the
    TN form as stored, dW as a split-K product that reads x untransposed; only dz^T (N x M) is materialised for it.  Everything
    else stays on the FFMA kernel."""

    @staticmethod
    def forward(ctx, x, w, b, act):
        lead = x.shape[:-1]
        x2 = x.contiguous().reshape(-1, x.shape[-1])
        w = w.contiguous()
        M, Kd = x2.shape
        N = w.shape[1]
        ctx.tc = _tc_shape(M, Kd, N) and act in (None, "linear", "relu", "sigmoid", "tanh")
        if ctx.tc:
            y = K.dense_fwd_t(x2, K.transpose(w), b, act)
        else:
            y = K.dense_fwd(x2, w, b, act)
        ctx.save_for_backward(x2, w, y)
        ctx.act, ctx.lead, ctx.has_bias = act, lead, b is not None
        return y.reshape(*lead, N)

    @staticmethod
    def backward(ctx, dy):
        x2, w, y = ctx.saved_tensors
        dy2 = dy.contiguous().reshape(-1, w.shape[1])
        dz = K.act_bwd(y, dy2, ctx.act) if ctx.act not in (None, "linear") else dy2
        if ctx.tc:
            dx = K.dense_bwd_x_t(dz, w)
            dw, db = K.dense_bwd_w_xn(x2, K.transpose(dz), want_bias=ctx.has_bias)
        else:
            dx = K.dense_bwd_x(dz, w)
            dw, db = K.dense_bwd_w(x2, dz, want_bias=ctx.has_bias)
        return dx.reshape(*ctx.lead, w.shape[0]), dw, (db if ctx.has_bias else None), None


class DiceFn(torch.autograd.Function):
    """layers/activation.py:27-42; mean/var are the layer's moving statistics (overwritten by batch statistics when training)."""

    @staticmethod
    def forward(ctx, x, alpha, mean, var, training, eps):
        x = x.contiguous()
        bm, bv = (torch.empty_like(mean), torch.empty_like(var)) if training else (mean, var)
        y = K.dice_fwd(x, alpha, bm, bv, training, eps)
        ctx.save_for_backward(x, alpha, bm, bv)
        ctx.training, ctx.eps = training, eps
        ctx.batch_stats = (bm, bv)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, alpha, bm, bv = ctx.saved_tensors
        dx, dalpha = K.dice_bwd(x, dy.contiguous(), alpha, bm, bv, ctx.training, ctx.eps)
        return dx, dalpha, None, None, None, None


class BatchNormFn(torch.autograd.Function):
    """Keras BatchNormalization on the last axis (layers/core.py:71-72)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, mean, var, training, eps):
        x = x.contiguous()
        units = x.shape[-1]
        rows = x.numel() // units
        bm, bv = (torch.empty_like(mean), torch.empty_like(var)) if training else (mean, var)
        y = torch.empty_like(x)
        call("hrb_batchnorm_fwd", K._p(x), rows, units, K._p(gamma), K._p(beta), K._p(bm), K._p(bv), eps, int(training), K._p(y), K._stream())
        ctx.save_for_backward(x, gamma, bm, bv)
        ctx.training, ctx.eps = training, eps
        ctx.batch_stats = (bm, bv)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, bm, bv = ctx.saved_tensors
        units = x.shape[-1]
        rows = x.numel() // units
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        dg, db = torch.empty_like(gamma), torch.empty_like(gamma)
        scratch = torch.empty(2 * units, device=x.device, dtype=torch.float32)
        call("hrb_batchnorm_bwd", K._p(x), K._p(dy), rows, units, K._p(gamma), K._p(bm), K._p(bv), ctx.eps, int(ctx.training), K._p(dx), K._p(dg),
             K._p(db), K._p(scratch), K._stream())
        return dx, dg, db, None, None, None, None


class DropoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, rate, seed):
        x = x.contiguous()
        y = torch.empty_like(x)
        call("hrb_dropout", K._p(x), x.numel(), float(rate), seed & 0xFFFFFFFF, K._p(y), K._stream())
        ctx.rate, ctx.seed = rate, seed
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = dy.contiguous()
        dx = torch.empty_like(dy)
        call("hrb_dropout", K._p(dy), dy.numel(), float(ctx.rate), ctx.seed & 0xFFFFFFFF, K._p(dx), K._stream())
        return dx, None, None


class AttInputFn(torch.autograd.Function):
    """[q, k, q-k, q*k] (layers/sequence.py:96-97)."""

    @staticmethod
    def forward(ctx, q, k):
        q, k = q.contiguous(), k.contiguous()
        B, T, D = k.shape
        out = torch.empty(B, T, 4 * D, device=k.device, dtype=torch.float32)
        call("hrb_att_input_fwd", K._p(q), K._p(k), B, T, D, K._p(out), K._stream())
        ctx.save_for_backward(q, k)
        return out

    @staticmethod
    def backward(ctx, g):
        q, k = ctx.saved_tensors
        B, T, D = k.shape
        dq, dk = torch.empty_like(q), torch.empty_like(k)
        call("hrb_att_input_bwd", K._p(q), K._p(k), K._p(g.contiguous()), B, T, D, K._p(dq), K._p(dk), K._stream())
        return dq, dk


class MaskScoresFn(torch.autograd.Function):
    """att_out * cast(mask) (layers/sequence.py:101); scores (B,T), mask (B,T) bool."""

    @staticmethod
    def forward(ctx, s, mask):
        s = s.contiguous()
        m = mask.contiguous().view(torch.uint8)
        out = torch.empty_like(s)
        call("hrb_mask_scores", K._p(s), K._p(m), s.numel(), K._p(out), K._stream())
        ctx.save_for_backward(m)
        return out

    @staticmethod
    def backward(ctx, g):
        (m,) = ctx.saved_tensors
        g = g.contiguous()
        out = torch.empty_like(g)
        call("hrb_mask_scores", K._p(g), K._p(m), g.numel(), K._p(out), K._stream())
        return out, None


class AttPoolFn(torch.autograd.Function):
    """tf.matmul(att (B,1,T), keys (B,T,D)) (models/ranking/sequential/DIN.py:93)."""

    @staticmethod
    def forward(ctx, s, k):
        s, k = s.contiguous(), k.contiguous()
        B, T, D = k.shape
        out = torch.empty(B, 1, D, device=k.device, dtype=torch.float32)
        call("hrb_att_pool_fwd", K._p(s), K._p(k), B, T, D, K._p(out), K._stream())
        ctx.save_for_backward(s, k)
        return out

    @staticmethod
    def backward(ctx, g):
        s, k = ctx.saved_tensors
        B, T, D = k.shape
        ds, dk = torch.empty_like(s), torch.empty_like(k)
        call("hrb_att_pool_bwd", K._p(s), K._p(k), K._p(g.contiguous()), B, T, D, K._p(ds), K._p(dk), K._stream())
        return ds, dk


class SigmoidBCEFn(torch.autograd.Function):
    """mean sigmoid cross-entropy with logits (Keras binary_crossentropy on a sigmoid output uses the cached logits).  With
    `weight` (one float32 per sample, on the device): Keras' weighted loss, sum(w * l) / B."""

    @staticmethod
    def forward(ctx, logit, label, weight=None):
        logit = logit.contiguous().reshape(-1)
        label = label.contiguous().reshape(-1).to(torch.float32)
        B = logit.numel()
        dl = torch.empty_like(logit)
        ls = torch.zeros(1, device=logit.device, dtype=torch.float32)
        K.sigmoid_bce(logit, None, label, 1.0 / B, None, dl, ls, weight=weight)
        ctx.save_for_backward(dl)
        return (ls / B).reshape(())

    @staticmethod
    def backward(ctx, g):
        (dl,) = ctx.saved_tensors
        return (dl * g).reshape(-1, 1), None, None


class ClippedBCEFn(torch.autograd.Function):
    """mean binary cross-entropy on probabilities clipped to [1e-7, 1-1e-7] (Keras' path without cached logits).  With `weight`:
    sum(w * l) / n, as SigmoidBCEFn."""

    @staticmethod
    def forward(ctx, prob, label, weight=None):
        shape = prob.shape
        prob = prob.contiguous().reshape(-1)
        label = label.contiguous().reshape(-1).to(torch.float32)
        n = prob.numel()
        dp = torch.empty_like(prob)
        ls = torch.zeros(1, device=prob.device, dtype=torch.float32)
        if weight is None:
            call("hrb_clipped_bce", K._p(prob), K._p(label), n, 1e-7, 1.0 / n, K._p(dp), K._p(ls), K._stream())
        else:
            if K._chk(weight, torch.float32, "weight").numel() != n:
                raise ValueError(f"binary_crossentropy: {weight.numel()} sample weights for {n} predictions")
            call("hrb_clipped_bce_weighted", K._p(prob), K._p(label), K._p(weight), n, 1e-7, 1.0 / n, K._p(dp), K._p(ls), K._stream())
        ctx.save_for_backward(dp)
        ctx.shape = shape
        return (ls / n).reshape(())

    @staticmethod
    def backward(ctx, g):
        (dp,) = ctx.saved_tensors
        return (dp * g).reshape(ctx.shape), None, None


_loss_ws = {}  # (device index, raw stream) -> the layer path's hrb_regression_loss workspace


def _regression_workspace(n: int, device: torch.device) -> torch.Tensor:
    """The hrb_regression_loss workspace of the current stream, zeroed once when it is allocated (or grown for a larger batch); the
    kernel leaves it zeroed, so later calls need no memset."""
    need = ctypes.c_size_t(0)
    call("hrb_regression_loss_workspace", n, ctypes.byref(need))
    key = (device.index, K._stream().value)
    ws = _loss_ws.get(key)
    if ws is None or ws.numel() < need.value:
        ws = _loss_ws[key] = torch.zeros(need.value, device=device, dtype=torch.uint8)
    return ws


class RegressionLossFn(torch.autograd.Function):
    """Keras mean_squared_error / mean_absolute_error / huber (`loss`, kernels.REG_LOSS): the mean over the last axis per sample,
    then the batch mean; with `weight`, sum(w * l) / B as SigmoidBCEFn.  `label` has the shape of `pred` (the caller applies Keras'
    (B,) -> (B, 1) rule)."""

    @staticmethod
    def forward(ctx, pred, label, loss, delta, weight=None):
        shape = pred.shape
        B = shape[0] if pred.dim() else 1
        cols = pred.numel() // B if B else 1
        p = pred.contiguous().reshape(-1)
        y = label.contiguous().reshape(-1).to(torch.float32)
        dp = torch.empty_like(p)
        ls = torch.empty(1, device=p.device, dtype=torch.float32)
        K.regression_loss(loss, delta, p, None, y, B, cols, 1.0 / max(B, 1), None, dp, ls, weight=weight,
                          workspace=_regression_workspace(p.numel(), p.device))
        ctx.save_for_backward(dp)
        ctx.shape = shape
        return (ls / max(B, 1)).reshape(())

    @staticmethod
    def backward(ctx, g):
        (dp,) = ctx.saved_tensors
        return (dp * g).reshape(ctx.shape), None, None, None, None


class ActivationFn(torch.autograd.Function):
    """Stand-alone Keras Activation(name) for relu / sigmoid / tanh (element-wise)."""

    @staticmethod
    def forward(ctx, x, act):
        x2 = x.contiguous().reshape(-1, 1)
        # y = act(x * 1 + 0): the dense kernel with a 1x1 identity weight is the element-wise activation
        one = torch.ones(1, 1, device=x.device, dtype=torch.float32)
        y = K.dense_fwd(x2, one, None, act, mode=_lib.GEMM_FP32)
        ctx.save_for_backward(y)
        ctx.act = act
        return y.reshape(x.shape)

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        return K.act_bwd(y, dy.contiguous().reshape(-1, 1), ctx.act).reshape(dy.shape), None


# ---------------------------------------------------------------------------------------------
# (f1) retrieval loss pieces: SampledSoftmaxLayer (layers/tools.py:32-84), DSSM cosine scaling (DSSM.py:105-106)
# ---------------------------------------------------------------------------------------------
class MatmulNTFn(torch.autograd.Function):
    """a (M,K) @ b (N,K)^T -> (M,N): the sampled logits `inputs @ sampled_w^T`.  The three products are the dense layer's GEMMs
    with the roles swapped (hrb_dense_bwd_x computes A.B^T, hrb_dense_fwd A.B, hrb_dense_bwd_w A^T.B)."""

    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        ctx.save_for_backward(a, b)
        return K.dense_bwd_x(a, b, mode=_lib.GEMM_FP32)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.contiguous()
        da = K.dense_fwd(g, b, None, None, mode=_lib.GEMM_FP32)                 # (M,N) @ (N,K)
        db, _ = K.dense_bwd_w(g, a, want_bias=False, mode=_lib.GEMM_FP32)       # (M,N)^T @ (M,K) -> (N,K)
        return da, db


class RowDotFn(torch.autograd.Function):
    """out[m] = <a[m,:], b[m,:]>: the true-class logits."""

    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        M, Kd = a.shape
        out = torch.empty(M, device=a.device, dtype=torch.float32)
        call("hrb_rowdot", K._p(a), Kd, K._p(b), Kd, M, Kd, K._p(out), K._stream())
        ctx.save_for_backward(a, b)
        return out

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.contiguous()
        M, Kd = a.shape
        da, db = torch.empty_like(a), torch.empty_like(b)
        call("hrb_rowscale", K._p(b), Kd, K._p(g), M, Kd, K._p(da), Kd, K._stream())
        call("hrb_rowscale", K._p(a), Kd, K._p(g), M, Kd, K._p(db), Kd, K._stream())
        return da, db


class SampledSoftmaxFn(torch.autograd.Function):
    """- log Q, accidental-hit mask and softmax cross-entropy against the true class, fused (hrb_sampled_softmax)."""

    @staticmethod
    def forward(ctx, true_logit, sampled_logit, labels, sampled, true_expected, sampled_expected, num_tries, range_max, remove_hits):
        true_logit, sampled_logit = true_logit.contiguous(), sampled_logit.contiguous()
        B, S = sampled_logit.shape
        loss = torch.empty(B, device=true_logit.device, dtype=torch.float32)
        ctx.save_for_backward(true_logit, sampled_logit, labels, sampled, true_expected, sampled_expected)
        ctx.cfg = (float(num_tries), int(range_max), int(bool(remove_hits)))
        call("hrb_sampled_softmax", K._p(true_logit), K._p(sampled_logit), S, K._p(labels), K._p(sampled), B, S, K._p(true_expected),
             K._p(sampled_expected), float(num_tries), int(range_max), int(bool(remove_hits)), None, K._p(loss), None, None, K._stream())
        return loss

    @staticmethod
    def backward(ctx, g):
        true_logit, sampled_logit, labels, sampled, te, se = ctx.saved_tensors
        nt, rm, rh = ctx.cfg
        B, S = sampled_logit.shape
        g = g.contiguous()
        dt, ds = torch.empty_like(true_logit), torch.empty_like(sampled_logit)
        call("hrb_sampled_softmax", K._p(true_logit), K._p(sampled_logit), S, K._p(labels), K._p(sampled), B, S, K._p(te), K._p(se), nt, rm, rh,
             K._p(g), None, K._p(dt), K._p(ds), K._stream())
        return dt, ds, None, None, None, None, None, None, None


class L2NormalizeFn(torch.autograd.Function):
    """tf.nn.l2_normalize(x) over the WHOLE tensor (no axis), as DSSM.py:105-106 calls it."""

    @staticmethod
    def forward(ctx, x, eps):
        x = x.contiguous()
        y = torch.empty_like(x)
        stat = torch.empty(1, device=x.device, dtype=torch.float32)
        scratch = torch.empty(256, device=x.device, dtype=torch.float32)
        call("hrb_l2_normalize_fwd", K._p(x), x.numel(), float(eps), K._p(y), K._p(stat), K._p(scratch), K._stream())
        ctx.save_for_backward(y, stat)
        return y

    @staticmethod
    def backward(ctx, dy):
        y, stat = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(dy)
        scratch = torch.empty(256, device=dy.device, dtype=torch.float32)
        call("hrb_l2_normalize_bwd", K._p(y), K._p(dy), dy.numel(), K._p(stat), K._p(dx), K._p(scratch), K._stream())
        return dx, None


class LAUFirstLayerFn(torch.autograd.Function):
    """First Dense of the local-activation MLP applied to [q, k, q-k, q*k] WITHOUT building that (B,T,4D) tensor
    (layers/sequence.py:96-99 + the Dense(4D) core.py:57 prepends):  q.(Wa+Wc) + b  per sample, plus  [k | q*k].[Wb-Wc; Wd]  as one
    B*T-row tcgen05 GEMM over 2D columns, the per-sample term added in its epilogue (hrb200.h, a10 training path)."""

    @staticmethod
    def forward(ctx, q, keys, W, b, act):
        q, keys, W = q.contiguous(), keys.contiguous(), W.contiguous()
        B, T, D = keys.shape
        U = W.shape[1]
        dev = q.device
        wq = torch.empty(D, U, device=dev)
        wp = torch.empty(2 * D, U, device=dev)
        wpt = torch.empty(U, 2 * D, device=dev)
        call("hrb_lau_split_weights", K._p(W), U, D, U, K._p(wq), K._p(wp), K._p(wpt), K._stream())
        qterm = K.dense_fwd(q, wq, b, None, mode=_lib.GEMM_FP32)                       # (B, U): the part that does not depend on t
        A = torch.empty(B * T, 2 * D, device=dev)
        call("hrb_lau_pack_fwd", K._p(q), K._p(keys), B, T, D, K._p(A), K._stream())
        y = torch.empty(B * T, U, device=dev)
        call("hrb_dense_fwd_t_grouped", K._p(A), 2 * D, K._p(wpt), 2 * D, K._p(qterm), U, T, B * T, 2 * D, U, ACT[act], K._p(y), U, K._stream())
        ctx.save_for_backward(q, keys, A, wq, wp, y)
        ctx.act, ctx.has_bias, ctx.shape = act, b is not None, (B, T, D, U)
        return y.reshape(B, T, U)

    @staticmethod
    def backward(ctx, dy):
        q, keys, A, wq, wp, y = ctx.saved_tensors
        B, T, D, U = ctx.shape
        dy2 = dy.contiguous().reshape(B * T, U)
        dz = K.act_bwd(y, dy2, ctx.act) if ctx.act not in (None, "linear") else dy2
        dA = K.dense_bwd_x_t(dz, wp)                                                    # (B*T, 2D)
        dwp, _ = K.dense_bwd_w_xn(A, K.transpose(dz), want_bias=False)                  # (2D, U)
        dqterm = torch.empty(B, U, device=dz.device)
        call("hrb_group_sum", K._p(dz), U, B, T, U, K._p(dqterm), K._stream())
        dq = K.dense_bwd_x(dqterm, wq, mode=_lib.GEMM_FP32)                            # (B, D): through the per-sample term
        dwq, db = K.dense_bwd_w(q, dqterm, want_bias=ctx.has_bias, mode=_lib.GEMM_FP32)
        dk = torch.empty_like(keys)
        call("hrb_lau_pack_bwd", K._p(q), K._p(keys), K._p(dA), B, T, D, 1, K._p(dq), K._p(dk), K._stream())
        dW = torch.empty(4 * D, U, device=dz.device)
        call("hrb_lau_merge_wgrads", K._p(dwq), K._p(dwp), D, U, K._p(dW), U, K._stream())
        return dq, dk, dW, (db if ctx.has_bias else None), None
