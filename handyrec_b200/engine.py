"""Fused DeepFM training / inference engine on top of the C ABI.

This is the execution plan that ``handyrec_b200.models.DeepFM`` runs when the FM group and the
DNN group hold the same features (the reference's shipped configs, e.g.
/root/reference/tests/ml-1m-test/DeepFM_cfg.yaml and examples/DeepFM/DeepFM_cfg.yaml): every
table is looked up ONCE (the reference does it twice, DeepFM.py:62-63), the pooled (B, F, D) block
is written once and serves as FM input and as the tail of the DNN input row, and the embedding
gradient of both paths meets in one sorted-segment update.

Data layout of one batch in HBM (all fp32, row-major):
  X0   (B, K0p)   [dense (n_dense) | zero pad to a multiple of 4 | F pooled embeddings of D floats]
  A_i  (B, ld_i)  activations of Dense layer i (ld_i = round-up-4(units_i))
  params          ONE flat buffer: W_0 | b_0 | ... | W_n | b_n | fm_w (D) | fm_w0 (1), every block padded
                  to 4 floats; W_i is (K_i_padded, ld_i) with zero rows/columns at the padding
  grads / adam m,v  same layout as params (Adagrad: its accumulator in the place of m, no v; Ftrl: accumulator in m, linear in v,
                  and grads ends with one touched flag per row of the dense-updated tables)
Reference order of the DNN input is kept (dense first, layers/utils.py:70-84); the padding rows of
W_0 multiply zero columns of X0 and receive zero gradients, so they stay zero.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from . import kernels as K
from ._lib import call


def _r4(n: int) -> int:
    return (n + 3) // 4 * 4


def launch_count() -> int:
    c = ctypes.c_int64(0)
    call("hrb_launch_count", ctypes.byref(c))
    return c.value


class DeepFMEngine:
    """DeepFM (models/ranking/context_aware/DeepFM.py) with shared FM / DNN feature groups.

    fields: list of (table_index, seq_len, pool) in reference order (sparse features first, then
    sequence features, features/group.py:319-334); all tables must share one embedding dim.

    Embedding optimiser.  Tables listed in `dense_update_tables` (default: every table with at most
    `dense_table_max_rows` rows) are "dense-updated": the engine re-homes them at the end of its flat parameter
    buffer (`engine.tables[t]` is the live table), their row gradients are reduced into the flat gradient buffer and
    they take the same optimiser step as the dense parameters -- exactly Keras' treatment of an IndexedSlices
    gradient (dense moment decay and dense l2_embd).  Every other table gets the touched-rows-only update.

    optimizer: "adam", "sgd", "adagrad" (Keras Adagrad; accumulators start at `initial_accumulator_value`) or "ftrl" (Keras Ftrl
    with Keras' hyperparameter names: learning_rate_power, initial_accumulator_value, l1, l2, l2_shrinkage, beta).  Under
    Adagrad and Ftrl the touched-rows-only update is exactly Keras' step whenever l2_embd = 0 (DESIGN.md 3).  Under Ftrl a
    zero-gradient step is not a no-op, so with l2_embd = 0 the dense-updated tables step only the rows the batch gathers
    (padding id 0 of pooled fields included): `plan.mark_rows` flags them in the tail of the flat gradient buffer.

    lr: the learning rate of every step, or None when `lr_step` gives each step its own (a Keras schedule).

    task: "binary" (sigmoid head, binary_crossentropy) or "regression" (the raw `dnn + fm`, DeepFM.py:86-88 without the sigmoid),
    trained with `loss` "mean_squared_error", "mean_absolute_error" or "huber" (`huber_delta`); `prob` then holds the predictions.
    """

    def __init__(
        self,
        tables: Sequence[torch.Tensor],
        fields: Sequence[Tuple[int, int, str]],
        n_dense: int,
        dnn_hidden_units: Sequence[int] = (64, 32, 1),
        dnn_activation: str = "relu",
        batch_size: int = 4096,
        optimizer: str = "adam",
        lr: Optional[float] = 1e-3,
        l2_embd: float = 0.0,
        l2_dnn: float = 0.0,
        embedding_optimizer: Optional[str] = None,
        seed: int = 2022,
        gemm_mode: int = _lib.GEMM_AUTO,
        task: str = "binary",
        dense_table_max_rows: int = 0,
        dense_update_tables: Optional[Sequence[int]] = None,
        initial_accumulator_value: float = 0.1,
        learning_rate_power: float = -0.5,
        l1: float = 0.0,
        l2: float = 0.0,
        l2_shrinkage: float = 0.0,
        beta: float = 0.0,
        clipvalue: Optional[float] = None,
        clipnorm: Optional[float] = None,
        global_clipnorm: Optional[float] = None,
        loss: Optional[str] = None,
        huber_delta: float = 1.0,
    ):
        if dnn_hidden_units[-1] != 1:  # DeepFM.py:59-60
            raise ValueError("Output size of dnn should be 1")
        if dnn_activation not in ("relu", "sigmoid", "tanh", "linear", None):
            raise ValueError(f"fused engine supports relu/sigmoid/tanh/linear DNN activations, got {dnn_activation!r}")
        if task == "binary" and loss not in (None, "binary_crossentropy"):
            raise ValueError(f"task='binary' trains binary_crossentropy, got loss={loss!r}")
        if task == "regression" and loss not in K.REG_LOSS:
            raise ValueError(f"task='regression' trains one of {sorted(K.REG_LOSS)}, got loss={loss!r}")
        if task not in ("binary", "regression"):
            raise ValueError(f"fused engine implements task='binary' and task='regression', got {task!r}")
        self.task, self.loss, self.huber_delta = task, loss or "binary_crossentropy", float(huber_delta)
        if initial_accumulator_value < 0:
            raise ValueError(f"initial_accumulator_value must be non-negative, got {initial_accumulator_value}")
        if learning_rate_power > 0 or min(l1, l2, l2_shrinkage) < 0:
            raise ValueError(f"Ftrl needs learning_rate_power <= 0 and non-negative l1 / l2 / l2_shrinkage, got {learning_rate_power}, "
                             f"{l1}, {l2}, {l2_shrinkage}")
        self.dev = tables[0].device
        self.tables = list(tables)
        self.D = int(tables[0].shape[1])
        if any(int(t.shape[1]) != self.D for t in tables):
            raise ValueError("FM needs one embedding dim for every field (Concatenate(axis=1), layers/utils.py:40)")
        self.F = len(fields)
        self.n_dense = int(n_dense)
        self.nd_pad = _r4(self.n_dense)
        self.B = int(batch_size)
        self.act = dnn_activation or "linear"
        self.optimizer = optimizer
        self.emb_opt = embedding_optimizer or {"adam": "adam_lazy", "adagrad": "adagrad", "ftrl": "ftrl"}.get(optimizer, "sgd")
        self.l2_embd, self.l2_dnn = float(l2_embd), float(l2_dnn)
        self.beta1, self.beta2, self.eps = 0.9, 0.999, 1e-7  # Keras Adam defaults (eps: also Keras Adagrad's)
        self.initial_accumulator_value = float(initial_accumulator_value)
        self.lr_power, self.l1, self.l2_shrinkage, self.beta = float(learning_rate_power), float(l1), float(l2_shrinkage), float(beta)
        self.ftrl_l2_reg = float(l2)
        self.set_lr(lr)
        self.gemm_mode = gemm_mode
        self.step_count = 0

        # ---- lookup plan: ids columns are packed in field order, outputs follow the dense block ----
        plan_fields, col = [], 0
        for f, (ti, L, pool) in enumerate(fields):
            plan_fields.append((ti, L, pool if (L > 1 or pool not in (None, "none")) else "none", col, self.nd_pad + f * self.D))
            col += L
        self.ids_cols = col
        self.plan_fields = plan_fields
        if dense_update_tables is None:
            dense_update_tables = [t for t, w in enumerate(self.tables) if w.shape[0] <= dense_table_max_rows]
        self.dense_tables = sorted(set(int(t) for t in dense_update_tables))

        # ---- dense parameters: one flat buffer ----
        self.K0 = self.n_dense + self.F * self.D           # logical DNN input width
        self.K0p = self.nd_pad + self.F * self.D           # padded row width of X0
        units = [self.K0] + [int(u) for u in dnn_hidden_units]  # core.py:57 prepends Dense(in)
        self.units = units
        self.layer_Kl = [self.K0] + units[:-1]                      # logical input widths
        self.layer_ld = [_r4(u) if u > 1 else 1 for u in units]  # the 1-unit logit layer stays contiguous
        self.layer_K = [self.K0p] + self.layer_ld[:-1]
        offs, off, self._segments = [], 0, []
        for Kp, ld in zip(self.layer_K, self.layer_ld):
            wo = off
            off = _r4(off + Kp * ld)
            bo = off
            off = _r4(off + ld)
            offs.append((wo, bo))
            self._segments.append((wo, bo - wo, True))   # kernel: l2_dnn applies (core.py:63)
            self._segments.append((bo, off - bo, False))  # bias: no regulariser
        self.fm_off = off
        off += _r4(self.D + 1)
        self._segments.append((self.fm_off, off - self.fm_off, False))
        self.n_dense_params = off
        self._table_off = {}
        # dense-updated tables live behind the dense parameters, rows on 128-byte lines like any table (under Ftrl also on a
        # multiple of D floats, so that the whole table block is rows of D floats for the touched flags)
        align = 32 if optimizer != "ftrl" else 32 * self.D // math.gcd(32, self.D)
        for t in self.dense_tables:
            off = (off + align - 1) // align * align
            self._table_off[t] = off
            off += self.tables[t].numel()
        self.n_params = off
        self.tab0 = min(self._table_off.values()) if self._table_off else off  # first float of the table block
        # Ftrl: one touched flag per D floats of the table block at the tail of the gradient buffer, then the sharded engine's
        # padding flags (zeroed with the table gradients, all-reduced with them by the sharded engine)
        n_touched = (off - self.tab0) // self.D if optimizer == "ftrl" else 0
        self.params = torch.zeros(off, device=self.dev, dtype=torch.float32)
        self.grads = torch.zeros(off + n_touched + self._n_pad_flags, device=self.dev, dtype=torch.float32)
        self.touched = self.grads[off : off + n_touched] if n_touched else None
        self.opt_m = torch.zeros(off, device=self.dev, dtype=torch.float32) if optimizer == "adam" else None
        self.opt_v = torch.zeros(off, device=self.dev, dtype=torch.float32) if optimizer == "adam" else None
        if optimizer in ("adagrad", "ftrl"):  # opt_m is the accumulator (Ftrl: opt_v the linear slot)
            self.opt_m = torch.full((off,), self.initial_accumulator_value, device=self.dev, dtype=torch.float32)
        if optimizer == "ftrl":
            self.opt_v = torch.zeros(off, device=self.dev, dtype=torch.float32)
        self.W, self.b, self.dW, self.db = [], [], [], []
        for (wo, bo), Kp, ld in zip(offs, self.layer_K, self.layer_ld):
            self.W.append(self.params[wo : wo + Kp * ld].view(Kp, ld))
            self.b.append(self.params[bo : bo + ld])
            self.dW.append(self.grads[wo : wo + Kp * ld].view(Kp, ld))
            self.db.append(self.grads[bo : bo + ld])
        self.fm_w = self.params[self.fm_off : self.fm_off + self.D]
        self.fm_w0 = self.params[self.fm_off + self.D : self.fm_off + self.D + 1]
        self.d_fm = self.grads[self.fm_off : self.fm_off + self.D + 1]
        self._init_dense(seed)
        table_grads: List[Optional[torch.Tensor]] = [None] * len(self.tables)
        for t, o in self._table_off.items():
            n = self.tables[t].numel()
            live = self.params[o : o + n].view_as(self.tables[t])
            live.copy_(self.tables[t])
            self.tables[t] = live
            table_grads[t] = self.grads[o : o + n].view_as(live)
        self.table_grads = table_grads
        self.adam_m = self.adam_v = self.accum = self.linear = None
        if self.emb_opt == "adam_lazy":
            self.adam_m = [None if t in self._table_off else torch.zeros_like(w) for t, w in enumerate(self.tables)]
            self.adam_v = [None if t in self._table_off else torch.zeros_like(w) for t, w in enumerate(self.tables)]
        elif self.emb_opt in ("adagrad", "ftrl"):
            self.accum = [None if t in self._table_off else torch.full_like(w, self.initial_accumulator_value) for t, w in enumerate(self.tables)]
        if self.emb_opt == "ftrl":
            self.linear = [None if t in self._table_off else torch.zeros_like(w) for t, w in enumerate(self.tables)]
        self.plan = K.LookupPlan(self.tables, plan_fields, self.adam_m, self.adam_v, accum=self.accum, linear=self.linear)
        self.table_touched: List[Optional[torch.Tensor]] = [None] * len(self.tables)  # Ftrl: touched flags of the dense-updated tables
        if self.touched is not None:
            for t, o in self._table_off.items():
                r0 = (o - self.tab0) // self.D
                self.table_touched[t] = self.touched[r0 : r0 + self.tables[t].shape[0]]
        if self.dense_tables:
            self.plan.set_dense_grads(table_grads)

        # ---- batch buffers ----
        B = self.B
        f32 = dict(device=self.dev, dtype=torch.float32)
        self.X0 = torch.zeros(B, self.K0p, **f32)
        self.A = [torch.zeros(B, ld, **f32) for ld in self.layer_ld]
        self.dZ = [torch.zeros(B, ld, **f32) for ld in self.layer_ld]
        self.dX0 = torch.zeros(B, self.K0p, **f32)
        self.fm_out = torch.empty(B, **f32)
        self.fm_sum = torch.empty(B, self.D, **f32)
        self.prob = torch.empty(B, **f32)
        self.loss_sum = torch.zeros(1, **f32)
        self._loss_ws = K.regression_loss_workspace(B, self.dev) if task == "regression" else None
        # tcgen05 path: transposed copies (W^T, dZ^T) so that every GEMM operand has its reduction dim contiguous; the activations are
        # read untransposed by the weight-gradient GEMM (hrb_dense_bwd_w_xn)
        self.use_tc = gemm_mode != _lib.GEMM_FP32 and B >= 512 and B % 4 == 0
        self.tc_layer = [self.use_tc and u >= 16 for u in self.units]
        if self.use_tc:
            self.Wt = [torch.zeros(ld, Kp, **f32) if tc else None for ld, Kp, tc in zip(self.layer_ld, self.layer_K, self.tc_layer)]
            self.dZt = [torch.zeros(ld, B, **f32) for ld in self.layer_ld]
            # relu sign bits of every hidden activation (1 bit/element) for the activation-gradient epilogue
            self.relu_mask = [torch.zeros(B, (u + 31) // 32, device=self.dev, dtype=torch.int32) if self.act == "relu" else None for u in self.units]
            self._refresh_wt()
        self.ids_dev = torch.zeros(B, self.ids_cols, device=self.dev, dtype=torch.int32)
        self.dense_dev = torch.zeros(B, max(self.n_dense, 1), **f32)
        self.label_dev = torch.zeros(B, **f32)
        self.loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        self._ws_emb = torch.empty(self.plan.workspace_bytes(B), device=self.dev, dtype=torch.uint8)
        self.clip = None
        if clipvalue is not None or clipnorm is not None or global_clipnorm is not None:
            self._init_clip((clipvalue, clipnorm, global_clipnorm))

    def _init_clip(self, args) -> None:
        """Keras gradient clipping (handyrec_b200.clip): one variable per Dense kernel / bias, FM kernel, FM w_0 and table.  With
        l2_embd = 0 the tables' gradients are their lookups' IndexedSlices, clipped per position in dX0 (the FM part apart, in
        fm_dx); with l2_embd > 0 they are dense, so every table must be dense-updated and its block is clipped like a Dense kernel."""
        from .clip import GradClip

        if self.l2_embd > 0.0 and len(self.dense_tables) != len(self.tables):
            raise ValueError("gradient clipping with l2_embd > 0 needs every table dense-updated (dense_table_max_rows): Keras' "
                             "clipped gradient of a regularised table covers every row, which the touched-rows update never forms")
        segs = self._segments[:-1] + [(self.fm_off, self.D, False), (self.fm_off + self.D, 1, False)]
        self._clip_nd = len(segs)
        cg, cw, cl, cv = [], [], [], []
        for k, (o, n, reg) in enumerate(segs):
            cg.append(self.grads[o : o + n])
            cw.append(self.params[o : o + n])
            cl.append(2.0 * self.l2_dnn if reg else 0.0)
            cv.append(k)
        if self.l2_embd > 0.0:
            for t, o in self._table_off.items():
                n = self.tables[t].numel()
                cg.append(self.grads[o : o + n])
                cw.append(self.params[o : o + n])
                cl.append(2.0 * self.l2_embd)
                cv.append(self._clip_nd + t)
        else:
            self.fm_dx = torch.zeros(self.B, self.F * self.D, device=self.dev, dtype=torch.float32)
        self._clip_segs = (cg, cw, cl, cv)
        self.clip = GradClip(args, self._clip_nd + len(self.tables), len(self.tables), self.dev)

    def _clip_gradients(self, ids: torch.Tensor, B: int) -> None:
        """Keras' _transform_gradients in place, once every gradient of the step is known and before anything steps; the
        optimisers then run with l2 = 0 where the prepare pass folded 2*l2*w in."""
        c, nd = self.clip, self._clip_nd
        cg, cw, cl, cv = self._clip_segs
        c.begin()
        if self.l2_embd == 0.0:
            self.plan.clip_grads(ids, self.dX0[:B], self.fm_dx[:B], c.value, c.sumsq[nd:] if c.scales else None, c.ws)
        c.prepare(cg, cw, cl, cv)
        c.finish()
        c.apply(cg, cv)
        if self.l2_embd == 0.0 and c.scales:
            self.plan.clip_apply(self.dX0[:B], B, c.scale[nd:])
        self._mark("clip")

    # When set, a callable giving the learning rate of every training step, called once per step by train_step_on_device before
    # anything launches (lowering.FusedDeepFM: a Keras schedule / decay, counted in the optimizer's `iterations`).  The rate reaches
    # the kernels as a launch argument: no extra launch, no host sync, no rebuild.
    lr_step = None

    def set_lr(self, lr: Optional[float]) -> None:
        """The learning rate of the following steps, with the l2 Keras hands its Ftrl kernel at that rate (l2 + beta / (2*lr)).
        None: no rate until `lr_step` gives the first step its own."""
        from .schedules import ftrl_kernel_l2

        self.lr = None if lr is None else float(lr)
        self.ftrl_l2 = None if lr is None else ftrl_kernel_l2(self.ftrl_l2_reg, self.beta, self.lr)

    _n_pad_flags = 0  # floats the sharded engine keeps behind the touched flags
    metrics = None  # handyrec_b200.metrics.MetricSet: counted from every training step's probabilities (one launch), None: nothing

    # ------------------------------------------------------------------------------------------
    _marks = None  # when a list: (phase name, cuda event) recorded after every phase of a step

    _timeline = None  # when a list: (name, event) recorded on whatever stream is current, WITHOUT serialising the streams

    def _mark(self, name: str) -> None:
        if self._timeline is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self._timeline.append((name, e))
        if self._marks is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self._marks.append((name, e))

    def profile_step(self, ids, dense, label) -> "OrderedDict[str, float]":
        """Run one train step with a CUDA event after every phase; returns ms per phase (launching stream)."""
        from collections import OrderedDict

        self._marks = []
        self._mark("start")
        self.train_step_on_device(ids, dense, label)
        torch.cuda.current_stream().synchronize()
        marks, self._marks = self._marks, None
        out = OrderedDict()
        for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
            out[n1] = out.get(n1, 0.0) + e0.elapsed_time(e1)
        return out

    def timeline_step(self, ids, dense, label) -> "OrderedDict[str, float]":
        """One NORMAL step (side streams and overlap as in production) with an event after every phase on the stream the
        phase runs on; returns the completion time of every phase in ms since the start of the step."""
        from collections import OrderedDict

        torch.cuda.synchronize()
        self._timeline = []
        self._mark("start")
        self.train_step_on_device(ids, dense, label)
        self._mark("end")
        torch.cuda.synchronize()
        tl, self._timeline = self._timeline, None
        e0 = tl[0][1]
        return OrderedDict((n, round(e0.elapsed_time(e), 4)) for n, e in tl[1:])

    def _refresh_wt(self) -> None:
        """W_i^T for the tensor-core forward (the optimiser updates W_i; 1.3 MB of transposes per step)."""
        if not getattr(self, "use_tc", False):
            return
        st = K._stream()
        for i, tc in enumerate(self.tc_layer):
            if tc:
                call("hrb_transpose", K._p(self.W[i]), self.layer_K[i], self.layer_ld[i], self.layer_ld[i], K._p(self.Wt[i]), self.layer_K[i], st)

    def _init_dense(self, seed: int) -> None:
        """Keras Dense defaults: glorot-uniform kernels, zero biases; FM Dense(1) glorot, w0 zeros."""
        g = torch.Generator().manual_seed(seed)
        for i, (Kl, u) in enumerate(zip(self.layer_Kl, self.units)):
            lim = math.sqrt(6.0 / (Kl + u))
            w = (torch.rand(Kl, u, generator=g) * 2 - 1) * lim
            self.set_dense_weights(i, w, torch.zeros(u))
        lim = math.sqrt(6.0 / (self.D + 1))
        self.fm_w.copy_(((torch.rand(self.D, generator=g) * 2 - 1) * lim).to(self.dev))
        self.fm_w0.zero_()

    def set_dense_weights(self, i: int, w: torch.Tensor, b: torch.Tensor) -> None:
        """w in the reference layout (K_logical, units): rows of layer 0 are [dense | embeddings]."""
        Kl, u = self.layer_Kl[i], self.units[i]
        assert tuple(w.shape) == (Kl, u) and tuple(b.shape) == (u,)
        W = torch.zeros(self.layer_K[i], self.layer_ld[i])
        if i == 0:
            W[: self.n_dense, :u] = w[: self.n_dense]
            W[self.nd_pad :, :u] = w[self.n_dense :]
        else:
            W[:Kl, :u] = w
        self.W[i].copy_(W.to(self.dev))
        bb = torch.zeros(self.layer_ld[i])
        bb[:u] = b
        self.b[i].copy_(bb.to(self.dev))
        self._refresh_wt()

    def get_dense_weights(self, i: int) -> Tuple[torch.Tensor, torch.Tensor]:
        Kl, u = self.layer_Kl[i], self.units[i]
        W = self.W[i].cpu()
        if i == 0:
            w = torch.cat([W[: self.n_dense, :u], W[self.nd_pad :, :u]], 0)
        else:
            w = W[:Kl, :u]
        return w.clone(), self.b[i][:u].cpu().clone()

    def get_dense_grads(self, i: int) -> Tuple[torch.Tensor, torch.Tensor]:
        Kl, u = self.layer_Kl[i], self.units[i]
        W = self.dW[i].cpu()
        w = torch.cat([W[: self.n_dense, :u], W[self.nd_pad :, :u]], 0) if i == 0 else W[:Kl, :u]
        return w.clone(), self.db[i][:u].cpu().clone()

    # ------------------------------------------------------------------------------------------
    def forward(self, ids: torch.Tensor, dense: Optional[torch.Tensor], training: bool = False) -> torch.Tensor:
        """ids (B, ids_cols) int32, dense (B, n_dense) fp32|int32 on device -> logits in self.A[-1], probabilities."""
        B = ids.shape[0]
        assert B <= self.B
        st = K._stream()
        if self.n_dense:
            call("hrb_pack_dense", K._p(dense), int(dense.dtype == torch.int32), dense.stride(0), B, self.n_dense, self.nd_pad,
                 K._p(self.X0), self.K0p, st)
            self._mark("pack_dense")
        self._lookup_fm_forward(ids, B, st)
        x, ldx = self.X0, self.K0p
        n = len(self.units)
        for i in range(n):
            act = self.act if i + 1 != n else "linear"  # core.py:66-69 with output_activation="linear"
            if self.units[i] == 1 and self.layer_K[i] % 4 == 0:
                call("hrb_dense1_fwd", K._p(x), ldx, K._p(self.W[i]), K._p(self.b[i]), B, self.layer_K[i], K._p(self.A[i]), st)
            elif self.use_tc and self.tc_layer[i] and B == self.B:
                call("hrb_dense_fwd_t", K._p(x), ldx, K._p(self.Wt[i]), self.layer_K[i], K._p(self.b[i]), B, self.layer_K[i], self.units[i],
                     _lib.ACT[act], K._p(self.A[i]), self.layer_ld[i], None, B,
                     K._p(self.relu_mask[i]) if (training and act == "relu") else None, st)
            else:
                call("hrb_dense_fwd", K._p(x), ldx, K._p(self.W[i]), self.layer_ld[i], K._p(self.b[i]), B, self.layer_K[i], self.units[i],
                     _lib.ACT[act], K._p(self.A[i]), self.layer_ld[i], _lib.GEMM_FP32, st)
            self._mark(f"dense_fwd_{i}")
            x, ldx = self.A[i], self.layer_ld[i]
        return self.A[-1]

    def _lookup_fm_forward(self, ids, B, st) -> None:
        """ids -> pooled embeddings in X0[:, nd_pad:], FM logit and field sum (overridden by the sharded engine)."""
        call("hrb_lookup_fm_fwd", self.plan._h, K._p(ids), ids.stride(0), B, K._p(self.X0), self.K0p, None, K._p(self.fm_w),
             K._p(self.fm_w0), K._p(self.fm_out), K._p(self.fm_sum), None, st)
        self._mark("lookup_fm_fwd")

    def _zero_table_grads(self) -> None:
        if self.grads.numel() > self.n_dense_params:
            self.grads[self.n_dense_params :].zero_()

    def _mark_touched(self, plan, ids, tables) -> None:
        """Ftrl with l2_embd = 0: flag the rows of the dense-updated tables among `tables` (the plan's tables, in order) that the
        batch gathers; the flat step then steps those rows only (with l2_embd > 0 Keras' table gradient is dense: every row steps)."""
        if self.touched is not None and self.l2_embd == 0.0:
            plan.mark_rows(ids, [self.table_touched[t] for t in tables])

    # The library has two implementations of the embedding backward (hrb200.h: hrb_bwd_algo); which one is faster depends on the
    # id distribution (spread ids: UNITS, a few very hot rows: SORT).  The engine times both on the caller's own data during
    # its first steps (steps 3-6, one host sync each) and keeps the faster one; both are deterministic and agree to rounding.
    autotune_embedding_bwd = True
    _bwd_trials: Optional[list] = None
    bwd_algo = "auto"

    def _embedding_backward(self, ids, B, st, op) -> None:
        self._zero_table_grads()
        self._mark_touched(self.plan, ids, range(len(self.tables)))
        trial = None
        n_trials = len(self._bwd_trials or [])
        if self.autotune_embedding_bwd and self._marks is None and B == self.B and self.step_count >= 3 and n_trials < 4 and self.bwd_algo == "auto":
            trial = _lib.BWD_UNITS if n_trials % 2 == 0 else _lib.BWD_SORT
            call("hrb_plan_set_bwd_algo", self.plan._h, trial)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        call("hrb_lookup_bwd_update", self.plan._h, K._p(ids), ids.stride(0), B, K._p(self.dX0), self.K0p, None, ctypes.byref(op),
             K._p(self._ws_emb), self._ws_emb.numel(), st)
        if trial is not None:
            e1.record()
            e1.synchronize()
            self._bwd_trials = (self._bwd_trials or []) + [(trial, e0.elapsed_time(e1))]
            if len(self._bwd_trials) == 4:
                best = {}
                for algo, ms in self._bwd_trials:
                    best[algo] = min(best.get(algo, 1e30), ms)
                pick = min(best, key=best.get)
                call("hrb_plan_set_bwd_algo", self.plan._h, pick)
                self.bwd_algo = "units" if pick == _lib.BWD_UNITS else "sort"
                self.bwd_algo_ms = {("units" if a == _lib.BWD_UNITS else "sort"): round(m, 4) for a, m in best.items()}
        self._mark("embedding_bwd_update")

    def _pre_embedding_backward(self) -> None:
        """Sharded engine: finish the routing exchange (host sync on data that is ready since the forward)."""

    def _sync_dense_grads(self) -> None:
        """Replicated dense parameters: the sharded engine all-reduces the flat gradient buffer here."""

    grad_scale_div = 1  # number of ranks the batch mean is taken over
    overlap_embedding_bwd = False  # sharded engine: run the row exchange/update beside the layer-0 weight gradient
    _side = None
    _side_pending = False

    def predict_on_device(self, ids: torch.Tensor, dense: Optional[torch.Tensor]) -> torch.Tensor:
        B = ids.shape[0]
        self.forward(ids, dense)
        if self.task == "regression":
            K.regression_loss(self.loss, self.huber_delta, self.A[-1], self.fm_out, None, B, 1, 0.0, pred=self.prob)
            return self.prob[:B]
        call("hrb_sigmoid_bce", K._p(self.A[-1]), K._p(self.fm_out), K._p(self.label_dev), B, 0.0, K._p(self.prob), None, None, K._stream())
        return self.prob[:B]

    def train_step_on_device(self, ids: torch.Tensor, dense: Optional[torch.Tensor], label: torch.Tensor,
                             weight: Optional[torch.Tensor] = None) -> None:
        """One full step: forward, loss (BCE, or the regression loss of task="regression"), backward, embedding row updates, dense
        optimiser.  Loss sum -> self.loss_sum.  `weight` (B float32, Keras' sample weights): the loss sum becomes sum(w * l) and dlogit
        w * dl/dlogit / (B * ranks), and the weighted metrics sum the weights; everything after dlogit runs unchanged."""
        B = ids.shape[0]
        st = K._stream()
        self.step_count += 1
        if self.lr_step is not None:
            self.set_lr(self.lr_step())
        self.forward(ids, dense, training=True)
        self.loss_sum.zero_()
        dlogit = self.dZ[-1]  # (B, 1): the logit layer has one unit (DeepFM.py:59-60)
        if self.task == "regression":  # prediction dnn + fm, loss sum and dlogit in one launch, as the sigmoid head
            K.regression_loss(self.loss, self.huber_delta, self.A[-1], self.fm_out, label, B, 1, 1.0 / (B * self.grad_scale_div), self.prob,
                              dlogit, self.loss_sum, weight=weight, workspace=self._loss_ws)
        elif weight is None:
            call("hrb_sigmoid_bce", K._p(self.A[-1]), K._p(self.fm_out), K._p(label), B, 1.0 / (B * self.grad_scale_div), K._p(self.prob), K._p(dlogit), K._p(self.loss_sum), st)
        else:
            call("hrb_sigmoid_bce_weighted", K._p(self.A[-1]), K._p(self.fm_out), K._p(label), K._p(weight), B, 1.0 / (B * self.grad_scale_div),
                 K._p(self.prob), K._p(dlogit), K._p(self.loss_sum), st)
        self._mark("sigmoid_bce" if self.task == "binary" else "regression_loss")
        if self.metrics is not None:  # Keras counts its metrics from the training forward, before the weight update
            self.metrics.update(self.prob[:B], label, weight)
            self._mark("metric_update")
        self._backward(ids, B, st)

    def _backward(self, ids: torch.Tensor, B: int, st) -> None:
        n = len(self.units)
        need = ctypes.c_size_t(0)
        dz, lddz = self.dZ[-1], self.layer_ld[-1]
        tc_step = self.use_tc and B == self.B
        op = _lib.OptParams()
        op.opt = {"sgd": _lib.OPT_SGD, "adagrad": _lib.OPT_ADAGRAD, "ftrl": _lib.OPT_FTRL}.get(self.emb_opt, _lib.OPT_ADAM_LAZY)
        op.lr, op.beta1, op.beta2, op.eps, op.l2_scale = self.lr, self.beta1, self.beta2, self.eps, 2.0 * self.l2_embd
        op.bias_corr1, op.bias_corr2 = 1.0 - self.beta1 ** self.step_count, 1.0 - self.beta2 ** self.step_count
        op.l1, op.l2, op.lr_power, op.l2_shrinkage = self.l1, self.ftrl_l2, self.lr_power, self.l2_shrinkage
        self._op = op
        emb_done = [False]

        def bwd_x_0(dz0, lddz0) -> None:
            # (adding the FM term in the epilogue of this GEMM instead of the separate fm_bwd pass was measured: the epilogue becomes the
            # GEMM's bottleneck, +110 us against the 43 us the pass costs -- profiles/r02_experiments.md)
            Kp0, N0 = self.layer_K[0], self.units[0]
            call("hrb_dense_bwd_x_t", K._p(dz0), lddz0, K._p(self.W[0]), self.layer_ld[0], B, Kp0, N0, None, 0, 0, None, K._p(self.dX0), self.K0p,
                 None, 0, st)

        def emb_part(side: bool) -> None:
            """dX0 is complete: add the FM path, then reduce + apply the embedding-row gradients (a13).  With `side`, the
            row exchange / update runs on a second stream while the main stream finishes the layer-0 weight gradient."""
            emb_done[0] = True
            emb_x = self.X0[:, self.nd_pad :]
            emb_dx = self.dX0[:, self.nd_pad :]
            if self.clip is not None and self.l2_embd == 0.0:
                # clipping: the FM part stays apart (Keras clips the FM and the DNN lookup's values separately), then dX0 takes both
                call("hrb_fm_bwd", K._p(emb_x), self.K0p, B, self.F, self.D, K._p(self.fm_w), K._p(self.dZ[-1]), K._p(self.fm_dx), self.F * self.D,
                     0, K._p(self.d_fm), K._stream())
                self._mark("fm_bwd")
                self._clip_gradients(ids, B)
            else:
                # FM path adds dlogit * (w + S - x) into the embedding columns of dX0 (interaction.py:26-39)
                call("hrb_fm_bwd", K._p(emb_x), self.K0p, B, self.F, self.D, K._p(self.fm_w), K._p(self.dZ[-1]), K._p(emb_dx), self.K0p, 1,
                     K._p(self.d_fm), K._stream())
                self._mark("fm_bwd")
            if side and self._marks is None:
                main = torch.cuda.current_stream()
                if self._side is None:
                    self._side = torch.cuda.Stream()
                with torch.cuda.stream(self._side):
                    self._pre_embedding_backward()  # host-synchronising preparation that does not depend on the gradients
                self._side.wait_stream(main)
                with torch.cuda.stream(self._side):
                    self._embedding_backward(ids, B, K._stream(), op)
                self._side_pending = True
            else:
                self._embedding_backward(ids, B, K._stream(), op)

        for i in range(n - 1, -1, -1):
            x, ldx = (self.A[i - 1], self.layer_ld[i - 1]) if i > 0 else (self.X0, self.K0p)
            Kp, N = self.layer_K[i], self.units[i]
            if N == 1 and i > 0 and Kp % 4 == 0 and Kp <= 1024:
                call("hrb_dense1_bwd_workspace", B, Kp, ctypes.byref(need))
                ws = self._dense_ws(need.value)
                call("hrb_dense1_bwd", K._p(x), ldx, K._p(self.W[i]), K._p(dz), B, Kp, _lib.ACT[self.act], K._p(self.dZ[i - 1]), self.layer_ld[i - 1],
                     K._p(self.dZt[i - 1]) if tc_step else None, B, K._p(self.dW[i]), K._p(self.db[i]), K._p(ws), ws.numel(), st)
                dz, lddz = self.dZ[i - 1], self.layer_ld[i - 1]
                self._mark(f"dense_bwd_{i}_logit")
                continue
            if tc_step and self.tc_layer[i] and i == 0 and self.overlap_embedding_bwd:
                # layer 0, overlapped order: dX0 first, then the embedding exchange/update on the side stream || dW0 here
                bwd_x_0(dz, lddz)
                self._mark("dense_bwd_x_0")
                emb_part(side=True)
                call("hrb_dense_bwd_w_t_workspace", B, Kp, N, ctypes.byref(need))
                ws = self._dense_ws(need.value)
                call("hrb_dense_bwd_w_xn", K._p(self.X0), self.K0p, K._p(self.dZt[0]), B, B, Kp, N, K._p(self.dW[0]), self.layer_ld[0],
                     K._p(self.db[0]), K._p(ws), ws.numel(), st)
                self._mark("dense_bwd_w_0")
                continue
            if tc_step and self.tc_layer[i]:
                call("hrb_dense_bwd_w_t_workspace", B, Kp, N, ctypes.byref(need))
                ws = self._dense_ws(need.value)
                # x is read as the forward stored it: the GEMM transposes the tile on its way into tensor memory (no X0^T / A_i^T copies)
                call("hrb_dense_bwd_w_xn", K._p(x), ldx, K._p(self.dZt[i]), B, B, Kp, N, K._p(self.dW[i]), self.layer_ld[i],
                     K._p(self.db[i]), K._p(ws), ws.numel(), st)
                self._mark(f"dense_bwd_w_{i}")
                if i > 0:
                    use_mask = self.act == "relu" and self.tc_layer[i - 1]  # the mask was written by the tensor-core forward of layer i-1
                    call("hrb_dense_bwd_x_t", K._p(dz), lddz, K._p(self.W[i]), self.layer_ld[i], B, Kp, N, K._p(self.A[i - 1]), self.layer_ld[i - 1],
                         _lib.ACT[self.act], K._p(self.relu_mask[i - 1]) if use_mask else None, K._p(self.dZ[i - 1]), self.layer_ld[i - 1],
                         K._p(self.dZt[i - 1]), B, st)
                    dz, lddz = self.dZ[i - 1], self.layer_ld[i - 1]
                else:
                    bwd_x_0(dz, lddz)
                self._mark(f"dense_bwd_x_{i}")
                continue
            call("hrb_dense_bwd_w_workspace", B, Kp, N, ctypes.byref(need))
            ws = self._dense_ws(need.value)
            call("hrb_dense_bwd_w", K._p(x), ldx, K._p(dz), lddz, B, Kp, N, K._p(self.dW[i]), self.layer_ld[i], K._p(self.db[i]),
                 K._p(ws), ws.numel(), _lib.GEMM_FP32, st)
            self._mark(f"dense_bwd_w_{i}")
            if i > 0:
                call("hrb_dense_bwd_x", K._p(dz), lddz, K._p(self.W[i]), self.layer_ld[i], B, Kp, N, K._p(self.A[i - 1]), self.layer_ld[i - 1],
                     _lib.ACT[self.act], K._p(self.dZ[i - 1]), self.layer_ld[i - 1], _lib.GEMM_FP32, st)
                dz, lddz = self.dZ[i - 1], self.layer_ld[i - 1]
                if tc_step:  # the next (tensor-core) weight gradient wants dz^T
                    call("hrb_transpose", K._p(dz), B, self.units[i - 1], lddz, K._p(self.dZt[i - 1]), B, st)
            else:
                call("hrb_dense_bwd_x", K._p(dz), lddz, K._p(self.W[0]), self.layer_ld[0], B, Kp, N, None, 0, 0, K._p(self.dX0), self.K0p,
                     _lib.GEMM_FP32, st)
            self._mark(f"dense_bwd_x_{i}")
        if not emb_done[0]:
            emb_part(side=False)
        self._sync_dense_grads()
        if self.clip is not None and self.l2_embd != 0.0:  # the table block holds the tables' dense gradients now
            self._clip_gradients(ids, B)
        # dense parameters (a clip folded every regulariser into the gradients)
        fold = self.clip is not None
        segs = [(o_, n_, 2.0 * self.l2_dnn if reg and not fold else 0.0) for o_, n_, reg in self._segments]
        ftrl_rows = self.optimizer == "ftrl" and self.touched is not None and self.l2_embd == 0.0
        if self.n_params > self.n_dense_params and not ftrl_rows:  # dense-updated tables: Keras adds d(l2_embd*sum w^2) for every row (group.py:289)
            segs.append((self.n_dense_params, self.n_params - self.n_dense_params, 0.0 if fold else 2.0 * self.l2_embd))
        merged = [segs[0]]
        for o_, n_, l2_ in segs[1:]:  # neighbouring segments with the same regulariser take one launch
            po, pn, pl = merged[-1]
            if pl == l2_ and po + pn == o_:
                merged[-1] = (po, pn + n_, pl)
            else:
                merged.append((o_, n_, l2_))
        for off, length, l2s in merged:
            o = off * 4
            pp = lambda t: ctypes.c_void_p(t.data_ptr() + o)
            if self.optimizer == "adam":
                call("hrb_adam_step", pp(self.params), pp(self.grads), pp(self.opt_m), pp(self.opt_v), length, self.lr, self.beta1,
                     self.beta2, self.eps, op.bias_corr1, op.bias_corr2, l2s, st)
            elif self.optimizer == "adagrad":
                call("hrb_adagrad_step", pp(self.params), pp(self.grads), pp(self.opt_m), length, self.lr, self.eps, l2s, st)
            elif self.optimizer == "ftrl":
                call("hrb_ftrl_step", pp(self.params), pp(self.grads), pp(self.opt_m), pp(self.opt_v), length, self.lr, self.l1, self.ftrl_l2,
                     self.lr_power, self.l2_shrinkage, l2s, None, 0, st)
            else:
                call("hrb_sgd_step", pp(self.params), pp(self.grads), length, self.lr, l2s, st)
        if ftrl_rows:  # the table block: only the rows the batch gathered (IndexedSlices) step
            o = self.tab0 * 4
            pp = lambda t: ctypes.c_void_p(t.data_ptr() + o)
            call("hrb_ftrl_step", pp(self.params), pp(self.grads), pp(self.opt_m), pp(self.opt_v), self.n_params - self.tab0, self.lr, self.l1,
                 self.ftrl_l2, self.lr_power, self.l2_shrinkage, 0.0, K._p(self.touched), self.D, st)
        self._refresh_wt()
        if self._side_pending:  # the next step's lookup must see the updated rows
            torch.cuda.current_stream().wait_stream(self._side)
            self._side_pending = False
        self._mark("dense_optimizer")

    _dws: Optional[torch.Tensor] = None

    def _dense_ws(self, nbytes: int) -> torch.Tensor:
        if self._dws is None or self._dws.numel() < nbytes:
            self._dws = torch.empty(max(nbytes, 1 << 20), device=self.dev, dtype=torch.uint8)
        return self._dws

    # ------------------------------------------------------------------------------------------
    # public, host-facing API (what Model.train_on_batch / predict call)
    # ------------------------------------------------------------------------------------------
    _weight_dev: Optional[torch.Tensor] = None  # the sample weights of train_on_batch / predict, allocated at the first weighted call

    def _weights_to_device(self, weight_host: Optional[torch.Tensor], B: int) -> Optional[torch.Tensor]:
        if weight_host is None:
            return None
        if self._weight_dev is None:
            self._weight_dev = torch.zeros(self.B, device=self.dev, dtype=torch.float32)
        self._weight_dev[:B].copy_(weight_host, non_blocking=True)
        return self._weight_dev[:B]

    def train_on_batch(self, ids_host: torch.Tensor, dense_host: Optional[torch.Tensor], label_host: torch.Tensor,
                       weight_host: Optional[torch.Tensor] = None) -> float:
        """Host (pinned) tensors in, mean loss out (with `weight_host`: sum(w * l) / B).  Includes the H2D copies and a D2H
        read of the loss."""
        B = ids_host.shape[0]
        self.ids_dev[:B].copy_(ids_host, non_blocking=True)
        if self.n_dense:
            self.dense_dev[:B].copy_(dense_host, non_blocking=True)
        self.label_dev[:B].copy_(label_host, non_blocking=True)
        weight = self._weights_to_device(weight_host, B)
        self.train_step_on_device(self.ids_dev[:B], self.dense_dev[:B] if self.n_dense else None, self.label_dev[:B], weight)
        self.loss_host.copy_(self.loss_sum, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(self.loss_host[0]) / B

    def fit_batches(self, batches, on_step=None) -> List[float]:
        """Keras-`fit`-like loop over host batches `(ids, dense, label)` or `(ids, dense, label, weight)` (pinned tensors; weight
        None or Keras' sample weights) with input prefetch: the H2D copies of batch t+1 run on a copy stream while batch t
        computes, and every step's loss is copied back asynchronously; the host waits once, at the end.  Returns the per-step
        mean losses.

        `on_step(t, loss)` (Keras callbacks with batch hooks): called with loss None before step t is issued, and with step t's mean
        loss once it is on the host -- after step t has been issued and batch t+1 fetched and its copy started, so the packing
        thread and the prefetch run on while the hook does.  A true return stops the loop before step t+1 is issued.  This costs
        one host sync per step; without `on_step` the loop issues exactly what it issued before."""
        main = torch.cuda.current_stream()
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream()
            f32 = dict(device=self.dev, dtype=torch.float32)
            self._stage = [(torch.zeros(self.B, self.ids_cols, device=self.dev, dtype=torch.int32), torch.zeros(self.B, max(self.n_dense, 1), **f32),
                            torch.zeros(self.B, **f32)) for _ in range(2)]
            self._stage_ready = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_free = [torch.cuda.Event(), torch.cuda.Event()]
        it = iter(batches)
        losses_host: List[torch.Tensor] = []
        sizes: List[int] = []
        pool: List[torch.Tensor] = []  # pinned read-back slots are carved from 256-float chunks kept across calls (pinning costs ~1 ms)
        if getattr(self, "_loss_pool", None) is None:
            self._loss_pool = []

        def upload(slot, batch):
            packed = batch if hasattr(batch, "views") else None  # lowering.HostBatch: a reusable pinned slot
            ids_h, dense_h, label_h, *weight_h = packed.views() if packed is not None else batch
            weight_h = weight_h[0] if weight_h else None
            B = ids_h.shape[0]
            if weight_h is not None and getattr(self, "_stage_w", None) is None:  # staged next to the label, from the first weighted batch
                self._stage_w = [torch.zeros(self.B, device=self.dev, dtype=torch.float32) for _ in range(2)]
            weighted[slot] = weight_h is not None
            with torch.cuda.stream(self._copy_stream):
                self._copy_stream.wait_event(self._stage_free[slot])  # the previous user of this slot has finished
                ids_d, dense_d, label_d = self._stage[slot]
                ids_d[:B].copy_(ids_h[:, : self.ids_cols], non_blocking=True)
                if self.n_dense:
                    dense_d[:B].copy_(dense_h[:, : self.n_dense], non_blocking=True)
                label_d[:B].copy_(label_h, non_blocking=True)
                if weight_h is not None:
                    self._stage_w[slot][:B].copy_(weight_h, non_blocking=True)
                self._stage_ready[slot].record(self._copy_stream)
                if packed is not None:  # the producer may refill the pinned slot once these copies have left it
                    packed.copied = torch.cuda.Event()
                    packed.copied.record(self._copy_stream)
            return B

        weighted = [False, False]
        for e in self._stage_free:
            e.record(main)
        nxt = next(it, None)
        slot = 0
        if nxt is not None:
            nB = upload(slot, nxt)
        step_done = torch.cuda.Event() if on_step is not None else None
        while nxt is not None:
            cur_slot, B = slot, nB
            if on_step is not None:
                on_step(len(losses_host), None)
            main.wait_event(self._stage_ready[cur_slot])
            ids_d, dense_d, label_d = self._stage[cur_slot]
            self.train_step_on_device(ids_d[:B], dense_d[:B] if self.n_dense else None, label_d[:B],
                                      self._stage_w[cur_slot][:B] if weighted[cur_slot] else None)
            self._stage_free[cur_slot].record(main)
            k = len(losses_host) % 256
            if k == 0:
                chunk = len(losses_host) // 256
                if chunk >= len(self._loss_pool):
                    self._loss_pool.append(torch.empty(256, dtype=torch.float32).pin_memory())
                pool.append(self._loss_pool[chunk])
            lh = pool[-1][k : k + 1]
            lh.copy_(self.loss_sum, non_blocking=True)  # D2H of this step's loss, not waited for here
            losses_host.append(lh)
            sizes.append(B)
            # the next batch is fetched AFTER this step has been issued: the GPU never waits for the producer of batch t+1 before it
            # may start batch t (the copy still overlaps step t: it only needs the other stage slot, free since step t-1)
            if on_step is not None:
                step_done.record(main)
            nxt = next(it, None)
            if nxt is not None:
                slot ^= 1
                nB = upload(slot, nxt)
            if on_step is not None:
                step_done.synchronize()
                if on_step(len(losses_host) - 1, float(lh[0]) / B):
                    break
        main.synchronize()
        return [float(l[0]) / b for l, b in zip(losses_host, sizes)]

    def predict(self, ids_host: torch.Tensor, dense_host: Optional[torch.Tensor], label_host: Optional[torch.Tensor] = None,
                metrics=None, weight_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Probabilities (task="regression": predictions) of one host batch; with `metrics` (a MetricSet) and the batch's labels,
        also counts them (one launch; with the batch's sample weights `weight_host`, the weighted update)."""
        B = ids_host.shape[0]
        self.ids_dev[:B].copy_(ids_host, non_blocking=True)
        if self.n_dense:
            self.dense_dev[:B].copy_(dense_host, non_blocking=True)
        weight = None
        if metrics is not None:
            self.label_dev[:B].copy_(label_host, non_blocking=True)
            weight = self._weights_to_device(weight_host, B)
        prob = self.predict_on_device(self.ids_dev[:B], self.dense_dev[:B] if self.n_dense else None)
        if metrics is not None:
            metrics.update(prob, self.label_dev[:B], weight)
        return prob.cpu().reshape(B, 1)

    def h2d_bytes_per_step(self, B: int) -> int:
        return B * (self.ids_cols * 4 + self.n_dense * 4 + 4)
