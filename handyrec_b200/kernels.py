"""Thin torch-tensor front end of the C ABI (include/hrb200.h).

PyTorch is used for device memory and streams only; every computation below is a call into
libhrb200.so on the current CUDA stream.  Nothing here computes on the CPU and nothing falls
back: tensors must be CUDA tensors, and a missing library raises (handyrec_b200._lib.lib).
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ACT, POOL, FieldDesc, OptParams, TableDesc, call

__all__ = [
    "init_uniform", "embedding_fwd", "embedding_bwd_dense", "seq_pool_fwd", "seq_pool_bwd", "LookupPlan",
    "fm_fwd", "fm_bwd", "dense_fwd", "dense_bwd_x", "dense_bwd_w", "act_bwd", "dice_fwd", "dice_bwd",
    "lau_fwd", "lau_pack_params", "sigmoid_bce", "regression_loss", "regression_loss_workspace", "adam_step", "sgd_step",
    "adam_step_multi", "sgd_step_multi",
    "adagrad_step", "adagrad_step_multi", "ftrl_step", "ftrl_step_multi", "metric_scratch_bytes", "metric_weighted_scratch_bytes",
    "metric_update",
    "clip_workspace", "clip_prepare_multi", "clip_scales", "clip_apply_multi",
]


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> ctypes.c_void_p:
    """The current torch stream of the current device as a raw cudaStream_t (called once per kernel launch: the raw getter
    costs ~0.3 us against ~8 us for building a torch.cuda.Stream object)."""
    if _raw_stream is not None:
        return ctypes.c_void_p(_raw_stream(torch.cuda.current_device()))
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _chk(t: torch.Tensor, dtype, name: str, contiguous: bool = True) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name} must be a CUDA tensor (handyrec_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if contiguous and not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def _row_major_2d(t: torch.Tensor, name: str) -> int:
    """Leading dimension of a 2-D row-major (possibly column-sliced) view."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"{name} must be a 2-D view with unit column stride")
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def init_uniform(table: torch.Tensor, seed: int, lo: float = -0.05, hi: float = 0.05, row_start: int = 0, row_step: int = 1) -> torch.Tensor:
    _chk(table, torch.float32, "table")
    call("hrb_init_uniform", _p(table), table.shape[0], table.shape[1], seed & 0xFFFFFFFF, lo, hi, row_start, row_step, _stream())
    return table


_oob_pending: Optional[list] = None  # a list while a `deferred_id_checks()` block is open


def _raise_if_oob(oob: torch.Tensor, what: str) -> None:
    if _oob_pending is not None:
        _oob_pending.append((oob, what))
        return
    flag = oob.tolist()
    if flag[0]:
        raise IndexError(f"{what}: id out of range (near flat sample index {flag[1]})")


class deferred_id_checks:
    """Reading a lookup's out-of-range flag is a host sync.  Inside this block the flags of all lookups are collected and read
    together when the block closes (one sync, normally shared with the step's loss read-back); an out-of-range id still raises
    IndexError from the same user call, only after the step's kernels have been issued (such a position reads as a zero row)."""

    def __enter__(self):
        global _oob_pending
        self.prev, _oob_pending = _oob_pending, []
        return self

    def __exit__(self, et, ev, tb):
        global _oob_pending
        pending, _oob_pending = _oob_pending, self.prev
        if et is None and pending:
            for flag, (_, what) in zip(torch.stack([o for o, _ in pending]).tolist(), pending):
                if flag[0]:
                    raise IndexError(f"{what}: id out of range (near flat sample index {flag[1]})")
        return False


# --------------------------------------------------------------------------------------------
# a5 / a13 (layer face)
# --------------------------------------------------------------------------------------------
def embedding_fwd(table: torch.Tensor, ids: torch.Tensor, mask_zero: bool, check_ids: bool = True):
    """layers/tools.py:87-101.  ids (...,) int32 -> out (..., D) fp32, mask (..., D) bool or None."""
    _chk(table, torch.float32, "table")
    _chk(ids, torch.int32, "ids")
    V, D = table.shape
    n = ids.numel()
    out = torch.empty(*ids.shape, D, device=table.device, dtype=torch.float32)
    mask = torch.empty(*ids.shape, D, device=table.device, dtype=torch.uint8) if mask_zero else None
    oob = torch.zeros(2, device=table.device, dtype=torch.int32) if check_ids else None
    call("hrb_embedding_fwd", _p(table), V, D, _p(ids), n, _p(out), _p(mask), _p(oob), _stream())
    if check_ids:
        _raise_if_oob(oob, "hrb_embedding_fwd")
    return out, (mask.view(torch.bool) if mask is not None else None)


def embedding_bwd_dense(ids: torch.Tensor, dout: torch.Tensor, vocab: int, table: Optional[torch.Tensor] = None, l2_scale: float = 0.0) -> torch.Tensor:
    _chk(ids, torch.int32, "ids")
    _chk(dout, torch.float32, "dout")
    D = dout.shape[-1]
    n = ids.numel()
    need = ctypes.c_size_t(0)
    call("hrb_embedding_bwd_dense_workspace", n, D, ctypes.byref(need))
    ws = torch.empty(need.value, device=dout.device, dtype=torch.uint8)
    dtable = torch.empty(vocab, D, device=dout.device, dtype=torch.float32)
    call("hrb_embedding_bwd_dense", _p(ids), n, _p(dout), vocab, D, _p(table), float(l2_scale), _p(dtable), _p(ws), need.value, _stream())
    return dtable


# --------------------------------------------------------------------------------------------
# a6 (layer face)
# --------------------------------------------------------------------------------------------
def _mask_u8(mask: torch.Tensor) -> torch.Tensor:
    if mask.dtype == torch.bool:
        mask = mask.view(torch.uint8)
    return _chk(mask, torch.uint8, "mask")


def seq_pool_fwd(x: torch.Tensor, mask: Optional[torch.Tensor], method: str) -> torch.Tensor:
    assert method in ["mean", "max", "sum"], "Pooling method should be `mean`, `max`, or `sum`"
    if mask is None:
        raise ValueError("Embedding layer should set `mask_zero` as True")
    _chk(x, torch.float32, "x")
    B, L, D = x.shape
    out = torch.empty(B, 1, D, device=x.device, dtype=torch.float32)
    call("hrb_seq_pool_fwd", _p(x), _p(_mask_u8(mask)), B, L, D, POOL[method], _p(out), _stream())
    return out


def seq_pool_bwd(x: torch.Tensor, mask: torch.Tensor, dout: torch.Tensor, method: str) -> torch.Tensor:
    _chk(x, torch.float32, "x")
    _chk(dout, torch.float32, "dout")
    B, L, D = x.shape
    dx = torch.empty_like(x)
    call("hrb_seq_pool_bwd", _p(x), _p(_mask_u8(mask)), _p(dout), B, L, D, POOL[method], _p(dx), _stream())
    return dx


# --------------------------------------------------------------------------------------------
# a7 / a13 fused plan
# --------------------------------------------------------------------------------------------
class LookupPlan:
    """Device plan of one feature group: tables + (table, seq_len, pool, ids_col, out_col) per field.

    Optimiser state per table (None entries for tables without): `adam_m` / `adam_v` for lazy Adam, `accum` for Adagrad, or
    `accum` and `linear` for Ftrl (they take the ABI's adam_m / adam_v slots, so they cannot be given with the Adam moments)."""

    def __init__(self, tables: Sequence[torch.Tensor], fields: Sequence[Tuple[int, int, str, int, int]],
                 adam_m: Optional[Sequence[torch.Tensor]] = None, adam_v: Optional[Sequence[torch.Tensor]] = None,
                 accum: Optional[Sequence[torch.Tensor]] = None, linear: Optional[Sequence[torch.Tensor]] = None):
        self.tables = [_chk(t, torch.float32, "table") for t in tables]
        if accum is not None:
            if adam_m is not None:
                raise ValueError("LookupPlan: pass either adam_m (Adam) or accum (Adagrad / Ftrl), not both")
            adam_m = accum
        if linear is not None:
            if adam_v is not None:
                raise ValueError("LookupPlan: pass either adam_v (Adam) or linear (Ftrl), not both")
            adam_v = linear
        self.adam_m = list(adam_m) if adam_m is not None else None
        self.adam_v = list(adam_v) if adam_v is not None else None
        self.fields = [tuple(f) for f in fields]
        self.n_fields = len(self.fields)
        self.device = self.tables[0].device
        td = (TableDesc * len(self.tables))()
        for i, t in enumerate(self.tables):
            td[i].weight = t.data_ptr()
            td[i].adam_m = self.adam_m[i].data_ptr() if self.adam_m is not None and self.adam_m[i] is not None else 0
            td[i].adam_v = self.adam_v[i].data_ptr() if self.adam_v is not None and self.adam_v[i] is not None else 0
            td[i].rows, td[i].dim = t.shape[0], t.shape[1]
        fd = (FieldDesc * self.n_fields)()
        self.ids_cols = 0
        self.out_cols = 0
        self.pos_cols = 0
        for i, (ti, L, pool, ids_col, out_col) in enumerate(self.fields):
            fd[i].table, fd[i].seq_len, fd[i].pool, fd[i].ids_col, fd[i].out_col = ti, L, POOL[pool], ids_col, out_col
            self.ids_cols = max(self.ids_cols, ids_col + L)
            self.out_cols = max(self.out_cols, out_col + self.tables[ti].shape[1])
            self.pos_cols += L
        self._h = ctypes.c_void_p(0)
        with torch.cuda.device(self.device):
            call("hrb_plan_create", td, len(self.tables), fd, self.n_fields, ctypes.byref(self._h))
        self._ws = None

    def set_dense_grads(self, grads: Sequence[Optional[torch.Tensor]]) -> None:
        """grads[t] (rows, dim) fp32 or None: the backward ADDS table t's row-gradient sums there instead of updating the rows."""
        assert len(grads) == len(self.tables)
        self._dense_grads = list(grads)  # keep the buffers alive
        arr = (ctypes.c_void_p * len(grads))(*[(g.data_ptr() if g is not None else None) for g in grads])
        call("hrb_plan_set_dense_grads", self._h, arr)

    def mark_rows(self, ids: torch.Tensor, touched: Sequence[Optional[torch.Tensor]]) -> None:
        """touched[t] (rows,) fp32 or None: store 1.0 at every row of table t that the batch names (every in-range id of a plain
        field, every position of a pooled field, padding id 0 included) -- the rows Keras' IndexedSlices gradient lists."""
        assert len(touched) == len(self.tables)
        ids_ld = self._ids_ld(ids)
        for t in touched:
            if t is not None:
                _chk(t, torch.float32, "touched")
        arr = (ctypes.c_void_p * len(touched))(*[(t.data_ptr() if t is not None else None) for t in touched])
        call("hrb_plan_mark_rows", self._h, _p(ids), ids_ld, ids.shape[0], arr, _stream())

    def pad_flags(self, ids: torch.Tensor, flags: torch.Tensor) -> None:
        """flags (2 * n_tables,) fp32, caller-zeroed: flags[2t] = 1 where a pooled field of table t holds padding, flags[2t+1] = 1
        where a valid position names row 0 of table t (hrb_plan_pad_flags)."""
        _chk(flags, torch.float32, "flags")
        call("hrb_plan_pad_flags", self._h, _p(ids), self._ids_ld(ids), ids.shape[0], _p(flags), _stream())

    def ftrl_pad_step(self, flags: torch.Tensor, op: OptParams) -> None:
        """Row 0 of every row-updated table whose flags show padding and no valid id 0 takes its zero-gradient Ftrl step."""
        call("hrb_plan_ftrl_pad_step", self._h, _p(flags), ctypes.byref(op), _stream())

    def clip_grads(self, ids: torch.Tensor, dx: torch.Tensor, fm: Optional[torch.Tensor], clipvalue: float,
                   sumsq: Optional[torch.Tensor], workspace: torch.Tensor) -> None:
        """hrb_plan_clip_grads: the DNN part (dx, the plan's column layout) and the FM part (fm, field f at column out_col_f -
        out_col_0) of every field's gradient clamped per position, dx <- their sum; sumsq[t] += the table's squared norm."""
        B = ids.shape[0]
        dx_ld = _row_major_2d(_chk(dx, torch.float32, "dx", contiguous=False), "dx")
        fm_ld = _row_major_2d(_chk(fm, torch.float32, "fm", contiguous=False), "fm") if fm is not None else 0
        if sumsq is not None:
            _chk(sumsq, torch.float32, "sumsq")
        call("hrb_plan_clip_grads", self._h, _p(ids), self._ids_ld(ids), B, _p(dx), dx_ld, _p(fm), fm_ld, float(clipvalue), _p(sumsq),
             _p(workspace), workspace.numel(), _stream())

    def clip_apply(self, dx: torch.Tensor, batch: int, scale: torch.Tensor) -> None:
        """hrb_plan_clip_apply: dx[:, columns of field f] *= scale[table of f]."""
        dx_ld = _row_major_2d(_chk(dx, torch.float32, "dx", contiguous=False), "dx")
        call("hrb_plan_clip_apply", self._h, _p(dx), dx_ld, batch, _p(_chk(scale, torch.float32, "scale")), _stream())

    def __del__(self):
        try:  # module globals may already be gone at interpreter shutdown
            h = getattr(self, "_h", None)
            if h is not None and h.value:
                _lib.lib().hrb_plan_destroy(h)
                self._h = None
        except Exception:
            pass

    def _ids_ld(self, ids: torch.Tensor) -> int:
        _chk(ids, torch.int32, "ids", contiguous=False)
        return _row_major_2d(ids, "ids")

    def forward(self, ids: torch.Tensor, out: Optional[torch.Tensor] = None, want_inv_count: bool = False,
                check_ids: bool = False, fm: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, want_fm_sum: bool = False):
        """ids (B, >=ids_cols) int32 -> out (B, >=out_cols).  With fm=(w (D,1|D), w0 (1,)) also the FM logit (B,)."""
        B = ids.shape[0]
        ids_ld = self._ids_ld(ids)
        if out is None:
            out = torch.empty(B, self.out_cols, device=self.device, dtype=torch.float32)
        out_ld = _row_major_2d(_chk(out, torch.float32, "out", contiguous=False), "out")
        inv = torch.empty(B, self.n_fields, device=self.device, dtype=torch.float32) if want_inv_count else None
        oob = torch.zeros(2, device=self.device, dtype=torch.int32) if check_ids else None
        res = {"out": out, "inv_count": inv}
        if fm is None:
            call("hrb_lookup_fwd", self._h, _p(ids), ids_ld, B, _p(out), out_ld, _p(inv), _p(oob), _stream())
        else:
            w, w0 = fm
            D = self.tables[0].shape[1]
            fm_out = torch.empty(B, device=self.device, dtype=torch.float32)
            fm_sum = torch.empty(B, D, device=self.device, dtype=torch.float32) if want_fm_sum else None
            call("hrb_lookup_fm_fwd", self._h, _p(ids), ids_ld, B, _p(out), out_ld, _p(inv), _p(w), _p(w0), _p(fm_out), _p(fm_sum), _p(oob), _stream())
            res["fm_out"], res["fm_sum"] = fm_out, fm_sum
        if check_ids:
            _raise_if_oob(oob, "hrb_lookup_fwd")
        return res

    def workspace_bytes(self, batch: int) -> int:
        need = ctypes.c_size_t(0)
        call("hrb_lookup_bwd_workspace", self._h, self.ids_cols, batch, ctypes.byref(need))
        return need.value

    def backward_update(self, ids: torch.Tensor, dout: torch.Tensor, opt: str = "sgd", lr: float = 0.01, l2_scale: float = 0.0,
                        beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-7, step: int = 1,
                        workspace: Optional[torch.Tensor] = None, autotune: bool = False, l1: float = 0.0, l2: float = 0.0,
                        lr_power: float = -0.5, l2_shrinkage: float = 0.0) -> None:
        """Segment-reduce the gradient rows per table row and update the touched rows of every table in place.

        opt: "sgd", "adam" (lazy Adam: beta1, beta2, eps, step), "adagrad" (eps; the plan's `accum`) or "ftrl" (l1, l2 with
        Keras' beta / (2*lr) added, lr_power, l2_shrinkage; the plan's `accum` and `linear`)."""
        B = ids.shape[0]
        ids_ld = self._ids_ld(ids)
        dout_ld = _row_major_2d(_chk(dout, torch.float32, "dout", contiguous=False), "dout")
        need = self.workspace_bytes(B)
        if workspace is None:
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(need, device=self.device, dtype=torch.uint8)
            workspace = self._ws
        op = OptParams()
        op.opt = {"sgd": _lib.OPT_SGD, "adagrad": _lib.OPT_ADAGRAD, "ftrl": _lib.OPT_FTRL}.get(opt, _lib.OPT_ADAM_LAZY)
        op.lr, op.beta1, op.beta2, op.eps, op.l2_scale = lr, beta1, beta2, eps, l2_scale
        op.bias_corr1, op.bias_corr2 = 1.0 - beta1 ** step, 1.0 - beta2 ** step
        op.l1, op.l2, op.lr_power, op.l2_shrinkage = l1, l2, lr_power, l2_shrinkage
        trial = self._next_bwd_trial(B) if autotune else None
        if trial is not None:
            call("hrb_plan_set_bwd_algo", self._h, _lib.BWD_UNITS if trial == "units" else _lib.BWD_SORT)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        call("hrb_lookup_bwd_update", self._h, _p(ids), ids_ld, B, _p(dout), dout_ld, None, ctypes.byref(op), _p(workspace), workspace.numel(), _stream())
        if trial is not None:
            e1.record()
            e1.synchronize()
            self._finish_bwd_trial(trial, e0.elapsed_time(e1))

    # Which implementation of the backward is faster depends on the ids (uniform: the partition path; a few rows collecting most
    # positions: the sorted path with its run-time long-row pass).  With autotune=True calls 3..6 of a plan at one batch size time
    # both (two trials each, one host sync per trial) and the faster one is kept; both give the same result to rounding.
    _bwd_trial_log = None
    bwd_algo = "auto"

    def _next_bwd_trial(self, B: int) -> Optional[str]:
        if self.bwd_algo != "auto":
            return None
        if self._bwd_trial_log is None or self._bwd_trial_log["B"] != B:
            self._bwd_trial_log = {"B": B, "calls": 0, "units": [], "sort": []}
        log = self._bwd_trial_log
        log["calls"] += 1
        if log["calls"] <= 2:
            return None
        return "units" if len(log["units"]) <= len(log["sort"]) else "sort"

    def _finish_bwd_trial(self, trial: str, ms: float) -> None:
        log = self._bwd_trial_log
        log[trial].append(ms)
        if len(log["units"]) >= 2 and len(log["sort"]) >= 2:
            self.bwd_algo = "units" if min(log["units"]) <= min(log["sort"]) else "sort"
            self.bwd_algo_ms = {"units": min(log["units"]), "sort": min(log["sort"])}
            call("hrb_plan_set_bwd_algo", self._h, _lib.BWD_UNITS if self.bwd_algo == "units" else _lib.BWD_SORT)


# --------------------------------------------------------------------------------------------
# a9 FM
# --------------------------------------------------------------------------------------------
def fm_fwd(x: torch.Tensor, w: torch.Tensor, w0: torch.Tensor, want_sum: bool = False):
    """x (B,F,D) (row stride may exceed F*D) -> (B,1)."""
    _chk(x, torch.float32, "x", contiguous=False)
    B, F, D = x.shape
    if x.stride(2) != 1 or x.stride(1) != D:
        raise ValueError("x must be a (B,F,D) view with contiguous (F,D) blocks")
    x_ld = x.stride(0) if B > 1 else F * D
    out = torch.empty(B, 1, device=x.device, dtype=torch.float32)
    s = torch.empty(B, D, device=x.device, dtype=torch.float32) if want_sum else None
    call("hrb_fm_fwd", _p(x), x_ld, B, F, D, _p(w), _p(w0), _p(out), _p(s), _stream())
    return (out, s) if want_sum else out


def fm_bwd(x: torch.Tensor, w: torch.Tensor, dout: torch.Tensor, dx: Optional[torch.Tensor] = None, accumulate: bool = False):
    B, F, D = x.shape
    x_ld = x.stride(0) if B > 1 else F * D
    if dx is None:
        dx = torch.empty(B, F, D, device=x.device, dtype=torch.float32)
        accumulate = False
    dx_ld = dx.stride(0) if B > 1 else F * D
    dwb = torch.empty(D + 1, device=x.device, dtype=torch.float32)
    call("hrb_fm_bwd", _p(x), x_ld, B, F, D, _p(w), _p(dout), _p(dx), dx_ld, int(accumulate), _p(dwb), _stream())
    return dx, dwb[:D].reshape(D, 1), dwb[D:]


# --------------------------------------------------------------------------------------------
# a11 Dense / Dice
# --------------------------------------------------------------------------------------------
def dense_fwd(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], act: Optional[str] = None,
              out: Optional[torch.Tensor] = None, mode: int = _lib.GEMM_AUTO) -> torch.Tensor:
    M, K = x.shape
    N = w.shape[1]
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=torch.float32)
    call("hrb_dense_fwd", _p(x), _row_major_2d(x, "x"), _p(w), _row_major_2d(w, "w"), _p(bias), M, K, N, ACT[act], _p(out), _row_major_2d(out, "out"), mode, _stream())
    return out


def dense_bwd_x(dz: torch.Tensor, w: torch.Tensor, a_prev: Optional[torch.Tensor] = None, act_prev: Optional[str] = None,
                out: Optional[torch.Tensor] = None, mode: int = _lib.GEMM_AUTO) -> torch.Tensor:
    M, N = dz.shape
    K = w.shape[0]
    if out is None:
        out = torch.empty(M, K, device=dz.device, dtype=torch.float32)
    call("hrb_dense_bwd_x", _p(dz), _row_major_2d(dz, "dz"), _p(w), _row_major_2d(w, "w"), M, K, N, _p(a_prev),
         _row_major_2d(a_prev, "a_prev") if a_prev is not None else 0, ACT[act_prev], _p(out), _row_major_2d(out, "out"), mode, _stream())
    return out


_dense_ws = {}


def dense_bwd_w(x: torch.Tensor, dz: torch.Tensor, dw: Optional[torch.Tensor] = None, dbias: Optional[torch.Tensor] = None,
                want_bias: bool = True, mode: int = _lib.GEMM_AUTO):
    M, K = x.shape
    N = dz.shape[1]
    need = ctypes.c_size_t(0)
    call("hrb_dense_bwd_w_workspace", M, K, N, ctypes.byref(need))
    key = (x.device.index, _stream().value)
    ws = _dense_ws.get(key)
    if ws is None or ws.numel() < need.value:
        ws = torch.empty(need.value, device=x.device, dtype=torch.uint8)
        _dense_ws[key] = ws
    if dw is None:
        dw = torch.empty(K, N, device=x.device, dtype=torch.float32)
    if dbias is None and want_bias:
        dbias = torch.empty(N, device=x.device, dtype=torch.float32)
    call("hrb_dense_bwd_w", _p(x), _row_major_2d(x, "x"), _p(dz), _row_major_2d(dz, "dz"), M, K, N, _p(dw), _row_major_2d(dw, "dw"), _p(dbias), _p(ws), ws.numel(), mode, _stream())
    return dw, dbias


def act_bwd(y: torch.Tensor, dy: torch.Tensor, act: Optional[str]) -> torch.Tensor:
    dz = torch.empty_like(dy)
    call("hrb_act_bwd", _p(y.contiguous()), _p(dy.contiguous()), dy.numel(), ACT[act], _p(dz), _stream())
    return dz


def dice_fwd(x: torch.Tensor, alpha: torch.Tensor, mean: torch.Tensor, var: torch.Tensor, training: bool, eps: float = 1e-9):
    """layers/activation.py:27-42.  training=True overwrites mean/var with the batch statistics."""
    units = x.shape[-1]
    rows = x.numel() // units
    y = torch.empty_like(x)
    call("hrb_dice_fwd", _p(_chk(x, torch.float32, "x")), rows, units, _p(alpha), _p(mean), _p(var), eps, int(training), _p(y), _stream())
    return y


def dice_bwd(x: torch.Tensor, dy: torch.Tensor, alpha: torch.Tensor, mean: torch.Tensor, var: torch.Tensor, training: bool, eps: float = 1e-9):
    units = x.shape[-1]
    rows = x.numel() // units
    dx = torch.empty_like(x)
    dalpha = torch.empty(units, device=x.device, dtype=torch.float32)
    scratch = torch.empty(2 * units, device=x.device, dtype=torch.float32)
    call("hrb_dice_bwd", _p(x), _p(_chk(dy, torch.float32, "dy")), rows, units, _p(alpha), _p(mean), _p(var), eps, int(training), _p(dx), _p(dalpha), _p(scratch), _stream())
    return dx, dalpha


# --------------------------------------------------------------------------------------------
# a10 LAU
# --------------------------------------------------------------------------------------------
def lau_pack_params(Ws: Sequence[torch.Tensor], bs: Sequence[torch.Tensor], dice: Optional[Sequence[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]] = None) -> torch.Tensor:
    """Pack [W_i, b_i, (alpha_i, mean_i, var_i)] back to back, padded to 4 floats per layer (hrb200.h a10)."""
    chunks: List[torch.Tensor] = []
    n = len(Ws)
    total = 0
    for i, (W, b) in enumerate(zip(Ws, bs)):
        parts = [W.reshape(-1), b.reshape(-1)]
        if dice is not None and i != n - 1:
            parts += [t.reshape(-1) for t in dice[i]]
        for p in parts:
            chunks.append(p.to(torch.float32))
            total += p.numel()
        pad = (-total) % 4
        if pad:
            chunks.append(torch.zeros(pad, device=Ws[0].device, dtype=torch.float32))
            total += pad
    return torch.cat(chunks).contiguous()


def lau_fwd(table: torch.Tensor, query_ids: torch.Tensor, key_ids: torch.Tensor, params: torch.Tensor, layer_out: Sequence[int],
            act: Optional[str], want_pooled: bool = True):
    """-> score (B,1,T), pooled (B,1,D)."""
    V, D = table.shape
    B, T = key_ids.shape
    score = torch.empty(B, 1, T, device=table.device, dtype=torch.float32)
    pooled = torch.empty(B, 1, D, device=table.device, dtype=torch.float32) if want_pooled else None
    lo = (ctypes.c_int32 * len(layer_out))(*layer_out)
    call("hrb_lau_fwd", _p(table), V, D, _p(_chk(query_ids, torch.int32, "query_ids")), _p(_chk(key_ids, torch.int32, "key_ids")), B, T,
         _p(params), lo, len(layer_out), ACT[act], _p(score), _p(pooled), _stream())
    return score, pooled


# --------------------------------------------------------------------------------------------
# head / optimisers
# --------------------------------------------------------------------------------------------
def sigmoid_bce(dnn_logit: torch.Tensor, fm_logit: Optional[torch.Tensor], label: torch.Tensor, grad_scale: float,
                prob: Optional[torch.Tensor] = None, dlogit: Optional[torch.Tensor] = None, loss_sum: Optional[torch.Tensor] = None,
                weight: Optional[torch.Tensor] = None):
    """With `weight` (one fp32 per sample): Keras' weighted loss, loss_sum += w*l and dlogit = (p-y)*w*grad_scale."""
    B = dnn_logit.numel()
    if weight is None:
        call("hrb_sigmoid_bce", _p(dnn_logit), _p(fm_logit), _p(label), B, grad_scale, _p(prob), _p(dlogit), _p(loss_sum), _stream())
    else:
        if _chk(weight, torch.float32, "weight").numel() != B:
            raise ValueError(f"sigmoid_bce: {weight.numel()} weights for {B} samples")
        call("hrb_sigmoid_bce_weighted", _p(dnn_logit), _p(fm_logit), _p(label), _p(weight), B, grad_scale, _p(prob), _p(dlogit),
             _p(loss_sum), _stream())


REG_LOSS = {"mean_squared_error": 0, "mean_absolute_error": 1, "huber": 2}  # hrb_regression_loss's `loss`


def regression_loss_workspace(n: int, device) -> torch.Tensor:
    """A zeroed workspace for hrb_regression_loss over n elements (it stays zeroed between calls)."""
    nb = ctypes.c_size_t(0)
    call("hrb_regression_loss_workspace", n, ctypes.byref(nb))
    return torch.zeros(nb.value, device=device, dtype=torch.uint8)


def regression_loss(loss: str, delta: float, a: torch.Tensor, b: Optional[torch.Tensor], label: Optional[torch.Tensor], batch: int,
                    cols: int, grad_scale: float, pred: Optional[torch.Tensor] = None, dpred: Optional[torch.Tensor] = None,
                    loss_sum: Optional[torch.Tensor] = None, weight: Optional[torch.Tensor] = None,
                    workspace: Optional[torch.Tensor] = None):
    """Keras MSE / MAE / Huber of pred = a (+ b) over the first batch * cols elements: loss_sum = sum(w * l) (l the mean over cols),
    dpred = dl/dpred * w * grad_scale / cols.  `weight`: one fp32 per sample, or None."""
    ws = (_p(workspace), workspace.numel()) if workspace is not None else (None, 0)
    if weight is None:
        call("hrb_regression_loss", REG_LOSS[loss], delta, _p(a), _p(b), _p(label), batch, cols, grad_scale, _p(pred), _p(dpred), _p(loss_sum),
             *ws, _stream())
    else:
        if _chk(weight, torch.float32, "weight").numel() != batch:
            raise ValueError(f"{loss}: {weight.numel()} sample weights for {batch} samples")
        call("hrb_regression_loss_weighted", REG_LOSS[loss], delta, _p(a), _p(b), _p(label), _p(weight), batch, cols, grad_scale, _p(pred),
             _p(dpred), _p(loss_sum), *ws, _stream())


def adam_step(param, grad, m, v, lr, beta1=0.9, beta2=0.999, eps=1e-7, step=1, l2_scale=0.0):
    call("hrb_adam_step", _p(param), _p(grad), _p(m), _p(v), param.numel(), lr, beta1, beta2, eps, 1.0 - beta1 ** step, 1.0 - beta2 ** step, l2_scale, _stream())


def sgd_step(param, grad, lr, l2_scale=0.0):
    call("hrb_sgd_step", _p(param), _p(grad), param.numel(), lr, l2_scale, _stream())


def adagrad_step(param, grad, acc, lr, eps=1e-7, l2_scale=0.0):
    call("hrb_adagrad_step", _p(param), _p(grad), _p(acc), param.numel(), lr, eps, l2_scale, _stream())


def ftrl_step(param, grad, acc, lin, lr, l1=0.0, l2=0.0, lr_power=-0.5, l2_shrinkage=0.0, l2_scale=0.0, row_touched=None, dim=0):
    """Keras Ftrl over every element (l2 with beta / (2*lr) added); with row_touched (one float per row of `dim` elements) the
    rows flagged 0 keep their bits."""
    if row_touched is not None:
        _chk(row_touched, torch.float32, "row_touched")
    call("hrb_ftrl_step", _p(param), _p(grad), _p(acc), _p(lin), param.numel(), lr, l1, l2, lr_power, l2_shrinkage, l2_scale,
         _p(row_touched), dim, _stream())


def _ptr_array(tensors):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def adam_step_multi(params, grads, ms, vs, l2_scales, lr, beta1=0.9, beta2=0.999, eps=1e-7, step=1):
    """hrb_adam_step for a list of tensors in one launch (per HRB_MULTI_MAX tensors)."""
    n = len(params)
    if n == 0:
        return
    for t in list(params) + list(grads) + list(ms) + list(vs):
        _chk(t, torch.float32, "tensor")
    call("hrb_adam_step_multi", n, _ptr_array(params), _ptr_array(grads), _ptr_array(ms), _ptr_array(vs),
         (ctypes.c_int64 * n)(*[p.numel() for p in params]), (ctypes.c_float * n)(*l2_scales), lr, beta1, beta2, eps,
         1.0 - beta1 ** step, 1.0 - beta2 ** step, _stream())


def sgd_step_multi(params, grads, l2_scales, lr):
    n = len(params)
    if n == 0:
        return
    for t in list(params) + list(grads):
        _chk(t, torch.float32, "tensor")
    call("hrb_sgd_step_multi", n, _ptr_array(params), _ptr_array(grads), (ctypes.c_int64 * n)(*[p.numel() for p in params]),
         (ctypes.c_float * n)(*l2_scales), lr, _stream())


def adagrad_step_multi(params, grads, accs, l2_scales, lr, eps=1e-7):
    """hrb_adagrad_step for a list of tensors in one launch (per HRB_MULTI_MAX tensors)."""
    n = len(params)
    if n == 0:
        return
    for t in list(params) + list(grads) + list(accs):
        _chk(t, torch.float32, "tensor")
    call("hrb_adagrad_step_multi", n, _ptr_array(params), _ptr_array(grads), _ptr_array(accs),
         (ctypes.c_int64 * n)(*[p.numel() for p in params]), (ctypes.c_float * n)(*l2_scales), lr, eps, _stream())


def ftrl_step_multi(params, grads, accs, lins, l2_scales, lr, l1=0.0, l2=0.0, lr_power=-0.5, l2_shrinkage=0.0):
    """hrb_ftrl_step for a list of tensors in one launch (per HRB_MULTI_MAX tensors), every element stepping."""
    n = len(params)
    if n == 0:
        return
    for t in list(params) + list(grads) + list(accs) + list(lins):
        _chk(t, torch.float32, "tensor")
    call("hrb_ftrl_step_multi", n, _ptr_array(params), _ptr_array(grads), _ptr_array(accs), _ptr_array(lins),
         (ctypes.c_int64 * n)(*[p.numel() for p in params]), (ctypes.c_float * n)(*l2_scales), lr, l1, l2, lr_power, l2_shrinkage,
         _stream())


# --------------------------------------------------------------------------------------------
# gradient clipping (Keras OptimizerV2 clipvalue / clipnorm / global_clipnorm), in place
# --------------------------------------------------------------------------------------------
def clip_workspace(n_tables: int, device) -> torch.Tensor:
    """A zeroed workspace for the clip entries (every call leaves it zeroed; calls sharing it must be stream-ordered)."""
    need = ctypes.c_size_t(0)
    call("hrb_clip_workspace_bytes", int(n_tables), ctypes.byref(need))
    return torch.zeros(need.value, device=device, dtype=torch.uint8)


def clip_prepare_multi(grads: Sequence[torch.Tensor], weights: Optional[Sequence[Optional[torch.Tensor]]], l2_scales: Optional[Sequence[float]],
                       var: Sequence[int], clipvalue: float, sumsq: Optional[torch.Tensor], workspace: torch.Tensor) -> None:
    """hrb_clip_prepare_multi: g <- clamp(g + l2_scale * w, -clipvalue, clipvalue) in place; sumsq[var[i]] += sum g^2."""
    n = len(grads)
    if n == 0:
        return
    for t in grads:
        _chk(t, torch.float32, "grad")
    if sumsq is not None:
        _chk(sumsq, torch.float32, "sumsq")
    w = None if weights is None else (ctypes.c_void_p * n)(*[(t.data_ptr() if t is not None else None) for t in weights])
    call("hrb_clip_prepare_multi", n, _ptr_array(grads), w, (ctypes.c_int64 * n)(*[g.numel() for g in grads]),
         None if l2_scales is None else (ctypes.c_float * n)(*l2_scales), (ctypes.c_int32 * n)(*var), float(clipvalue), _p(sumsq),
         _p(workspace), workspace.numel(), _stream())


def clip_scales(sumsq: torch.Tensor, clipnorm: float, global_norm: bool, scale: torch.Tensor) -> None:
    """hrb_clip_scales: scale[k] = c / max(||g_k||, c), or one scale from the global norm (NaN when it is not finite)."""
    _chk(sumsq, torch.float32, "sumsq")
    _chk(scale, torch.float32, "scale")
    call("hrb_clip_scales", _p(sumsq), sumsq.numel(), float(clipnorm), int(global_norm), _p(scale), _stream())


def clip_apply_multi(grads: Sequence[torch.Tensor], var: Sequence[int], scale: torch.Tensor) -> None:
    """hrb_clip_apply_multi: g *= scale[var[i]] in place."""
    n = len(grads)
    if n == 0:
        return
    for t in grads:
        _chk(t, torch.float32, "grad")
    call("hrb_clip_apply_multi", n, _ptr_array(grads), (ctypes.c_int64 * n)(*[g.numel() for g in grads]), (ctypes.c_int32 * n)(*var),
         _p(_chk(scale, torch.float32, "scale")), _stream())


# --------------------------------------------------------------------------------------------
# tcgen05 "TN" Dense variants (3xTF32): every operand has its reduction dim contiguous
# --------------------------------------------------------------------------------------------
def transpose(src: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    rows, cols = src.shape
    if out is None:
        out = torch.empty(cols, rows, device=src.device, dtype=torch.float32)
    call("hrb_transpose", _p(src), rows, cols, _row_major_2d(src, "src"), _p(out), _row_major_2d(out, "out"), _stream())
    return out


def dense_fwd_t(x, wt, bias, act=None, out=None, out_t=None, relu_mask=None):
    """y = act(x @ wt.T + bias); wt is (N, K).  out_t (N, M) optionally receives y^T."""
    M, Kd = x.shape
    N = wt.shape[0]
    if out is None:
        out = torch.empty(M, N, device=x.device, dtype=torch.float32)
    call("hrb_dense_fwd_t", _p(x), _row_major_2d(x, "x"), _p(wt), _row_major_2d(wt, "wt"), _p(bias), M, Kd, N, ACT[act], _p(out),
         _row_major_2d(out, "out"), _p(out_t), _row_major_2d(out_t, "out_t") if out_t is not None else 0, _p(relu_mask), _stream())
    return out


def dense_bwd_x_t(dz, w, a_prev=None, act_prev=None, out=None, out_t=None, relu_mask=None):
    """dx = (dz @ w.T) * act'(a_prev); w is (K, N) row-major as in the forward."""
    M, N = dz.shape
    Kd = w.shape[0]
    if out is None:
        out = torch.empty(M, Kd, device=dz.device, dtype=torch.float32)
    call("hrb_dense_bwd_x_t", _p(dz), _row_major_2d(dz, "dz"), _p(w), _row_major_2d(w, "w"), M, Kd, N, _p(a_prev),
         _row_major_2d(a_prev, "a_prev") if a_prev is not None else 0, ACT[act_prev], _p(relu_mask), _p(out), _row_major_2d(out, "out"), _p(out_t),
         _row_major_2d(out_t, "out_t") if out_t is not None else 0, _stream())
    return out


def dense_bwd_w_t(xt, dzt, dz=None, dw=None, dbias=None):
    """dw (K, N) = xt (K, M) @ dzt (N, M).T ; dbias = column sums of dz (M, N)."""
    Kd, M = xt.shape
    N = dzt.shape[0]
    need = ctypes.c_size_t(0)
    call("hrb_dense_bwd_w_t_workspace", M, Kd, N, ctypes.byref(need))
    key = ("t", xt.device.index, _stream().value)
    ws = _dense_ws.get(key)
    if ws is None or ws.numel() < need.value:
        ws = torch.empty(need.value, device=xt.device, dtype=torch.uint8)
        _dense_ws[key] = ws
    if dw is None:
        dw = torch.empty(Kd, N, device=xt.device, dtype=torch.float32)
    if dbias is None and dz is not None:
        dbias = torch.empty(N, device=xt.device, dtype=torch.float32)
    call("hrb_dense_bwd_w_t", _p(xt), _row_major_2d(xt, "xt"), _p(dzt), _row_major_2d(dzt, "dzt"), _p(dz),
         _row_major_2d(dz, "dz") if dz is not None else 0, M, Kd, N, _p(dw), _row_major_2d(dw, "dw"), _p(dbias), _p(ws), ws.numel(), _stream())
    return dw, dbias


def dense_bwd_w_xn(x, dzt, dw=None, want_bias=True):
    """dw (K, N) = x (M, K).T @ dz with dz given transposed (dzt (N, M)); x is read as stored, no x^T copy.  dbias = row sums of dzt."""
    M, Kd = x.shape
    N = dzt.shape[0]
    need = ctypes.c_size_t(0)
    call("hrb_dense_bwd_w_t_workspace", M, Kd, N, ctypes.byref(need))
    key = ("t", x.device.index, _stream().value)
    ws = _dense_ws.get(key)
    if ws is None or ws.numel() < need.value:
        ws = torch.empty(need.value, device=x.device, dtype=torch.uint8)
        _dense_ws[key] = ws
    if dw is None:
        dw = torch.empty(Kd, N, device=x.device, dtype=torch.float32)
    dbias = torch.empty(N, device=x.device, dtype=torch.float32) if want_bias else None
    call("hrb_dense_bwd_w_xn", _p(x), _row_major_2d(x, "x"), _p(dzt), _row_major_2d(dzt, "dzt"), M, Kd, N, _p(dw), _row_major_2d(dw, "dw"),
         _p(dbias), _p(ws), ws.numel(), _stream())
    return dw, dbias


def dense1_fwd(x, w, bias, out=None):
    """The 1-unit logit layer: y (M,) = x (M,K) @ w (K,) + bias."""
    M, Kd = x.shape
    if out is None:
        out = torch.empty(M, 1, device=x.device, dtype=torch.float32)
    call("hrb_dense1_fwd", _p(x), _row_major_2d(x, "x"), _p(w), _p(bias), M, Kd, _p(out), _stream())
    return out


def dense1_bwd(x, w, dy, act_prev=None, want_t=False):
    M, Kd = x.shape
    need = ctypes.c_size_t(0)
    call("hrb_dense1_bwd_workspace", M, Kd, ctypes.byref(need))
    ws = torch.empty(need.value, device=x.device, dtype=torch.uint8)
    ld = (Kd + 3) // 4 * 4
    dz = torch.zeros(M, ld, device=x.device, dtype=torch.float32)
    dzt = torch.zeros(ld, M, device=x.device, dtype=torch.float32) if want_t else None
    dw = torch.empty(Kd, device=x.device, dtype=torch.float32)
    db = torch.empty(1, device=x.device, dtype=torch.float32)
    call("hrb_dense1_bwd", _p(x), _row_major_2d(x, "x"), _p(w), _p(dy), M, Kd, ACT[act_prev], _p(dz), ld, _p(dzt), M, _p(dw), _p(db), _p(ws), ws.numel(), _stream())
    return dz[:, :Kd], (dzt[:Kd] if want_t else None), dw, db


# --------------------------------------------------------------------------------------------
# Keras metrics: confusion / accuracy variables counted on the device (one launch per update)
# --------------------------------------------------------------------------------------------
METRIC_TP, METRIC_FP, METRIC_TN, METRIC_FN, METRIC_CORRECT, METRIC_COUNT = 0, 1, 2, 3, 4, 5
METRIC_WTP, METRIC_WFP, METRIC_WTN, METRIC_WFN, METRIC_WCORRECT, METRIC_WCOUNT = 6, 7, 8, 9, 10, 11
METRIC_MAX_THRESHOLDS = 8192


def metric_scratch_bytes(n_thr: int) -> int:
    need = ctypes.c_size_t(0)
    call("hrb_metric_scratch_bytes", int(n_thr), ctypes.byref(need))
    return need.value


def metric_weighted_scratch_bytes(n_thr: int) -> int:
    need = ctypes.c_size_t(0)
    call("hrb_metric_weighted_scratch_bytes", int(n_thr), ctypes.byref(need))
    return need.value


def metric_update(prob: torch.Tensor, label: torch.Tensor, thresholds: torch.Tensor, var_kind: torch.Tensor, var_thr: torch.Tensor,
                  vars: torch.Tensor, scratch: torch.Tensor, flags: Optional[torch.Tensor] = None,
                  weight: Optional[torch.Tensor] = None) -> None:
    """vars[v] += the batch's count of kind var_kind[v] at thresholds[var_thr[v]], one fp32 rounding per variable (hrb200.h:
    hrb_metric_update).  thresholds ascending and distinct; scratch from metric_scratch_bytes, zeroed once; flags (int32, one per
    variable, nullable): set for the TP / FP / TN / FN variables when a prob is outside [0, 1] or NaN.
    With `weight` (fp32, one per sample): hrb_metric_update_weighted, which also takes the weighted kinds METRIC_WTP..WCOUNT;
    scratch from metric_weighted_scratch_bytes."""
    _chk(prob, torch.float32, "prob")
    _chk(label, torch.float32, "label")
    _chk(thresholds, torch.float32, "thresholds")
    _chk(var_kind, torch.int32, "var_kind")
    _chk(var_thr, torch.int32, "var_thr")
    _chk(vars, torch.float32, "vars")
    _chk(scratch, torch.uint8, "scratch")
    if prob.numel() != label.numel():
        raise ValueError(f"metric_update: {prob.numel()} predictions but {label.numel()} labels")
    if not (var_kind.numel() == var_thr.numel() == vars.numel()):
        raise ValueError("metric_update: var_kind, var_thr and vars must have one entry per variable")
    if flags is not None and (_chk(flags, torch.int32, "flags").numel() != vars.numel()):
        raise ValueError("metric_update: flags must have one entry per variable")
    if weight is not None:
        if _chk(weight, torch.float32, "weight").numel() != prob.numel():
            raise ValueError(f"metric_update: {prob.numel()} predictions but {weight.numel()} weights")
        if scratch.numel() < metric_weighted_scratch_bytes(thresholds.numel()):
            raise ValueError("metric_update: scratch too small (metric_weighted_scratch_bytes)")
        call("hrb_metric_update_weighted", _p(prob), _p(label), _p(weight), prob.numel(), _p(thresholds), thresholds.numel(), _p(var_kind),
             _p(var_thr), vars.numel(), _p(vars), _p(scratch), _p(flags), _stream())
        return
    if scratch.numel() < metric_scratch_bytes(thresholds.numel()):
        raise ValueError("metric_update: scratch too small (metric_scratch_bytes)")
    call("hrb_metric_update", _p(prob), _p(label), prob.numel(), _p(thresholds), thresholds.numel(), _p(var_kind), _p(var_thr),
         vars.numel(), _p(vars), _p(scratch), _p(flags), _stream())
