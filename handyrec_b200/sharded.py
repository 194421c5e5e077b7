"""Row-sharded embedding tables: owner(r) = r % N, local row r // N  (SURVEY.md §8e).

The reference is single-device; this is the multi-GPU face of the same lookup.  One process per GPU.
Per step and per rank (requester = the rank that owns the SAMPLE, owner = the rank that owns the ROW):

  forward   route ids (owner + owner-side key per position, grouped by owner)      [hrb_route_ids]
            all-to-all #0  counts            (N int64, equal split)     -> ONE host sync for the split sizes
            all-to-all #1  keys              (4 B per valid position)
            owner gathers its rows                                              [hrb_rows_by_key]
            all-to-all #2  rows              (4*D B per valid position)
            requester scatters / pools them into the group's output block       [hrb_scatter_rows]
  backward  requester gathers per-position gradients in the same order          [hrb_gather_grads]
            all-to-all #3  gradient rows
            owner: sort -> segment-reduce -> row update of its shard            [hrb_keyed_bwd_update]
  dense parameters are replicated; their flat gradient buffer is all-reduced once.

`RowExchange` holds the protocol; the arithmetic lives behind a small provider object so that the protocol can
be exercised under gloo on CPU tensors by the tests (tests/ supplies an oracle-backed provider; the product has
only the CUDA provider below -- there is no CPU fallback in this package).
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from . import kernels as K
from ._lib import call
from .engine import DeepFMEngine


def shard_rows(vocab: int, rank: int, n_ranks: int) -> int:
    """Rows of a `vocab`-row table held by `rank` (at least 1 so that every shard is a valid table)."""
    return max(1, (vocab - rank + n_ranks - 1) // n_ranks)


def key_base_table(vocabs: Sequence[int], n_ranks: int) -> torch.Tensor:
    """key_base[r, t] = first key of table t in rank r's shard key space (uint32 stored as int64 on host)."""
    kb = torch.zeros(n_ranks, len(vocabs), dtype=torch.int64)
    for r in range(n_ranks):
        acc = 0
        for t, v in enumerate(vocabs):
            kb[r, t] = acc
            acc += shard_rows(v, r, n_ranks)
    return kb


class CudaShardProvider:
    """The arithmetic of the exchange on this rank's GPU (C ABI calls only)."""

    def __init__(self, plan: K.LookupPlan, vocabs: Sequence[int], n_ranks: int, batch: int):
        self.plan, self.N, self.dev = plan, n_ranks, plan.device
        self.D = plan.tables[0].shape[1]
        self.kb = key_base_table(vocabs, n_ranks).to(torch.int32).to(self.dev)  # values < 2^31
        # the plan's tables are SHARDS: give the routing kernels the full vocabulary sizes so that an out-of-vocabulary id is
        # dropped here exactly like on the single-GPU path instead of landing in another table's key range
        call("hrb_plan_set_full_rows", plan._h, (ctypes.c_int64 * len(vocabs))(*[int(v) for v in vocabs]))
        need = ctypes.c_size_t(0)
        call("hrb_route_workspace", plan._h, batch, ctypes.byref(need))
        self.ws_route = torch.empty(need.value, device=self.dev, dtype=torch.uint8)
        n = batch * plan.pos_cols
        self.perm = torch.empty(max(n, 1), device=self.dev, dtype=torch.int32)
        self.send_keys = torch.empty(max(n, 1), device=self.dev, dtype=torch.int32)
        self.counts = torch.zeros(n_ranks + 1, device=self.dev, dtype=torch.int64)
        self.pos_rows = None if all(f[1] == 1 and f[2] in ("none", None) for f in plan.fields) else torch.zeros(max(n, 1), self.D, device=self.dev)
        self._ws_bwd = None

    def route(self, ids: torch.Tensor):
        B = ids.shape[0]
        call("hrb_route_ids", self.plan._h, K._p(ids), ids.stride(0), B, self.N, K._p(self.kb), K._p(self.perm), K._p(self.send_keys),
             K._p(self.counts), K._p(self.ws_route), self.ws_route.numel(), K._stream())
        return self.perm, self.send_keys, self.counts

    def rows_by_key(self, keys: torch.Tensor, n: int) -> torch.Tensor:
        out = torch.empty(max(n, 1), self.D, device=self.dev, dtype=torch.float32)
        call("hrb_rows_by_key", self.plan._h, K._p(keys), n, K._p(out), K._stream())
        return out[:n]

    def scatter_rows(self, ids, perm, n, rows, out):
        call("hrb_scatter_rows", self.plan._h, K._p(ids), ids.stride(0), ids.shape[0], K._p(perm), n, K._p(rows), K._p(out), out.stride(0),
             K._p(self.pos_rows), K._stream())

    def gather_grads(self, ids, perm, n, dout) -> torch.Tensor:
        send = torch.empty(max(n, 1), self.D, device=self.dev, dtype=torch.float32)
        call("hrb_gather_grads", self.plan._h, K._p(ids), ids.stride(0), K._p(perm), n, K._p(dout), dout.stride(0), K._p(send), K._stream())
        return send[:n]

    def scatter_grads_to_owners(self, ids, perm, send_keys, dout, send_counts, dst_off, rx: "ReceiveBuffers") -> None:
        n = self.N
        call("hrb_scatter_grads_to_owners", self.plan._h, K._p(ids), ids.stride(0), K._p(perm), K._p(send_keys), K._p(dout), dout.stride(0), n,
             (ctypes.c_int64 * n)(*send_counts), (ctypes.c_int64 * n)(*dst_off), (ctypes.c_void_p * n)(*rx.peer_grads),
             (ctypes.c_void_p * n)(*rx.peer_keys), K._stream())

    def keyed_update(self, keys, grads, n, op: _lib.OptParams):
        need = ctypes.c_size_t(0)
        call("hrb_keyed_bwd_workspace", self.plan._h, n, ctypes.byref(need))
        if self._ws_bwd is None or self._ws_bwd.numel() < need.value:
            self._ws_bwd = torch.empty(int(need.value * 1.25) + 1024, device=self.dev, dtype=torch.uint8)
        call("hrb_keyed_bwd_update", self.plan._h, K._p(keys), K._p(grads), n, ctypes.byref(op), K._p(self._ws_bwd), self._ws_bwd.numel(), K._stream())


def exchange_offsets(count_matrix: Sequence[Sequence[int]], rank: int) -> Tuple[List[int], List[int], List[int]]:
    """count_matrix[s][d] = entries rank s has for owner d  ->  (send_counts, recv_counts, dst_off) of `rank`:
    dst_off[d] = first row `rank` writes in owner d's receive buffers = the entries of lower-ranked senders for d, so that every
    owner's buffer ends up ordered by sender -- the layout of an all-to-all -- without the senders talking to each other."""
    n = len(count_matrix)
    send = [int(x) for x in count_matrix[rank]]
    recv = [int(count_matrix[s][rank]) for s in range(n)]
    off = [sum(int(count_matrix[s][d]) for s in range(rank)) for d in range(n)]
    return send, recv, off


class ReceiveBuffers:
    """This rank's receive blocks + the addresses of every rank's blocks as mapped here + the symmetric-memory handle (barriers)."""

    def __init__(self, arena, hdl, grads, keys, peer_grads: List[int], peer_keys: List[int]):
        self.arena, self.hdl, self.grads, self.keys, self.peer_grads, self.peer_keys = arena, hdl, grads, keys, peer_grads, peer_keys

    def barrier(self, channel: int) -> None:
        """Cross-GPU barrier on the CURRENT stream (signal pads in symmetric memory, release/acquire at system scope): stores
        issued to peers by earlier kernels of this stream are visible to kernels the peers launch behind their barrier."""
        self.hdl.barrier(channel=channel)


class TorchDistComm:
    """torch.distributed plumbing (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, group=None):
        import torch.distributed as dist

        self.dist, self.group = dist, group
        self.N, self.rank = dist.get_world_size(group), dist.get_rank(group)

    def all_to_all_equal(self, send: torch.Tensor) -> torch.Tensor:
        recv = torch.empty_like(send)
        self.dist.all_to_all_single(recv, send, group=self.group)
        return recv

    def all_to_all_v(self, send: torch.Tensor, send_counts: List[int], recv_counts: List[int]) -> torch.Tensor:
        recv = torch.empty((sum(recv_counts),) + tuple(send.shape[1:]), device=send.device, dtype=send.dtype)
        self.dist.all_to_all_single(recv, send, output_split_sizes=recv_counts, input_split_sizes=send_counts, group=self.group)
        return recv

    def all_to_all_v_start(self, send: torch.Tensor, send_counts: List[int], recv_counts: List[int]):
        """Non-blocking variant: -> (recv, wait) where wait() makes the CURRENT stream wait for the transfer."""
        recv = torch.empty((sum(recv_counts),) + tuple(send.shape[1:]), device=send.device, dtype=send.dtype)
        work = self.dist.all_to_all_single(recv, send, output_split_sizes=recv_counts, input_split_sizes=send_counts, group=self.group, async_op=True)
        return recv, work.wait

    def all_gather_equal(self, send: torch.Tensor) -> torch.Tensor:
        """-> (N, len(send)): row r = rank r's `send`."""
        out = torch.empty((self.N,) + tuple(send.shape), device=send.device, dtype=send.dtype)
        self.dist.all_gather_into_tensor(out, send.contiguous(), group=self.group)
        return out

    def all_reduce_sum(self, t: torch.Tensor) -> None:
        self.dist.all_reduce(t, group=self.group)

    def alloc_receive_buffers(self, rows: int, dim: int, device) -> Optional["ReceiveBuffers"]:
        """Owner-side receive buffers of the gradient exchange in symmetric memory: every rank maps every other rank's
        [rows, dim] fp32 gradient block and [rows] key block and stores into them over NVLink (hrb_scatter_grads_to_owners).
        None under gloo (CPU tests): the exchange then runs as all-to-alls."""
        if self.dist.get_backend(self.group) != "nccl":
            return None
        import torch.distributed._symmetric_memory as symm_mem

        g_elems = (rows * dim + 63) // 64 * 64
        arena = symm_mem.empty((g_elems + rows,), dtype=torch.float32, device=device)
        hdl = symm_mem.rendezvous(arena, group=self.group if self.group is not None else self.dist.group.WORLD)
        grads = arena[: rows * dim].view(rows, dim)
        keys = arena[g_elems : g_elems + rows].view(torch.int32)
        base = [int(p) for p in hdl.buffer_ptrs]
        return ReceiveBuffers(arena, hdl, grads, keys, base, [b + g_elems * 4 for b in base])

    _dense_group = None

    def all_reduce_dense(self, t: torch.Tensor) -> None:
        """All-reduce of the replicated parameters' gradients on a communicator of its own (NCCL only), so that it does not
        queue behind the embedding exchange of the same step on the process group's stream."""
        if self._dense_group is None:
            nccl = self.dist.get_backend(self.group) == "nccl"
            ranks = None if self.group is None else self.dist.get_process_group_ranks(self.group)
            self._dense_group = self.dist.new_group(ranks=ranks) if nccl else self.group
        self.dist.all_reduce(t, group=self._dense_group)

    def alloc_tables(self, vocabs: Sequence[int], dim: int, device, replicate_max_rows: int = 0) -> Tuple[List[torch.Tensor], Optional[List[List[int]]]]:
        """Allocate this rank's shards in ONE symmetric-memory arena (torch.distributed._symmetric_memory: CUDA VMM
        allocations exported to every rank of the node and mapped over NVLink) -> (tables, peer_ptrs[r][t]).
        Tables with at most `replicate_max_rows` rows are not sharded: every rank gets a full copy (plain allocation, peer
        pointer 0).  With the gloo backend (CPU tests) plain tensors are returned and peer_ptrs is None."""
        rep = [v <= replicate_max_rows for v in vocabs]
        rows = [v if r else shard_rows(v, self.rank, self.N) for v, r in zip(vocabs, rep)]
        if self.dist.get_backend(self.group) != "nccl":
            return [torch.zeros(r, dim) for r in rows], None
        import torch.distributed._symmetric_memory as symm_mem

        offs, off = [], 0
        for v, r in zip(vocabs, rep):
            offs.append(off)
            if not r:
                off += (shard_rows(v, 0, self.N) * dim + 63) // 64 * 64  # identical layout on every rank, 256-byte aligned table starts
        arena = symm_mem.empty((max(off, 64),), dtype=torch.float32, device=device)
        hdl = symm_mem.rendezvous(arena, group=self.group if self.group is not None else self.dist.group.WORLD)
        self._arena, self._arena_hdl = arena, hdl  # keep the mapping alive
        tables = [torch.zeros(n, dim, device=device) if r else arena[o : o + n * dim].view(n, dim) for o, n, r in zip(offs, rows, rep)]
        peer_ptrs = [[0 if r else int(hdl.buffer_ptrs[rk]) + o * 4 for o, r in zip(offs, rep)] for rk in range(self.N)]
        return tables, peer_ptrs


class RowExchange:
    """The requester/owner protocol of one rank.  `provider` does the arithmetic, `comm` moves the bytes."""

    def __init__(self, provider, comm):
        self.p, self.comm = provider, comm
        self.N = comm.N
        self.rx: Optional[ReceiveBuffers] = None  # set -> the backward exchange stores straight into the owners' buffers (no all-to-all)

    def route_async(self, ids: torch.Tensor) -> None:
        """Launch the routing of `ids` (owner + key per position, grouped by owner) and the exchange of the per-rank counts;
        nothing waits on the host.  Routing depends on the ids only, so it can run long before its results are needed."""
        self.perm, self.send_keys, counts = self.p.route(ids)
        self._counts_dev = counts
        if self.rx is not None:  # every rank needs the whole N x N count matrix: its write offset at owner d = entries of lower ranks for d
            self._count_matrix_dev = self.comm.all_gather_equal(counts[: self.N])
        else:
            self._recv_counts_dev = self.comm.all_to_all_equal(counts[: self.N].contiguous())
        self._routed = False
        # the routing may have been issued on a side stream: whoever consumes perm / send_keys / the counts first makes ITS
        # stream wait for this event (finish_route), so a caller on another stream never reads them half-written
        self._route_done = None
        if self.perm.is_cuda:
            self._route_done = torch.cuda.Event()
            self._route_done.record()

    def finish_route(self) -> None:
        if self._routed:
            return
        if getattr(self, "_route_done", None) is not None:
            torch.cuda.current_stream().wait_event(self._route_done)
        if self.rx is not None:
            C = self._count_matrix_dev.tolist()  # the one host sync of the step
            self.send_counts, self.recv_counts, self.dst_off = exchange_offsets(C, self.comm.rank)
            self.n_send, self.n_recv = sum(self.send_counts), sum(self.recv_counts)
            if self.n_recv > self.rx.keys.shape[0]:
                raise RuntimeError(f"gradient exchange: {self.n_recv} rows for this owner exceed the receive buffer ({self.rx.keys.shape[0]})")
            self.recv_keys = None  # keys travel with the gradient rows
            self._routed = True
            return
        both = torch.cat([self._counts_dev[: self.N], self._recv_counts_dev]).tolist()  # the one host sync of the step
        self.send_counts, self.recv_counts = [int(x) for x in both[: self.N]], [int(x) for x in both[self.N :]]
        self.n_send, self.n_recv = sum(self.send_counts), sum(self.recv_counts)
        self.recv_keys = self.comm.all_to_all_v(self.send_keys[: self.n_send], self.send_counts, self.recv_counts)
        self._routed = True

    def forward(self, ids: torch.Tensor, out: torch.Tensor) -> None:
        if self.rx is not None:
            raise RuntimeError("the all-to-all forward needs the keys exchanged: do not attach receive buffers in this mode")
        self.route_async(ids)
        self.finish_route()
        rows = self.p.rows_by_key(self.recv_keys, self.n_recv)
        got = self.comm.all_to_all_v(rows, self.recv_counts, self.send_counts)
        self.p.scatter_rows(ids, self.perm, self.n_send, got, out)

    def backward_start(self, ids: torch.Tensor, dout: torch.Tensor) -> None:
        """Gather this rank's per-position gradient rows and put them on the wire; work issued to the current stream after
        this call overlaps the transfer."""
        self.finish_route()
        if getattr(self, "_route_done", None) is not None:  # finish_route may have run earlier, on another stream
            torch.cuda.current_stream().wait_event(self._route_done)
        if self.rx is not None:
            # fused gather + exchange: one kernel stores rows and keys into the owners' buffers over NVLink
            self.p.scatter_grads_to_owners(ids, self.perm, self.send_keys, dout, self.send_counts, self.dst_off, self.rx)
            self._grad_send = self._grad_recv = self._grad_wait = None
            return
        self._grad_send = self.p.gather_grads(ids, self.perm, self.n_send, dout)
        start = getattr(self.comm, "all_to_all_v_start", None)
        if start is not None:
            self._grad_recv, self._grad_wait = start(self._grad_send, self.send_counts, self.recv_counts)
        else:
            self._grad_recv, self._grad_wait = self.comm.all_to_all_v(self._grad_send, self.send_counts, self.recv_counts), None

    def backward_finish(self, op, mark=None) -> None:
        if self.rx is not None:
            self.rx.barrier(0)  # every rank's stores have landed (and this rank's have left) once all have passed this point
            if mark is not None:
                mark("grad_rows_p2p_scatter")
            self.p.keyed_update(self.rx.keys, self.rx.grads, self.n_recv, op)
            if mark is not None:
                mark("keyed_update")
            return
        if self._grad_wait is not None:
            self._grad_wait()
        if mark is not None:
            mark("grad_rows_all_to_all")
        if self._grad_recv.is_cuda:  # this may run on another stream than the one the buffers were allocated on
            cur = torch.cuda.current_stream()
            self._grad_recv.record_stream(cur)
            self._grad_send.record_stream(cur)
            self.recv_keys.record_stream(cur)
        self.p.keyed_update(self.recv_keys, self._grad_recv, self.n_recv, op)
        self._grad_send = self._grad_recv = self._grad_wait = None
        if mark is not None:
            mark("keyed_update")

    def backward_update(self, ids: torch.Tensor, dout: torch.Tensor, op, mark=None) -> None:
        self.backward_start(ids, dout)
        self.backward_finish(op, mark)


class ShardedDeepFMEngine(DeepFMEngine):
    """DeepFMEngine over the ranks of `comm`: large tables row-sharded, small tables replicated.

    `vocabs` are the full vocabulary sizes.  `tables[t]` is this rank's SHARD of table t (rows r with r % N == rank, in
    order) -- or, for t in `replicated` (default: vocab <= `replicate_max_rows`), a full copy that is identical on every
    rank.  Replicated tables are read locally, their row gradients are reduced into the flat gradient buffer, all-reduced
    together with the dense parameters' gradients and stepped by the dense optimiser (DeepFMEngine: dense-updated tables);
    only the sharded tables take part in the row exchange.  The per-rank batch is fixed (weak scaling); gradients are
    averaged over the global batch.
    """

    def __init__(self, tables, vocabs, fields, n_dense, comm, peer_ptrs=None, replicate_max_rows: int = 0, replicated=None,
                 p2p_grad_exchange: bool = True, **kw):
        if replicated is None:
            replicated = [t for t, v in enumerate(vocabs) if v <= replicate_max_rows]
        self.replicated = sorted(set(int(t) for t in replicated))
        n_sharded = len(tables) - len(self.replicated)
        pooled = any(pool not in (None, "none") for ti, L, pool in fields if ti not in self.replicated)
        self._n_pad_flags = 2 * n_sharded if kw.get("optimizer") == "ftrl" and pooled else 0
        for t in self.replicated:
            if tables[t].shape[0] != vocabs[t]:
                raise ValueError(f"replicated table {t} must be a full copy ({vocabs[t]} rows), got {tables[t].shape[0]}")
        super().__init__(tables, fields, n_dense, dense_update_tables=self.replicated, **kw)
        self.comm = comm
        self.world = comm.N
        n_t = len(self.tables)
        self.sharded = [t for t in range(n_t) if t not in self.replicated]
        # sub-plans over the same id / output matrices: the sharded fields feed the row exchange, the replicated ones the
        # local gradient reduction
        def sub_plan(tabs, with_moments):
            remap = {t: i for i, t in enumerate(tabs)}
            flds = [(remap[f[0]],) + tuple(f[1:]) for f in self.plan_fields if f[0] in remap]
            if not flds:
                return None
            m = [self.adam_m[t] for t in tabs] if (with_moments and self.adam_m is not None) else None
            v = [self.adam_v[t] for t in tabs] if (with_moments and self.adam_v is not None) else None
            acc = [self.accum[t] for t in tabs] if (with_moments and self.accum is not None) else None
            lin = [self.linear[t] for t in tabs] if (with_moments and self.linear is not None) else None
            return K.LookupPlan([self.tables[t] for t in tabs], flds, m, v, accum=acc, linear=lin)

        if self.replicated:
            self.plan_shard = sub_plan(self.sharded, True)
            self.plan_rep = sub_plan(self.replicated, False)
            if self.plan_rep is not None:
                self.plan_rep.set_dense_grads([self.table_grads[t] for t in self.replicated])
                self._ws_rep = torch.empty(self.plan_rep.workspace_bytes(self.B), device=self.dev, dtype=torch.uint8)
        else:
            self.plan_shard, self.plan_rep = self.plan, None
        # Ftrl: padding positions of pooled fields name row 0, which the row exchange does not route.  Every rank flags, per
        # row-sharded table, padding seen / a valid id 0 seen in the tail of the flat gradient buffer (after the touched flags);
        # the gradient all-reduce sums them and the owner of row 0 (rank 0) gives row 0 its zero-gradient step where needed.
        self._pad_flags = self.grads[-self._n_pad_flags :] if self._n_pad_flags else None
        self.exchange = None
        if self.plan_shard is not None:
            self.provider = CudaShardProvider(self.plan_shard, [vocabs[t] for t in self.sharded], comm.N, self.B)
            self.exchange = RowExchange(self.provider, comm)
        self.grad_scale_div = comm.N
        self.overlap_embedding_bwd = True
        self.peer_lookup = False
        self._rep_done = None
        self._barrier_buf = torch.zeros(1, device=self.dev)
        plain = all(f[1] == 1 and f[2] in ("none", None) for f in fields)
        if self.exchange is None and plain:
            self.peer_lookup = True  # everything is replicated: the local fused lookup is the whole forward
        elif peer_ptrs is not None and plain:
            # forward without any all-to-all: every rank maps every other rank's shards (comm.alloc_tables: symmetric memory over
            # NVLink) and the fused lookup+FM kernel gathers row `id` from rank id % N at local row id // N
            ptrs = (ctypes.c_void_p * (comm.N * n_t))(
                *[(None if t in self.replicated else int(peer_ptrs[r][t])) for r in range(comm.N) for t in range(n_t)])
            full = (ctypes.c_int64 * n_t)(*[int(v) for v in vocabs])
            call("hrb_plan_set_peers", self.plan._h, comm.N, ptrs, full)
            self.peer_lookup = True
            if p2p_grad_exchange and hasattr(comm, "alloc_receive_buffers"):
                # worst case for one owner: every position of every rank's batch
                self.exchange.rx = comm.alloc_receive_buffers(comm.N * self.B * self.plan_shard.pos_cols, self.D, self.dev)

    _fwd_training = False

    def forward(self, ids, dense, training: bool = False):
        self._fwd_training = training
        return super().forward(ids, dense, training)

    def _lookup_fm_forward(self, ids, B, st):
        if self.peer_lookup:
            super()._lookup_fm_forward(ids, B, st)
            # the routing needed by the BACKWARD exchange depends on the ids only: it is issued right behind the lookup, on the side
            # stream, so that it fills in beside the dense forward instead of delaying the lookup
            if self.exchange is not None and self._fwd_training:
                main = torch.cuda.current_stream()
                if self._side is None:
                    self._side = torch.cuda.Stream()
                if self._marks is None:
                    self._side.wait_stream(main)
                    with torch.cuda.stream(self._side):
                        self.exchange.route_async(ids)
                else:
                    self.exchange.route_async(ids)
                    self._mark("route_ids")
            return
        if self.exchange is not None:
            self.exchange.forward(ids, self.X0)  # the plan's out_col already includes the dense block
        if self.plan_rep is not None:
            call("hrb_lookup_fwd", self.plan_rep._h, K._p(ids), ids.stride(0), B, K._p(self.X0), self.K0p, None, None, st)
        self._mark("sharded_lookup_fwd")
        emb = self.X0[:, self.nd_pad :]
        call("hrb_fm_fwd", K._p(emb), self.K0p, B, self.F, self.D, K._p(self.fm_w), K._p(self.fm_w0), K._p(self.fm_out), K._p(self.fm_sum), st)
        self._mark("fm_fwd")

    def _pre_embedding_backward(self):
        if self.peer_lookup and self.exchange is not None:
            self.exchange.finish_route()
            if self._timeline is not None:
                self._mark("route_keys_all_to_all")

    _side2 = None

    def _embedding_backward(self, ids, B, st, op):
        cur = torch.cuda.current_stream()
        own_stream = False
        if self.exchange is not None:  # gradient rows of the sharded tables go on the wire first: the transfer runs beside the local reduction
            self.exchange.backward_start(ids, self.dX0)
            # the owner-side row update of the sharded tables only needs the all-to-all: it gets a stream of its own so that it
            # starts the moment the rows land instead of queueing behind the replicated tables' reduction (round 1: 0.23 ms of tail)
            own_stream = self._marks is None and self.plan_rep is not None and self.dX0.is_cuda
            if own_stream:
                if self._side2 is None:
                    self._side2 = torch.cuda.Stream()
                self._side2.wait_stream(cur)
                with torch.cuda.stream(self._side2):
                    self._finish_sharded(op)
        if self.plan_rep is None and self._pad_flags is not None:
            self._zero_table_grads()
            self.plan_shard.pad_flags(ids, self._pad_flags)
            self._rep_done = torch.cuda.Event()  # the gradient all-reduce carries the flags
            self._rep_done.record()
        if self.plan_rep is not None:  # replicated tables: local reduction into the flat gradient buffer
            self._zero_table_grads()
            self._mark_touched(self.plan_rep, ids, self.replicated)
            if self._pad_flags is not None:
                self.plan_shard.pad_flags(ids, self._pad_flags)
            call("hrb_lookup_bwd_update", self.plan_rep._h, K._p(ids), ids.stride(0), B, K._p(self.dX0), self.K0p, None, ctypes.byref(op),
                 K._p(self._ws_rep), self._ws_rep.numel(), K._stream())
            self._rep_done = torch.cuda.Event()
            self._rep_done.record()
            self._mark("replicated_embedding_bwd")
        if self.exchange is not None:
            if own_stream:
                cur.wait_stream(self._side2)
            else:
                self._finish_sharded(op)
            self._mark("sharded_embedding_bwd_update")

    def _finish_sharded(self, op):
        self.exchange.backward_finish(op, mark=self._mark if self._timeline is not None else None)
        if self.peer_lookup:
            # peers read this shard in the next forward (and write this rank's receive buffers in the next backward): nobody may
            # start it before every rank has finished updating
            if self.exchange.rx is not None:
                self.exchange.rx.barrier(1)
            else:
                self.comm.all_reduce_sum(self._barrier_buf)

    def _sync_dense_grads(self):
        if self._rep_done is not None:  # recorded on the side stream when the embedding backward is overlapped
            torch.cuda.current_stream().wait_event(self._rep_done)
            self._rep_done = None
        getattr(self.comm, "all_reduce_dense", self.comm.all_reduce_sum)(self.grads)
        self._mark("dense_allreduce")
        if self._pad_flags is not None and self.comm.rank == 0:  # local row 0 of rank 0's shards is row 0 of every sharded table
            self.plan_shard.ftrl_pad_step(self._pad_flags, self._op)
