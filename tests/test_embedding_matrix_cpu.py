"""CPU: the float64 pieces behind tests/test_gpu_embedding_matrix.py -- the restatement of the sort-free backward's unit
decomposition (build_units / unit_path_supported of csrc/embedding_bwd.cu) against hand-worked plans, the per-table gradient
sums against autograd of the oracle layers, lazy Adam against the dense Keras formula, and the row-list table hash."""
import numpy as np
import torch

import oracle
from oracle.embedding_ref import plan_grad_sums, table_units, unit_counts, unit_path_taken
from oracle.optim_ref import adam_lazy_sparse


def _summary(units):
    return [(u["lo"], u["hi"], u["slices"], u["expect"]) for u in units]


def test_units_of_a_uniform_table():
    # 65536 positions over 100 rows: range 4 is the largest power of two whose share (2621) stays <= 3686; range 8 would be 5242
    u = table_units(100, 1, 65536)
    assert len(u) == 25 and {x["shift"] for x in u} == {2}
    assert _summary(u)[0] == (0, 4, 1, 2621) and _summary(u)[-1] == (96, 100, 1, 2621)
    # 2^20 rows: 2^15-row units of 2048 expected positions
    u = table_units(1 << 20, 1, 65536)
    assert len(u) == 32 and u[0]["shift"] == 15 and u[0]["expect"] == 2048


def test_units_short_last_unit():
    # 100003 rows at 20000 positions: range 2^14 (3276 expected), the 7th unit holds the last 1699 rows only
    u = table_units(100003, 1, 20000)
    assert len(u) == 7 and u[0]["shift"] == 14
    assert _summary(u)[0] == (0, 16384, 1, 3276)
    assert _summary(u)[-1] == (98304, 100003, 1, 339)


def test_single_row_units_and_slices():
    # 6 rows at 20000: one row per unit (range 2 would expect 6666), 3333 positions each -> not sliced
    assert _summary(table_units(6, 1, 20000)) == [(r, r + 1, 1, 3333) for r in range(6)]
    # 2 rows at 20000: 10000 > 2 * 4096 -> ceil(10000 / 4096) = 3 slices per row
    assert _summary(table_units(2, 1, 20000)) == [(0, 1, 3, 10000), (1, 2, 3, 10000)]
    # 2 rows under a 10-long field at 65536: 327680 expected positions per row -> 80 slices, capped at 64
    assert _summary(table_units(2, 10, 65536)) == [(0, 1, 64, 327680), (1, 2, 64, 327680)]


def test_unit_limit_256_bins():
    # 8 columns at 65536 (524288 positions): 256 rows still fit (one row per unit), 257 rows need 257 units -> sorted path
    assert len(table_units(256, 8, 65536)) == 256
    assert table_units(257, 8, 65536) is None
    f = [(0, 8, "sum", 0, 0)]
    assert unit_path_taken([(256, 16)], f, 65536) and not unit_path_taken([(257, 16)], f, 65536)


def test_unit_path_conditions():
    plain = [(0, 1, "none", 0, 0)]
    assert unit_path_taken([(1000, 128)], plain, 4096)
    for d in (12, 24, 96, 256, 1024):  # G not a power of two, or G > 32
        assert not unit_path_taken([(1000, d)], plain, 4096)
    assert unit_path_taken([(5000, 16)], [(0, 256, "mean", 0, 0)], 2048)
    assert not unit_path_taken([(5000, 16)], [(0, 257, "mean", 0, 0)], 2048)  # 257 position columns in one table
    assert not unit_path_taken([(5000, 16)], [(0, 256, "mean", 0, 0), (0, 1, "none", 256, 16)], 2048)
    assert not unit_path_taken([(5000, 16)], [(0, 3, "max", 0, 0)], 4097)
    assert not unit_path_taken([(1 << 30, 16)], plain, 1 << 24) and not unit_path_taken([(1000, 16)], plain, 0)


def test_unit_counts():
    u = table_units(1 << 20, 1, 65536)
    ids = np.array([0, 32767, 32768, (1 << 20) - 1])
    c = unit_counts(u, ids)
    assert c[0] == 2 and c[1] == 1 and c[31] == 1 and c.sum() == 4


def test_plan_grad_sums_match_autograd_of_the_oracle_layers():
    g = torch.Generator().manual_seed(0)
    B, D, V, W = 37, 8, 11, 5
    t0, t1 = torch.randn(V, D, generator=g, dtype=torch.float64), torch.randn(W, D, generator=g, dtype=torch.float64)
    plain = torch.randint(0, V, (B, 1), generator=g)
    hist = torch.randint(0, V, (B, 4), generator=g)
    hist[::3] = 0  # all-padding rows
    seq = torch.randint(0, W, (B, 3), generator=g)
    ids = torch.cat([plain, hist, seq], 1)
    fields = [(0, 1, "none", 0, 0), (0, 4, "mean", 1, D), (1, 3, "sum", 5, 2 * D)]
    dout = torch.randn(B, 3 * D, generator=g, dtype=torch.float64)
    l0, l1 = t0.clone().requires_grad_(True), t1.clone().requires_grad_(True)
    e0, _ = oracle.custom_embedding(l0, plain, False)
    e1 = oracle.sequence_pooling(*oracle.custom_embedding(l0, hist, True), "mean")
    e2 = oracle.sequence_pooling(*oracle.custom_embedding(l1, seq, True), "sum")
    (torch.cat([e0[:, 0], e1[:, 0], e2[:, 0]], 1) * dout).sum().backward()
    sums = plan_grad_sums([(V, D), (W, D)], fields, ids, dout)
    for s, leaf in zip(sums, (l0, l1)):
        want = leaf.grad
        touched = want.abs().sum(1) > 0
        assert set(s["rows"].tolist()) >= set(torch.nonzero(touched).reshape(-1).tolist())
        np.testing.assert_allclose(s["grad"].numpy(), want[s["rows"]].numpy(), rtol=1e-6, atol=1e-7)  # the oracle layers scale in float32
    assert sums[0]["pad"] and sums[1]["pad"] == bool((seq == 0).any())
    # a dropped plain id takes its gradient row away from the row it replaced and lands nowhere
    bad = ids.clone()
    bad[2, 0] = V + 7
    sb = plan_grad_sums([(V, D), (W, D)], fields, bad, dout)
    assert int(((sb[0]["rows"] < 0) | (sb[0]["rows"] >= V)).sum()) == 0
    full = torch.zeros(V, D, dtype=torch.float64)
    full[sums[0]["rows"]] = sums[0]["grad"]
    full[plain[2, 0]] -= dout[2, :D]
    got = torch.zeros(V, D, dtype=torch.float64)
    got[sb[0]["rows"]] = sb[0]["grad"]
    assert torch.allclose(got, full, rtol=0, atol=1e-12)
    # a negative id inside a mean-pooled row is dropped from the row's n_valid too
    bad = ids.clone()
    bad[1, 1:5] = torch.tensor([-3, 4, 0, V])
    sb = plan_grad_sums([(V, D), (W, D)], fields, bad, dout)
    got = torch.zeros(V, D, dtype=torch.float64)
    got[sb[0]["rows"]] = sb[0]["grad"]
    want = torch.zeros(V, D, dtype=torch.float64)
    for ii in (ids.clone(),):
        ii[1, 1:5] = torch.tensor([0, 4, 0, 0])  # the same sample with the dropped ids as padding
        s2 = plan_grad_sums([(V, D), (W, D)], fields, ii, dout)
        want[s2[0]["rows"]] = s2[0]["grad"]
    assert torch.allclose(got, want, rtol=0, atol=1e-12)


def test_adam_lazy_sparse_is_dense_adam_on_the_listed_rows():
    g = torch.Generator().manual_seed(1)
    V, D, step = 9, 4, 5
    w, m = torch.randn(V, D, generator=g, dtype=torch.float64), torch.randn(V, D, generator=g, dtype=torch.float64) * 0.01
    v = torch.rand(V, D, generator=g, dtype=torch.float64) * 1e-3 + 1e-4
    idx = torch.tensor([3, 1, 3, 7])
    vals = torch.randn(4, D, generator=g, dtype=torch.float64)
    nw, nm, nv = adam_lazy_sparse(w, m, v, idx, vals, lr=0.01, step=step, l2_scale=0.02)
    rows = torch.tensor([1, 3, 7])
    gs = torch.zeros(V, D, dtype=torch.float64).index_add_(0, idx, vals)[rows] + 0.02 * w[rows]
    mm = 0.9 * m[rows] + 0.1 * gs
    vv = 0.999 * v[rows] + 0.001 * gs * gs
    ww = w[rows] - 0.01 * np.sqrt(1 - 0.999 ** step) / (1 - 0.9 ** step) * mm / (vv.sqrt() + 1e-7)
    assert torch.allclose(nw[rows], ww, rtol=1e-14, atol=0) and torch.allclose(nm[rows], mm) and torch.allclose(nv[rows], vv)
    rest = torch.tensor([r for r in range(V) if r not in (1, 3, 7)])
    assert torch.equal(nw[rest], w[rest]) and torch.equal(nm[rest], m[rest]) and torch.equal(nv[rest], v[rest])


def test_hash_uniform_rows_is_a_row_gather_of_the_table():
    t = oracle.hash_uniform_table(300, 12, seed=5, lo=1e-4, hi=1e-3)
    rows = np.array([299, 0, 17, 17, 150])
    assert np.array_equal(oracle.hash_uniform_rows(rows, 12, seed=5, lo=1e-4, hi=1e-3), t[rows])
    # rows past 2^32 / D use the high word of the element index like hrb_init_uniform
    big = np.array([(1 << 30) + 3])
    assert oracle.hash_uniform_rows(big, 8, seed=1).shape == (1, 8)
