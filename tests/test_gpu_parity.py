"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical inputs/weights.

Tolerances (BASELINE.json north_star): bit-exact for id mapping, gathers and masks; <= 1e-5 relative
for fp32 forward (pooling, FM, attention); <= 1e-4 for gradients.  "relative" is taken against the
magnitude of the tensor (atol = tol * max|ref|) because sums with cancellation have no meaningful
element-wise relative error.
"""
import numpy as np
import pytest
import torch

import oracle
from oracle import kat

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-5
GRAD_TOL = 1e-4


def K():
    from handyrec_b200 import kernels

    return kernels


def close(got, want, tol):
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    want = want.detach().cpu().numpy() if isinstance(want, torch.Tensor) else np.asarray(want)
    assert got.shape == want.shape, (got.shape, want.shape)
    scale = max(float(np.abs(want).max()), 1e-30) if want.size else 1.0
    np.testing.assert_allclose(got, want, rtol=tol, atol=tol * scale)


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def rand_ids(B, L, V, seed=0, pad_frac=0.4, pre_pad=True):
    """History-like ids: random length per row, zero padding in front (data/utils.py:46-49)."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1, V, (B, L), generator=g, dtype=torch.int32)
    lens = torch.randint(0, L + 1, (B,), generator=g)
    lens[torch.rand(B, generator=g) < 0.1] = 0  # some all-padding rows
    pos = torch.arange(L).unsqueeze(0)
    keep = pos >= (L - lens).unsqueeze(1) if pre_pad else pos < lens.unsqueeze(1)
    return torch.where(keep, ids, torch.zeros_like(ids))


# ------------------------------------------------------------------------------------------------
# known-answer vectors through the C ABI
# ------------------------------------------------------------------------------------------------
def test_kat_pool_and_mask(dev):
    k = K()
    table = torch.from_numpy(kat.POOL_TABLE).to(dev)
    ids = torch.from_numpy(kat.POOL_IDS).to(dev)
    seq, mask = k.embedding_fwd(table, ids, mask_zero=True)
    assert np.array_equal(seq.cpu().numpy(), kat.POOL_TABLE[kat.POOL_IDS])
    assert mask.dtype == torch.bool and np.array_equal(mask.cpu().numpy(), np.repeat(kat.POOL_MASK[..., None], 4, -1))
    for method, want in (("mean", kat.POOL_MEAN), ("sum", kat.POOL_SUM), ("max", kat.POOL_MAX)):
        got = k.seq_pool_fwd(seq, mask, method)
        assert got.shape == (3, 1, 4)
        np.testing.assert_allclose(got[:, 0].cpu().numpy(), want, rtol=1e-6)
        plan = k.LookupPlan([table], [(0, 3, method, 0, 0)])
        fused = plan.forward(ids)["out"]
        np.testing.assert_allclose(fused.cpu().numpy(), want, rtol=1e-6)
    _, nomask = k.embedding_fwd(table, ids, mask_zero=False)
    assert nomask is None
    with pytest.raises(ValueError):
        k.seq_pool_fwd(seq, None, "mean")
    with pytest.raises(AssertionError):
        k.seq_pool_fwd(seq, mask, "median")


def test_kat_fm(dev):
    k = K()
    x = torch.from_numpy(kat.FM_X).to(dev)
    w = torch.from_numpy(kat.FM_W).to(dev)
    w0 = torch.from_numpy(kat.FM_W0).to(dev)
    # D = 2 is not a multiple of 4: exercises the direct kernel
    out = k.fm_fwd(x, w, w0)
    np.testing.assert_allclose(out.cpu().numpy(), kat.FM_OUT, rtol=1e-6)


def test_kat_dice(dev):
    k = K()
    x = torch.from_numpy(kat.DICE_X).to(dev)
    y = k.dice_fwd(x, torch.full((4,), 0.25, device=dev), torch.zeros(4, device=dev), torch.ones(4, device=dev), training=False)
    np.testing.assert_allclose(y.cpu().numpy(), kat.DICE_OUT, rtol=1e-6, atol=1e-7)


def test_kat_lau(dev):
    k = K()
    # table rows: 0 -> pad key [0,0] (padded to D=4), 1 -> q [1,2], 2 -> [1,1], 3 -> [2,-1]
    table = torch.tensor([[0, 0, 0, 0], [1, 2, 0, 0], [1, 1, 0, 0], [2, -1, 0, 0]], dtype=torch.float32)
    qid = torch.tensor([1], dtype=torch.int32)
    kid = torch.tensor([[0, 2, 3]], dtype=torch.int32)
    # stand-in MLP on the padded 16-wide input: identity Dense(16) then Dense(1) of 0.1s, act = linear
    Ws = [torch.eye(16), torch.full((16, 1), 0.1)]
    bs = [torch.zeros(16), torch.zeros(1)]
    params = k.lau_pack_params([w.to(dev) for w in Ws], [b.to(dev) for b in bs])
    score, pooled = k.lau_fwd(table.to(dev), qid.to(dev), kid.to(dev), params, [16, 1], "linear")
    np.testing.assert_allclose(score.cpu().numpy(), kat.LAU_ATT, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(pooled.cpu().numpy()[:, :, :2], kat.LAU_POOLED, rtol=1e-6, atol=1e-7)


# ------------------------------------------------------------------------------------------------
# a5 / a6: gather, mask, pooling (layer face)
# ------------------------------------------------------------------------------------------------
def test_init_uniform_bit_exact(dev):
    k = K()
    for (V, D, seed) in ((1000, 16, 7), (257, 8, 123456789), (5, 32, 0)):
        t = torch.empty(V, D, device=dev)
        k.init_uniform(t, seed)
        assert np.array_equal(t.cpu().numpy(), oracle.hash_uniform_table(V, D, seed))
    t = torch.empty(25, 16, device=dev)
    k.init_uniform(t, 7, row_start=3, row_step=4)
    assert np.array_equal(t.cpu().numpy(), oracle.hash_uniform_table(100, 16, 7)[3::4])


@pytest.mark.parametrize("V,D,shape", [(3953, 32, (64, 50)), (19, 8, (5, 3)), (100003, 16, (4096, 1)), (7, 4, (1, 1)), (50, 64, (33, 7))])
def test_embedding_gather_and_mask_bit_exact(dev, V, D, shape):
    k = K()
    table = rnd(V, D, seed=V)
    ids = rand_ids(shape[0], shape[1], V, seed=D)
    out, mask = k.embedding_fwd(table.to(dev), ids.to(dev), mask_zero=True)
    want, wmask = oracle.custom_embedding(table, ids, True)
    assert np.array_equal(out.cpu().numpy(), want.numpy())
    assert np.array_equal(mask.cpu().numpy(), wmask.numpy())


def test_embedding_empty_and_out_of_range(dev):
    k = K()
    table = rnd(10, 8).to(dev)
    out, mask = k.embedding_fwd(table, torch.zeros(0, 3, dtype=torch.int32, device=dev), True)
    assert out.shape == (0, 3, 8) and mask.shape == (0, 3, 8)
    with pytest.raises(IndexError):  # TF-CPU raises InvalidArgumentError; oracle raises IndexError
        k.embedding_fwd(table, torch.tensor([[1, 10]], dtype=torch.int32, device=dev), True)
    with pytest.raises(IndexError):
        oracle.custom_embedding(table.cpu(), torch.tensor([[1, 10]]), True)
    from handyrec_b200._lib import HrbError

    with pytest.raises(HrbError):  # dim % 4 != 0 is declared unsupported, not silently mishandled
        k.embedding_fwd(rnd(10, 6).to(dev), torch.zeros(1, 1, dtype=torch.int32, device=dev), True)


@pytest.mark.parametrize("method", ["mean", "sum", "max"])
@pytest.mark.parametrize("B,L,D", [(64, 50, 32), (5, 2, 8), (5, 3, 8), (257, 6, 8), (3, 1, 4)])
def test_seq_pool_fwd_bwd(dev, method, B, L, D):
    k = K()
    V = 101
    table = rnd(V, D, seed=3, scale=0.05)
    ids = rand_ids(B, L, V, seed=B + L)
    x, mask = oracle.custom_embedding(table, ids, True)
    x = x.clone().requires_grad_(True)
    want = oracle.sequence_pooling(x, mask, method)
    got = k.seq_pool_fwd(x.detach().to(dev), mask.to(dev), method)
    close(got, want, FWD_TOL)
    dout = rnd(B, 1, D, seed=9)
    want.backward(dout)
    dx = k.seq_pool_bwd(x.detach().to(dev), mask.to(dev), dout.reshape(B, D).to(dev), method)
    close(dx, x.grad, GRAD_TOL)


# ------------------------------------------------------------------------------------------------
# a7: fused group lookup
# ------------------------------------------------------------------------------------------------
def _c1_like_group(seed=0, B=5, pool="mean"):
    """tests/ml-1m-test/DeepFM_cfg.yaml shape: 6 sparse + hist_movie (L=2, shares movie_id) + genres (L=3), D=8."""
    vocabs = {"user_id": 6, "gender": 3, "occupation": 21, "zip": 6, "age": 57, "movie_id": 11, "genre_id": 19}
    D = 8
    names = list(vocabs)
    tables = {n: rnd(v, D, seed=seed + i, scale=0.05) for i, (n, v) in enumerate(vocabs.items())}
    g = torch.Generator().manual_seed(seed)
    sparse = ["user_id", "gender", "occupation", "zip", "age", "movie_id"]
    cols = [torch.randint(0, vocabs[n], (B, 1), generator=g, dtype=torch.int32) for n in sparse]
    hist = rand_ids(B, 2, vocabs["movie_id"], seed=seed + 1)
    genres = rand_ids(B, 3, vocabs["genre_id"], seed=seed + 2, pre_pad=False)
    ids = torch.cat(cols + [hist, genres], 1)
    # plan: table index, L, pool, ids_col, out_col
    fields = [(names.index(n), 1, "none", i, i * D) for i, n in enumerate(sparse)]
    fields.append((names.index("movie_id"), 2, pool, 6, 6 * D))
    fields.append((names.index("genre_id"), 3, pool, 8, 7 * D))
    # movie_id is the unit of a seq feature in this group -> mask_zero=True (group.py:273,292); values unaffected
    o_sparse = {n: (tables[n], ids[:, i : i + 1], n == "movie_id") for i, n in enumerate(sparse)}
    o_seq = {"hist_movie": (tables["movie_id"], hist), "genres": (tables["genre_id"], genres)}
    return names, tables, ids, fields, o_sparse, o_seq, D


@pytest.mark.parametrize("pool", ["mean", "sum", "max"])
@pytest.mark.parametrize("B", [5, 1, 300])
def test_group_lookup_c1_shape(dev, pool, B):
    k = K()
    names, tables, ids, fields, o_sparse, o_seq, D = _c1_like_group(seed=B, B=B, pool=pool)
    plan = k.LookupPlan([tables[n].to(dev) for n in names], fields)
    res = plan.forward(ids.to(dev), want_inv_count=True, check_ids=True)
    from collections import OrderedDict

    want = oracle.concat([], oracle.group_embedding_lookup(OrderedDict(o_sparse), OrderedDict(o_seq), pool))
    got = res["out"]
    assert got.shape == want.shape
    # plain lookups are bit-exact
    assert np.array_equal(got[:, : 6 * D].cpu().numpy(), want[:, : 6 * D].numpy())
    close(got[:, 6 * D :], want[:, 6 * D :], FWD_TOL)


def test_group_lookup_mixed_dims_and_fm_requirements(dev):
    k = K()
    t32, t8 = rnd(3953, 32, seed=1, scale=0.05), rnd(19, 8, seed=2, scale=0.05)
    B = 129
    hist = rand_ids(B, 50, 3953, seed=4)
    genres = rand_ids(B, 6, 19, seed=5)
    ids = torch.cat([hist, genres], 1)
    plan = k.LookupPlan([t32.to(dev), t8.to(dev)], [(0, 50, "mean", 0, 0), (1, 6, "mean", 50, 32)])
    got = plan.forward(ids.to(dev))["out"]
    w1 = oracle.sequence_pooling(*oracle.custom_embedding(t32, hist, True), "mean")
    w2 = oracle.sequence_pooling(*oracle.custom_embedding(t8, genres, True), "mean")
    close(got, torch.cat([w1, w2], -1)[:, 0], FWD_TOL)
    from handyrec_b200._lib import HrbError

    with pytest.raises(HrbError):  # FM needs equal dims (layers/utils.py Concatenate(axis=1) would fail too)
        plan.forward(ids.to(dev), fm=(rnd(32, 1).to(dev), torch.zeros(1, device=dev)))


@pytest.mark.parametrize("B,F,D", [(4096, 26, 16), (5, 3, 8), (1000, 7, 32), (64, 2, 4), (333, 5, 64)])
def test_fused_lookup_fm_criteo_shape(dev, B, F, D):
    k = K()
    vocabs = [max(4, int(10 ** (1 + 4 * f / max(F - 1, 1)))) for f in range(F)]
    tables = [torch.from_numpy(oracle.hash_uniform_table(v, D, seed=7 + f)) for f, v in enumerate(vocabs)]
    g = torch.Generator().manual_seed(B)
    ids = torch.stack([torch.randint(0, v, (B,), generator=g, dtype=torch.int32) for v in vocabs], 1)
    w, w0 = rnd(D, 1, seed=1, scale=0.1), torch.tensor([0.3])
    dtab = []
    for f, v in enumerate(vocabs):
        t = torch.empty(v, D, device=dev)
        k.init_uniform(t, 7 + f)
        dtab.append(t)
    plan = k.LookupPlan(dtab, [(f, 1, "none", f, f * D) for f in range(F)])
    res = plan.forward(ids.to(dev), fm=(w.to(dev), w0.to(dev)), want_fm_sum=True)
    x = torch.stack([tables[f][ids[:, f].long()] for f in range(F)], 1)
    assert np.array_equal(res["out"].cpu().numpy().reshape(B, F, D), x.numpy())  # gathers: bit-exact
    close(res["fm_out"], oracle.fm(x, w, w0)[:, 0], FWD_TOL)
    close(res["fm_sum"], x.sum(1), FWD_TOL)
    # unfused pair: items kernel + staged FM kernel give the same answers
    res2 = plan.forward(ids.to(dev))
    assert torch.equal(res2["out"], res["out"])
    fm2 = k.fm_fwd(res2["out"].view(B, F, D), w.to(dev), w0.to(dev))
    close(fm2, oracle.fm(x, w, w0), FWD_TOL)


def test_fused_lookup_fm_with_sequences(dev):
    k = K()
    names, tables, ids, fields, o_sparse, o_seq, D = _c1_like_group(seed=3, B=77)
    from collections import OrderedDict

    plan = k.LookupPlan([tables[n].to(dev) for n in names], fields)
    w, w0 = rnd(D, 1, seed=5, scale=0.1), torch.tensor([-0.1])
    res = plan.forward(ids.to(dev), fm=(w.to(dev), w0.to(dev)))
    embds = oracle.group_embedding_lookup(OrderedDict(o_sparse), OrderedDict(o_seq), "mean")
    x = oracle.concat([], embds, axis=1, keepdims=True)
    close(res["out"].view(77, 8, D), x, FWD_TOL)
    close(res["fm_out"], oracle.fm(x, w, w0)[:, 0], FWD_TOL)


# ------------------------------------------------------------------------------------------------
# a9: FM on a materialised tensor, forward + backward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,F,D,pad", [(4096, 26, 16, 0), (100, 8, 8, 0), (257, 3, 32, 0), (64, 26, 16, 16), (1, 1, 4, 0), (50, 4, 128, 0), (31, 5, 6, 0)])
def test_fm_fwd_bwd(dev, B, F, D, pad):
    k = K()
    buf = rnd(B, F * D + pad, seed=B, scale=0.3)
    x = buf[:, pad:].reshape(B, F, D).clone().requires_grad_(True)
    w = rnd(D, 1, seed=1, scale=0.2).requires_grad_(True)
    w0 = torch.tensor([0.1], requires_grad=True)
    want = oracle.fm(x, w, w0)
    dbuf = buf.to(dev)
    xv = dbuf[:, pad:].view(B, F, D) if pad else dbuf.view(B, F, D)
    got, s = k.fm_fwd(xv, w.detach().to(dev), w0.detach().to(dev), want_sum=True)
    close(got, want, FWD_TOL)
    close(s, x.detach().sum(1), FWD_TOL)
    if D % 4 == 0 and (D // 4) & (D // 4 - 1) == 0:
        dout = rnd(B, 1, seed=4)
        want.backward(dout)
        dx, dw, dw0 = k.fm_bwd(xv, w.detach().to(dev), dout.reshape(B).to(dev))
        close(dx, x.grad, GRAD_TOL)
        close(dw, w.grad, GRAD_TOL)
        close(dw0, w0.grad, GRAD_TOL)
        # accumulate into an existing gradient
        base = rnd(B, F, D, seed=8).to(dev)
        dx2, _, _ = k.fm_bwd(xv, w.detach().to(dev), dout.reshape(B).to(dev), dx=base.clone(), accumulate=True)
        close(dx2, x.grad + base.cpu(), GRAD_TOL)


def test_kat_fm_gradient(dev):
    k = K()
    # KAT-FM dX on a D=4 padded copy (zero columns do not change sums)
    x = torch.zeros(2, 3, 4)
    x[:, :, :2] = torch.from_numpy(kat.FM_X)
    w = torch.zeros(4, 1)
    w[:2] = torch.from_numpy(kat.FM_W)
    dx, _, _ = k.fm_bwd(x.to(dev), w.to(dev), torch.ones(2, device=dev))
    np.testing.assert_allclose(dx.cpu().numpy()[:, :, :2], kat.FM_DX, rtol=1e-6, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# a13: embedding backward (sorted segments)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("V,D,n", [(50, 8, 5000), (100003, 16, 20000), (7, 4, 1), (3, 32, 4097), (1000, 64, 999)])
def test_embedding_bwd_dense(dev, V, D, n):
    k = K()
    g = torch.Generator().manual_seed(n)
    ids = torch.randint(0, V, (n,), generator=g, dtype=torch.int32)
    dout = rnd(n, D, seed=V)
    table = rnd(V, D, seed=2)
    want = oracle.embedding_grad_dense(V, ids, dout, table, l2=1e-3)
    got = k.embedding_bwd_dense(ids.to(dev), dout.to(dev), V, table.to(dev), l2_scale=2e-3)
    close(got, want, GRAD_TOL)
    got0 = k.embedding_bwd_dense(ids.to(dev), dout.to(dev), V)
    close(got0, oracle.embedding_grad_dense(V, ids, dout), GRAD_TOL)
    # deterministic: bitwise identical on a second run
    assert torch.equal(got0, k.embedding_bwd_dense(ids.to(dev), dout.to(dev), V))


@pytest.mark.parametrize("V,D,n,dist", [(3953, 32, 204800, "zipf"), (1000, 16, 50000, "one"), (300000, 64, 120000, "zipf"), (5000, 8, 3000, "two")])
def test_embedding_bwd_dense_long_runs(dev, V, D, n, dist):
    """Skewed ids put 10^3..10^5 positions on one row: those runs leave the chunk/merge chain for the run-time long-row pass
    (lookup.cu: bwd_long_detect_kernel + slice kernels).  Same sums as index_add, bit-reproducible."""
    k = K()
    if dist == "zipf":
        ids = _zipf_ids(n, V, 1.05, 5)
    elif dist == "one":
        ids = torch.full((n,), 7, dtype=torch.int32)
        ids[::9] = 8
    else:  # two runs of 257..511 positions (the boundary of the classification) between short ones
        g = torch.Generator().manual_seed(1)
        ids = torch.randint(0, V, (n,), generator=g, dtype=torch.int32)
        ids[:300] = 11
        ids[300:811] = 12
    dout = rnd(n, D, seed=V, scale=1.0 / 64)
    want = oracle.embedding_grad_dense(V, ids, dout)
    got = k.embedding_bwd_dense(ids.to(dev), dout.to(dev), V)
    close(got, want, GRAD_TOL)
    assert torch.equal(got, k.embedding_bwd_dense(ids.to(dev), dout.to(dev), V))


@pytest.mark.parametrize("pool", ["mean", "sum"])
@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_group_lookup_bwd_update(dev, pool, opt):
    """One optimiser step on every table == autograd of the oracle lookup + the same update rule."""
    k = K()
    B = 513
    names, tables, ids, fields, o_sparse, o_seq, D = _c1_like_group(seed=11, B=B, pool=pool)
    from collections import OrderedDict

    leaf = {n: t.clone().requires_grad_(True) for n, t in tables.items()}
    o_sparse = OrderedDict((n, (leaf[n], v[1], v[2])) for n, v in o_sparse.items())
    o_seq = OrderedDict((("hist_movie", (leaf["movie_id"], o_seq["hist_movie"][1])), ("genres", (leaf["genre_id"], o_seq["genres"][1]))))
    out = oracle.concat([], oracle.group_embedding_lookup(o_sparse, o_seq, pool))
    dout = rnd(B, out.shape[1], seed=5)
    (out * dout).sum().backward()
    lr = 0.1
    dev_tables = [tables[n].clone().to(dev) for n in names]
    if opt == "sgd":
        plan = k.LookupPlan(dev_tables, fields)
        plan.backward_update(ids.to(dev), dout.to(dev), opt="sgd", lr=lr)
        for i, n in enumerate(names):
            want = tables[n] - lr * leaf[n].grad
            close(dev_tables[i], want, GRAD_TOL)
    else:
        ms = [torch.zeros_like(t) for t in dev_tables]
        vs = [torch.zeros_like(t) for t in dev_tables]
        plan = k.LookupPlan(dev_tables, fields, adam_m=ms, adam_v=vs)
        plan.backward_update(ids.to(dev), dout.to(dev), opt="adam", lr=lr, step=1)
        for i, n in enumerate(names):
            gr = leaf[n].grad
            m = 0.1 * gr
            v = 0.001 * gr * gr
            lr_t = lr * np.sqrt(1 - 0.999) / (1 - 0.9)
            # untouched rows have m = v = 0 -> no movement: the lazy row update equals dense Keras Adam at step 1
            want = tables[n] - lr_t * m / (v.sqrt() + 1e-7)
            close(dev_tables[i], want, 2e-4)


def test_group_lookup_bwd_hot_rows(dev):
    """Tiny vocabularies -> thousands of duplicates per row: long segments crossing many chunks."""
    k = K()
    B, D = 20000, 16
    vocabs = [2, 3, 5, 40000]
    tables = [rnd(v, D, seed=v, scale=0.05) for v in vocabs]
    g = torch.Generator().manual_seed(1)
    ids = torch.stack([torch.randint(0, v, (B,), generator=g, dtype=torch.int32) for v in vocabs], 1)
    dout = rnd(B, 4 * D, seed=2)
    dev_tables = [t.clone().to(dev) for t in tables]
    plan = k.LookupPlan(dev_tables, [(f, 1, "none", f, f * D) for f in range(4)])
    plan.backward_update(ids.to(dev), dout.to(dev), opt="sgd", lr=1.0)
    for f, v in enumerate(vocabs):
        want = tables[f] - oracle.embedding_grad_dense(v, ids[:, f], dout[:, f * D : (f + 1) * D])
        close(dev_tables[f], want, GRAD_TOL)


def test_shared_table_two_fields_bwd(dev):
    """movie_id as a sparse feature AND as the unit of hist_movie: gradients of both fields meet in one row."""
    k = K()
    B, D, V = 300, 8, 20
    table = rnd(V, D, seed=1, scale=0.05)
    g = torch.Generator().manual_seed(3)
    mid = torch.randint(0, V, (B, 1), generator=g, dtype=torch.int32)
    hist = rand_ids(B, 4, V, seed=4)
    ids = torch.cat([mid, hist], 1)
    leaf = table.clone().requires_grad_(True)
    e1, _ = oracle.custom_embedding(leaf, mid, True)
    e2 = oracle.sequence_pooling(*oracle.custom_embedding(leaf, hist, True), "mean")
    out = oracle.concat([], [e1, e2])
    dout = rnd(B, 2 * D, seed=6)
    (out * dout).sum().backward()
    dt = table.clone().to(dev)
    plan = k.LookupPlan([dt], [(0, 1, "none", 0, 0), (0, 4, "mean", 1, D)])
    plan.backward_update(ids.to(dev), dout.to(dev), opt="sgd", lr=0.5)
    close(dt, table - 0.5 * leaf.grad, GRAD_TOL)


def _zipf_ids(B, V, a, seed):
    """Zipf(a) over [1, V): inverse CDF of the continuous approximation (bench.py --ids zipf)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(B, generator=g, dtype=torch.float64)
    x = ((V ** (1 - a) - 1) * u + 1) ** (1 / (1 - a))
    return x.long().clamp_(1, V - 1).to(torch.int32)


@pytest.mark.parametrize("algo", ["units", "sort"])
@pytest.mark.parametrize("opt", ["sgd", "adam"])
@pytest.mark.parametrize("B,dist", [(65536, "zipf"), (30001, "uniform"), (65536, "onehot")])
def test_group_lookup_bwd_unit_path_skew(dev, opt, B, dist, algo):
    """The sort-free backward (embedding_bwd.cu) under skew: Zipf ids (histogram splits, single hot rows inside big tables),
    one id for the whole batch (a row with 65536 positions), tiny tables (slices), a batch that is not a multiple of 16;
    a dense-updated table next to in-place ones; deterministic bit for bit."""
    k = K()
    D = 16
    vocabs = [4, 11, 300, 5000, 250000, 2000000]
    tables = [rnd(v, D, seed=v, scale=0.05) for v in vocabs]
    if dist == "zipf":
        ids = torch.stack([_zipf_ids(B, v, 1.05, 10 + f) for f, v in enumerate(vocabs)], 1)
    elif dist == "uniform":
        g = torch.Generator().manual_seed(2)
        ids = torch.stack([torch.randint(0, v, (B,), generator=g, dtype=torch.int32) for v in vocabs], 1)
    else:
        ids = torch.stack([torch.full((B,), min(3, v - 1), dtype=torch.int32) for v in vocabs], 1)
        ids[::7, 5] = 123456
    dout = rnd(B, len(vocabs) * D, seed=3, scale=1.0 / 256)
    fields = [(f, 1, "none", f, f * D) for f in range(len(vocabs))]
    lr = 0.5

    def run():
        dt = [t.clone().to(dev) for t in tables]
        ms = [torch.zeros_like(t) for t in dt] if opt == "adam" else None
        vs = [torch.zeros_like(t) for t in dt] if opt == "adam" else None
        plan = k.LookupPlan(dt, fields, adam_m=ms, adam_v=vs)
        dense_g = torch.zeros_like(dt[3])
        plan.set_dense_grads([None, None, None, dense_g, None, None])  # table 3 is "dense-updated": gradient sums only
        from handyrec_b200 import _lib

        _lib.call("hrb_plan_set_bwd_algo", plan._h, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT)
        plan.backward_update(ids.to(dev), dout.to(dev), opt=opt, lr=lr, step=1)
        torch.cuda.synchronize()
        return dt, dense_g

    dt, dense_g = run()
    for f, v in enumerate(vocabs):
        gr = oracle.embedding_grad_dense(v, ids[:, f], dout[:, f * D : (f + 1) * D])
        if f == 3:
            close(dense_g, gr, GRAD_TOL)
            assert torch.equal(dt[3].cpu(), tables[3])
        elif opt == "sgd":
            close(dt[f], tables[f] - lr * gr, GRAD_TOL)
        else:
            lr_t = lr * np.sqrt(1 - 0.999) / (1 - 0.9)
            want = tables[f] - lr_t * (0.1 * gr) / ((0.001 * gr * gr).sqrt() + 1e-7)
            touched = torch.zeros(v, dtype=torch.bool)
            touched[ids[:, f].long()] = True
            # rows whose summed gradient is ~0 make m/(sqrt(v)+eps) ill-conditioned: compare the well-conditioned ones
            ok = (gr.abs() > 1e-6).all(1) | ~touched
            close(dt[f].cpu()[ok], want[ok], 5e-4)
            assert torch.equal(dt[f].cpu()[~touched], tables[f][~touched])
    dt2, dense_g2 = run()
    assert all(torch.equal(a, b) for a, b in zip(dt, dt2)) and torch.equal(dense_g, dense_g2), "backward is not deterministic"


def test_group_lookup_bwd_unit_path_mixed_dims_and_sequences(dev):
    """Tables of different widths (G = 2 and 8), a long mean-pooled history sharing its table with a plain feature, and a
    sum-pooled one: every position of every column is reduced into the right row with the right 1/n_valid scale."""
    k = K()
    B = 4099
    Vm, Vg, Vu = 3953, 19, 6041
    Dm, Dg = 32, 8
    t_m, t_g, t_u = rnd(Vm, Dm, seed=1, scale=0.05), rnd(Vg, Dg, seed=2, scale=0.05), rnd(Vu, Dm, seed=3, scale=0.05)
    g = torch.Generator().manual_seed(5)
    uid = torch.randint(0, Vu, (B, 1), generator=g, dtype=torch.int32)
    mid = torch.randint(0, Vm, (B, 1), generator=g, dtype=torch.int32)
    hist = rand_ids(B, 50, Vm, seed=6)
    genres = rand_ids(B, 6, Vg, seed=7)
    ids = torch.cat([uid, mid, hist, genres], 1)
    leaf = [t.clone().requires_grad_(True) for t in (t_u, t_m, t_g)]
    e_u, _ = oracle.custom_embedding(leaf[0], uid, False)
    e_m, _ = oracle.custom_embedding(leaf[1], mid, True)
    e_h = oracle.sequence_pooling(*oracle.custom_embedding(leaf[1], hist, True), "mean")
    e_g = oracle.sequence_pooling(*oracle.custom_embedding(leaf[2], genres, True), "sum")
    out = torch.cat([e_u[:, 0], e_m[:, 0], e_h[:, 0], e_g[:, 0]], 1)
    dout = rnd(B, out.shape[1], seed=8)
    (out * dout).sum().backward()
    dt = [t.clone().to(dev) for t in (t_u, t_m, t_g)]
    fields = [(0, 1, "none", 0, 0), (1, 1, "none", 1, Dm), (1, 50, "mean", 2, 2 * Dm), (2, 6, "sum", 52, 3 * Dm)]
    plan = k.LookupPlan(dt, fields)
    plan.backward_update(ids.to(dev), dout.to(dev), opt="sgd", lr=0.25)
    for got, t0, lf in zip(dt, (t_u, t_m, t_g), leaf):
        close(got, t0 - 0.25 * lf.grad, GRAD_TOL)


# ------------------------------------------------------------------------------------------------
# a11: Dense, Dice
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,Kd,N,act", [(1024, 429, 429, "relu"), (1000, 429, 256, "relu"), (513, 128, 1, None), (5, 57, 8, "sigmoid"), (300, 84, 128, "tanh"), (128, 16, 432, "relu")])
def test_dense_fwd_bwd(dev, M, Kd, N, act):
    k = K()
    x = rnd(M, Kd, seed=1).requires_grad_(True)
    W = (rnd(Kd, N, seed=2) / np.sqrt(Kd)).requires_grad_(True)
    b = rnd(N, seed=3, scale=0.1).requires_grad_(True)
    y = oracle.activation(act, oracle.dense(x.double(), W.double(), b.double()))
    got = k.dense_fwd(x.detach().to(dev), W.detach().to(dev), b.detach().to(dev), act)
    close(got, y.float(), FWD_TOL)
    dy = rnd(M, N, seed=4)
    y.backward(dy.double())
    dz = k.act_bwd(got, dy.to(dev), act)
    dx = k.dense_bwd_x(dz, W.detach().to(dev))
    dw, db = k.dense_bwd_w(x.detach().to(dev), dz)
    close(dx, x.grad, GRAD_TOL)
    close(dw, W.grad, GRAD_TOL)
    close(db, b.grad, GRAD_TOL)


def test_dense_bwd_x_fused_activation_grad_and_padded_ld(dev):
    k = K()
    M, Kd, N = 777, 429, 256
    ld = 432
    a_prev_buf = torch.zeros(M, ld)
    a_prev = torch.relu(rnd(M, Kd, seed=1))
    a_prev_buf[:, :Kd] = a_prev
    W = rnd(Kd, N, seed=2) / 20
    dz = rnd(M, N, seed=3)
    want = (dz.double() @ W.double().T) * (a_prev > 0)
    dbuf = a_prev_buf.to(dev)
    out = torch.zeros(M, ld, device=dev)
    k.dense_bwd_x(dz.to(dev), W.to(dev), a_prev=dbuf[:, :Kd], act_prev="relu", out=out[:, :Kd])
    close(out[:, :Kd], want.float(), GRAD_TOL)
    assert float(out[:, Kd:].abs().max()) == 0.0  # padding columns untouched


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("shape", [(4096, 128), (64, 50, 32), (7, 36), (204800, 128), (4096, 50, 32)])
def test_dice_fwd_bwd(dev, training, shape):
    k = K()
    units = shape[-1]
    x = rnd(*shape, seed=1).double().requires_grad_(True)
    alpha = rnd(units, seed=2, scale=0.3).double().requires_grad_(True)
    mm, mv = rnd(units, seed=3, scale=0.1), torch.rand(units, generator=torch.Generator().manual_seed(4)) + 0.5
    want = oracle.dice(x, alpha, mm.double(), mv.double(), training=training)
    dmean, dvar = mm.clone().to(dev), mv.clone().to(dev)
    got = k.dice_fwd(x.detach().float().to(dev), alpha.detach().float().to(dev), dmean, dvar, training)
    close(got, want, FWD_TOL)
    if training:
        red = tuple(range(len(shape) - 1))
        close(dmean, x.detach().mean(red), FWD_TOL)
        close(dvar, x.detach().var(red, unbiased=False), 1e-4)
    dy = rnd(*shape, seed=5)
    want.backward(dy.double())
    dx, dalpha = k.dice_bwd(x.detach().float().to(dev), dy.to(dev), alpha.detach().float().to(dev), dmean, dvar, training)
    close(dx, x.grad, GRAD_TOL)
    close(dalpha, alpha.grad, GRAD_TOL)


# ------------------------------------------------------------------------------------------------
# a10: DIN local activation unit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("act", ["sigmoid", "relu", "dice"])
@pytest.mark.parametrize("B,T,D,hidden", [(64, 50, 32, (32, 1)), (5, 2, 8, (36, 1)), (130, 7, 16, (64, 32, 1)), (33, 7, 4, (16, 1)),
                                         (200, 1, 32, (32, 1)), (50, 13, 64, (64, 8, 1))])
def test_lau_fwd(dev, act, B, T, D, hidden):
    k = K()
    V = 3953
    table = rnd(V, D, seed=1, scale=0.05)
    g = torch.Generator().manual_seed(2)
    qid = torch.randint(1, V, (B, 1), generator=g, dtype=torch.int32)
    kid = rand_ids(B, T, V, seed=3)
    p = oracle.dnn_init(4 * D, hidden, seed=4)
    for i in range(len(p.units)):
        p.b[i] = rnd(p.units[i], seed=10 + i, scale=0.1)
        p.dice_alpha[i] = rnd(p.units[i], seed=20 + i, scale=0.3)
        p.dice_mean[i] = rnd(p.units[i], seed=30 + i, scale=0.1)
        p.dice_var[i] = torch.rand(p.units[i], generator=g) + 0.5
    q, _ = oracle.custom_embedding(table, qid, True)
    keys, kmask = oracle.custom_embedding(table, kid, True)
    keys, kmask2 = oracle.squeeze_mask(keys, kmask)
    want_score = oracle.local_activation_unit(q, keys, kmask2, p, act=act, training=False)
    want_pooled = oracle.din_attention_pool(want_score, keys)
    dice = [(p.dice_alpha[i].to(dev), p.dice_mean[i].to(dev), p.dice_var[i].to(dev)) for i in range(len(p.units))] if act == "dice" else None
    params = k.lau_pack_params([w.to(dev) for w in p.W], [b.to(dev) for b in p.b], dice)
    score, pooled = k.lau_fwd(table.to(dev), qid.reshape(B).to(dev), kid.to(dev), params, p.units, act)
    assert score.shape == (B, 1, T) and pooled.shape == (B, 1, D)
    close(score, want_score, FWD_TOL)
    close(pooled, want_pooled, FWD_TOL)
    # mask is exact: padded positions score exactly 0
    assert np.array_equal(score.cpu().numpy()[:, 0][kid.numpy() == 0], np.zeros(int((kid == 0).sum()), np.float32))


# ------------------------------------------------------------------------------------------------
# head, optimisers
# ------------------------------------------------------------------------------------------------
def test_sigmoid_bce_and_optimisers(dev):
    k = K()
    B = 10007
    a, b = rnd(B, seed=1, scale=3), rnd(B, seed=2)
    y = (torch.rand(B, generator=torch.Generator().manual_seed(3)) < 0.25).float()
    logit = (a + b).clone().requires_grad_(True)
    loss = oracle.bce_from_logits(logit, y)
    loss.backward()
    prob, dl, ls = torch.empty(B, device=dev), torch.empty(B, device=dev), torch.zeros(1, device=dev)
    k.sigmoid_bce(a.to(dev), b.to(dev), y.to(dev), 1.0 / B, prob, dl, ls)
    close(prob, torch.sigmoid(logit.detach()), FWD_TOL)
    close(dl, logit.grad, GRAD_TOL)
    close(ls / B, loss.detach().reshape(1), FWD_TOL)
    p0, g0 = rnd(5000, seed=4), rnd(5000, seed=5)
    p, m, v = p0.clone().to(dev), torch.zeros(5000, device=dev), torch.zeros(5000, device=dev)
    ref, rm, rv = p0.double(), torch.zeros(5000, dtype=torch.float64), torch.zeros(5000, dtype=torch.float64)
    for step in (1, 2, 3):  # Keras Adam: lr_t = lr*sqrt(1-b2^t)/(1-b1^t); w -= lr_t*m/(sqrt(v)+eps)
        gg = g0.double() * step
        rm = 0.9 * rm + 0.1 * gg
        rv = 0.999 * rv + 0.001 * gg * gg
        ref = ref - 1e-2 * np.sqrt(1 - 0.999 ** step) / (1 - 0.9 ** step) * rm / (rv.sqrt() + 1e-7)
        k.adam_step(p, (g0 * step).to(dev), m, v, lr=1e-2, step=step)
    close(p, ref.float(), FWD_TOL)
    q = p0.clone().to(dev)
    k.sgd_step(q, g0.to(dev), lr=0.1, l2_scale=2e-3)
    close(q, p0 - 0.1 * (g0 + 2e-3 * p0), FWD_TOL)


def test_multi_tensor_optimizer_steps_match_the_single_tensor_ones(dev):
    """hrb_adam_step_multi / hrb_sgd_step_multi: 37 tensors of odd sizes (two launches of <= 32) == one hrb_adam_step / hrb_sgd_step each."""
    k = K()
    sizes = [1, 3, 7, 128, 1000, 4097, 65536 + 5] + [11 * i + 1 for i in range(30)]
    ps = [rnd(n, seed=100 + i) for i, n in enumerate(sizes)]
    gs = [rnd(n, seed=300 + i) for i, n in enumerate(sizes)]
    l2 = [0.0 if i % 3 else 2e-3 for i in range(len(sizes))]
    a = [p.clone().to(dev) for p in ps]
    am, av = [torch.zeros_like(t) for t in a], [torch.zeros_like(t) for t in a]
    b = [p.clone().to(dev) for p in ps]
    bm, bv = [torch.zeros_like(t) for t in b], [torch.zeros_like(t) for t in b]
    gd = [g.to(dev) for g in gs]
    for step in (1, 2):
        k.adam_step_multi(a, gd, am, av, l2, 1e-2, step=step)
        for i in range(len(sizes)):
            k.adam_step(b[i], gd[i], bm[i], bv[i], lr=1e-2, step=step, l2_scale=l2[i])
    for i in range(len(sizes)):  # same formulas; the two kernels may contract a*b+c differently, so equal to rounding, not bit for bit
        close(a[i], b[i], 1e-6)
        close(am[i], bm[i], 1e-6)
        close(av[i], bv[i], 1e-6)
    c = [p.clone().to(dev) for p in ps]
    d = [p.clone().to(dev) for p in ps]
    k.sgd_step_multi(c, gd, l2, 0.1)
    for i in range(len(sizes)):
        k.sgd_step(d[i], gd[i], lr=0.1, l2_scale=l2[i])
        close(c[i], d[i], 1e-6)
    k.adam_step_multi([], [], [], [], [], 1e-2)  # nothing to do


# ------------------------------------------------------------------------------------------------
# a11: BatchNormalization / Dropout inside DNN (layers/core.py:71-73)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(777, 37), (64, 50, 36), (4096, 128), (3, 5), (204800, 128), (4096, 50, 32)])
@pytest.mark.parametrize("training", [True, False])
def test_batchnorm_fwd_bwd(dev, shape, training):
    """hrb_batchnorm_fwd/bwd against oracle.batch_norm + autograd: training (biased batch statistics over every axis but the
    last) and inference (moving statistics), 2-D and 3-D inputs, affine parameters, Keras eps = 1e-3."""
    from handyrec_b200.autograd_ops import BatchNormFn

    u = shape[-1]
    x = (rnd(*shape, seed=1) * 1.7 + 0.3).double().requires_grad_(True)
    gamma = (1.0 + 0.2 * rnd(u, seed=2)).double().requires_grad_(True)
    beta = (0.1 * rnd(u, seed=3)).double().requires_grad_(True)
    mm, mv = 0.2 * rnd(u, seed=4), 0.5 + rnd(u, seed=5).abs()
    dy = rnd(*shape, seed=6)
    y, bm, bv = oracle.batch_norm(x, mm.double(), mv.double(), gamma, beta, 1e-3, training)
    (y * dy.double()).sum().backward()
    xd = x.detach().float().to(dev).requires_grad_(True)
    gd, bd = gamma.detach().float().to(dev).requires_grad_(True), beta.detach().float().to(dev).requires_grad_(True)
    yd = BatchNormFn.apply(xd, gd, bd, mm.to(dev), mv.to(dev), training, 1e-3)
    close(yd, y, FWD_TOL)
    if training:
        got_m, got_v = yd.grad_fn.batch_stats
        close(got_m, bm, FWD_TOL)
        close(got_v, bv, FWD_TOL)
    (yd * dy.to(dev)).sum().backward()
    close(xd.grad, x.grad, GRAD_TOL)
    close(gd.grad, gamma.grad, GRAD_TOL)
    close(bd.grad, beta.grad, GRAD_TOL)


@pytest.mark.parametrize("training", [True, False])
def test_batchnorm_bwd_empty_batch_zeroes_parameter_gradients(dev, training):
    """rows = 0: the gradients of gamma and beta are sums over no rows, i.e. 0 -- written, not left as whatever the output buffers
    held (BatchNormFn allocates them uninitialised)."""
    from handyrec_b200._lib import call

    k = K()
    u = 37
    x, dy, dx, dgamma, dbeta, scratch = (torch.full((n,), float("nan"), device=dev) for n in (u, u, u, u, u, 2 * u))
    gamma, mean, var = torch.ones(u, device=dev), torch.zeros(u, device=dev), torch.ones(u, device=dev)
    call("hrb_batchnorm_bwd", k._p(x), k._p(dy), 0, u, k._p(gamma), k._p(mean), k._p(var), 1e-3, int(training), k._p(dx), k._p(dgamma),
         k._p(dbeta), k._p(scratch), k._stream())
    assert torch.equal(dgamma.cpu(), torch.zeros(u)) and torch.equal(dbeta.cpu(), torch.zeros(u))
    assert bool(dx.isnan().all())  # no rows: nothing else is written


@pytest.mark.parametrize("rate", [0.1, 0.5, 0.9])
def test_dropout_mask_scale_and_backward(dev, rate):
    """hrb_dropout: survivors are scaled by exactly 1/(1-rate) (Keras Dropout in training mode), the keep mask is a pure function
    of (seed, element index) -- so the backward (the same call on dy) uses the SAME mask, a second call reproduces it bit for
    bit, another seed gives another mask -- and the keep fraction is 1-rate within sampling error."""
    from handyrec_b200.autograd_ops import DropoutFn

    n = 1 << 20
    x = (rnd(n, seed=1).abs() + 0.5).to(dev).requires_grad_(True)
    y = DropoutFn.apply(x, rate, 1234)
    keep = y != 0
    frac = float(keep.float().mean())
    assert abs(frac - (1 - rate)) < 4 * np.sqrt(rate * (1 - rate) / n) + 1e-4, frac
    want = torch.where(keep, x.detach() * np.float32(1.0 / (1.0 - rate)), torch.zeros_like(y))
    assert torch.allclose(y.detach(), want, rtol=1e-6, atol=0)
    assert torch.equal(y.detach(), DropoutFn.apply(x.detach(), rate, 1234))
    assert not torch.equal(keep, DropoutFn.apply(x.detach(), rate, 1235) != 0)
    dy = rnd(n, seed=2).to(dev)
    y.backward(dy)
    want_dx = torch.where(keep, dy * np.float32(1.0 / (1.0 - rate)), torch.zeros_like(dy))
    assert torch.allclose(x.grad, want_dx, rtol=1e-6, atol=0)


def test_clipped_bce_matches_keras_probability_path(dev):
    """Keras binary_crossentropy without cached logits: clip to [1e-7, 1-1e-7], mean over the batch, gradient 0 where clipped."""
    from handyrec_b200.autograd_ops import ClippedBCEFn

    g = torch.Generator().manual_seed(0)
    p = torch.rand(5000, 1, generator=g)
    p[:5] = torch.tensor([[0.0], [1.0], [1e-9], [1 - 1e-9], [0.5]])
    y = (torch.rand(5000, 1, generator=g) < 0.3).float()
    pl = p.clone().requires_grad_(True)
    # Keras clips in fp32 with fp32 constants (1 - 1e-7 rounds to 1 - 1.19e-7); the sums are taken in float64 here
    pc = torch.clamp(pl, float(np.float32(1e-7)), float(np.float32(1.0) - np.float32(1e-7)))
    want = -(y * torch.log(pc.double()) + (1 - y) * torch.log1p(-pc.double())).mean()
    want.backward()
    pd = p.to(dev).requires_grad_(True)
    got = ClippedBCEFn.apply(pd, y.to(dev))
    assert abs(float(got.detach()) - float(want.detach())) < 1e-5 * max(1.0, abs(float(want.detach())))
    got.backward()
    inner = (p > 1e-6) & (p < 1 - 1e-6)
    close(pd.grad[inner], pl.grad[inner].float(), GRAD_TOL)
    assert float(pd.grad[0]) == 0.0 and float(pd.grad[1]) == 0.0
