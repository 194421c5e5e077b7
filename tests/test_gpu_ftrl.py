"""GPU: Keras Ftrl -- the dense steps, the touched-rows embedding update on both backward algorithms (Keras' sparse Ftrl, padding
row 0 of pooled fields included), the fused and sharded DeepFM engines, and the Model API."""
import numpy as np
import pytest
import torch

import oracle
from oracle.ftrl_ref import ftrl_dense
from tests.test_gpu_adagrad import _zipf_ids
from tests.test_gpu_api import _deepfm_data, _deepfm_model, _retrieval_data, _retrieval_groups
from tests.test_gpu_engine import _oracle_step
from tests.test_gpu_parity import close, rand_ids, rnd

pytestmark = pytest.mark.gpu

HYPER = dict(l1=0.05, l2=0.01, lr_power=-0.5, l2_shrinkage=0.0)


def _near_l1(lin, l1):
    """Elements whose |linear| lies within fp32 rounding of l1: the select may go either way there."""
    return (lin.abs() - l1).abs() <= 1e-5 * max(l1, 1.0)


# ---- 1. dense steps --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lr_power,l1,l2,shrink,l2_scale", [(-0.5, 0.0, 0.0, 0.0, 0.0), (-0.5, 0.02, 0.1, 0.0, 1e-2),
                                                            (0.0, 0.01, 0.0, 0.05, 0.0), (-1.0, 0.0, 0.3, 0.0, 0.0)])
def test_ftrl_step_matches_the_oracle(dev, lr_power, l1, l2, shrink, l2_scale):
    from handyrec_b200 import kernels as K

    n, lr = 100_003, 0.05
    p0 = rnd(n, seed=1)
    p, acc, lin = p0.to(dev), torch.full((n,), 0.1, device=dev), torch.zeros(n, device=dev)
    wp, wa, wl = p0.double(), torch.full((n,), 0.1, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    amb = torch.zeros(n, dtype=torch.bool)
    kw = dict(l1=l1, l2=l2, lr_power=lr_power, l2_shrinkage=shrink)
    for s in range(3):
        g = rnd(n, seed=10 + s)
        K.ftrl_step(p, g.to(dev), acc, lin, lr, l2_scale=l2_scale, **kw)
        wp, wa, wl = ftrl_dense(wp, wa, wl, g, lr, l2_scale=l2_scale, **kw)
        amb |= _near_l1(wl, l1)
    ok = ~amb
    close(p.cpu()[ok], wp[ok], 1e-5)
    close(acc.cpu()[ok], wa[ok], 1e-5)
    close(lin.cpu()[ok], wl[ok], 1e-5)


def test_ftrl_step_row_touched_leaves_other_rows_bit_identical(dev):
    from handyrec_b200 import kernels as K

    rows, D = 5001, 12
    p0 = rnd(rows, D, seed=2)
    p, acc, lin = p0.clone().to(dev), torch.full((rows, D), 0.1, device=dev), rnd(rows, D, seed=3).to(dev)
    acc0, lin0 = acc.clone(), lin.clone()
    touched = (torch.rand(rows, generator=torch.Generator().manual_seed(4)) < 0.3).float()
    g = rnd(rows, D, seed=5).to(dev)
    K.ftrl_step(p, g, acc, lin, 0.1, row_touched=touched.to(dev), dim=D, **HYPER)
    full = [p0.clone().to(dev), acc0.clone(), lin0.clone()]
    K.ftrl_step(full[0], g, full[1], full[2], 0.1, **HYPER)
    t = touched.bool()
    assert torch.equal(p.cpu()[~t], p0[~t]) and torch.equal(acc[~t.to(dev)], acc0[~t.to(dev)]) and torch.equal(lin[~t.to(dev)], lin0[~t.to(dev)])
    for a, b in zip((p, acc, lin), full):  # touched rows: exactly the unmasked step
        assert torch.equal(a[t.to(dev)], b[t.to(dev)])


def test_ftrl_step_multi_matches_the_single_tensor_kernel(dev):
    """37 tensors of odd sizes (two launches of <= 32) == one hrb_ftrl_step each, bit for bit."""
    from handyrec_b200 import kernels as K

    sizes = [1, 3, 7, 128, 1000, 4097, 65536 + 5] + [11 * i + 1 for i in range(30)]
    ps = [rnd(n, seed=100 + i) for i, n in enumerate(sizes)]
    l2s = [0.0 if i % 3 else 2e-3 for i in range(len(sizes))]
    a = [[p.clone().to(dev), torch.full((p.numel(),), 0.1, device=dev), torch.zeros(p.numel(), device=dev)] for p in ps]
    b = [[p.clone().to(dev), torch.full((p.numel(),), 0.1, device=dev), torch.zeros(p.numel(), device=dev)] for p in ps]
    for step in range(3):
        gd = [rnd(n, seed=300 + 50 * step + i).to(dev) for i, n in enumerate(sizes)]
        K.ftrl_step_multi([x[0] for x in a], gd, [x[1] for x in a], [x[2] for x in a], l2s, 1e-2, **HYPER)
        for i in range(len(sizes)):
            K.ftrl_step(b[i][0], gd[i], b[i][1], b[i][2], 1e-2, l2_scale=l2s[i], **HYPER)
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            assert torch.equal(u, v)


# ---- 2. the embedding backward: touched rows == Keras' sparse Ftrl --------------------------------------------------------------
def _oracle_sparse_grads(shapes, fields, ids, dout):
    """Per-table gradient sums and touched rows in float64: plain fields name every in-range id; pooled fields name every position
    (padding id 0 included, with a zero gradient), the valid ones taking 1/n_valid (mean) of the row."""
    G = [torch.zeros(v, d, dtype=torch.float64) for v, d in shapes]
    T = [torch.zeros(v, dtype=torch.bool) for v, _ in shapes]
    dout = dout.double()
    for ti, L, pool, ids_col, out_col in fields:
        d = shapes[ti][1]
        cols = ids[:, ids_col : ids_col + L].long()
        g = dout[:, out_col : out_col + d]
        T[ti][cols.reshape(-1)] = True
        if pool == "none":
            for l in range(L):
                G[ti].index_add_(0, cols[:, l], g)
            continue
        valid = cols != 0
        n = valid.sum(1, keepdim=True).double()
        scale = torch.where(n > 0, 1.0 / n.clamp(min=1), torch.zeros_like(n)) if pool == "mean" else torch.ones_like(n)
        for l in range(L):
            keep = valid[:, l]
            G[ti].index_add_(0, cols[keep, l], g[keep] * scale[keep])
    return G, T


def _run_bwd_case(dev, shapes, fields, batches, algo, lr=0.01, acc0=0.1, hyper=HYPER):
    """Three backward_update(opt="ftrl") steps from one initial state, run twice (bit-equal); checked against float64 Keras sparse
    Ftrl stepping exactly the touched rows of each batch."""
    from handyrec_b200 import kernels as K
    from handyrec_b200._lib import call

    g = torch.Generator().manual_seed(len(shapes))
    tables0 = [(torch.rand(v, d, generator=g) - 0.5) * 0.1 for v, d in shapes]

    def run():
        w = [t.to(dev) for t in tables0]
        acc = [torch.full_like(t, acc0) for t in w]
        lin = [torch.zeros_like(t) for t in w]
        plan = K.LookupPlan(w, fields, accum=acc, linear=lin)
        call("hrb_plan_set_bwd_algo", plan._h, algo)
        for ids, dout in batches:
            plan.backward_update(ids.to(dev), dout.to(dev), opt="ftrl", lr=lr, **hyper)
        torch.cuda.synchronize()
        return [t.cpu() for t in w], [a.cpu() for a in acc], [l.cpu() for l in lin]

    r1, r2 = run(), run()
    for x, y in zip(sum(r1, []), sum(r2, [])):
        assert torch.equal(x, y)  # deterministic
    w1, a1, l1_ = r1
    ww = [t.double() for t in tables0]
    wa = [torch.full(t.shape, acc0, dtype=torch.float64) for t in tables0]
    wl = [torch.zeros(t.shape, dtype=torch.float64) for t in tables0]
    amb = [torch.zeros(t.shape, dtype=torch.bool) for t in tables0]
    ever = [torch.zeros(v, dtype=torch.bool) for v, _ in shapes]
    for ids, dout in batches:
        G, T = _oracle_sparse_grads(shapes, fields, ids, dout)
        for t in range(len(shapes)):
            r = T[t]
            ever[t] |= r
            nw, na, nl = ftrl_dense(ww[t][r], wa[t][r], wl[t][r], G[t][r], lr, **hyper)
            ww[t][r], wa[t][r], wl[t][r] = nw, na, nl
            amb[t][r] |= _near_l1(nl, hyper["l1"])
    zeroed = 0
    for t in range(len(shapes)):
        ok = ~amb[t]
        close(w1[t][ok], ww[t][ok], 1e-4)
        close(a1[t][ok], wa[t][ok], 1e-4)
        close(l1_[t][ok], wl[t][ok], 1e-4)
        un = ~ever[t]
        assert torch.equal(w1[t][un], tables0[t][un]) and bool((a1[t][un] == acc0).all()) and bool((l1_[t][un] == 0).all())
        zeroed += int(((w1[t] == 0) & ever[t][:, None]).sum())
    return zeroed


@pytest.mark.parametrize("dist", ["uniform", "zipf", "one"])
@pytest.mark.parametrize("algo", ["units", "sort"])
def test_backward_update_ftrl_is_keras_sparse_ftrl(dev, algo, dist):
    from handyrec_b200 import _lib

    B, D = 30001, 16
    vocabs = [4, 1000, 100_000, 2_000_000]
    shapes = [(v, D) for v in vocabs]
    fields = [(t, 1, "none", t, t * D) for t in range(len(vocabs))]
    batches = []
    for step in range(3):
        cols = []
        for t, v in enumerate(vocabs):
            if dist == "uniform":
                c = torch.randint(0, v, (B,), generator=torch.Generator().manual_seed(100 * step + t), dtype=torch.int32)
            elif dist == "zipf":
                c = _zipf_ids(B, v, 100 * step + t)
            else:
                c = torch.full((B,), (7 * step + 1) % v, dtype=torch.int32)
            cols.append(c)
        batches.append((torch.stack(cols, 1).contiguous(), rnd(B, len(vocabs) * D, seed=50 + step, scale=0.1)))
    zeroed = _run_bwd_case(dev, shapes, fields, batches, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT)
    if dist != "one":  # one id per table sums a whole batch of gradient rows: its |linear| is far above l1
        assert zeroed > 0  # l1 set some touched elements to exactly 0


@pytest.mark.parametrize("shrink", [0.0, 0.2])
@pytest.mark.parametrize("plain_zero", [False, True])
@pytest.mark.parametrize("algo", ["units", "sort"])
def test_backward_update_ftrl_padding_steps_row_zero_once(dev, algo, plain_zero, shrink):
    """A mean-pooled field with padding: row 0 of its table takes exactly one step per batch -- with the gradient of a plain field
    that also names id 0 (plain_zero), else with a zero gradient."""
    from handyrec_b200 import _lib

    B = 4099
    shapes = [(1000, 8), (300_000, 16), (20, 4)]
    fields = [(0, 1, "none", 0, 0), (1, 4, "mean", 1, 8), (1, 1, "none", 5, 24), (2, 3, "mean", 6, 40)]
    batches = []
    for step in range(3):
        g = torch.Generator().manual_seed(step)
        plain = torch.randint(1, 300_000, (B, 1), generator=g, dtype=torch.int32)
        if plain_zero:
            plain[:: 7] = 0
        ids = torch.cat([torch.randint(0, 1000, (B, 1), generator=g, dtype=torch.int32), rand_ids(B, 4, 300_000, seed=10 + step),
                         plain, rand_ids(B, 3, 20, seed=20 + step)], 1).contiguous()
        ids[:, 1:5][ids[:, 1:5] == 0] = 1
        ids[::3, 3:5] = 0  # padding in every third sample
        batches.append((ids, rnd(B, 52, seed=30 + step, scale=0.1)))
    hyper = dict(HYPER, l2_shrinkage=shrink)
    _run_bwd_case(dev, shapes, fields, batches, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT, hyper=hyper)


def test_ftrl_without_slots_raises(dev):
    from handyrec_b200 import kernels as K
    from handyrec_b200._lib import HrbError

    w = [torch.zeros(100, 8, device=dev)]
    ids = torch.randint(0, 50, (64, 1), dtype=torch.int32, device=dev)
    plan = K.LookupPlan(w, [(0, 1, "none", 0, 0)], accum=[torch.zeros_like(w[0])])
    with pytest.raises(HrbError, match="Ftrl"):
        plan.backward_update(ids, torch.ones(64, 8, device=dev), opt="ftrl", lr=0.1)


# ---- 3. the fused DeepFM engine ------------------------------------------------------------------------------------------------
def test_engine_ftrl_dense_updated_tables_step_touched_rows_only(dev):
    """l2_embd = 0: the dense-updated tables step the rows the batch gathers (the padding row 0 of a pooled field included) and
    nothing else; the in-place tables likewise.  Two steps against the oracle."""
    from handyrec_b200.engine import DeepFMEngine

    B, D, n_dense, hidden, lr, acc0 = 64, 8, 2, (8, 1), 0.05, 0.1
    vocabs = [7, 50, 1000]
    tables = [rnd(v, D, seed=20 + i, scale=0.05) for i, v in enumerate(vocabs)]
    fields = [(0, 1, "none"), (2, 1, "none"), (1, 3, "mean")]  # reference order: plain fields first, then sequences
    kw = dict(l1=0.001, l2=0.01, learning_rate_power=-0.5, l2_shrinkage=0.0, beta=0.1)
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer="ftrl", lr=lr,
                       dense_table_max_rows=50, **kw)
    assert eng.dense_tables == [0, 1] and eng.touched is not None
    k_l2 = kw["l2"] + kw["beta"] / (2 * lr)
    hyp = dict(l1=kw["l1"], l2=k_l2, lr_power=-0.5)
    slots = [(torch.full_like(t, acc0).double(), torch.zeros_like(t).double()) for t in tables]
    cur = [t.clone() for t in tables]
    ever = [torch.zeros(v, dtype=torch.bool) for v in vocabs]
    for step in (1, 2):
        g = torch.Generator().manual_seed(100 + step)
        ids = torch.cat([torch.randint(0, 7, (B, 1), generator=g, dtype=torch.int32), torch.randint(0, 1000, (B, 1), generator=g, dtype=torch.int32),
                         torch.randint(1, 50, (B, 3), generator=g, dtype=torch.int32)], 1)
        ids[::4, 3:5] = 0  # padding
        dense, label = rnd(B, n_dense, seed=step), (torch.rand(B, generator=g) < 0.3).float()
        leaf, *_ = _oracle_step(eng, cur, fields, ids, dense, label, B, hidden)
        eng.train_step_on_device(ids.to(dev), dense.to(dev), label.to(dev))
        col = {0: ids[:, 0:1], 1: ids[:, 2:5], 2: ids[:, 1:2]}
        for t in range(3):
            rows = torch.zeros(vocabs[t], dtype=torch.bool)
            rows[col[t].long().reshape(-1)] = True
            ever[t] |= rows
            a, l = slots[t]
            nw, na, nl = ftrl_dense(cur[t][rows], a[rows], l[rows], leaf[t].grad[rows], lr, **hyp)
            want = cur[t].double().clone()
            want[rows], a[rows], l[rows] = nw, na, nl
            got = eng.tables[t].cpu()
            close(got, want, 2e-4)
            assert torch.equal(got[~ever[t]], tables[t][~ever[t]])  # never-touched rows keep their bits
            if t not in eng.dense_tables:
                close(eng.accum[t], a, 2e-4)
                close(eng.linear[t], l, 2e-4)
        cur = [t_.cpu().clone() for t_ in eng.tables]
    assert bool(ever[1][0])  # row 0 of the pooled table was stepped through its padding


def test_engine_ftrl_step_at_bench_configuration(dev):
    """ONE Ftrl step of the bench.py configuration (B = 65536, 26 plain fields, D = 16, 429-256-128-1, tcgen05, 17 dense-updated
    tables) against the oracle: every touched row is the float64 Ftrl step of its oracle gradient, every other row keeps its bits.
    learning_rate_power = 0: the 1/B-scaled row gradients are ~1e-7, and with lr_power = -0.5 the fp32 accumulator 0.1 + g^2 rounds
    to 0.1 or its neighbour, which decides sqrt(acc') - sqrt(acc) entirely (the other tests cover lr_power = -0.5)."""
    from handyrec_b200.engine import DeepFMEngine

    B, D, n_dense, hidden = 65536, 16, 13, (256, 128, 1)
    criteo = [40_000_000, 40_000_000, 10_000_000, 5_000_000, 3_000_000, 2_000_000, 1_000_000, 500_000, 300_000, 100_000,
              50_000, 20_000, 12_000, 10_000, 7_000, 5_000, 2_000, 1_500, 1_000, 600, 300, 100, 30, 20, 10, 4]
    vocabs = [min(v + 1, 200_000) for v in criteo]
    tables = [torch.from_numpy(oracle.hash_uniform_table(v, D, seed=7 + f)) for f, v in enumerate(vocabs)]
    fields = [(f, 1, "none") for f in range(len(vocabs))]
    g = torch.Generator().manual_seed(1234)
    ids = torch.stack([torch.randint(0, v, (B,), generator=g, dtype=torch.int32) for v in vocabs], 1)
    dense = torch.log1p(torch.empty(B, n_dense).exponential_(1.0, generator=g))
    label = (torch.rand(B, generator=g) < 0.25).float()
    lr = 0.05
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer="ftrl", lr=lr,
                       dense_table_max_rows=131072, learning_rate_power=0.0)
    assert eng.use_tc and len(eng.dense_tables) == 17
    leaf, p, fm_w, fm_w0, logit, loss = _oracle_step(eng, tables, fields, ids, dense, label, B, hidden)
    eng.train_step_on_device(ids.to(dev), dense.to(dev), label.to(dev))
    torch.cuda.synchronize()
    close(eng.loss_sum / B, loss.detach().reshape(1), 1e-5)
    with torch.no_grad():  # samples whose ReLU pre-activation lies within rounding of 0 are left out (see the Adagrad test)
        x = torch.cat([dense] + [tables[t][ids[:, t].long()] for t in range(len(vocabs))], 1)
        amb = torch.zeros(B, dtype=torch.bool)
        for i in range(len(eng.units) - 1):
            z = x @ p.W[i].detach() + p.b[i].detach()
            amb |= (z.abs() < 2e-6 * z.abs().max()).any(1)
            x = torch.relu(z)
    assert int(amb.sum()) < B // 20
    for t, lf in enumerate(leaf):
        got = eng.tables[t].cpu()
        touched = torch.zeros(vocabs[t], dtype=torch.bool)
        touched[ids[:, t].long()] = True
        clean = touched.clone()
        clean[ids[amb, t].long()] = False
        want, _, _ = ftrl_dense(tables[t][clean], torch.full((int(clean.sum()), D), 0.1), torch.zeros(int(clean.sum()), D), lf.grad[clean], lr,
                                lr_power=0.0)
        close(got[clean], want, 1e-4)
        assert torch.equal(got[~touched], tables[t][~touched])


# ---- 4. Model API --------------------------------------------------------------------------------------------------------------
def test_model_fit_with_ftrl_fused_matches_the_layer_path(dev):
    from handyrec_b200 import keras_lite as KL

    n, bs = 700, 256
    x, y = _deepfm_data(n)
    fused, plain = _deepfm_model(), _deepfm_model()
    plain.fuse = False
    opt = lambda: KL.Ftrl(learning_rate=0.1, l1_regularization_strength=1e-3, l2_regularization_strength=1e-3, beta=0.1)
    fused.compile(optimizer=opt(), loss=KL.binary_crossentropy)
    plain.compile(optimizer=opt(), loss=KL.binary_crossentropy)
    assert fused._fused is not None and plain._fused is None
    hf = fused.fit(x, y, batch_size=bs, epochs=2)
    hp = plain.fit(x, y, batch_size=bs, epochs=2)
    assert fused._fused.engine.optimizer == "ftrl" and fused._fused.engine.step_count == 6
    np.testing.assert_allclose(hf.history["loss"], hp.history["loss"], rtol=2e-4)
    pf, pp = fused.predict(x, batch_size=300), plain.predict(x, batch_size=300)
    np.testing.assert_allclose(pf, pp, rtol=2e-3, atol=2e-5)
    for lf, lp in zip(fused.layers, plain.layers):
        for a, b in zip(lf.get_weights(), lp.get_weights()):
            close(a, b, 2e-3)


# ---- 5. sharded engine on emulated ranks ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("rep", [0, 60])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_engine_ftrl_matches_single_gpu_engine(dev, world, rep):
    """Two Ftrl steps of N emulated ranks (a mean-pooled field with padding on a row-sharded table; tables <= rep rows replicated
    with their touched flags all-reduced) == one engine on the concatenated batches."""
    from handyrec_b200.engine import DeepFMEngine
    from handyrec_b200.sharded import ShardedDeepFMEngine
    from tests import shard_helpers as H
    from tests.test_gpu_sharded import _run_threads

    b, D, n_dense, hidden = 64, 8, 3, (16, 1)
    g = torch.Generator().manual_seed(1)
    vocabs = [11, 50, 300]
    tables = [(torch.rand(v, D, generator=g) - 0.5) * 0.1 for v in vocabs]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 3, "mean")]
    kw = dict(optimizer="ftrl", lr=0.1, seed=7, l1=1e-3, l2=1e-3, l2_shrinkage=0.01)
    steps = []
    for _ in range(2):
        ids = []
        for _ in range(world):
            i = torch.cat([torch.randint(0, 11, (b, 1), generator=g, dtype=torch.int32), torch.randint(1, 50, (b, 1), generator=g, dtype=torch.int32),
                           torch.randint(1, 300, (b, 3), generator=g, dtype=torch.int32)], 1)
            i[::3, 3:5] = 0
            ids.append(i)
        dense = [torch.randn(b, n_dense, generator=g) for _ in range(world)]
        label = [(torch.rand(b, generator=g) < 0.3).float() for _ in range(world)]
        steps.append((ids, dense, label))
    ref = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=b * world, dense_table_max_rows=rep, **kw)
    for ids, dense, label in steps:
        ref.train_step_on_device(torch.cat(ids).to(dev), torch.cat(dense).to(dev), torch.cat(label).to(dev))
    torch.cuda.synchronize()
    shared = H.ThreadComm.Shared(world)
    engines = [None] * world

    def rank_fn(r):
        sh = [(full if v <= rep else s_).to(dev) for full, s_, v in zip(tables, H.shards_of(tables, r, world), vocabs)]
        comm = H.ThreadComm(shared, r)
        eng = ShardedDeepFMEngine(sh, vocabs, fields, n_dense, comm, dnn_hidden_units=hidden, dnn_activation="relu", batch_size=b,
                                  replicate_max_rows=rep, **kw)
        engines[r] = eng
        for ids, dense, label in steps:
            eng.train_step_on_device(ids[r].to(dev), dense[r].to(dev), label[r].to(dev))
        torch.cuda.synchronize()
        return float(eng.loss_sum)

    losses = _run_threads(world, rank_fn)
    assert abs(sum(losses) - float(ref.loss_sum)) < 1e-4 * abs(float(ref.loss_sum))
    for r in range(world):
        close(engines[r].params, ref.params, 1e-4)
        close(engines[r].opt_m, ref.opt_m, 1e-4)
        close(engines[r].opt_v, ref.opt_v, 1e-4)
        for t in range(len(vocabs)):
            ws = ref.tables[t] if vocabs[t] <= rep else ref.tables[t][r::world]
            close(engines[r].tables[t][: ws.shape[0]], ws, 1e-4)
            if vocabs[t] > rep:
                close(engines[r].accum[t][: ws.shape[0]], ref.accum[t][r::world], 1e-4)
                close(engines[r].linear[t][: ws.shape[0]], ref.linear[t][r::world], 1e-4)


# ---- 6. the layer-by-layer models ----------------------------------------------------------------------------------------------
def test_din_fits_with_ftrl(dev):
    from handyrec_b200.config import ConfigLoader
    from handyrec_b200.keras_lite import Ftrl, binary_crossentropy
    from handyrec_b200.models import DIN
    from tests.test_gpu_models import _data
    from tests.test_mirror_cpu import DIN_CFG, FEATURE_DIM

    g = ConfigLoader(DIN_CFG).prepare_features(FEATURE_DIM)
    model = DIN(g["item_seq_feat_group"], g["other_feature_group"], dnn_hidden_units=(8,), lau_dnn_hidden_units=(8, 1))
    x, y = _data(200, seed=3)
    model.compile(optimizer=Ftrl(learning_rate=0.1), loss=binary_crossentropy)
    h = model.fit(x=x, y=y, batch_size=50, epochs=2)
    loss = h.history["loss"]
    assert np.isfinite(loss).all() and loss[1] < loss[0]
    assert len(model.optimizer.state) > 0


def test_youtube_match_dnn_fits_with_ftrl(dev):
    import handyrec_b200.models as M
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding, SampledSoftmaxLayer
    from handyrec_b200.layers.utils import sampledsoftmaxloss

    n_items, B = 60, 100
    ug, ig, _ = _retrieval_groups(n_items)
    m = M.YouTubeMatchDNN(ug, ig, dnn_hidden_units=(16, 8), num_sampled=10)
    m.compile(optimizer=KL.Ftrl(0.5), loss=sampledsoftmaxloss)
    x = _retrieval_data(B, n_items)
    ssl = [l for l in m.layers if isinstance(l, SampledSoftmaxLayer)][0]
    sampled, tries = oracle.log_uniform_sample(10, n_items, np.random.RandomState(5))
    ssl.sampled_values = (sampled, oracle.unique_expected_count(oracle.log_uniform_prob(x["movie_id"].reshape(-1), n_items), tries),
                          oracle.unique_expected_count(oracle.log_uniform_prob(sampled, n_items), tries))
    h = m.fit(x=[(x, np.zeros(B))] * 4, epochs=2)
    loss = h.history["loss"]
    assert np.isfinite(loss).all() and loss[1] < loss[0]
    cat = [l for l in m.layers if isinstance(l, CustomEmbedding) and l.input_dim == n_items]
    assert any(getattr(l, "_linear", None) is not None for l in cat)  # l2 = 0 under Ftrl: touched-rows update at any size
