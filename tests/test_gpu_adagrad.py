"""GPU: Keras Adagrad -- the dense steps, the touched-rows-only embedding update on both backward algorithms (exactly Keras'
sparse Adagrad), the fused and sharded DeepFM engines, and the Model API."""
import numpy as np
import pytest
import torch

import oracle
from oracle.optim_ref import adagrad_dense
from tests.test_gpu_api import _deepfm_data, _deepfm_model, _retrieval_data, _retrieval_groups
from tests.test_gpu_engine import _oracle_step
from tests.test_gpu_parity import close, rand_ids, rnd

pytestmark = pytest.mark.gpu


# ---- 1. dense steps --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("l2", [0.0, 1e-2])
def test_adagrad_step_matches_the_formula(dev, l2):
    from handyrec_b200 import kernels as K

    n, lr = 100_003, 0.05
    p0 = rnd(n, seed=1)
    p, acc = p0.to(dev), torch.full((n,), 0.1, device=dev)
    want_p, want_acc = p0.double(), torch.full((n,), 0.1, dtype=torch.float64)
    for s in range(3):
        g = rnd(n, seed=10 + s)
        K.adagrad_step(p, g.to(dev), acc, lr, eps=1e-7, l2_scale=l2)
        want_p, want_acc = adagrad_dense(want_p, want_acc, g, lr, 1e-7, l2)
    close(p, want_p, 1e-5)
    close(acc, want_acc, 1e-5)


def test_adagrad_step_multi_matches_the_single_tensor_kernel(dev):
    """37 tensors of odd sizes (two launches of <= 32) == one hrb_adagrad_step each."""
    from handyrec_b200 import kernels as K

    sizes = [1, 3, 7, 128, 1000, 4097, 65536 + 5] + [11 * i + 1 for i in range(30)]
    ps = [rnd(n, seed=100 + i) for i, n in enumerate(sizes)]
    l2 = [0.0 if i % 3 else 2e-3 for i in range(len(sizes))]
    a = [p.clone().to(dev) for p in ps]
    b = [p.clone().to(dev) for p in ps]
    aa = [torch.full_like(t, 0.1) for t in a]
    ba = [torch.full_like(t, 0.1) for t in b]
    for step in range(3):
        gd = [rnd(n, seed=300 + 50 * step + i).to(dev) for i, n in enumerate(sizes)]
        K.adagrad_step_multi(a, gd, aa, l2, 1e-2, eps=1e-7)
        for i in range(len(sizes)):
            K.adagrad_step(b[i], gd[i], ba[i], 1e-2, eps=1e-7, l2_scale=l2[i])
    for i in range(len(sizes)):
        close(a[i], b[i], 1e-6)
        close(aa[i], ba[i], 1e-6)
    K.adagrad_step_multi([], [], [], [], 1e-2)  # nothing to do


# ---- 2. the embedding backward: touched rows only == Keras' dense Adagrad over every row --------------------------------------
def _oracle_table_grads(shapes, fields, ids, dout):
    """Per-table gradient sums in float64 (plain fields: every id; mean-pooled fields: ids != 0, each 1/n_valid of the row)."""
    G = [torch.zeros(v, d, dtype=torch.float64) for v, d in shapes]
    dout = dout.double()
    for ti, L, pool, ids_col, out_col in fields:
        d = shapes[ti][1]
        cols = ids[:, ids_col : ids_col + L].long()
        g = dout[:, out_col : out_col + d]
        if pool == "none":
            G[ti].index_add_(0, cols[:, 0], g)
            continue
        valid = cols != 0
        n = valid.sum(1, keepdim=True).double()
        scale = torch.where(n > 0, 1.0 / n.clamp(min=1), torch.zeros_like(n))
        for l in range(L):
            keep = valid[:, l]
            G[ti].index_add_(0, cols[keep, l], g[keep] * scale[keep])
    return G


def _zipf_ids(B, V, seed):
    z = np.random.RandomState(seed).zipf(1.05, B)
    return torch.from_numpy(((z - 1) % V).astype(np.int32))


def _run_bwd_case(dev, shapes, fields, batches, algo, dense_t=None, lr=0.01, eps=1e-7, acc0=0.1):
    """Three backward_update(opt="adagrad") steps from one initial state, run twice; checked against float64 Keras Adagrad applied
    densely to every row of every table."""
    from handyrec_b200 import kernels as K
    from handyrec_b200._lib import call

    g = torch.Generator().manual_seed(len(shapes))
    tables0 = [(torch.rand(v, d, generator=g) - 0.5) * 0.1 for v, d in shapes]

    def run():
        w = [t.to(dev) for t in tables0]
        acc = [None if i == dense_t else torch.full_like(t, acc0) for i, t in enumerate(w)]
        plan = K.LookupPlan(w, fields, accum=acc)
        call("hrb_plan_set_bwd_algo", plan._h, algo)
        gbuf, gsums = None, []
        if dense_t is not None:
            gbuf = torch.zeros_like(w[dense_t])
            plan.set_dense_grads([gbuf if i == dense_t else None for i in range(len(w))])
        for ids, dout in batches:
            if gbuf is not None:
                gbuf.zero_()
            plan.backward_update(ids.to(dev), dout.to(dev), opt="adagrad", lr=lr, eps=eps)
            if gbuf is not None:
                gsums.append(gbuf.cpu())
        torch.cuda.synchronize()
        return [t.cpu() for t in w], [a.cpu() if a is not None else None for a in acc], gsums

    w1, a1, gs1 = run()
    w2, a2, gs2 = run()
    for x, y in zip(w1 + [a for a in a1 if a is not None] + gs1, w2 + [a for a in a2 if a is not None] + gs2):
        assert torch.equal(x, y)  # deterministic: fixed summation order, no atomics
    want_w = [t.double() for t in tables0]
    want_a = [torch.full(t.shape, acc0, dtype=torch.float64) for t in tables0]
    touched = [torch.zeros(v, dtype=torch.bool) for v, _ in shapes]
    for step, (ids, dout) in enumerate(batches):
        G = _oracle_table_grads(shapes, fields, ids, dout)
        for t in range(len(shapes)):
            touched[t] |= G[t].abs().sum(1) > 0
            if t == dense_t:
                close(gs1[step], G[t], 1e-4)
            else:
                want_w[t], want_a[t] = adagrad_dense(want_w[t], want_a[t], G[t], lr, eps)
    for t in range(len(shapes)):
        if t == dense_t:
            assert torch.equal(w1[t], tables0[t])  # a dense-gradient table only receives its gradient sum
            continue
        close(w1[t], want_w[t], 1e-4)
        close(a1[t], want_a[t], 1e-4)
        un = ~touched[t]
        assert torch.equal(w1[t][un], tables0[t][un])
        assert bool((a1[t][un] == torch.tensor(acc0, dtype=torch.float32)).all())


@pytest.mark.parametrize("dist", ["uniform", "zipf", "one"])
@pytest.mark.parametrize("B", [30001, 65536])
@pytest.mark.parametrize("algo", ["units", "sort"])
def test_backward_update_adagrad_is_keras_adagrad(dev, algo, B, dist):
    from handyrec_b200 import _lib

    D = 16
    vocabs = [4, 1000, 100_000, 2_000_000, 50]  # the last one is dense-gradient (reduced, not updated)
    shapes = [(v, D) for v in vocabs]
    fields = [(t, 1, "none", t, t * D) for t in range(len(vocabs))]
    batches = []
    for step in range(3):  # three steps on different ids
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
    _run_bwd_case(dev, shapes, fields, batches, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT, dense_t=len(vocabs) - 1)


@pytest.mark.parametrize("algo", ["units", "sort"])
def test_backward_update_adagrad_mixed_dims_and_mean_pooling(dev, algo):
    from handyrec_b200 import _lib

    B = 30001
    shapes = [(1000, 8), (300_000, 16), (50_000, 32), (20, 4)]
    # (table, seq_len, pool, ids_col, out_col): plain fields and mean-pooled sequences (id 0 = padding), table 1 shared
    fields = [(0, 1, "none", 0, 0), (1, 1, "none", 1, 8), (2, 5, "mean", 2, 24), (1, 3, "mean", 7, 56), (3, 1, "none", 10, 72)]
    batches = []
    for step in range(3):
        g = torch.Generator().manual_seed(step)
        ids = torch.cat([torch.randint(0, 1000, (B, 1), generator=g, dtype=torch.int32),
                         torch.randint(0, 300_000, (B, 1), generator=g, dtype=torch.int32),
                         rand_ids(B, 5, 50_000, seed=10 + step), rand_ids(B, 3, 300_000, seed=20 + step),
                         torch.randint(0, 20, (B, 1), generator=g, dtype=torch.int32)], 1).contiguous()
        batches.append((ids, rnd(B, 76, seed=30 + step, scale=0.1)))
    _run_bwd_case(dev, shapes, fields, batches, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT)


# ---- 3. a row-updated table without an accumulator -----------------------------------------------------------------------------
def test_adagrad_without_accumulator_raises(dev):
    from handyrec_b200 import kernels as K
    from handyrec_b200._lib import HrbError

    w = [torch.zeros(100, 8, device=dev), torch.zeros(50, 8, device=dev)]
    ids = torch.randint(0, 50, (64, 2), dtype=torch.int32, device=dev)
    dout = torch.ones(64, 16, device=dev)
    fields = [(0, 1, "none", 0, 0), (1, 1, "none", 1, 8)]
    for acc in (None, [torch.zeros_like(w[0]), None]):
        plan = K.LookupPlan(w, fields, accum=acc)
        with pytest.raises(HrbError, match="Adagrad"):
            plan.backward_update(ids, dout, opt="adagrad", lr=0.1)
    with pytest.raises(ValueError):
        K.LookupPlan(w, fields, adam_m=[torch.zeros_like(t) for t in w], accum=[torch.zeros_like(t) for t in w])


# ---- 4./5. the fused DeepFM engine ---------------------------------------------------------------------------------------------
def test_engine_adagrad_dense_updated_and_in_place_tables(dev):
    """With l2_embd > 0 the dense-updated tables step every row (Keras: dense gradient) while in-place tables step only the touched
    rows.  Two steps on different batches, every table and accumulator against the oracle."""
    from handyrec_b200.engine import DeepFMEngine

    B, D, n_dense, hidden, lr, l2, acc0 = 64, 8, 2, (8, 1), 0.05, 0.01, 0.1
    vocabs = [7, 50, 1000]
    tables = [rnd(v, D, seed=20 + i, scale=0.05) for i, v in enumerate(vocabs)]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 1, "none")]
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer="adagrad", lr=lr,
                       l2_embd=l2, dense_table_max_rows=50)
    assert eng.dense_tables == [0, 1] and eng.opt_v is None and eng.initial_accumulator_value == acc0
    assert eng.accum[0] is None and eng.accum[1] is None and bool((eng.accum[2] == acc0).all())
    acc = [torch.full_like(t, acc0) for t in tables]
    cur = [t.clone() for t in tables]
    for step in (1, 2):
        g = torch.Generator().manual_seed(100 + step)
        ids = torch.cat([torch.randint(0, vv, (B, 1), generator=g, dtype=torch.int32) for vv in vocabs], 1)
        dense, label = rnd(B, n_dense, seed=step), (torch.rand(B, generator=g) < 0.3).float()
        leaf, *_ = _oracle_step(eng, cur, fields, ids, dense, label, B, hidden)
        eng.train_step_on_device(ids.to(dev), dense.to(dev), label.to(dev))
        for t in range(3):
            touched = torch.zeros(vocabs[t], dtype=torch.bool)
            touched[ids[:, t].long()] = True
            rows = torch.ones_like(touched) if t in eng.dense_tables else touched
            gt = (leaf[t].grad + 2 * l2 * cur[t]) * rows[:, None]
            acc[t] = acc[t] + gt * gt
            cur[t] = cur[t] - lr * gt / (acc[t].sqrt() + 1e-7)
            close(eng.tables[t], cur[t], 2e-4)
            if t not in eng.dense_tables:
                close(eng.accum[t], acc[t], 2e-4)
                assert torch.equal(eng.tables[t].cpu()[~rows], cur[t][~rows])
        cur = [t_.cpu().clone() for t_ in eng.tables]  # the next oracle step starts from the engine's state


def test_engine_adagrad_step_at_bench_configuration(dev):
    """ONE Adagrad step of the bench.py configuration (B = 65536, 26 plain fields, D = 16, 429-256-128-1, tcgen05, 17 dense-updated
    tables next to in-place ones) against the oracle.  lr is large so that the 1/B-scaled row gradients move the fp32 rows visibly;
    with acc = 0.1 + g^2 (g ~ 1e-7) the row step is lr * g / sqrt(0.1) to rounding."""
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
    lr = 1000.0 * float(np.sqrt(0.1))  # the same row movement as the SGD case's lr = 1000
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer="adagrad", lr=lr,
                       dense_table_max_rows=131072)
    assert eng.use_tc and len(eng.dense_tables) == 17
    leaf, p, fm_w, fm_w0, logit, loss = _oracle_step(eng, tables, fields, ids, dense, label, B, hidden)
    prob = eng.predict_on_device(ids.to(dev), dense.to(dev))
    close(prob, torch.sigmoid(logit[:, 0]), 1e-5)
    eng.train_step_on_device(ids.to(dev), dense.to(dev), label.to(dev))
    torch.cuda.synchronize()
    close(eng.loss_sum / B, loss.detach().reshape(1), 1e-5)
    for i in range(len(eng.units)):
        dw, db = eng.get_dense_grads(i)
        close(dw, p.W[i].grad, 1e-4)
        close(db, p.b[i].grad, 1e-4)
    close(eng.d_fm[: eng.D], fm_w.grad[:, 0], 1e-4)
    # samples whose ReLU pre-activation lies within rounding of 0 are left out (test_engine_step_at_bench_configuration explains why)
    with torch.no_grad():
        x = torch.cat([dense] + [tables[t][ids[:, t].long()] for t in range(len(vocabs))], 1)
        amb = torch.zeros(B, dtype=torch.bool)
        for i in range(len(eng.units) - 1):
            z = x @ p.W[i].detach() + p.b[i].detach()
            amb |= (z.abs() < 2e-6 * z.abs().max()).any(1)
            x = torch.relu(z)
    assert int(amb.sum()) < B // 20
    for t, lf in enumerate(leaf):
        gr = lf.grad
        got = eng.tables[t].cpu()
        touched = torch.zeros(vocabs[t], dtype=torch.bool)
        touched[ids[:, t].long()] = True
        clean = torch.ones(vocabs[t], dtype=torch.bool)
        clean[ids[amb, t].long()] = False
        step_to_grad = (gr.double() ** 2 + 0.1).sqrt() + 1e-7
        close((((tables[t] - got).double() * step_to_grad) / lr)[clean], gr[clean].double(), 1e-4)
        assert torch.equal(got[~touched], tables[t][~touched])
        if t not in eng.dense_tables:
            close(eng.accum[t].cpu()[clean], (0.1 + gr.double() ** 2)[clean], 1e-6)


# ---- 6. Model API --------------------------------------------------------------------------------------------------------------
def test_model_fit_with_adagrad_fused_matches_the_layer_path(dev):
    from handyrec_b200 import keras_lite as KL

    n, bs = 700, 256
    x, y = _deepfm_data(n)
    fused, plain = _deepfm_model(), _deepfm_model()
    plain.fuse = False
    fused.compile(optimizer=KL.Adagrad(learning_rate=0.1), loss=KL.binary_crossentropy)
    plain.compile(optimizer=KL.Adagrad(learning_rate=0.1), loss=KL.binary_crossentropy)
    assert fused._fused is not None and plain._fused is None
    hf = fused.fit(x, y, batch_size=bs, epochs=2)
    hp = plain.fit(x, y, batch_size=bs, epochs=2)
    assert fused._fused.engine is not None and fused._fused.engine.optimizer == "adagrad" and fused._fused.engine.step_count == 6
    np.testing.assert_allclose(hf.history["loss"], hp.history["loss"], rtol=2e-4)
    pf, pp = fused.predict(x, batch_size=300), plain.predict(x, batch_size=300)
    np.testing.assert_allclose(pf, pp, rtol=2e-3, atol=2e-5)
    for lf, lp in zip(fused.layers, plain.layers):
        for a, b in zip(lf.get_weights(), lp.get_weights()):
            close(a, b, 2e-3)


def test_sparse_row_updates_equal_the_dense_adagrad_step(dev):
    """Tables above SPARSE_UPDATE_MIN_ROWS take the touched-rows-only update (apply_sparse), the others Keras' dense step: with
    l2 = 0 the two agree at every step (for Adam only at step 1)."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding

    x, y = _deepfm_data(300)
    res = {}
    for thr in (10, 1 << 30):
        CustomEmbedding.SPARSE_UPDATE_MIN_ROWS = thr
        try:
            m = _deepfm_model(hidden=(8, 1))
            m.fuse = False
            m.compile(optimizer=KL.Adagrad(0.1), loss=KL.binary_crossentropy)
            losses = [m.train_on_batch({k: v[s : s + 100] for k, v in x.items()}, y[s : s + 100]) for s in (0, 100, 200)]
            embs = [lay for lay in m.layers if isinstance(lay, CustomEmbedding)]
            if thr == 10:
                assert any(getattr(lay, "_accum", None) is not None for lay in embs)
            res[thr] = (losses, {lay.name: lay.get_weights()[0] for lay in embs})
        finally:
            CustomEmbedding.SPARSE_UPDATE_MIN_ROWS = 131072
    np.testing.assert_allclose(res[10][0], res[1 << 30][0], rtol=1e-4)
    for k in res[10][1]:
        close(res[10][1][k], res[1 << 30][1][k], 1e-4)


# ---- 7. sharded engine on emulated ranks ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("rep", [0, 60])
@pytest.mark.parametrize("peer", [True, False])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_engine_adagrad_matches_single_gpu_engine(dev, world, peer, rep):
    """Two Adagrad steps of N emulated ranks (large tables row-sharded with their accumulators, tables <= rep rows replicated with
    theirs in the flat buffer) == one engine on the concatenated batches."""
    from handyrec_b200.engine import DeepFMEngine
    from handyrec_b200.sharded import ShardedDeepFMEngine
    from tests import shard_helpers as H
    from tests.test_gpu_sharded import _run_threads

    b, D, n_dense, hidden = 64, 8, 3, (16, 1)
    g = torch.Generator().manual_seed(1)
    vocabs = [11, 50, 300]
    tables = [(torch.rand(v, D, generator=g) - 0.5) * 0.1 for v in vocabs]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 1, "none")]
    steps = []
    for _ in range(2):
        ids = [torch.stack([torch.randint(0, v, (b,), generator=g, dtype=torch.int32) for v in vocabs], 1) for _ in range(world)]
        dense = [torch.randn(b, n_dense, generator=g) for _ in range(world)]
        label = [(torch.rand(b, generator=g) < 0.3).float() for _ in range(world)]
        steps.append((ids, dense, label))
    ref = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=b * world, optimizer="adagrad", lr=0.1,
                       seed=7, dense_table_max_rows=rep)
    for ids, dense, label in steps:
        ref.train_step_on_device(torch.cat(ids).to(dev), torch.cat(dense).to(dev), torch.cat(label).to(dev))
    torch.cuda.synchronize()
    shared = H.ThreadComm.Shared(world)
    engines = [None] * world

    def rank_fn(r):
        sh = [(full if v <= rep else s_).to(dev) for full, s_, v in zip(tables, H.shards_of(tables, r, world), vocabs)]
        comm = H.ThreadComm(shared, r)
        peer_ptrs = comm.share_ptrs(sh) if peer else None
        eng = ShardedDeepFMEngine(sh, vocabs, fields, n_dense, comm, peer_ptrs=peer_ptrs, dnn_hidden_units=hidden, dnn_activation="relu",
                                  batch_size=b, optimizer="adagrad", lr=0.1, seed=7, replicate_max_rows=rep)
        assert eng.peer_lookup == peer
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
        for t in range(len(vocabs)):
            ws = ref.tables[t] if vocabs[t] <= rep else ref.tables[t][r::world]
            if ws.shape[0]:
                close(engines[r].tables[t][: ws.shape[0]], ws, 1e-4)
            if vocabs[t] > rep:
                wa = ref.accum[t][r::world]
                close(engines[r].accum[t][: wa.shape[0]], wa, 1e-4)


# ---- 8. the layer-by-layer models ----------------------------------------------------------------------------------------------
def test_din_fits_with_adagrad(dev):
    from handyrec_b200.config import ConfigLoader
    from handyrec_b200.keras_lite import Adagrad, binary_crossentropy
    from handyrec_b200.models import DIN
    from tests.test_gpu_models import _data
    from tests.test_mirror_cpu import DIN_CFG, FEATURE_DIM

    g = ConfigLoader(DIN_CFG).prepare_features(FEATURE_DIM)
    model = DIN(g["item_seq_feat_group"], g["other_feature_group"], dnn_hidden_units=(8,), lau_dnn_hidden_units=(8, 1))
    x, y = _data(200, seed=3)
    model.compile(optimizer=Adagrad(learning_rate=0.1), loss=binary_crossentropy)
    h = model.fit(x=x, y=y, batch_size=50, epochs=2)
    loss = h.history["loss"]
    assert np.isfinite(loss).all() and loss[1] < loss[0]
    assert len(model.optimizer.state) > 0


def test_youtube_match_dnn_fits_with_adagrad_and_the_catalogue_takes_apply_sparse(dev):
    import handyrec_b200.models as M
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding, SampledSoftmaxLayer
    from handyrec_b200.layers.utils import sampledsoftmaxloss

    n_items, B = 60, 100
    CustomEmbedding.SPARSE_UPDATE_MIN_ROWS = n_items  # the catalogue (n_items rows) takes the touched-rows-only update
    try:
        ug, ig, _ = _retrieval_groups(n_items)
        m = M.YouTubeMatchDNN(ug, ig, dnn_hidden_units=(16, 8), num_sampled=10)
        m.compile(optimizer=KL.Adagrad(0.5), loss=sampledsoftmaxloss)
        x = _retrieval_data(B, n_items)
        ssl = [l for l in m.layers if isinstance(l, SampledSoftmaxLayer)][0]
        sampled, tries = oracle.log_uniform_sample(10, n_items, np.random.RandomState(5))
        ssl.sampled_values = (sampled, oracle.unique_expected_count(oracle.log_uniform_prob(x["movie_id"].reshape(-1), n_items), tries),
                              oracle.unique_expected_count(oracle.log_uniform_prob(sampled, n_items), tries))
        h = m.fit(x=[(x, np.zeros(B))] * 4, epochs=2)  # candidates pinned: a fixed objective
        loss = h.history["loss"]
        assert np.isfinite(loss).all() and loss[1] < loss[0]
        cat = [l for l in m.layers if isinstance(l, CustomEmbedding) and l.input_dim == n_items]
        assert any(getattr(l, "_accum", None) is not None for l in cat)
    finally:
        CustomEmbedding.SPARSE_UPDATE_MIN_ROWS = 131072
