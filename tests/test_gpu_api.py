"""GPU: the reference-shaped API (feature groups -> model constructor -> compile / fit / predict) on the fused paths, and the
retrieval loss pieces against the oracle."""
import numpy as np
import pytest
import torch

import oracle
from tests.test_gpu_parity import close, rand_ids, rnd

pytestmark = pytest.mark.gpu


def _deepfm_model(seed=0, hidden=(16, 8, 1), dense=True):
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature, SparseSeqFeature
    from handyrec_b200.models import DeepFM

    torch.manual_seed(seed)
    sparse = [SparseFeature("user_id", 40, 8), SparseFeature("gender", 3, 8), SparseFeature("movie_id", 50, 8),
              SparseSeqFeature(SparseFeature("movie_id", 50, 8), "hist_movie", 4), SparseSeqFeature(SparseFeature("genre_id", 19, 8), "genres", 3)]
    pool = FeaturePool()
    fm = FeatureGroup("fm", sparse, pool, l2_embd=0.0)
    dnn = FeatureGroup("dnn", ([DenseFeature("age"), DenseFeature("score", dim=2)] if dense else []) + sparse, pool, l2_embd=0.0)
    return DeepFM(fm, dnn, dnn_hidden_units=hidden)


def _deepfm_data(n, seed=1):
    g = np.random.RandomState(seed)
    x = {"user_id": g.randint(0, 40, (n, 1)).astype(np.int32), "gender": g.randint(0, 3, (n,)).astype(np.int64),
         "movie_id": g.randint(1, 50, (n, 1)).astype(np.int32), "hist_movie": rand_ids(n, 4, 50, seed=2).numpy(),
         "genres": rand_ids(n, 3, 19, seed=3).numpy().astype(np.int64), "age": g.rand(n, 1).astype(np.float32),
         "score": g.randint(0, 5, (n, 2)).astype(np.float64)}
    y = (g.rand(n) < 0.3).astype(np.float32)
    return x, y


@pytest.mark.parametrize("opt", ["adam", "sgd"])
def test_model_fit_runs_on_the_fused_engine_and_matches_the_layer_path(dev, opt):
    """`DeepFM(...).compile(); .fit(dict of arrays)` is lowered onto DeepFMEngine (one lookup, fused backward, host batches packed
    by hrb_host_pack_*); the same model with `fuse = False` runs layer by layer.  Same initial weights -> same losses, weights and
    predictions (the dense optimiser step of the engine IS Keras' step for these small tables)."""
    from handyrec_b200 import keras_lite as KL

    n, bs = 700, 256  # the last batch is partial
    x, y = _deepfm_data(n)
    mk = (lambda: KL.Adam(learning_rate=0.01)) if opt == "adam" else (lambda: KL.SGD(learning_rate=0.5))
    fused, plain = _deepfm_model(), _deepfm_model()
    plain.fuse = False
    fused.compile(optimizer=mk(), loss=KL.binary_crossentropy)
    plain.compile(optimizer=mk(), loss=KL.binary_crossentropy)
    assert fused._fused is not None and plain._fused is None
    hf = fused.fit(x, y, batch_size=bs, epochs=2)
    hp = plain.fit(x, y, batch_size=bs, epochs=2)
    assert fused._fused.engine is not None and fused._fused.engine.step_count == 6
    np.testing.assert_allclose(hf.history["loss"], hp.history["loss"], rtol=2e-4)
    pf, pp = fused.predict(x, batch_size=300), plain.predict(x, batch_size=300)
    assert pf.shape == (n, 1)
    np.testing.assert_allclose(pf, pp, rtol=2e-3, atol=2e-5)
    for lf, lp in zip(fused.layers, plain.layers):
        for a, b in zip(lf.get_weights(), lp.get_weights()):
            close(a, b, 2e-3)
    # train_on_batch goes through the same binding; the layers see the engine's weights after sync()
    l1 = fused.train_on_batch({k: v[:bs] for k, v in x.items()}, y[:bs])
    l2 = plain.train_on_batch({k: v[:bs] for k, v in x.items()}, y[:bs])
    assert abs(l1 - l2) <= 2e-4 * max(1.0, abs(l2))


def test_model_without_dense_features_and_tuple_input(dev):
    from handyrec_b200 import keras_lite as KL

    x, y = _deepfm_data(300)
    x = {k: v for k, v in x.items() if k not in ("age", "score")}
    m = _deepfm_model(dense=False, hidden=(8, 1))
    m.compile(optimizer=KL.Adam(1e-2), loss=KL.binary_crossentropy)
    assert m._fused is not None and m._fused.n_dense == 0
    h = m.fit((x, y), batch_size=128, epochs=3)
    assert h.history["loss"][-1] < h.history["loss"][0]
    assert m.predict(x).shape == (300, 1)


def test_host_pack_matches_numpy(dev):
    """hrb_host_pack_i32 / _f32: per-feature arrays of mixed dtypes and widths -> one packed matrix, any row window."""
    import ctypes

    from handyrec_b200._lib import call
    from handyrec_b200.lowering import _ColumnSet

    g = np.random.RandomState(0)
    n = 70000
    cols = [g.randint(0, 1000, (n, 1)).astype(np.int32), g.randint(0, 1 << 40, (n,)).astype(np.int64) % 100000, g.randint(0, 50, (n, 7)).astype(np.int32),
            g.rand(n, 3).astype(np.float64) * 100]
    cs = _ColumnSet(cols)
    for start, rows in ((0, n), (12345, 4097), (n - 5, 5), (100, 0)):
        dst = torch.full((max(rows, 1), cs.total + 2), -7, dtype=torch.int32)
        call("hrb_host_pack_i32", cs.ptrs, cs.dtype, cs.width, cs.ld, cs.n, start, rows, ctypes.c_void_p(dst.data_ptr()), dst.shape[1], 0)
        want = np.concatenate([np.asarray(c).reshape(n, -1)[start : start + rows].astype(np.int32) for c in cols], 1)
        if rows:
            assert np.array_equal(dst.numpy()[:rows, : cs.total], want) and (dst.numpy()[:, cs.total :] == -7).all()
        dstf = torch.zeros(max(rows, 1), cs.total, dtype=torch.float32)
        call("hrb_host_pack_f32", cs.ptrs, cs.dtype, cs.width, cs.ld, cs.n, start, rows, ctypes.c_void_p(dstf.data_ptr()), dstf.shape[1], 3)
        wantf = np.concatenate([np.asarray(c).reshape(n, -1)[start : start + rows].astype(np.float32) for c in cols], 1)
        if rows:
            assert np.array_equal(dstf.numpy()[:rows], wantf)


# ------------------------------------------------------------------------------------------------
# (f1) sampled softmax / l2_normalize / lazy catalogue
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,D,B,S", [(500, 16, 64, 20), (3883, 32, 257, 100), (40, 8, 33, 5)])
def test_sampled_softmax_layer_matches_oracle_with_injected_samples(dev, C, D, B, S):
    """SampledSoftmaxLayer == tf.nn.sampled_softmax_loss restated (oracle) on the same candidates: loss and the gradients w.r.t.
    the item matrix and the user vectors, including accidental hits (the label among the sampled ids)."""
    from handyrec_b200.layers import SampledSoftmaxLayer

    rng = np.random.RandomState(C)
    W = rnd(C, D, seed=1, scale=0.3)
    U = rnd(B, D, seed=2, scale=0.3)
    labels = torch.from_numpy(rng.randint(0, C, (B, 1)).astype(np.int32))
    sampled, tries = oracle.log_uniform_sample(S, C, rng)
    labels[: min(B, S), 0] = torch.from_numpy(sampled[: min(B, S)])  # force accidental hits
    te = oracle.unique_expected_count(oracle.log_uniform_prob(labels.numpy().reshape(-1), C), tries).astype(np.float32)
    se = oracle.unique_expected_count(oracle.log_uniform_prob(sampled, C), tries).astype(np.float32)
    Wl, Ul = W.clone().requires_grad_(True), U.clone().requires_grad_(True)
    want = oracle.sampled_softmax_loss(Wl, torch.zeros(C), labels, Ul, torch.from_numpy(sampled), torch.from_numpy(te), torch.from_numpy(se))
    gsc = rnd(B, seed=3)
    (want * gsc).sum().backward()
    layer = SampledSoftmaxLayer(num_sampled=S)
    Wd, Ud = W.to(dev).requires_grad_(True), U.to(dev).requires_grad_(True)
    layer.build([(C, D), (None, D), (None, 1)])
    layer.sampled_values = (sampled, te, se)
    got = layer.call([Wd, Ud, labels.to(dev)])
    assert got.shape == (B, 1)
    close(got[:, 0], want, 1e-5)
    (got[:, 0] * gsc.to(dev)).sum().backward()
    close(Ud.grad, Ul.grad, 1e-4)
    close(Wd.grad, Wl.grad, 1e-4)
    # the kernel's own log Q (from id and number of tries) equals the injected expected counts
    from handyrec_b200.autograd_ops import MatmulNTFn, RowDotFn, SampledSoftmaxFn

    lab = labels.reshape(-1).to(dev)
    smp = torch.from_numpy(sampled).to(dev)
    tl, sl = RowDotFn.apply(U.to(dev), W.to(dev)[lab.long()]), MatmulNTFn.apply(U.to(dev), W.to(dev)[smp.long()])
    own = SampledSoftmaxFn.apply(tl, sl, lab, smp, None, None, float(tries), C, True)
    close(own, want, 2e-5)


def test_l2_normalize_whole_tensor(dev):
    from handyrec_b200.autograd_ops import L2NormalizeFn

    x = rnd(3000, 32, seed=4)
    xl = x.clone().requires_grad_(True)
    want = oracle.l2_normalize(xl)
    g = rnd(3000, 32, seed=5)
    (want * g).sum().backward()
    xd = x.to(dev).requires_grad_(True)
    got = L2NormalizeFn.apply(xd, 1e-12)
    close(got, want, 1e-5)
    (got * g.to(dev)).sum().backward()
    close(xd.grad, xl.grad, 1e-4)
    assert torch.equal(got, L2NormalizeFn.apply(xd.detach(), 1e-12))  # fixed-order reduction: reproducible


def _retrieval_groups(n_items=60, seed=0):
    from handyrec_b200.features import EmbdFeatureGroup, FeatureGroup, FeaturePool, SparseFeature, SparseSeqFeature

    torch.manual_seed(seed)
    movie, genre = SparseFeature("movie_id", n_items, 8), SparseFeature("genre_id", 19, 8)
    values = {"movie_id": np.arange(n_items), "genres": np.random.RandomState(0).randint(0, 19, (n_items, 3))}
    values["genres"][::4, 0] = 0
    pool = FeaturePool()
    item_group = EmbdFeatureGroup("item", "movie_id", [movie, SparseSeqFeature(genre, "genres", 3)], pool, values, embd_dim=8, l2_embd=0.0)
    user = [SparseFeature("user_id", 40, 8), SparseFeature("gender", 3, 4), SparseSeqFeature(SparseFeature("movie_id", n_items, 8), "hist_movie", 4)]
    return FeatureGroup("user", user, pool, l2_embd=0.0), item_group, values


def _retrieval_data(n, n_items, seed=1):
    g = np.random.RandomState(seed)
    return {"user_id": g.randint(0, 40, (n, 1)).astype(np.int32), "gender": g.randint(0, 3, (n, 1)).astype(np.int32),
            "hist_movie": rand_ids(n, 4, n_items, seed=2).numpy(), "movie_id": g.randint(1, n_items, (n, 1)).astype(np.int32)}


@pytest.mark.parametrize("name", ["DSSM", "YouTubeMatchDNN"])
def test_lazy_catalogue_equals_full_catalogue(dev, name):
    """Evaluating the item side for the B + S rows a step reads (row_tower) gives the same loss and the same weight update as
    evaluating all n items (the reference's get_embd), candidates pinned on both sides."""
    import handyrec_b200.models as M
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import SampledSoftmaxLayer
    from handyrec_b200.layers.utils import sampledsoftmaxloss

    n_items, B, S = 60, 50, 7
    x = _retrieval_data(B, n_items)
    rng = np.random.RandomState(3)
    sampled, tries = oracle.log_uniform_sample(S, n_items, rng)
    te = oracle.unique_expected_count(oracle.log_uniform_prob(x["movie_id"].reshape(-1), n_items), tries).astype(np.float32)
    se = oracle.unique_expected_count(oracle.log_uniform_prob(sampled, n_items), tries).astype(np.float32)
    kw = dict(user_dnn_hidden_units=(16, 8), item_dnn_hidden_units=(16, 8)) if name == "DSSM" else dict(dnn_hidden_units=(16, 8))
    results = []
    for lazy in (True, False):
        ug, ig, _ = _retrieval_groups(n_items)
        m = getattr(M, name)(ug, ig, num_sampled=S, lazy_catalogue=lazy, **kw)
        ssl = [l for l in m.layers if isinstance(l, SampledSoftmaxLayer)][0]
        assert (ssl.item_rows is not None) == lazy
        ssl.sampled_values = (sampled, te, se)
        m.compile(optimizer=KL.SGD(0.5), loss=sampledsoftmaxloss)
        loss = m.train_on_batch(x, np.zeros(B))
        loss2 = m.train_on_batch(x, np.zeros(B))  # depends on every weight the first step moved
        # inference handles like the reference's (DSSM.py:116-119): user tower + item rows of the full catalogue
        users = KL.Model(inputs=m.user_input, outputs=m.user_embedding).predict(x, batch_size=16)
        items = KL.Model(inputs=m.item_input, outputs=m.item_embedding).predict({"movie_id": np.arange(n_items).reshape(-1, 1)}, batch_size=n_items)
        assert users.shape == (B, 8) and items.shape == (n_items, 8)
        results.append((loss, loss2, users, items, sum(p.numel() for p, _ in m.weights_with_l2())))
    (la, la2, ua, ia, na), (lb, lb2, ub, ib, nb) = results
    assert na == nb  # the same parameters are trained either way
    assert abs(la - lb) <= 1e-5 * max(1.0, abs(lb)) and abs(la2 - lb2) <= 1e-4 * max(1.0, abs(lb2))
    close(ua, ub, 1e-4)
    close(ia, ib, 1e-4)


def test_retrieval_models_fit_like_the_reference_tests(dev):
    """tests/models/retrieval/test_DSSM.py / test_YouTubeMatchDnn.py flows: constructor errors, compile with sampledsoftmaxloss,
    fit two epochs on tf.data-like batches, loss goes down; DSSM with BatchNorm + cosine scaling runs the full-catalogue path."""
    import handyrec_b200.models as M
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers.utils import sampledsoftmaxloss

    n_items, n = 60, 400
    x = _retrieval_data(n, n_items)
    ug, ig, _ = _retrieval_groups(n_items)
    with pytest.raises(ValueError):
        M.DSSM(ug, ug, num_sampled=1)
    m = M.DSSM(ug, ig, user_dnn_hidden_units=(16, 8), item_dnn_hidden_units=(16, 8), dnn_dropout=0.1, dnn_bn=True, num_sampled=5, cos_sim=True)
    m.compile(optimizer=KL.Adam(5e-3), loss=sampledsoftmaxloss)
    batches = [({k: v[s : s + 100] for k, v in x.items()}, np.zeros(100)) for s in range(0, n, 100)]
    h = m.fit(x=batches, epochs=3)
    assert np.isfinite(h.history["loss"]).all()
    ug2, ig2, _ = _retrieval_groups(n_items, seed=1)
    with pytest.raises(ValueError):
        M.YouTubeMatchDNN(ug2, ug2)
    m2 = M.YouTubeMatchDNN(ug2, ig2, dnn_hidden_units=(16, 8), num_sampled=10)
    m2.compile(optimizer=KL.Adam(2e-2), loss=sampledsoftmaxloss)
    h2 = m2.fit(x=batches, epochs=2)  # fresh candidates every step (the layer's own log-uniform sampler)
    assert np.isfinite(h2.history["loss"]).all()
    # with the candidates pinned the objective is fixed, and training on one batch must bring it down
    from handyrec_b200.layers import SampledSoftmaxLayer

    ssl = [l for l in m2.layers if isinstance(l, SampledSoftmaxLayer)][0]
    sampled, tries = oracle.log_uniform_sample(10, n_items, np.random.RandomState(5))
    lab = batches[0][0]["movie_id"].reshape(-1)
    ssl.sampled_values = (sampled, oracle.unique_expected_count(oracle.log_uniform_prob(lab, n_items), tries),
                          oracle.unique_expected_count(oracle.log_uniform_prob(sampled, n_items), tries))
    losses = [m2.train_on_batch(*batches[0]) for _ in range(15)]
    assert losses[-1] < 0.8 * losses[0]


def test_large_table_takes_sparse_row_updates(dev):
    """A table above SPARSE_UPDATE_MIN_ROWS keeps its gradient as (ids, rows) and gets the sorted-segment row update: identical to the
    dense path for SGD, and for Adam on the touched rows at step 1."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding

    x, y = _deepfm_data(300)
    res = {}
    for thr in (10, 1 << 30):
        CustomEmbedding.SPARSE_UPDATE_MIN_ROWS = thr
        try:
            m = _deepfm_model(hidden=(8, 1))
            m.fuse = False
            m.compile(optimizer=KL.SGD(0.5), loss=KL.binary_crossentropy)
            l = m.train_on_batch(x, y)
            res[thr] = (l, {lay.name: lay.get_weights()[0] for lay in m.layers if isinstance(lay, CustomEmbedding)})
        finally:
            CustomEmbedding.SPARSE_UPDATE_MIN_ROWS = 131072
    assert abs(res[10][0] - res[1 << 30][0]) < 1e-6
    for k in res[10][1]:
        close(res[10][1][k], res[1 << 30][1][k], 1e-4)


def test_save_and_load_weights_round_trip(dev, tmp_path):
    """model.save_weights / load_weights (Quickstart.md:250-262): a trained fused DeepFM -> row-sharded .npy files -> a freshly
    constructed model predicts the same; pre-trained tables go back in through FeaturePool(pre_embd) like group.py:283-291."""
    from handyrec_b200 import checkpoint
    from handyrec_b200 import keras_lite as KL

    x, y = _deepfm_data(600)
    m = _deepfm_model(seed=3)
    m.compile(optimizer=KL.Adam(1e-2), loss=KL.binary_crossentropy)
    m.fit(x, y, batch_size=200, epochs=2)
    want = m.predict(x)
    d = str(tmp_path / "ckpt")
    old = checkpoint.SHARD_ROWS
    man = checkpoint.save_weights(m, d, shard_rows=16)  # force row shards for the 40- and 50-row tables
    assert any(len(v["files"]) > 1 for v in man["weights"].values())
    m2 = _deepfm_model(seed=99)
    m2.compile(optimizer=KL.Adam(1e-2), loss=KL.binary_crossentropy)
    assert not np.allclose(m2.predict(x), want)
    m2.load_weights(d)
    np.testing.assert_allclose(m2.predict(x), want, rtol=1e-5, atol=1e-6)
    # a model that already owns a fused engine takes the loaded weights too
    m.fit(x, y, batch_size=200, epochs=1)
    m.load_weights(d)
    np.testing.assert_allclose(m.predict(x), want, rtol=1e-5, atol=1e-6)
    pre = checkpoint.export_pre_embd(m)
    assert set(pre) >= {"user_id", "gender", "movie_id", "genre_id"} and pre["movie_id"].shape == (50, 8)


def test_din_predict_takes_the_fused_attention_kernel(dev):
    """DIN inference: LocalActivationUnit hands (table, query ids, history ids) to hrb_lau_fwd (fused gather + [q,k,q-k,q*k] + MLP
    + mask, no (B,T,4D) tensor); the layer-by-layer forward with gradients enabled is the comparison."""
    import bench_models
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import LocalActivationUnit

    torch.manual_seed(0)
    m = bench_models.build_din()
    for l in m._all_layers():  # make Dice non-trivial: alpha != 0, moving statistics != (0, 1)
        if type(l).__name__ == "Dice":
            l.alphas.data.uniform_(-0.3, 0.3)
            l.moving_mean.data.uniform_(-0.2, 0.2)
            l.moving_variance.data.uniform_(0.5, 1.5)
    assert [l for l in m._all_layers() if isinstance(l, LocalActivationUnit)][0].dnn.activation == "dice"
    x, _ = bench_models.din_data(257)
    calls = []
    from handyrec_b200 import kernels as K

    orig = K.lau_fwd
    K.lau_fwd = lambda *a, **k: (calls.append(1), orig(*a, **k))[1]
    try:
        fused = m.predict(x)
    finally:
        K.lau_fwd = orig
    assert calls, "predict did not reach hrb_lau_fwd"
    plain = m(x, training=False).detach().cpu().numpy()  # gradients enabled -> the layer-by-layer path
    np.testing.assert_allclose(fused, plain, rtol=2e-4, atol=2e-6)


def test_din_inference_too_wide_for_the_fused_kernel_takes_the_layer_path(dev):
    """A 128-wide movie embedding makes the attention MLP's input 4D = 512 wide: more than hrb_lau_fwd's shared-memory tiles hold.
    The kernel declares that unsupported before launching anything, and inference (predict, and evaluate through it) falls back to
    the layer path instead of raising: the same probabilities as the forward with gradients enabled."""
    import bench_models
    from bench_models import DIN_T, GENRES_L, ML
    from handyrec_b200 import _lib
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200 import kernels as K
    from handyrec_b200.features import FeatureGroup, FeaturePool, SparseFeature, SparseSeqFeature
    from handyrec_b200.models import DIN

    torch.manual_seed(0)
    movie = SparseFeature("movie_id", ML["movie_id"][0], 128)  # bench_models.build_din with a wider movie embedding
    pool = FeaturePool()
    seq_group = FeatureGroup("item_seq", [SparseSeqFeature(movie, "hist_movie", DIN_T)], pool, l2_embd=0.0)
    other = [SparseFeature(k, *ML[k]) for k in ("user_id", "gender", "occupation", "zip", "age")] + [movie, SparseFeature("year", *ML["year"])]
    other.append(SparseSeqFeature(SparseFeature("genre_id", *ML["genre_id"]), "genres", GENRES_L))
    m = DIN(seq_group, FeatureGroup("other_feats", other, pool, l2_embd=0.0), dnn_hidden_units=(64, 32), dnn_activation="dice",
            lau_dnn_hidden_units=(32, 1), lau_dnn_activation="dice")
    m.compile(optimizer=KL.Adam(learning_rate=1e-3), loss=KL.binary_crossentropy)
    for l in m._all_layers():
        if type(l).__name__ == "Dice":
            l.alphas.data.uniform_(-0.3, 0.3)
            l.moving_mean.data.uniform_(-0.2, 0.2)
            l.moving_variance.data.uniform_(0.5, 1.5)
    x, _ = bench_models.din_data(257)
    declined = []
    orig = K.lau_fwd

    def lau_fwd(*a, **k):
        try:
            return orig(*a, **k)
        except _lib.HrbError as e:
            declined.append(e.status)
            raise

    K.lau_fwd = lau_fwd
    try:
        fused = m.predict(x)
    finally:
        K.lau_fwd = orig
    assert declined == [_lib.HRB_UNSUPPORTED]
    plain = m(x, training=False).detach().cpu().numpy()
    np.testing.assert_allclose(fused, plain, rtol=2e-4, atol=2e-6)


@pytest.mark.parametrize("Q,N,D,n", [(7, 3883, 32, 100), (600, 20000, 64, 10), (3, 50, 8, 50), (33, 9000, 16, 1)])
def test_topn_inner_product_search_is_exact(dev, Q, N, D, n):
    """search_embedding == faiss.IndexFlatIP.search: exact top-n by inner product, best first, duplicates (ties) by lower index."""
    from handyrec_b200 import search

    items = rnd(N, D, seed=1)
    items[N // 2] = items[3]  # an exact tie
    users = rnd(Q, D, seed=2)
    sc = users.double() @ items.double().t()
    got_v, got_i = search.topn_inner_product(users.to(dev), items.to(dev), n)
    got_v, got_i = got_v.cpu(), got_i.cpu().long()
    assert got_i.shape == (Q, min(n, N))
    # returned scores are the scores of the returned items, sorted, and no better item was left out
    np.testing.assert_allclose(got_v.numpy(), torch.gather(sc, 1, got_i).numpy(), rtol=1e-4, atol=1e-5)
    assert (got_v[:, :-1] >= got_v[:, 1:]).all()
    kth = torch.topk(sc, min(n, N), dim=1).values[:, -1]
    assert (got_v[:, -1].double() >= kth - 1e-4 * kth.abs().clamp(min=1)).all()
    assert all(len(set(r.tolist())) == len(r) for r in got_i)
    cand = search.search_embedding(D, items.numpy(), users.numpy(), np.arange(N) + 1000, n)
    assert cand.shape == (Q, min(n, N)) and np.array_equal(cand, got_i.numpy() + 1000)


def test_ranking_metrics_match_reference_definitions():
    from handyrec_b200 import search

    actual = [[1, 2, 3], [4], [5, 6]]
    pred = [[1, 9, 3, 8], [7, 4, 4], [9, 9, 9]]
    assert abs(search.map_at_k(actual, pred, 3) - np.mean([(1 / 1 + 2 / 3) / 3, (1 / 2) / 1, 0.0])) < 1e-12
    assert abs(search.recall_at_k(actual, pred, 2) - np.mean([1 / 3, 1.0, 0.0])) < 1e-12
    assert abs(search.hr_at_k(actual, pred, 1) - 1 / 3) < 1e-12


@pytest.mark.parametrize("B,T,D,hidden,act", [
    (96, 50, 32, (32, 1), "dice"), (96, 50, 32, (32, 1), "relu"),
    (91, 45, 32, (32, 1), "dice"),          # B*T = 4095: one row short of the tensor-core path, the (B,T,4D) tensor is built
    (4096, 1, 32, (32, 1), "sigmoid"),      # T = 1, exactly 4096 rows
    (82, 50, 8, (16, 1), "dice"),           # 4100 rows; 2D = 16, less than one 32-wide k-block
    (100, 41, 16, (32, 1), "sigmoid"),
    (1000, 50, 32, (32, 1), "dice"),        # 50 000 rows: the last partial batch of a DIN fit
    (1000, 50, 64, (32, 1), "tanh"),
    (96, 50, 128, (64, 1), "sigmoid"),      # 4D = 512
])
def test_local_activation_unit_training_path_without_the_4d_tensor(dev, B, T, D, hidden, act):
    """B*T >= 4096 rows: the first LAU layer runs as a per-sample q-term + a [k | q*k] tensor-core GEMM (LAUFirstLayerFn); below that
    the (B,T,4D) tensor is materialised.  Scores and every gradient (query, keys, all MLP weights, Dice alphas) against float64
    autograd of the oracle's materialised [q,k,q-k,q*k] path, Dice in training mode.  Without Dice (whose column statistics use
    atomics) every reduction runs in fixed order: a second forward + backward gives the same bits."""
    from handyrec_b200.layers import LocalActivationUnit
    from handyrec_b200.layers.activation import Dice
    from handyrec_b200.layers.core import Dense

    torch.manual_seed(1)
    lau = LocalActivationUnit(hidden_units=hidden, activation=act)
    lau.build([(None, 1, D), (None, T, D)])
    dense = [l for l in lau.dnn.layers if isinstance(l, Dense)]
    dices = [l for l in lau.dnn.layers if isinstance(l, Dice)]
    for d in dense:
        d.bias.data.normal_(0, 0.1)
    for d in dices:
        d.alphas.data.uniform_(-0.3, 0.3)
    q, k = rnd(B, 1, D, seed=2, scale=0.5), rnd(B, T, D, seed=3, scale=0.5)
    mask = torch.from_numpy(rand_ids(B, T, 100, seed=4).numpy() != 0)
    p = oracle.dnn_init(4 * D, hidden)
    p.W = [d.kernel.detach().cpu().double().requires_grad_(True) for d in dense]
    p.b = [d.bias.detach().cpu().double().requires_grad_(True) for d in dense]
    p.dice_mean = [m.double() for m in p.dice_mean]
    p.dice_var = [v.double() for v in p.dice_var]
    for i, d in enumerate(dices):
        p.dice_alpha[i] = d.alphas.detach().cpu().double().requires_grad_(True)
    ql, kl = q.double().requires_grad_(True), k.double().requires_grad_(True)
    want = oracle.local_activation_unit(ql, kl, mask, p, act=act, training=True)
    g = rnd(B, 1, T, seed=5)
    (want * g.double()).sum().backward()

    def run():
        for d in dense:
            d.kernel.grad, d.bias.grad = None, None
        for d in dices:
            d.alphas.grad = None
        qd, kd = q.to(dev).requires_grad_(True), k.to(dev).requires_grad_(True)
        got = lau.call([qd, kd], mask=[None, mask.to(dev)], training=True)
        (got * g.to(dev)).sum().backward()
        return [got.detach(), qd.grad, kd.grad] + [t.grad for d in dense for t in (d.kernel, d.bias)] + [d.alphas.grad for d in dices]

    res = run()
    got, dq, dk = res[:3]
    close(got, want, 1e-5)
    close(dq, ql.grad, 1e-4)
    close(dk, kl.grad, 1e-4)
    for d, W, b in zip(dense, p.W, p.b):
        close(d.kernel.grad, W.grad, 1e-4)
        close(d.bias.grad, b.grad, 1e-4)
    for i, d in enumerate(dices):
        close(d.alphas.grad, p.dice_alpha[i].grad, 1e-4)
    if not dices:
        assert all(torch.equal(a, b) for a, b in zip(res, run()))
