"""GPU: Keras gradient clipping (clipvalue / clipnorm / global_clipnorm) -- the clip kernels against float64, the layer path
against a float64 DeepFM with Keras' IndexedSlices gradients, the fused engine against the layer path, inactive clips as exact
no-ops and bit-reproducible clipped runs."""
import math

import numpy as np
import pytest
import torch

import oracle
from oracle.clip_ref import IndexedSlices, clip_gradients, concat_slices, densify
from oracle.ftrl_ref import ftrl_dense, ftrl_sparse
from oracle.optim_ref import adagrad_dense
from tests.test_gpu_api import _deepfm_data
from tests.test_gpu_parity import close, rand_ids, rnd

pytestmark = pytest.mark.gpu


# ---- 1. kernels ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_w", [False, True])
@pytest.mark.parametrize("clipvalue", [math.inf, 0.5])
def test_clip_prepare_multi_matches_float64(dev, with_w, clipvalue):
    from handyrec_b200 import kernels as K

    sizes = [0, 1, 5, 4097, 1_000_000] + [7 * i + 3 for i in range(35)]  # 40 segments: two launches
    var = [i % 6 for i in range(len(sizes))]  # several segments per variable
    gs = [rnd(n, seed=10 + i) for i, n in enumerate(sizes)]
    ws = [rnd(n, seed=100 + i) for i, n in enumerate(sizes)]
    l2s = [0.02 * (i % 3) if with_w else 0.0 for i in range(len(sizes))]
    ws_ = K.clip_workspace(0, dev)
    outs, sums = [], []
    for _ in range(2):
        g = [t.to(dev) for t in gs]
        sumsq = torch.zeros(6, device=dev)
        K.clip_prepare_multi(g, [t.to(dev) for t in ws] if with_w else None, l2s if with_w else None, var, clipvalue, sumsq, ws_)
        torch.cuda.synchronize()
        outs.append([t.cpu() for t in g])
        sums.append(sumsq.cpu())
    assert all(torch.equal(a, b) for a, b in zip(outs[0], outs[1])) and torch.equal(sums[0], sums[1])  # bit-reproducible
    want_sum = np.zeros(6)
    for i in range(len(sizes)):
        want = gs[i].double() + (l2s[i] * ws[i].double() if with_w else 0.0)
        want = want.float().double().clamp(-clipvalue, clipvalue)
        close(outs[0][i], want, 1e-6)
        want_sum[var[i]] += float((outs[0][i].double() ** 2).sum())
    np.testing.assert_allclose(sums[0].double().numpy(), want_sum, rtol=1e-6)
    if clipvalue < math.inf:
        assert max(float(t.abs().max()) for t in outs[0] if t.numel()) == clipvalue
    # clipvalue alone: no sums, the clamp only
    g = [t.to(dev) for t in gs[:5]]
    K.clip_prepare_multi(g, None, None, var[:5], 0.25, None, ws_)
    for a, b in zip(g, gs[:5]):
        assert torch.equal(a.cpu(), b.clamp(-0.25, 0.25))


def _plan_case(dev, B=5000, D=8):
    from handyrec_b200 import kernels as K

    shapes = [(300, D), (1000, D), (40, D)]
    fields = [(0, 1, "none", 0, 0), (1, 4, "mean", 1, D), (2, 3, "sum", 5, 2 * D), (1, 1, "none", 8, 3 * D)]  # table 1 twice
    g = torch.Generator().manual_seed(5)
    ids = torch.cat([torch.randint(0, 300, (B, 1), generator=g, dtype=torch.int32), rand_ids(B, 4, 1000, seed=6),
                     rand_ids(B, 3, 40, seed=7), torch.randint(0, 1000, (B, 1), generator=g, dtype=torch.int32)], 1).contiguous()
    ids[::97, 0] = 300 + 5  # out of range: contributes nothing
    ids[1::89, 8] = -3
    plan = K.LookupPlan([torch.zeros(v, d, device=dev) for v, d in shapes], fields)
    dx = rnd(B, 4 * D, seed=8, scale=0.1)
    fm = rnd(B, 4 * D, seed=9, scale=0.1)
    return plan, shapes, fields, ids, dx, fm


def _plan_ref(shapes, fields, ids, dx, fm, v):
    """float32 emulation of the write-back, float64 sums."""
    out = dx.clone()
    sums = np.zeros(len(shapes))
    f32 = lambda a: a.to(torch.float32)
    for ti, L, pool, col, oc in fields:
        D = shapes[ti][1]
        c = ids[:, col : col + L].long()
        valid = (c >= 0) & (c < shapes[ti][0]) & ((c != 0) if pool != "none" else torch.ones_like(c, dtype=torch.bool))
        n = valid.sum(1, keepdim=True).to(torch.float32)
        inv = torch.where(n > 0, torch.tensor(1.0) / n.clamp(min=1), torch.zeros_like(n)) if pool == "mean" else torch.ones_like(n)
        nsc = n if pool == "mean" else torch.ones_like(n)
        parts, sq = [], 0.0
        for src in (dx[:, oc : oc + D], fm[:, oc : oc + D]):
            p = f32(src * inv)
            cl = p.clamp(-v, v)
            bound = (p > v) | (p < -v)
            parts.append(torch.where(bound, f32(cl * nsc), src))
            sq = sq + cl.double() ** 2
        out[:, oc : oc + D] = f32(parts[0] + parts[1])
        sums[ti] += float((n.double() * sq).sum())
    return out, sums


@pytest.mark.parametrize("v", [math.inf, 0.02])
def test_plan_clip_grads_matches_float64(dev, v):
    from handyrec_b200 import kernels as K

    plan, shapes, fields, ids, dx, fm = _plan_case(dev)
    ws = K.clip_workspace(len(shapes), dev)
    res = []
    for _ in range(2):
        d = dx.to(dev)
        sumsq = torch.zeros(len(shapes), device=dev)
        plan.clip_grads(ids.to(dev), d, fm.to(dev), v, sumsq, ws)
        torch.cuda.synchronize()
        res.append((d.cpu(), sumsq.cpu()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    want, sums = _plan_ref(shapes, fields, ids, dx, fm, v)
    if v == math.inf:
        assert torch.equal(res[0][0], dx + fm)  # nothing binds: exactly the FM part added, as fm_bwd's accumulate does
    else:
        assert not torch.equal(res[0][0], dx + fm)
    close(res[0][0], want, 1e-6)
    np.testing.assert_allclose(res[0][1].double().numpy(), sums, rtol=1e-6)
    # the scale pass: field blocks times the scale of their table
    scale = torch.tensor([0.5, 2.0, 0.25], device=dev)
    d = res[0][0].to(dev)
    plan.clip_apply(d, dx.shape[0], scale)
    want = res[0][0].clone()
    for ti, _, _, _, oc in fields:
        want[:, oc : oc + 8] *= float(scale[ti])
    assert torch.equal(d.cpu(), want)


def test_clip_scales(dev):
    from handyrec_b200 import kernels as K

    sumsq = torch.tensor([0.0, 4.0, 100.0, 25.0], device=dev)
    s = torch.empty(4, device=dev)
    K.clip_scales(sumsq, 5.0, False, s)
    assert s.cpu().tolist() == [1.0, 1.0, 0.5, 1.0]
    K.clip_scales(sumsq, 6.5, True, s)  # norm sqrt(129)
    close(s.cpu(), torch.full((4,), 6.5 / math.sqrt(129.0)), 1e-6)
    K.clip_scales(torch.tensor([1.0, math.inf], device=dev), 1.0, True, s[:2])
    assert torch.isnan(s[:2]).all()
    K.clip_scales(torch.tensor([0.0, 4.0], device=dev), 0.0, False, s[:2])
    assert math.isnan(float(s[0])) and float(s[1]) == 0.0


# ---- 2. the layer path against float64 --------------------------------------------------------------------------------------
def _model(seed=0, l2=0.0, l2_dnn=0.0):
    from handyrec_b200.features import DenseFeature, FeatureGroup, FeaturePool, SparseFeature, SparseSeqFeature
    from handyrec_b200.models import DeepFM

    torch.manual_seed(seed)
    sparse = [SparseFeature("user_id", 40, 8), SparseFeature("gender", 3, 8), SparseFeature("movie_id", 50, 8),
              SparseSeqFeature(SparseFeature("movie_id", 50, 8), "hist_movie", 4), SparseSeqFeature(SparseFeature("genre_id", 19, 8), "genres", 3)]
    pool = FeaturePool()
    fm = FeatureGroup("fm", sparse, pool, l2_embd=l2)
    dnn = FeatureGroup("dnn", [DenseFeature("age"), DenseFeature("score", dim=2)] + sparse, pool, l2_embd=l2)
    return DeepFM(fm, dnn, dnn_hidden_units=(16, 8, 1), l2_dnn=l2_dnn)


_TABLE_OF = {"user_id": 40, "gender": 3, "movie_id": 50, "hist_movie": 50, "genres": 19}


def _vars(m):
    """(name, parameter) of every trainable variable: the tables by vocabulary, the Dense kernels / biases, FM's two."""
    from handyrec_b200.layers import CustomEmbedding
    from handyrec_b200.layers.core import Dense
    from handyrec_b200.layers.interaction import FM

    out = [(f"t{l.input_dim}", l.embeddings) for l in m._all_layers() if isinstance(l, CustomEmbedding)]
    dn = [l for l in m._all_layers() if isinstance(l, Dense)]
    for i, d in enumerate(dn):
        out += [(f"W{i}", d.kernel), (f"b{i}", d.bias)]
    fm = next(l for l in m._all_layers() if isinstance(l, FM))
    return out + [("fmw", fm.linear), ("fmw0", fm.w_0)]


def _ref_grads(m, x, y):
    """float64 DeepFM, each table looked up once per group; a table's gradient is the concatenation of its lookups' gathered-output
    gradients (IndexedSlices values, one row per position), every other variable's is dense."""
    V = {k: p.detach().cpu().double().requires_grad_(True) for k, p in _vars(m)}
    B = len(y)
    taken = {}

    def lookup():
        outs = []
        for name in ("user_id", "gender", "movie_id", "hist_movie", "genres"):
            ids = torch.as_tensor(np.asarray(x[name])).reshape(B, -1).long()
            e = V[f"t{_TABLE_OF[name]}"][ids]
            e.retain_grad()
            taken.setdefault(_TABLE_OF[name], []).append((ids, e))
            outs.append(e if ids.shape[1] == 1 else oracle.sequence_pooling(e, (ids != 0)[..., None].expand_as(e), "mean"))
        return outs

    fm_e, dnn_e = lookup(), lookup()
    p = oracle.DNNParams(3 + 5 * 8, (16, 8, 1))  # units [in, 16, 8, 1]: core.py:57 puts a Dense(in) first
    for i in range(len(p.units)):
        p.W.append(V[f"W{i}"])
        p.b.append(V[f"b{i}"])
    dense = [torch.as_tensor(np.asarray(x["age"], dtype=np.float64)).reshape(B, 1), torch.as_tensor(np.asarray(x["score"], dtype=np.float64))]
    logit = oracle.deepfm_forward(dense, fm_e, dnn_e, p, V["fmw"], V["fmw0"], return_logit=True)
    oracle.bce_from_logits(logit[:, 0], torch.as_tensor(y, dtype=torch.float64)).backward()
    names = [k for k, _ in _vars(m)]
    grads = []
    for k in names:
        if k.startswith("t"):
            parts = taken[int(k[1:])]
            grads.append(concat_slices(*[IndexedSlices(i.reshape(-1).numpy(), e.grad.reshape(-1, 8).numpy()) for i, e in parts]))
        else:
            grads.append(V[k].grad.numpy())
    return names, {k: V[k].detach().numpy() for k in names}, grads


def _bind(grads, mode):
    """Clip arguments that bind for these gradients."""
    vals = [g.values if isinstance(g, IndexedSlices) else g for g in grads]
    norms = [float(np.sqrt((v ** 2).sum())) for v in vals]
    mx = max(float(np.abs(v).max()) for v in vals)
    kw = {"clipvalue": dict(clipvalue=0.3 * mx), "clipnorm": dict(clipnorm=0.5 * min(norms)),
          "global_clipnorm": dict(global_clipnorm=0.5 * math.sqrt(sum(n * n for n in norms))),
          "clipvalue+clipnorm": dict(clipvalue=0.3 * mx, clipnorm=0.2 * min(norms))}
    return kw[mode]


def _step_ref(opt, names, w0, grads, lr):
    out = {}
    for k, g in zip(names, grads):
        w = w0[k]
        if opt == "sgd":
            out[k] = w - lr * densify(g, w.shape[0])
        elif opt == "adam":  # Keras Adam, step 1 from zero moments (lazy Adam is the same on the touched rows at step 1)
            gd = densify(g, w.shape[0])
            m, v = 0.1 * gd, 0.001 * gd * gd
            out[k] = w - lr * math.sqrt(1 - 0.999) / (1 - 0.9) * m / (np.sqrt(v) + 1e-7)
        elif opt == "adagrad":
            out[k] = adagrad_dense(w, np.full(w.shape, 0.1), densify(g, w.shape[0]), lr)[0].numpy()
        elif isinstance(g, IndexedSlices):  # Ftrl: l2 = 0 tables step the listed rows only
            out[k] = ftrl_sparse(w, np.full(w.shape, 0.1), np.zeros(w.shape), g.indices, g.values, lr)[0].numpy()
        else:
            out[k] = ftrl_dense(w, np.full(w.shape, 0.1), np.zeros(w.shape), g, lr)[0].numpy()
    return out


_OPTS = {"sgd": ("SGD", 0.5), "adam": ("Adam", 0.01), "adagrad": ("Adagrad", 0.1), "ftrl": ("Ftrl", 0.1)}


def _opt(name, **kw):
    from handyrec_b200 import keras_lite as KL

    cls, lr = _OPTS[name]
    return getattr(KL, cls)(lr, **kw)


@pytest.mark.parametrize("mode,opt", [(m, "sgd") for m in ("clipvalue", "clipnorm", "global_clipnorm", "clipvalue+clipnorm")]
                         + [("clipnorm", "adam"), ("global_clipnorm", "adagrad"), ("clipvalue+clipnorm", "ftrl")])
def test_layer_path_step_matches_float64_keras(dev, monkeypatch, mode, opt):
    """One step of DeepFM with fuse = False: a small table (dense gradient), a table above SPARSE_UPDATE_MIN_ROWS shared by a plain
    and a mean-pooled field (touched-rows update), a second mean-pooled table."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding

    monkeypatch.setattr(CustomEmbedding, "SPARSE_UPDATE_MIN_ROWS", 45)
    x, y = _deepfm_data(300)
    m = _model()
    m.fuse = False
    names, w0, grads = _ref_grads(m, x, y)
    kw = _bind(grads, mode)
    m.compile(optimizer=_opt(opt, **kw), loss=KL.binary_crossentropy)
    m.train_on_batch(x, y)
    movie = next(l for l in m._all_layers() if isinstance(l, CustomEmbedding) and l.input_dim == 50)
    assert getattr(movie, "_plan", None) is not None  # the large table took the touched-rows update
    want = _step_ref(opt, names, w0, clip_gradients(grads, **kw), _OPTS[opt][1])
    # Ftrl's first step recomputes w from linear = g - sigma * w, a cancellation: fp32 keeps ~1e-3 of the small new weights
    tol = 1e-3 if opt == "ftrl" else 1e-4
    for k, p in _vars(m):
        close(p.detach().cpu(), torch.from_numpy(want[k]).float(), tol)


# ---- 3. the fused engine against the layer path ----------------------------------------------------------------------------
def _pair(opt, kw, l2=0.0, small=45, seed=0):
    from handyrec_b200 import keras_lite as KL

    fused, plain = _model(seed, l2), _model(seed, l2)
    plain.fuse = False
    fused.dense_table_max_rows = small
    fused.compile(optimizer=_opt(opt, **kw), loss=KL.binary_crossentropy)
    plain.compile(optimizer=_opt(opt, **kw), loss=KL.binary_crossentropy)
    assert fused._fused is not None and plain._fused is None
    return fused, plain


def _three_steps(m, x, y, bs=256, algo=None, check=None):
    from handyrec_b200 import _lib

    for s in range(3):
        xb = {k: v[s * bs : (s + 1) * bs] for k, v in x.items()}
        yb = y[s * bs : (s + 1) * bs]
        if s == 0 and m._fused is not None:
            m._fused.build(bs, m.optimizer)
            if algo is not None:
                eng = m._fused.engine
                eng.bwd_algo = algo
                _lib.call("hrb_plan_set_bwd_algo", eng.plan._h, _lib.BWD_UNITS if algo == "units" else _lib.BWD_SORT)
        m.train_on_batch(xb, yb)
        if s == 0 and check is not None:
            check(m)
    torch.cuda.synchronize()


def _weights(m):
    return [w for l in m.layers for w in l.get_weights()]


_MODES = {"clipvalue": dict(clipvalue=2e-3), "clipnorm": dict(clipnorm=1e-2), "global_clipnorm": dict(global_clipnorm=2e-2),
          "clipvalue+clipnorm": dict(clipvalue=2e-3, clipnorm=5e-3)}


def _bound(kw):
    def check(m):
        eng = m._fused.engine
        c = eng.clip
        if "clipnorm" in kw or "global_clipnorm" in kw:
            assert float(c.scale[: c.n_vars].min()) < 1.0  # a norm clip bound in step 1
        else:
            assert float(eng.grads[: eng.n_dense_params].abs().max()) == np.float32(kw["clipvalue"])  # the clamp bound
    return check


@pytest.mark.parametrize("algo", ["units", "sort"])
@pytest.mark.parametrize("opt", ["sgd", "adam", "adagrad", "ftrl"])
@pytest.mark.parametrize("mode", list(_MODES))
def test_fused_matches_the_layer_path(dev, monkeypatch, mode, opt, algo):
    from handyrec_b200.layers import CustomEmbedding

    monkeypatch.setattr(CustomEmbedding, "SPARSE_UPDATE_MIN_ROWS", 45)  # the same tables row-updated on both paths
    x, y = _deepfm_data(768)
    kw = _MODES[mode]
    fused, plain = _pair(opt, kw)
    _three_steps(fused, x, y, algo=algo, check=_bound(kw))
    _three_steps(plain, x, y)
    eng = fused._fused.engine
    assert eng.dense_tables and len(eng.dense_tables) < len(eng.tables)
    tol = 2e-4 if opt == "adam" else 1e-4
    for a, b in zip(_weights(fused), _weights(plain)):
        close(a, b, tol)


def test_fused_with_l2_embd_matches_the_layer_path(dev):
    """l2_embd > 0: every table dense-updated, its dense gradient (with 2*l2*w) clipped like a Dense kernel."""
    x, y = _deepfm_data(768)
    for kw in (dict(clipnorm=1e-2, clipvalue=2e-3), dict(global_clipnorm=2e-2)):
        fused, plain = _pair("sgd", kw, l2=1e-3, small=1000)
        assert fused._fused is not None
        _three_steps(fused, x, y)
        _three_steps(plain, x, y)
        assert fused._fused.engine.l2_embd > 0 and len(fused._fused.engine.dense_tables) == 4
        for a, b in zip(_weights(fused), _weights(plain)):
            close(a, b, 1e-4)


def test_flat_buffer_padding_contributes_nothing(dev):
    """The clip runs over whole padded segments of the flat buffer: their padding gradients must be exactly 0."""
    x, y = _deepfm_data(768)
    fused, _ = _pair("sgd", dict(clipnorm=1e-2))
    _three_steps(fused, x, y)
    eng = fused._fused.engine
    logical = torch.zeros(eng.n_dense_params, dtype=torch.bool)
    for i, ((o, n, _), Kl) in enumerate(zip(eng._segments[0::2], eng.layer_Kl)):
        w = logical[o : o + eng.layer_K[i] * eng.layer_ld[i]].view(eng.layer_K[i], eng.layer_ld[i])
        rows = list(range(eng.n_dense)) + list(range(eng.nd_pad, eng.K0p)) if i == 0 else list(range(Kl))
        w[rows, : eng.units[i]] = True
        bo = eng._segments[2 * i + 1][0]
        logical[bo : bo + eng.units[i]] = True
    logical[eng.fm_off : eng.fm_off + eng.D + 1] = True
    g = eng.grads[: eng.n_dense_params].cpu()
    assert bool((g[~logical] == 0).all()) and bool((g[logical] != 0).any())
    assert bool((eng.params[: eng.n_dense_params].cpu()[~logical] == 0).all())


# ---- 4. inactive clips, determinism -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("opt", ["sgd", "adam"])
@pytest.mark.parametrize("fuse", [True, False])
def test_inactive_clip_is_bit_exact(dev, monkeypatch, fuse, opt):
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding

    monkeypatch.setattr(CustomEmbedding, "SPARSE_UPDATE_MIN_ROWS", 45)
    x, y = _deepfm_data(768)
    runs = []
    for kw in ({}, dict(clipvalue=1e30, clipnorm=1e30), dict(global_clipnorm=1e30)):
        m = _model(l2=0.0, l2_dnn=1e-3)
        m.fuse = fuse
        m.dense_table_max_rows = 45
        m.compile(optimizer=_opt(opt, **kw), loss=KL.binary_crossentropy)
        _three_steps(m, x, y)
        runs.append(_weights(m))
    for r in runs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(runs[0], r))


def test_clipped_fused_runs_are_bit_identical(dev):
    x, y = _deepfm_data(768)
    runs = []
    for _ in range(2):
        fused, _ = _pair("adam", dict(clipvalue=2e-3, global_clipnorm=2e-2))
        _three_steps(fused, x, y, algo="units")
        runs.append(_weights(fused))
    assert all(np.array_equal(a, b) for a, b in zip(*runs))


def test_din_trains_with_clipping_and_an_inactive_clip_is_bit_exact(dev):
    from handyrec_b200.config import ConfigLoader
    from handyrec_b200.keras_lite import SGD, binary_crossentropy
    from handyrec_b200.models import DIN
    from tests.test_gpu_models import _data
    from tests.test_mirror_cpu import DIN_CFG, FEATURE_DIM

    x, y = _data(200, seed=3)
    res = []
    for kw in ({}, dict(clipvalue=1e30, clipnorm=1e30), dict(global_clipnorm=1e-3)):
        torch.manual_seed(0)
        g = ConfigLoader(DIN_CFG).prepare_features(FEATURE_DIM)
        model = DIN(g["item_seq_feat_group"], g["other_feature_group"], dnn_hidden_units=(8,), lau_dnn_hidden_units=(8, 1))
        model.compile(optimizer=SGD(0.1, **kw), loss=binary_crossentropy)
        h = model.fit(x=x, y=y, batch_size=50, epochs=1)
        assert np.isfinite(h.history["loss"]).all()
        res.append([w.detach().cpu().numpy() for w in model.trainable_weights])
        if "global_clipnorm" in kw:  # every step bound: the global norm of the applied update is lr * c
            assert float(model._clip_state.scale[0]) < 1.0
    assert all(np.array_equal(a, b) for a, b in zip(res[0], res[1]))
    assert not all(np.array_equal(a, b) for a, b in zip(res[0], res[2]))


# ---- 5. many tables: one workspace shared by the table and the dense reductions -------------------------------------------------
def test_plan_and_prepare_share_a_workspace_with_many_tables(dev):
    """40 tables at B = 65536: the plan reduction's partials (512 CTAs x 40 tables) reach far past the dense reduction's, and more
    than one warp of a CTA stores them.  Both sums stay exact, call after call, on one workspace."""
    from handyrec_b200 import kernels as K

    B, D, T = 65536, 8, 40
    shapes = [(1000, D)] * T
    fields = [(t, 1, "none", t, t * D) for t in range(T)]
    g = torch.Generator().manual_seed(11)
    ids = torch.randint(0, 1000, (B, T), generator=g, dtype=torch.int32)
    plan = K.LookupPlan([torch.zeros(v, d, device=dev) for v, d in shapes], fields)
    dx, fm = rnd(B, T * D, seed=12, scale=0.1), rnd(B, T * D, seed=13, scale=0.1)
    dense = [rnd(n, seed=20 + i) for i, n in enumerate((70_000, 333, 1, 5000))]
    ws = K.clip_workspace(T, dev)
    want_tab = _plan_ref(shapes, fields, ids, dx, fm, 0.05)[1]
    results = []
    for _ in range(3):
        sumsq = torch.zeros(T + 4, device=dev)
        plan.clip_grads(ids.to(dev), dx.to(dev), fm.to(dev), 0.05, sumsq[4:], ws)
        gd = [t.to(dev) for t in dense]
        K.clip_prepare_multi(gd, None, None, [0, 1, 2, 3], 0.05, sumsq, ws)
        torch.cuda.synchronize()
        results.append(sumsq.cpu())
    assert all(torch.equal(results[0], r) for r in results[1:])
    want_dense = [float((t.clamp(-0.05, 0.05).double() ** 2).sum()) for t in dense]
    np.testing.assert_allclose(results[0][:4].double().numpy(), want_dense, rtol=1e-6)
    np.testing.assert_allclose(results[0][4:].double().numpy(), want_tab, rtol=1e-6)


@pytest.mark.parametrize("mode", ["clipnorm", "global_clipnorm"])
def test_engine_dense_norms_with_many_tables(dev, mode):
    """The fused engine at a bench-like shape (40 tables, B = 65536, tcgen05 layers): the squared norm of every Dense kernel, bias
    and FM variable is the float64 norm of its gradient (an inactive clip leaves the gradients as they are)."""
    from handyrec_b200.engine import DeepFMEngine

    B, D, T, n_dense = 65536, 8, 40, 5
    g = torch.Generator().manual_seed(21)
    tables = [rnd(v, D, seed=30 + t, scale=0.05) for t, v in enumerate([50] * 20 + [3000] * 20)]
    eng = DeepFMEngine([t.to(dev) for t in tables], [(t, 1, "none") for t in range(T)], n_dense, (64, 16, 1), "relu", batch_size=B,
                       optimizer="sgd", lr=0.1, dense_table_max_rows=100, **{mode: 1e30})
    assert eng.use_tc and len(eng.dense_tables) == 20
    ids = torch.stack([torch.randint(0, v, (B,), generator=g, dtype=torch.int32) for v in [50] * 20 + [3000] * 20], 1)
    eng.train_step_on_device(ids.to(dev), rnd(B, n_dense, seed=40).to(dev), (torch.rand(B, generator=g) < 0.3).float().to(dev))
    torch.cuda.synchronize()
    c, nd = eng.clip, eng._clip_nd
    want = [float((t.double() ** 2).sum()) for t in (s.cpu() for s in eng._clip_segs[0])]
    assert min(want) > 0
    np.testing.assert_allclose(c.sumsq[:nd].cpu().double().numpy(), want, rtol=1e-6)
    assert bool((c.sumsq[nd : nd + T] > 0).all()) and bool((c.scale[: c.n_vars] == 1.0).all())
