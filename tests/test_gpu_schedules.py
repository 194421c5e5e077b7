"""GPU: Keras learning-rate schedules and time-based decay on both training paths -- the fused DeepFM engine, the layer path
(dense multi-tensor step and apply_sparse row updates) and a float64 DeepFM driven by the oracle's rates; constant schedules against
float rates; the step counter across fits; the sharded engine on emulated ranks."""
import math

import numpy as np
import pytest
import torch

import oracle
from oracle import schedule_ref as R
from tests.test_gpu_api import _deepfm_data
from tests.test_gpu_clip import _TABLE_OF, _model, _vars
from tests.test_gpu_parity import close

pytestmark = pytest.mark.gpu

BS, STEPS = 256, 5
SMALL = 45  # tables above this size take the row update on both paths (movie_id, 50 rows); the others are dense-updated
LR0 = {"sgd": 0.5, "adam": 0.02, "adagrad": 0.1, "ftrl": 0.2}
FTRL_KW = dict(beta=0.1, l2_regularization_strength=1e-3)


def _opt(name, lr, **kw):
    from handyrec_b200 import keras_lite as KL

    cls = {"sgd": KL.SGD, "adam": KL.Adam, "adagrad": KL.Adagrad, "ftrl": KL.Ftrl}[name]
    return cls(lr, **(dict(FTRL_KW, **kw) if name == "ftrl" else kw))


def _pin_units(m, bs=BS):
    """Build the engine now and pin its embedding backward to one algorithm (the autotune picks by timing)."""
    from handyrec_b200 import _lib

    m._fused.build(bs, m.optimizer)
    eng = m._fused.engine
    eng.bwd_algo = "units"
    _lib.call("hrb_plan_set_bwd_algo", eng.plan._h, _lib.BWD_UNITS)
    return eng


def _pair(name, make_opt, monkeypatch, seed=0):
    """A fused and a layer-path DeepFM with the same initial weights; movie_id takes the row update on both."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding

    monkeypatch.setattr(CustomEmbedding, "SPARSE_UPDATE_MIN_ROWS", SMALL)
    fused, plain = _model(seed), _model(seed)
    plain.fuse = False
    fused.dense_table_max_rows = SMALL
    fused.compile(optimizer=make_opt(), loss=KL.binary_crossentropy)
    plain.compile(optimizer=make_opt(), loss=KL.binary_crossentropy)
    assert fused._fused is not None and plain._fused is None
    return fused, plain


def _weights(m):
    return {k: p.detach().cpu().double() for k, p in _vars(m)}


# ---- the float64 DeepFM, stepped by the oracle's rates ----------------------------------------------------------------------
def _grads(W, x, y):
    """Dense float64 gradients of the mean BCE at weights W (names of tests.test_gpu_clip._vars) and, per table, the rows the
    batch gathers (padding id 0 of the pooled fields included, as Keras' IndexedSlices lists it)."""
    V = {k: w.clone().requires_grad_(True) for k, w in W.items()}
    B = len(y)
    touched = {k: torch.zeros(w.shape[0], dtype=torch.bool) for k, w in W.items() if k.startswith("t")}

    def lookup():
        outs = []
        for name in ("user_id", "gender", "movie_id", "hist_movie", "genres"):
            ids = torch.as_tensor(np.asarray(x[name])).reshape(B, -1).long()
            t = f"t{_TABLE_OF[name]}"
            touched[t][ids.reshape(-1)] = True
            e = V[t][ids]
            outs.append(e if ids.shape[1] == 1 else oracle.sequence_pooling(e, (ids != 0)[..., None].expand_as(e), "mean"))
        return outs

    fm_e, dnn_e = lookup(), lookup()
    p = oracle.DNNParams(3 + 5 * 8, (16, 8, 1))
    for i in range(len(p.units)):
        p.W.append(V[f"W{i}"])
        p.b.append(V[f"b{i}"])
    dense = [torch.as_tensor(np.asarray(x["age"], dtype=np.float64)).reshape(B, 1), torch.as_tensor(np.asarray(x["score"], dtype=np.float64))]
    logit = oracle.deepfm_forward(dense, fm_e, dnn_e, p, V["fmw"], V["fmw0"], return_logit=True)
    oracle.bce_from_logits(logit[:, 0], torch.as_tensor(y, dtype=torch.float64)).backward()
    return {k: v.grad.detach() for k, v in V.items()}, touched


def _oracle_run(name, W, x, y, rates):
    """Keras' optimizer on the float64 DeepFM, one step per batch at rates[i]: dense Adam on the dense-updated tables and the
    dense variables, lazy Adam on the row-updated table; Adagrad, SGD (dense == sparse); Ftrl stepping the gathered rows of every
    table (l2 = 0 tables, IndexedSlices) with l2 + beta / (2*lr_t)."""
    from oracle.ftrl_ref import ftrl_dense, kernel_l2
    from oracle.optim_ref import adagrad_dense

    W = {k: w.clone() for k, w in W.items()}
    S = {k: (torch.zeros_like(w), torch.zeros_like(w)) if name == "adam" else
         (torch.full_like(w, 0.1), torch.zeros_like(w)) for k, w in W.items()}
    for i, lr in enumerate(rates):
        xb = {k: v[i * BS : (i + 1) * BS] for k, v in x.items()}
        G, T = _grads(W, xb, y[i * BS : (i + 1) * BS])
        t = i + 1
        for k, g in G.items():
            w, (a, b) = W[k], S[k]
            if name == "sgd":
                W[k] = w - lr * g
            elif name == "adagrad":
                W[k], a = adagrad_dense(w, a, g, lr)
            elif name == "ftrl":
                l2 = kernel_l2(lr, FTRL_KW["l2_regularization_strength"], FTRL_KW["beta"])
                rows = T[k] if k in T else torch.ones(w.shape[0], dtype=torch.bool)
                w, a, b = w.clone(), a.clone(), b.clone()
                w[rows], a[rows], b[rows] = ftrl_dense(w[rows], a[rows], b[rows], g[rows], lr, l2=l2)
                W[k] = w
            else:
                rows = T[k] if k == "t50" else torch.ones(w.shape[0], dtype=torch.bool)  # movie_id (row update): lazy Adam
                a, b = a.clone(), b.clone()
                a[rows] = 0.9 * a[rows] + 0.1 * g[rows]
                b[rows] = 0.999 * b[rows] + 0.001 * g[rows] ** 2
                w = w.clone()
                w[rows] = w[rows] - lr * math.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t) * a[rows] / (torch.sqrt(b[rows]) + 1e-7)
                W[k] = w
            S[k] = (a, b)
    return W


def _schedule(kind, lr0):
    """A schedule whose rate changes at every step, and its float64 oracle."""
    from handyrec_b200.schedules import CosineDecayRestarts, ExponentialDecay

    if kind == "exponential":
        return ExponentialDecay(lr0, 2, 0.5), (lambda s: R.exponential_decay(s, lr0, 2, 0.5))
    return CosineDecayRestarts(lr0, 3, m_mul=0.8, alpha=0.2), (lambda s: R.cosine_decay_restarts(s, lr0, 3, m_mul=0.8, alpha=0.2))


@pytest.mark.parametrize("kind", ["exponential", "cosine_restarts"])
@pytest.mark.parametrize("name", ["sgd", "adam", "adagrad", "ftrl"])
def test_schedule_fused_layer_path_and_oracle_agree(dev, monkeypatch, name, kind):
    x, y = _deepfm_data(STEPS * BS)
    _, ref = _schedule(kind, LR0[name])
    fused, plain = _pair(name, lambda: _opt(name, _schedule(kind, LR0[name])[0]), monkeypatch)
    w0 = _weights(plain)
    eng = _pin_units(fused)
    fused.fit(x, y, batch_size=BS)
    plain.fit(x, y, batch_size=BS)
    assert fused._fused.engine is eng and fused.optimizer.iterations == STEPS and plain.optimizer.iterations == STEPS
    movie = next(l for l in plain._all_layers() if getattr(l, "input_dim", 0) == 50)
    assert getattr(movie, "_plan", None) is not None  # the layer path's large table took apply_sparse
    rates = [ref(s) for s in range(STEPS)]
    assert len(set(rates)) == STEPS
    assert abs(eng.lr - rates[-1]) <= 1e-6 * rates[-1]  # the engine ran its last step at the schedule's rate
    tol = {"sgd": 1e-4, "adagrad": 1e-4, "adam": 2e-4, "ftrl": 1e-3}[name]
    wf, wp = _weights(fused), _weights(plain)
    for k in wf:
        close(wf[k], wp[k], tol)
    want = _oracle_run(name, w0, x, y, rates)
    # Adam / Ftrl: m / sqrt(v) and Ftrl's linear - sigma * w amplify the fp32 rounding of small gradients over five steps
    otol = {"sgd": 2e-4, "adagrad": 2e-4, "adam": 2e-3, "ftrl": 2e-3}[name]
    for k in wp:
        close(wp[k], want[k], otol)


@pytest.mark.parametrize("name", ["sgd", "adam", "adagrad", "ftrl"])
@pytest.mark.parametrize("fuse", [True, False])
def test_constant_schedule_equals_the_float_rate(dev, monkeypatch, name, fuse):
    """ExponentialDecay(lr, 10, 1.0) is float32(lr) at every step: the kernels take the same float as with the float rate, so the
    weights are bit-equal.  Ftrl's beta / (2*lr) is formed in double from float32(lr) instead of lr: equal to rounding."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.layers import CustomEmbedding
    from handyrec_b200.schedules import ExponentialDecay

    monkeypatch.setattr(CustomEmbedding, "SPARSE_UPDATE_MIN_ROWS", SMALL)
    x, y = _deepfm_data(4 * BS)
    lr = LR0[name]
    runs = []
    for rate in (lr, ExponentialDecay(lr, 10, 1.0)):
        m = _model(0)
        m.fuse = fuse
        m.dense_table_max_rows = SMALL
        m.compile(optimizer=_opt(name, rate), loss=KL.binary_crossentropy)
        if fuse:
            _pin_units(m)
        m.fit(x, y, batch_size=BS)
        assert m.optimizer.iterations == 4
        runs.append(_weights(m))
    for k in runs[0]:
        if name == "ftrl":
            close(runs[1][k], runs[0][k], 1e-5)
        else:
            assert torch.equal(runs[0][k], runs[1][k]), k


def test_fit_keeps_the_engine_and_a_second_fit_continues_the_schedule(dev, monkeypatch):
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.schedules import CosineDecayRestarts

    x, y = _deepfm_data(8 * BS)
    half = 4 * BS
    runs = []
    for split in (False, True):
        m = _model(0)
        m.dense_table_max_rows = SMALL
        sched = CosineDecayRestarts(0.02, 3, t_mul=1.5, m_mul=0.8, alpha=0.1)
        m.compile(optimizer=KL.Adam(sched, decay=0.05), loss=KL.binary_crossentropy)
        eng = _pin_units(m)
        if split:
            m.fit({k: v[:half] for k, v in x.items()}, y[:half], batch_size=BS)
            assert m._fused.engine is eng and m.optimizer.iterations == 4 and eng.step_count == 4
            m.fit({k: v[half:] for k, v in x.items()}, y[half:], batch_size=BS)
        else:
            m.fit(x, y, batch_size=BS)
        assert m._fused.engine is eng and m.optimizer.iterations == 8 and eng.step_count == 8
        want_lr = float(np.float32(sched(7)) / (np.float32(1) + np.float32(0.05) * np.float32(7)))
        assert eng.lr == want_lr and m.optimizer.lr_t == want_lr
        runs.append(_weights(m))
    for k in runs[0]:
        assert torch.equal(runs[0][k], runs[1][k]), k


def test_layer_path_step_after_fused_fit_continues_the_schedule(dev, monkeypatch):
    """A train_on_batch through the engine, then through the layer path: the counter is shared, each step evaluated once."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.schedules import LearningRateSchedule

    calls = []

    class Halving(LearningRateSchedule):
        def __call__(self, step):
            calls.append(step)
            return 0.5 * 0.5 ** step

    x, y = _deepfm_data(3 * BS)
    m = _model(0)
    m.compile(optimizer=KL.SGD(Halving()), loss=KL.binary_crossentropy)
    m.fit({k: v[: 2 * BS] for k, v in x.items()}, y[: 2 * BS], batch_size=BS)
    m.sync()
    m._fused = None  # the layer path from here on
    m.train_on_batch({k: v[2 * BS :] for k, v in x.items()}, y[2 * BS :])
    assert calls == [0, 1, 2] and m.optimizer.iterations == 3 and m.optimizer.lr_t == 0.125


@pytest.mark.parametrize("name,kw", [("sgd", dict(decay=0.3)), ("ftrl", dict(decay=0.3)), ("adam", dict(decay=0.2, clipnorm=1e-2)),
                                     ("adagrad", dict(decay=0.2, clipnorm=1e-2))])
def test_time_based_decay(dev, monkeypatch, name, kw):
    """decay= alone (against the oracle too) and with clipnorm (fused against the layer path)."""
    x, y = _deepfm_data(STEPS * BS)
    lr = LR0[name]
    fused, plain = _pair(name, lambda: _opt(name, lr, **kw), monkeypatch)
    w0 = _weights(plain)
    _pin_units(fused)
    fused.fit(x, y, batch_size=BS)
    plain.fit(x, y, batch_size=BS)
    assert fused.optimizer.iterations == plain.optimizer.iterations == STEPS
    rates = [float(np.float32(lr) / (np.float32(1) + np.float32(kw["decay"]) * np.float32(s))) for s in range(STEPS)]
    assert fused._fused.engine.lr == rates[-1] and plain.optimizer.lr_t == rates[-1]
    tol = {"sgd": 1e-4, "adagrad": 1e-4, "adam": 2e-4, "ftrl": 1e-3}[name]
    wf, wp = _weights(fused), _weights(plain)
    for k in wf:
        close(wf[k], wp[k], tol)
    if "clipnorm" not in kw:
        want = _oracle_run(name, w0, x, y, [R.decayed_lr(lr, s, kw["decay"]) for s in range(STEPS)])
        for k in wp:
            close(wp[k], want[k], 2e-4 if name == "sgd" else 2e-3)


@pytest.mark.parametrize("opt", ["adam", "ftrl"])
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_engine_with_a_schedule_matches_single_gpu_engine(dev, world, opt):
    """Three steps of N emulated ranks whose rates come from a schedule (every rank its own optimizer, counting alike) == one engine
    on the concatenated batches with the same schedule.  Ftrl's beta / (2*lr_t) reaches the owner-side keyed update."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.engine import DeepFMEngine
    from handyrec_b200.lowering import _lr_step
    from handyrec_b200.schedules import ExponentialDecay
    from handyrec_b200.sharded import ShardedDeepFMEngine
    from tests import shard_helpers as H
    from tests.test_gpu_sharded import _run_threads

    b, D, n_dense, hidden, rep = 64, 8, 3, (16, 1), 60
    g = torch.Generator().manual_seed(1)
    vocabs = [11, 50, 300]
    tables = [(torch.rand(v, D, generator=g) - 0.5) * 0.1 for v in vocabs]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 3, "mean")]
    kw = dict(optimizer=opt, lr=0.1, seed=7) if opt == "adam" else dict(optimizer=opt, lr=0.1, seed=7, l1=1e-3, l2=1e-3, beta=0.5)
    make = (lambda: KL.Adam(ExponentialDecay(0.05, 1, 0.6))) if opt == "adam" else (lambda: KL.Ftrl(ExponentialDecay(0.3, 1, 0.6)))
    steps = []
    for _ in range(3):
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
    ref_opt = make()
    ref.lr_step = _lr_step(ref_opt)
    for ids, dense, label in steps:
        ref.train_step_on_device(torch.cat(ids).to(dev), torch.cat(dense).to(dev), torch.cat(label).to(dev))
    torch.cuda.synchronize()
    shared = H.ThreadComm.Shared(world)
    engines, opts = [None] * world, [make() for _ in range(world)]

    def rank_fn(r):
        sh = [(full if v <= rep else s_).to(dev) for full, s_, v in zip(tables, H.shards_of(tables, r, world), vocabs)]
        comm = H.ThreadComm(shared, r)
        eng = ShardedDeepFMEngine(sh, vocabs, fields, n_dense, comm, dnn_hidden_units=hidden, dnn_activation="relu", batch_size=b,
                                  replicate_max_rows=rep, **kw)
        eng.lr_step = _lr_step(opts[r])
        engines[r] = eng
        for ids, dense, label in steps:
            eng.train_step_on_device(ids[r].to(dev), dense[r].to(dev), label[r].to(dev))
        torch.cuda.synchronize()
        return float(eng.loss_sum)

    losses = _run_threads(world, rank_fn)
    assert all(o.iterations == 3 and o.lr_t == ref_opt.lr_t for o in opts) and ref_opt.iterations == 3
    assert ref.lr == ref_opt.lr_t and all(e.lr == ref.lr and e.ftrl_l2 == ref.ftrl_l2 for e in engines)
    assert abs(sum(losses) - float(ref.loss_sum)) < 1e-4 * abs(float(ref.loss_sum))
    for r in range(world):
        close(engines[r].params, ref.params, 1e-4)
        close(engines[r].opt_m, ref.opt_m, 1e-4)
        close(engines[r].opt_v, ref.opt_v, 1e-4)
        t = 2  # the row-sharded table
        ws = ref.tables[t][r::world]
        close(engines[r].tables[t][: ws.shape[0]], ws, 1e-4)
        if opt == "ftrl":
            close(engines[r].accum[t][: ws.shape[0]], ref.accum[t][r::world], 1e-4)
            close(engines[r].linear[t][: ws.shape[0]], ref.linear[t][r::world], 1e-4)
        else:
            close(engines[r].adam_m[t][: ws.shape[0]], ref.adam_m[t][r::world], 1e-4)
