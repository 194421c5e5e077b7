"""GPU: Keras sample weights -- the weighted metric kernel against exact and float64 sums, the weighted BCE kernels against the
oracle, DeepFM fit with sample_weight / class_weight on the fused and layer paths against each other and a float64 DeepFM,
evaluate((x, y, sample_weight)) and weighted_metrics on the fused and layer paths (DIN and a BatchNorm DNN too), the sharded engine on
emulated ranks, and the step's launches with and without weights."""
import numpy as np
import pytest
import torch

import oracle
from oracle import weights_ref as WR
from tests.test_gpu_api import _deepfm_data
from tests.test_gpu_parity import close

pytestmark = pytest.mark.gpu


# ---- 1. the weighted metric kernel -------------------------------------------------------------------------------------------------
def _set_with(T):
    """A MetricSet over T thresholds whose metrics are half weighted, half not."""
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet, Precision, Recall

    if T == 1:
        ms = [Precision(), Recall(), BinaryAccuracy(), Precision(), BinaryAccuracy()]
    else:
        a, b = AUC(num_thresholds=T), AUC(num_thresholds=T)
        t = float(a._thresholds[T // 2])
        ms = [a, BinaryAccuracy(threshold=t), b, BinaryAccuracy(threshold=t)]
    s = MetricSet(ms, weighted=ms[len(ms) // 2 :])
    assert len(s.thresholds) == T
    return s


def _increments(s, p, y, w, kinds):
    """One batch's float64 increment of every variable of MetricSet `s` under descriptor kinds `kinds` (histogram form)."""
    p = np.asarray(p, np.float32)
    thr = s.thresholds
    T = len(thr)
    bucket = np.where(np.isnan(p), 0, np.searchsorted(thr, p, side="left"))
    cls = np.where(y == 0, 0, np.where(y == 1, 1, 2))
    inc = np.zeros(len(kinds), np.float64)
    for weighted in (False, True):
        ww = w.astype(np.float64) if weighted else np.ones(len(p))
        hist = np.stack([np.bincount(bucket[cls == c], weights=ww[cls == c], minlength=T + 1) for c in range(3)])
        above = np.cumsum(hist[:, ::-1], axis=1)[:, ::-1][:, 1:]
        tot = hist.sum(1)
        for v, (k, j) in enumerate(zip(kinds, s.thr_index)):
            if (k >= 6) != weighted:
                continue
            a0, a1, a2 = above[0, j], above[1, j], above[2, j]
            inc[v] = [a1 + a2, a0, tot[0] - a0, tot[1] + tot[2] - a1 - a2, a1 + tot[0] - a0, tot.sum()][k % 6]
    return inc


def _batch(n, thr, seed, weights):
    from tests.test_gpu_metrics import _adversarial

    p, y = _adversarial(n, thr, seed)
    rng = np.random.RandomState(seed + 1)
    if weights == "int":
        w = rng.randint(-3, 8, n).astype(np.float32)
    elif weights == "float":
        w = (rng.randn(n) * 2).astype(np.float32)
        w[rng.rand(n) < 0.1] = 0.0
    else:
        w = np.ones(n, np.float32)
    return p, y, w


@pytest.mark.parametrize("T", [1, 200, 8192])
@pytest.mark.parametrize("n", [1, 255, 65_536, 1_000_003])
def test_weighted_kernel_variables(dev, n, T):
    from handyrec_b200 import kernels as K

    s = _set_with(T)
    wk = s.weighted_kinds
    for weights in ("int", "float", "ones"):
        p, y, w = _batch(n, s.thresholds, n % 97 + T, weights)
        pd, yd, wd = (torch.from_numpy(a).to(dev) for a in (p, y, w))
        s.reset()
        s.update(pd, yd, wd)
        got = s.variables.cpu().numpy()
        inc = _increments(s, p, y, w, wk)
        want = inc.astype(np.float32)
        counts = wk < 6
        assert np.array_equal(got[counts], want[counts])  # integer counts: exact
        if weights == "float":
            ulp = np.spacing(np.abs(want[~counts]))
            assert np.all(np.abs(got[~counts].astype(np.float64) - want[~counts]) <= ulp), weights
        else:
            assert np.array_equal(got, want), weights
        if weights == "ones":  # all-ones weights: the weighted variables are the counts
            assert np.array_equal(got[~counts], _increments(s, p, y, w, s.kinds).astype(np.float32)[~counts])
        # kinds 0..5 of the weighted launch == hrb_metric_update on the same batch
        v1 = torch.zeros(len(s.kinds), device=dev)
        b = s._buffers()
        K.metric_update(pd, yd, b["thresholds"], b["kinds"], b["thr_index"], v1, b["scratch"])
        assert np.array_equal(got[counts], v1.cpu().numpy()[counts])
        # two runs give the same bits
        s.reset()
        s.update(pd, yd, wd)
        assert np.array_equal(s.variables.cpu().numpy(), got)


def test_weighted_kernel_accumulates_and_flags(dev):
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet

    auc, acc = AUC(num_thresholds=50), BinaryAccuracy()
    s = MetricSet([auc, acc], weighted=[auc, acc])
    want = np.zeros(len(s.kinds), np.float32)
    for i in range(3):  # the scratch is left clean for the next call
        p, y, w = _batch(10_000, s.thresholds, i, "int")
        s.update(torch.from_numpy(p).to(dev), torch.from_numpy(y).to(dev), torch.from_numpy(w).to(dev))
        want = (want + _increments(s, p, y, w, s.weighted_kinds).astype(np.float32)).astype(np.float32)
    assert np.array_equal(s.variables.cpu().numpy(), want)
    s.update(torch.tensor([0.2, 1.5], device=dev), torch.tensor([0.0, 1.0], device=dev), torch.tensor([1.0, 2.0], device=dev))
    with pytest.raises(ValueError, match="'auc'"):
        auc.result()
    acc.result()  # accuracy is never flagged
    auc.reset_state()
    s.update(torch.tensor([0.3, 0.6], device=dev), torch.tensor([0.0, 1.0], device=dev), torch.tensor([2.0, 3.0], device=dev))
    assert auc.result() == pytest.approx(1.0)


def test_weighted_results_match_the_oracle(dev):
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet
    from oracle import metrics_ref as R

    rng = np.random.RandomState(3)
    y = (rng.rand(5000) < 0.3).astype(np.float32)
    p = np.clip(rng.beta(2, 5, 5000) + 0.2 * y, 0, 1).astype(np.float32)
    w = rng.rand(5000).astype(np.float32) * 3
    auc, acc = AUC(), BinaryAccuracy()
    s = MetricSet([auc, acc], weighted=[auc, acc])
    s.update(torch.from_numpy(p).to(dev), torch.from_numpy(y).to(dev), torch.from_numpy(w).to(dev))
    k, c = WR.weighted_binary_accuracy(p, y, w)
    assert float(acc.result()) == pytest.approx(k / c, rel=1e-6)
    c = WR.weighted_confusion(p, y, w, auc._thresholds)
    assert float(auc.result()) == pytest.approx(R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"]), rel=1e-5)


# ---- 2. the weighted BCE kernels ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 1000, 100_003])
def test_weighted_bce_kernels(dev, n):
    from handyrec_b200 import kernels as K
    from handyrec_b200._lib import call

    g = torch.Generator().manual_seed(n)
    a, b = torch.randn(n, generator=g) * 3, torch.randn(n, generator=g)
    y = (torch.rand(n, generator=g) < 0.3).float()
    w = torch.randn(n, generator=g) * 2
    w[torch.rand(n, generator=g) < 0.1] = 0.0
    A, Bd, Y, Wd = (t.to(dev) for t in (a, b, y, w))
    outs = {}
    for name, wt in (("w", Wd), ("ones", torch.ones(n, device=dev)), ("plain", None)):
        prob, dl, ls = torch.empty(n, device=dev), torch.empty(n, device=dev), torch.zeros(1, device=dev)
        K.sigmoid_bce(A, Bd, Y, 1.0 / n, prob, dl, ls, weight=wt)
        outs[name] = (prob.cpu(), dl.cpu(), float(ls) / n)
    loss, d = WR.weighted_bce_from_logits((a + b).double(), y, w)
    assert outs["w"][2] == pytest.approx(loss, rel=1e-5, abs=1e-6)
    close(outs["w"][1], d, 1e-4)
    assert torch.equal(outs["ones"][0], outs["plain"][0]) and torch.equal(outs["ones"][1], outs["plain"][1])
    # the clipped (probability) form, with probabilities at and beyond the clip
    pr = torch.sigmoid(a)
    pr[:: 7] = 0.0
    outs = {}
    for name, wt in (("w", Wd), ("ones", torch.ones(n, device=dev)), ("plain", None)):
        dp, ls = torch.empty(n, device=dev), torch.zeros(1, device=dev)
        if wt is None:
            call("hrb_clipped_bce", K._p(pr.to(dev)), K._p(Y), n, 1e-7, 1.0 / n, K._p(dp), K._p(ls), K._stream())
        else:
            call("hrb_clipped_bce_weighted", K._p(pr.to(dev)), K._p(Y), K._p(wt), n, 1e-7, 1.0 / n, K._p(dp), K._p(ls), K._stream())
        outs[name] = (dp.cpu(), float(ls) / n)
    loss, d = WR.weighted_bce_from_probs(pr.double(), y, w)
    assert outs["w"][1] == pytest.approx(loss, rel=1e-5, abs=1e-6)
    close(outs["w"][0], d, 1e-4)
    assert torch.equal(outs["ones"][0], outs["plain"][0])


# ---- 3. DeepFM fit with sample weights ------------------------------------------------------------------------------------------
def _weights_of(y, seed=5):
    rng = np.random.RandomState(seed)
    w = rng.rand(len(y)) * 2.0
    w[rng.rand(len(y)) < 0.1] = 0.0
    return w


@pytest.mark.parametrize("name", ["adam", "ftrl"])
def test_weighted_fit_fused_layer_and_oracle_agree(dev, monkeypatch, name):
    from tests import test_gpu_schedules as S

    steps = 3
    x, y = _deepfm_data(steps * S.BS)
    sw = _weights_of(y)
    fused, plain = S._pair(name, lambda: S._opt(name, S.LR0[name]), monkeypatch)
    w0 = S._weights(plain)
    S._pin_units(fused)
    fused.fit(x, y, batch_size=S.BS, sample_weight=sw)
    plain.fit(x, y, batch_size=S.BS, sample_weight=sw)
    tol = {"adam": 2e-4, "ftrl": 1e-3}[name]
    wf, wp = S._weights(fused), S._weights(plain)
    for k in wf:
        close(wf[k], wp[k], tol)
    # the float64 DeepFM: its mean BCE becomes Keras' weighted loss, batch by batch
    calls = iter(range(steps))
    w32 = sw.astype(np.float32).astype(np.float64)

    def weighted_bce(logit, yy):
        i = next(calls)
        ww = torch.as_tensor(w32[i * S.BS : (i + 1) * S.BS], dtype=logit.dtype)
        l = torch.nn.functional.binary_cross_entropy_with_logits(logit, yy.to(logit.dtype), reduction="none")
        return (ww * l).mean()

    monkeypatch.setattr(oracle, "bce_from_logits", weighted_bce)
    want = S._oracle_run(name, w0, x, y, [S.LR0[name]] * steps)
    otol = {"adam": 2e-3, "ftrl": 2e-3}[name]
    for k in wp:
        close(wp[k], want[k], otol)


def test_weighted_fit_with_clipnorm_fused_equals_layer_path(dev, monkeypatch):
    from tests import test_gpu_schedules as S

    x, y = _deepfm_data(3 * S.BS)
    sw = _weights_of(y, 7)
    fused, plain = S._pair("adam", lambda: S._opt("adam", 0.02, clipnorm=0.05), monkeypatch)
    S._pin_units(fused)
    fused.fit(x, y, batch_size=S.BS, sample_weight=sw)
    plain.fit(x, y, batch_size=S.BS, sample_weight=sw)
    wf, wp = S._weights(fused), S._weights(plain)
    for k in wf:
        close(wf[k], wp[k], 2e-4)


@pytest.mark.parametrize("fuse", [True, False])
def test_unit_weights_and_class_weight_are_bit_exact(dev, monkeypatch, fuse):
    """Weights of one leave every parameter bit-equal to an unweighted fit; class_weight equals the sample_weight it stands for."""
    from handyrec_b200 import keras_lite as KL
    from tests import test_gpu_schedules as S
    from tests.test_gpu_clip import _model

    x, y = _deepfm_data(3 * S.BS + 100)  # a partial last batch
    cw = {0: 0.5, 1: 3.0}
    runs = []
    for kw in ({}, dict(sample_weight=np.ones(len(y))), dict(class_weight={0: 1, 1: 1}), dict(class_weight=cw),
               dict(sample_weight=np.where(y == 1, 3.0, 0.5))):
        m = _model(0)
        m.fuse = fuse
        m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy, metrics=["AUC"])
        if fuse:
            S._pin_units(m)
        h = m.fit(x, y, batch_size=S.BS, **kw)
        runs.append((S._weights(m), h.history))
    for i, j in ((0, 1), (0, 2), (3, 4)):
        for k in runs[i][0]:
            assert torch.equal(runs[i][0][k], runs[j][0][k]), (i, j, k)
        assert runs[i][1] == runs[j][1]
    assert any(not torch.equal(runs[0][0][k], runs[3][0][k]) for k in runs[0][0])


# ---- 4. evaluate((x, y, sample_weight)) and weighted_metrics ------------------------------------------------------------------------------
def _check_weighted_evaluate(make, x, y, xv, yv, bs, logits=True):
    """fit with validation_data=(x, y, sw) -> evaluate((x, y, sw)) == val_loss; weighted metrics against the oracle;
    the unweighted metrics of the run equal to evaluating without weights.  Without logits (BatchNorm behind the sigmoid, so
    predictions leave [0, 1]) only accuracy, which has no range rule, is compiled."""
    from oracle import metrics_ref as R

    names = ["auc", "accuracy"] if logits else ["accuracy"]
    sw, swv = _weights_of(y, 1), _weights_of(yv, 2)
    m = make([n.upper() if n == "auc" else n for n in names], [n.upper() if n == "auc" else n for n in names])
    assert m.metrics_names == ["loss"] + names + ["weighted_" + n for n in names]
    h = m.fit(x, y, batch_size=bs, sample_weight=sw, validation_data=(xv, yv, swv))
    keys = names + ["weighted_" + n for n in names]
    assert list(h.history) == ["loss"] + keys + ["val_loss"] + ["val_" + k for k in keys]
    res = m.evaluate((xv, yv, swv), batch_size=bs, return_dict=True)
    assert res["loss"] == h.history["val_loss"][-1]
    for k in keys:
        assert res[k] == pytest.approx(h.history["val_" + k][-1], rel=1e-6)
    p = m.predict(xv, batch_size=bs).reshape(-1)
    w32 = swv.astype(np.float32)
    k, n = WR.weighted_binary_accuracy(p, yv, w32)
    assert res["weighted_accuracy"] == pytest.approx(k / n, rel=1e-5)
    if logits:
        lp = np.clip(p.astype(np.float64), 1e-7, 1 - 1e-7)
        want = -(yv * np.log(lp) + (1 - yv) * np.log1p(-lp)) * w32
        assert res["loss"] == pytest.approx(want.mean() if m._fused is not None else np.mean(
            [want[s : s + bs].sum() / len(want[s : s + bs]) for s in range(0, len(want), bs)]), rel=1e-4)
        c = WR.weighted_confusion(p, yv, w32, m.metrics[2]._thresholds)
        assert res["weighted_auc"] == pytest.approx(R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"]), rel=1e-4)
        c = R.confusion_counts(p, yv, m.metrics[0]._thresholds)
        assert res["auc"] == pytest.approx(R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"]), rel=1e-4)
    # the unweighted metrics never see the weights: the same values as evaluating without them
    plain = m.evaluate(xv, yv, batch_size=bs, return_dict=True)
    for k in names:
        assert plain[k] == res[k]
    k, n = R.binary_accuracy_counts(p, yv)
    assert plain["weighted_accuracy"] == pytest.approx(k / n, rel=1e-6)  # no weights: counted like an unweighted metric
    return m


@pytest.mark.parametrize("fuse", [True, False])
def test_weighted_evaluate_deepfm(dev, fuse):
    from handyrec_b200 import keras_lite as K
    from tests.test_gpu_api import _deepfm_model

    def make(metrics, weighted):
        m = _deepfm_model()
        m.fuse = fuse
        m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy, metrics=metrics, weighted_metrics=weighted)
        assert (m._fused is not None) == fuse
        return m

    x, y = _deepfm_data(600)
    xv, yv = _deepfm_data(333, seed=7)
    _check_weighted_evaluate(make, x, y, xv, yv, 128)
    # the unweighted metrics, counted by the weighted update of each training step, are bit-equal to a fit without weights
    a, b = make(["AUC", "accuracy"], ["AUC"]), make(["AUC", "accuracy"], None)
    ha = a.fit(x, y, batch_size=128, sample_weight=np.ones(600))
    hb = b.fit(x, y, batch_size=128)
    for k in ("loss", "auc", "accuracy"):
        assert ha.history[k] == hb.history[k]


def test_weighted_evaluate_din_layer_path(dev):
    from handyrec_b200 import keras_lite as K
    from handyrec_b200.config import ConfigLoader
    from handyrec_b200.models import DIN
    from tests.test_gpu_models import _data
    from tests.test_mirror_cpu import DIN_CFG, FEATURE_DIM

    def make(metrics, weighted):
        g = ConfigLoader(DIN_CFG).prepare_features(FEATURE_DIM)
        m = DIN(g["item_seq_feat_group"], g["other_feature_group"], dnn_hidden_units=(8,), lau_dnn_hidden_units=(8, 1))
        m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy, metrics=metrics, weighted_metrics=weighted)
        return m

    x, y = _data(200, seed=3)
    xv, yv = _data(120, seed=4)
    _check_weighted_evaluate(make, x, y, xv, yv, 50)


def test_weighted_evaluate_batchnorm_dnn_clipped_bce(dev):
    """A DNN with BatchNorm behind its sigmoid: binary_crossentropy takes the clipped-probability path, weighted."""
    from handyrec_b200 import keras_lite as K
    from handyrec_b200.layers.core import DNN

    def make(metrics, weighted):
        torch.manual_seed(0)
        inp = K.Input((6,), name="feat")
        out = DNN((8, 1), use_bn=True, output_activation="sigmoid")(inp)
        m = K.Model(inp, out)
        m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy, metrics=metrics, weighted_metrics=weighted)
        return m

    rng = np.random.RandomState(0)
    x = {"feat": rng.randn(300, 6).astype(np.float32)}
    y = (rng.rand(300) < 0.4).astype(np.float32)
    xv = {"feat": rng.randn(150, 6).astype(np.float32)}
    yv = (rng.rand(150) < 0.4).astype(np.float32)
    m = _check_weighted_evaluate(make, x, y, xv, yv, 50, logits=False)
    # the weighted clipped loss of one batch against the oracle
    sw = _weights_of(yv, 9)[:50]
    xb = {"feat": xv["feat"][:50]}
    p = m.predict(xb).reshape(-1)
    got = m.evaluate((xb, yv[:50], sw), batch_size=50)
    assert got[0] == pytest.approx(WR.weighted_bce_from_probs(p, yv[:50], sw.astype(np.float32))[0], rel=1e-5)


def test_iterable_batches_and_tuple_input_take_weights(dev):
    """fit over an iterable of (x, y, sw) batches or an (x, y, sw) tuple equals fit over the arrays with sample_weight (layer
    path); evaluate over a tuple equals evaluate over the batches."""
    from handyrec_b200 import keras_lite as K
    from tests.test_gpu_api import _deepfm_model
    from tests.test_gpu_clip import _vars

    x, y = _deepfm_data(512)
    sw = _weights_of(y, 4)
    out = []
    for mode in ("arrays", "iterable", "tuple"):
        m = _deepfm_model()
        m.fuse = False
        m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy)
        if mode == "arrays":
            m.fit(x, y, batch_size=128, sample_weight=sw)
        elif mode == "tuple":
            m.fit((x, y, sw), batch_size=128)
        else:
            m.fit([({k: v[s : s + 128] for k, v in x.items()}, y[s : s + 128], sw[s : s + 128]) for s in range(0, 512, 128)])
        out.append({k: p.detach().cpu().clone() for k, p in _vars(m)})
    for k in out[0]:
        assert torch.equal(out[0][k], out[1][k]) and torch.equal(out[0][k], out[2][k]), k
    # evaluate takes its weights with the data: a (x, y, sw) tuple and an iterable of (x, y, sw) batches give the same loss
    batches = [({k: v[s : s + 128] for k, v in x.items()}, y[s : s + 128], sw[s : s + 128]) for s in range(0, 512, 128)]
    assert m.evaluate((x, y, sw), batch_size=128) == m.evaluate(batches)
    assert m.evaluate((x, y, np.ones(512)), batch_size=128) == m.evaluate(x, y, batch_size=128)


def test_shim_fit_takes_sample_weight(dev):
    """`tf.keras` code through the compat shim: fit(sample_weight=...) reaches the weighted step."""
    from handyrec_b200 import compat
    from tests.test_gpu_api import _deepfm_model

    x, y = _deepfm_data(256)
    compat.install(force=True)
    try:
        import tensorflow as tf

        losses = []
        for sw in (None, np.where(y == 1, 4.0, 1.0)):
            m = _deepfm_model()
            m.compile(optimizer=tf.keras.optimizers.Adam(0.01), loss=tf.keras.losses.binary_crossentropy)
            losses.append(m.fit(x, y, batch_size=256, sample_weight=sw).history["loss"][0])
        assert losses[1] > losses[0] * 1.3
    finally:
        compat.uninstall()


# ---- 5. the sharded engine ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_weighted_step_equals_one_gpu(dev, world):
    from handyrec_b200.engine import DeepFMEngine
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet
    from handyrec_b200.sharded import ShardedDeepFMEngine
    from tests import shard_helpers as H
    from tests.test_gpu_sharded import _run_threads

    b, D, n_dense, hidden = 64, 8, 3, (16, 1)
    g = torch.Generator().manual_seed(1)
    vocabs = [11, 50, 300]
    tables = [(torch.rand(v, D, generator=g) - 0.5) * 0.1 for v in vocabs]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 1, "none")]
    ids = [torch.cat([torch.randint(0, v, (b, 1), generator=g, dtype=torch.int32) for v in vocabs], 1) for _ in range(world)]
    dense = [torch.randn(b, n_dense, generator=g) for _ in range(world)]
    label = [(torch.rand(b, generator=g) < 0.3).float() for _ in range(world)]
    weight = [torch.randint(0, 4, (b,), generator=g).float() for _ in range(world)]  # integer weights: exact sums in any order

    def mk():
        a, acc = AUC(num_thresholds=50), BinaryAccuracy()
        return MetricSet([a, acc], weighted=[a, acc])

    ref = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=b * world, seed=7, lr=0.1)
    ref.metrics = mk()
    ref.train_step_on_device(torch.cat(ids).to(dev), torch.cat(dense).to(dev), torch.cat(label).to(dev), torch.cat(weight).to(dev))
    torch.cuda.synchronize()
    shared = H.ThreadComm.Shared(world)
    engines, read, probs = [None] * world, [None] * world, [None] * world

    def rank_fn(r):
        sh = [s_.to(dev) for s_ in H.shards_of(tables, r, world)]
        comm = H.ThreadComm(shared, r)
        eng = ShardedDeepFMEngine(sh, vocabs, fields, n_dense, comm, dnn_hidden_units=hidden, dnn_activation="relu", batch_size=b, seed=7,
                                  lr=0.1)
        eng.metrics = mk()
        engines[r] = eng
        eng.train_step_on_device(ids[r].to(dev), dense[r].to(dev), label[r].to(dev), weight[r].to(dev))
        torch.cuda.synchronize()
        probs[r] = eng.prob[:b].cpu().numpy()
        read[r] = eng.metrics.read(comm)
        return float(eng.loss_sum)

    losses = _run_threads(world, rank_fn)
    assert abs(sum(losses) - float(ref.loss_sum)) < 1e-4 * abs(float(ref.loss_sum))
    for r in range(world):
        close(engines[r].params, ref.params, 1e-4)
        for t in range(len(vocabs)):
            ws = ref.tables[t][r::world]
            if ws.shape[0]:
                close(engines[r].tables[t][: ws.shape[0]], ws, 1e-4)
    ms = mk()
    want = _increments(ms, np.concatenate(probs), torch.cat(label).numpy(), torch.cat(weight).numpy(), ms.weighted_kinds)
    for r in range(world):
        assert np.array_equal(read[r], want.astype(np.float32))  # integer weights: the summed read is exact


# ---- 6. launches -----------------------------------------------------------------------------------------------------------------
def test_step_launches_with_and_without_weights(dev):
    from handyrec_b200.engine import DeepFMEngine, launch_count
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet

    g = torch.Generator().manual_seed(2)
    vocabs, D, B = [40, 70, 500], 8, 1024
    tables = [((torch.rand(v, D, generator=g) - 0.5) * 0.1).to(dev) for v in vocabs]
    eng = DeepFMEngine(tables, [(0, 1, "none"), (1, 1, "none"), (2, 2, "mean")], 4, (32, 16, 1), "relu", batch_size=B)
    eng.autotune_embedding_bwd = False
    ids = torch.cat([torch.randint(0, v, (B, 1 if i < 2 else 2), generator=g, dtype=torch.int32) for i, v in enumerate(vocabs)], 1).to(dev)
    dense = torch.randn(B, 4, generator=g).to(dev)
    label = (torch.rand(B, generator=g) < 0.3).float().to(dev)
    w = torch.rand(B, generator=g).to(dev)

    def step_launches(weight=None):
        c0 = launch_count()
        eng.train_step_on_device(ids, dense, label, weight)
        torch.cuda.synchronize()
        return launch_count() - c0

    step_launches()
    base = step_launches()
    assert step_launches(w) == base  # the weighted BCE replaces the BCE
    auc = AUC()
    eng.metrics = MetricSet([auc, BinaryAccuracy()])
    assert step_launches() == base + 1 and step_launches(w) == base + 1  # no weighted metric: the weights are not read
    auc_w = AUC()
    eng.metrics = MetricSet([AUC(), auc_w, BinaryAccuracy()], weighted=[auc_w])
    assert step_launches() == base + 1  # without weights: hrb_metric_update as before
    assert step_launches(w) == base + 2  # one weighted update: two launches for every metric of the set
    eng.metrics = None
    assert step_launches() == base
