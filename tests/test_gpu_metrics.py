"""GPU: Keras metrics counted by hrb_metric_update -- the variables bit-equal to a float32 emulation of Keras' confusion updates, the
results against the float64 oracle, the fused DeepFM step, fit / evaluate on the fused and layer paths, the sharded engine's
all-reduced read, and nothing changed (launches, history keys) without metrics."""
import numpy as np
import pytest
import torch

from oracle import metrics_ref as R

pytestmark = pytest.mark.gpu


def _increments(ms, p, y):
    """One batch's integer increments of every variable of MetricSet `ms`, by the oracle's rules (histogram form for big cases)."""
    p = np.asarray(p, np.float32).reshape(-1)
    y = np.asarray(y, np.float32).reshape(-1)
    thr = ms.thresholds
    bucket = np.where(np.isnan(p), 0, np.searchsorted(thr, p, side="left"))  # thresholds strictly below p
    cls = np.where(y == 0, 0, np.where(y == 1, 1, 2))
    T = len(thr)
    hist = np.stack([np.bincount(bucket[cls == c], minlength=T + 1) for c in range(3)]).astype(np.int64)
    suffix = np.cumsum(hist[:, ::-1], axis=1)[:, ::-1]
    above = suffix[:, 1:]  # above[c, j]
    tot = hist.sum(1)
    inc = np.zeros(len(ms.kinds), np.int64)
    for v, (k, j) in enumerate(zip(ms.kinds, ms.thr_index)):
        a0, a1, a2 = above[0, j], above[1, j], above[2, j]
        inc[v] = [a1 + a2, a0, tot[0] - a0, tot[1] + tot[2] - a1 - a2, a1 + tot[0] - a0, len(p)][k]
    return inc


def _adversarial(n, thr, seed):
    rng = np.random.RandomState(seed)
    pick = thr[(thr >= 0) & (thr <= 1)]
    specials = np.concatenate([pick, np.nextafter(pick, np.float32(2)), np.nextafter(pick, np.float32(-1)),
                               np.array([0.0, 1.0, 0.5, np.nextafter(np.float32(0.5), np.float32(1))], np.float32)]).astype(np.float32)
    specials = specials[(specials >= 0) & (specials <= 1)]
    p = rng.rand(n).astype(np.float32)
    k = min(n, len(specials))
    idx = rng.choice(n, k, replace=False)
    p[idx] = rng.choice(specials, k, replace=False) if len(specials) >= k else specials[:k]
    y = rng.choice(np.array([0, 1, 0.3, np.nan], np.float32), n, p=[0.45, 0.45, 0.05, 0.05])
    return p, y


def _set_with(T):
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet, Precision, Recall

    if T == 1:
        ms = [Precision(), Recall(), BinaryAccuracy()]
    else:
        a = AUC(num_thresholds=T)
        ms = [a, BinaryAccuracy(threshold=float(a._thresholds[T // 2]))]
    s = MetricSet(ms)
    assert len(s.thresholds) == T
    return s


# ---- 1. the kernel's variables are Keras' float32 counts ---------------------------------------------------------------------
def test_histogram_emulation_equals_the_oracle_counts():
    from handyrec_b200.metrics import AUC, MetricSet

    s = MetricSet([AUC(num_thresholds=7)])
    p, y = _adversarial(500, s.thresholds, 0)
    c = R.confusion_counts(p, y, s.thresholds)
    assert _increments(s, p, y).tolist() == np.concatenate([c["tp"], c["fp"], c["tn"], c["fn"]]).tolist()


@pytest.mark.parametrize("T", [1, 200, 8192])
@pytest.mark.parametrize("n", [1, 255, 65_536, 1_000_003])
def test_kernel_variables_bit_equal_float32_emulation(dev, n, T):
    s = _set_with(T)
    want = np.zeros(len(s.kinds), np.float32)
    for call in range(2):  # the second call must see a clean scratch
        p, y = _adversarial(n, s.thresholds, seed=10 * call + T % 7)
        s.update(torch.from_numpy(p).to(dev), torch.from_numpy(y).to(dev))
        want = R.accumulate_f32(want, _increments(s, p, y))
        got = s.variables.cpu().numpy()
        assert np.array_equal(got, want), f"call {call}: {np.flatnonzero(got != want)[:10]}"
    fresh = _set_with(T)
    fresh.update(torch.from_numpy(p).to(dev), torch.from_numpy(y).to(dev))
    assert np.array_equal(fresh.variables.cpu().numpy(), R.accumulate_f32(np.zeros(len(s.kinds), np.float32), _increments(s, p, y)))


def test_accumulation_over_300_batches_crosses_2_24(dev):
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet

    s = MetricSet([AUC(num_thresholds=10), BinaryAccuracy()])
    want = np.zeros(len(s.kinds), np.float32)
    rng = np.random.RandomState(5)
    for _ in range(300):
        p = rng.rand(65_536).astype(np.float32)
        y = (rng.rand(65_536) < 0.5).astype(np.float32)
        s.update(torch.from_numpy(p).to(dev), torch.from_numpy(y).to(dev))
        want = R.accumulate_f32(want, _increments(s, p, y))
    got = s.variables.cpu().numpy()
    assert want.max() > 2**24 and np.array_equal(got, want)


@pytest.mark.parametrize("bad", [-1e-8, 1.0000001, float("nan")])
def test_predictions_outside_unit_interval_raise_at_read(dev, bad):
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet

    auc, acc = AUC(), BinaryAccuracy()
    MetricSet([auc, acc])
    p = torch.tensor([0.2, bad, 0.7], device=dev)
    auc._set.update(p, torch.tensor([0.0, 1.0, 1.0], device=dev))
    with pytest.raises(ValueError, match="'auc'"):
        auc.result()
    assert float(acc.result()) == pytest.approx(1.0 if bad > 0.5 else 2 / 3)  # accuracy has no range rule (NaN > 0.5 is False)
    auc.reset_state()  # the public reset clears the metric's flags with its variables
    auc.update_state([0.0, 1.0], [0.3, 0.6])
    assert auc.result() == pytest.approx(1.0)
    solo = BinaryAccuracy()
    solo.update_state([1.0], [bad])
    solo.result()  # no ValueError: binary_accuracy asserts nothing
    # a standalone metric recovers after reset_state, as a Keras metric stays usable after its assertion failed
    own = AUC()
    own.update_state([0.0, 1.0], [0.2, bad])
    with pytest.raises(ValueError, match="'auc'"):
        own.result()
    own.reset_states()
    own.update_state([0.0, 1.0], [0.2, 0.9])
    assert own.result() == pytest.approx(1.0)


def test_a_bad_update_of_one_metric_leaves_the_others_of_its_set_readable(dev):
    from handyrec_b200 import keras_lite as K
    from tests.test_metrics_cpu import _tiny_model

    m = _tiny_model()
    m.compile(optimizer=K.SGD(0.1), loss=K.binary_crossentropy, metrics=["AUC", "Precision", "accuracy"])
    auc, prec, _ = m.metrics
    prec.update_state([1.0, 0.0], [1.5, 0.2])  # Precision alone counts the bad prediction
    with pytest.raises(ValueError, match="'precision'"):
        prec.result()
    auc.update_state([1.0, 0.0], [0.8, 0.2])
    assert auc.result() == pytest.approx(1.0)
    with pytest.raises(ValueError, match="'precision'"):  # the whole-model read names the metric that counted it
        m._metric_values()
    m.reset_metrics()
    assert m._metric_values()["precision"] == 0.0


# ---- 2. results against the float64 oracle -------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", ["ROC", "PR"])
@pytest.mark.parametrize("method", ["interpolation", "minoring", "majoring"])
def test_results_match_the_float64_oracle(dev, curve, method):
    from handyrec_b200.metrics import AUC, BinaryAccuracy, Precision, Recall

    rng = np.random.RandomState(1)
    n = 20_000
    y = (rng.rand(n) < 0.3).astype(np.float32)
    p = np.clip(rng.beta(2, 5, n) + 0.2 * y, 0, 1).astype(np.float32)
    auc, pr, rc, acc = AUC(curve=curve, summation_method=method), Precision(), Recall(thresholds=[0.3, 0.7]), BinaryAccuracy()
    for m in (auc, pr, rc, acc):
        m.update_state(torch.from_numpy(y).to(dev), p)  # device labels, host predictions
    c = R.confusion_counts(p, y, auc._thresholds)
    assert float(auc.result()) == pytest.approx(R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"], curve, method), rel=1e-6)
    c = R.confusion_counts(p, y, [0.5])
    assert float(pr.result()) == pytest.approx(float(R.precision_result(c["tp"], c["fp"])[0]), rel=1e-6)
    c = R.confusion_counts(p, y, [0.3, 0.7])
    np.testing.assert_allclose(rc.result(), R.recall_result(c["tp"], c["fn"]), rtol=1e-6)
    k, m = R.binary_accuracy_counts(p, y)
    assert float(acc.result()) == pytest.approx(k / m, rel=1e-6)
    acc.reset_states()
    assert float(acc.result()) == 0.0


# ---- 3. fused DeepFM: each training step counts its own forward ------------------------------------------------------------------
def _compiled_deepfm(fuse=True):
    from handyrec_b200 import keras_lite as K
    from tests.test_gpu_api import _deepfm_model

    m = _deepfm_model()
    m.fuse = fuse
    m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy,
              metrics=["AUC", "accuracy", K.Precision(), K.Recall(thresholds=[0.3, 0.7])])
    return m


def _slice(d, s, e):
    return {k: v[s:e] for k, v in d.items()}


def _check_counts(ms, p, y, slack=2):
    """The variables of `ms` after one batch == the oracle's counts from predictions `p`, except where a prediction lies within a
    few ulp of a threshold (two forwards may round differently there)."""
    got = ms.variables.cpu().numpy()
    want = _increments(ms, p, y).astype(np.float64)
    thr = ms.thresholds[ms.thr_index]
    p = np.asarray(p, np.float32).reshape(-1)
    near = np.abs(p[None, :].astype(np.float64) - thr[:, None]) <= slack * np.spacing(np.abs(thr[:, None]).astype(np.float32))
    amb = near.sum(1)
    amb[ms.kinds == 5] = 0
    assert np.all(np.abs(got - want) <= amb), np.flatnonzero(np.abs(got - want) > amb)


def test_fused_train_on_batch_counts_each_steps_forward(dev):
    from tests.test_gpu_api import _deepfm_data

    m = _compiled_deepfm()
    assert m._fused is not None
    x, y = _deepfm_data(1024)
    bs = 256
    m.train_on_batch(_slice(x, 0, bs), y[:bs])  # builds the engine
    for s in range(bs, 1024, bs):
        xb, yb = _slice(x, s, s + bs), y[s : s + bs]
        p = m.predict(xb, batch_size=bs)
        out = m.train_on_batch(xb, yb)
        assert len(out) == 5 and np.shape(out[4]) == (2,)
        _check_counts(m._metric_set, p, yb)
    d = m.train_on_batch(_slice(x, 0, bs), y[:bs], return_dict=True)
    assert list(d) == ["loss", "auc", "accuracy", "precision", "recall"]


def test_fused_fit_history_and_per_epoch_reset(dev):
    from tests.test_gpu_api import _deepfm_data

    m = _compiled_deepfm()
    x, y = _deepfm_data(700)
    xv, yv = _deepfm_data(300, seed=4)
    h = m.fit(x, y, batch_size=256, epochs=2, validation_data=(xv, yv))
    assert list(h.history) == ["loss", "auc", "accuracy", "precision", "recall", "val_loss", "val_auc", "val_accuracy", "val_precision",
                               "val_recall"]
    assert all(len(v) == 2 for v in h.history.values())
    # the state left behind is the last validation pass: 300 samples, not 700 or 1400
    acc = m.metrics[1]
    v = m._metric_set.variables.cpu().numpy()[m._metric_set.slices[1]]
    assert acc.name == "accuracy" and v[1] == 300
    h = m.fit(x, y, batch_size=256, epochs=2)
    v = m._metric_set.variables.cpu().numpy()[m._metric_set.slices[1]]
    assert v[1] == 700  # the second epoch's batches only: the metrics were reset at its start
    assert "val_loss" not in h.history and len(h.history["accuracy"]) == 2


# ---- 4. evaluate ---------------------------------------------------------------------------------------------------------------
def _check_evaluate(m, x, y, xv, yv, bs):
    h = m.fit(x, y, batch_size=bs, epochs=1, validation_data=(xv, yv))
    res = m.evaluate(xv, yv, batch_size=bs, return_dict=True)
    assert res["loss"] == h.history["val_loss"][-1]
    for k in ("auc", "accuracy"):
        assert res[k] == pytest.approx(h.history["val_" + k][-1], rel=1e-6)
    p = m.predict(xv, batch_size=bs).reshape(-1)
    auc = m.metrics[0]
    c = R.confusion_counts(p, yv, auc._thresholds)
    assert res["auc"] == pytest.approx(R.auc_result(c["tp"], c["fp"], c["tn"], c["fn"]), rel=1e-5)
    k, n = R.binary_accuracy_counts(p, yv)
    assert res["accuracy"] == pytest.approx(k / n, rel=1e-6)
    lst = m.evaluate(xv, yv, batch_size=bs)
    assert isinstance(lst, list) and lst[0] == res["loss"] and len(lst) == len(m.metrics_names)


@pytest.mark.parametrize("fuse", [True, False])
def test_evaluate_deepfm_equals_oracle_and_val_loss(dev, fuse):
    from tests.test_gpu_api import _deepfm_data

    m = _compiled_deepfm(fuse)
    assert (m._fused is not None) == fuse
    x, y = _deepfm_data(600)
    xv, yv = _deepfm_data(333, seed=7)
    _check_evaluate(m, x, y, xv, yv, 128)


def test_evaluate_din_layer_path(dev):
    from handyrec_b200 import keras_lite as K
    from handyrec_b200.config import ConfigLoader
    from handyrec_b200.models import DIN
    from tests.test_gpu_models import _data
    from tests.test_mirror_cpu import DIN_CFG, FEATURE_DIM

    g = ConfigLoader(DIN_CFG).prepare_features(FEATURE_DIM)
    m = DIN(g["item_seq_feat_group"], g["other_feature_group"], dnn_hidden_units=(8,), lau_dnn_hidden_units=(8, 1))
    m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy, metrics=["AUC", "accuracy"])
    x, y = _data(200, seed=3)
    xv, yv = _data(120, seed=4)
    _check_evaluate(m, x, y, xv, yv, 50)


def test_evaluate_without_metrics_returns_the_loss(dev):
    from handyrec_b200 import keras_lite as K
    from tests.test_gpu_api import _deepfm_data, _deepfm_model

    m = _deepfm_model()
    m.compile(optimizer=K.Adam(0.01), loss=K.binary_crossentropy)
    x, y = _deepfm_data(500)
    h = m.fit(x, y, batch_size=128, epochs=1, validation_data=(x, y))
    assert list(h.history) == ["loss", "val_loss"]
    assert m.evaluate(x, y, batch_size=128) == h.history["val_loss"][0]
    assert isinstance(m.train_on_batch(_slice(x, 0, 128), y[:128]), float)
    with pytest.raises(NotImplementedError):
        m.evaluate(x, y, sample_weight=np.ones(500))


# ---- 5. sharded engine: the read sums a copy over the ranks ----------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_read_sums_ranks_and_keeps_local_variables(dev, world):
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
    mk = lambda: MetricSet([AUC(num_thresholds=50), BinaryAccuracy()])
    ref = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=b * world, seed=7)
    ref.metrics = mk()
    ref.train_step_on_device(torch.cat(ids).to(dev), torch.cat(dense).to(dev), torch.cat(label).to(dev))
    p_ref = ref.prob[: b * world].cpu().numpy()
    torch.cuda.synchronize()
    shared = H.ThreadComm.Shared(world)
    local, read, probs = [None] * world, [None] * world, [None] * world

    def rank_fn(r):
        sh = [s_.to(dev) for s_ in H.shards_of(tables, r, world)]
        comm = H.ThreadComm(shared, r)
        eng = ShardedDeepFMEngine(sh, vocabs, fields, n_dense, comm, dnn_hidden_units=hidden, dnn_activation="relu", batch_size=b, seed=7)
        eng.metrics = mk()
        eng.train_step_on_device(ids[r].to(dev), dense[r].to(dev), label[r].to(dev))
        probs[r] = eng.prob[:b].cpu().numpy()
        before = eng.metrics.variables.clone()
        read[r] = eng.metrics.read(comm)
        local[r] = eng.metrics.variables.cpu().numpy()
        assert torch.equal(eng.metrics.variables, before)

    _run_threads(world, rank_fn)
    total = np.sum(np.stack(local).astype(np.float64), 0)
    for r in range(world):
        assert np.array_equal(read[r], total.astype(np.float32))
    ms = mk()
    lab = torch.cat(label).numpy()
    assert np.array_equal(total, _increments(ms, np.concatenate(probs), lab))
    # and the single-GPU engine over the concatenated batches, up to predictions that sit on a threshold
    _check_counts(ref.metrics, p_ref, lab)
    thr = ms.thresholds[ms.thr_index]
    near = (np.abs(np.concatenate(probs)[None, :] - thr[:, None]) <= 1e-6).sum(1) + (np.abs(p_ref[None, :] - thr[:, None]) <= 1e-6).sum(1)
    assert np.all(np.abs(total - ref.metrics.variables.cpu().numpy()) <= near)


# ---- 6. nothing changes without metrics; one launch with them -----------------------------------------------------------------
def test_step_launches_unchanged_without_metrics_and_one_more_with(dev):
    from handyrec_b200.engine import DeepFMEngine, launch_count
    from handyrec_b200.metrics import AUC, BinaryAccuracy, MetricSet, Precision

    g = torch.Generator().manual_seed(2)
    vocabs, D, B = [40, 70, 500], 8, 1024
    tables = [((torch.rand(v, D, generator=g) - 0.5) * 0.1).to(dev) for v in vocabs]
    eng = DeepFMEngine(tables, [(0, 1, "none"), (1, 1, "none"), (2, 2, "mean")], 4, (32, 16, 1), "relu", batch_size=B)
    eng.autotune_embedding_bwd = False
    ids = torch.cat([torch.randint(0, v, (B, 1 if i < 2 else 2), generator=g, dtype=torch.int32) for i, v in enumerate(vocabs)], 1).to(dev)
    dense = torch.randn(B, 4, generator=g).to(dev)
    label = (torch.rand(B, generator=g) < 0.3).float().to(dev)

    def step_launches():
        c0 = launch_count()
        eng.train_step_on_device(ids, dense, label)
        torch.cuda.synchronize()
        return launch_count() - c0

    step_launches()
    base = step_launches()
    assert step_launches() == base
    eng.metrics = MetricSet([AUC(), BinaryAccuracy(), Precision(thresholds=[0.2, 0.4])])
    assert step_launches() == base + 1
    eng.metrics = None
    assert step_launches() == base
