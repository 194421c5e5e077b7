"""GPU: Keras callbacks on the fused DeepFM engine, the layer path and the row-sharded engine (2 emulated ranks) -- the hook
sequence and logs, the unchanged training step (launches, weights), learning-rate callbacks without an engine rebuild,
EarlyStopping's restore through set_weights, ModelCheckpoint + load_weights, TerminateOnNaN, and identical decisions on every rank."""
import os

import numpy as np
import pytest
import torch

from tests.test_gpu_api import _deepfm_data
from tests.test_gpu_clip import _model
from tests.test_gpu_parity import close
from tests.test_gpu_schedules import SMALL, _pair, _pin_units, _weights

pytestmark = pytest.mark.gpu

BS = 256


def _C():
    from handyrec_b200 import callbacks

    return callbacks


class _Recorder:
    """Records every hook with its index and log keys; epoch-end logs and weights kept apart."""

    def __new__(cls, batch_hooks=True):
        C = _C()

        class Rec(C.Callback):
            def __init__(self):
                super().__init__()
                self.events, self.batch_losses, self.epoch_logs, self.weights = [], [], [], []

            def _ev(self, name, i=None, logs=None):
                self.events.append((name, i, tuple(sorted(logs)) if logs else ()))

            def on_train_begin(self, logs=None):
                self._ev("train_begin")

            def on_train_end(self, logs=None):
                self._ev("train_end", None, logs)

            def on_epoch_begin(self, epoch, logs=None):
                self._ev("epoch_begin", epoch)

            def on_epoch_end(self, epoch, logs=None):
                self._ev("epoch_end", epoch, logs)
                self.epoch_logs.append(dict(logs))
                self.weights.append(self.model.get_weights())

            def on_test_begin(self, logs=None):
                self._ev("test_begin")

            def on_test_end(self, logs=None):
                self._ev("test_end", None, logs)

        if batch_hooks:

            class RecB(Rec):
                def on_train_batch_begin(self, batch, logs=None):
                    self._ev("batch_begin", batch, logs)

                def on_train_batch_end(self, batch, logs=None):
                    self._ev("batch_end", batch, logs)
                    self.batch_losses.append(logs["loss"])

                def on_test_batch_begin(self, batch, logs=None):
                    self._ev("test_batch_begin", batch, logs)

                def on_test_batch_end(self, batch, logs=None):
                    self._ev("test_batch_end", batch, logs)

            return RecB()
        return Rec()


def _compiled_pair(monkeypatch, opt, metrics=None):
    from handyrec_b200 import keras_lite as KL

    fused, plain = _pair("adam", opt, monkeypatch)
    if metrics:
        for m in (fused, plain):
            m.compile(optimizer=opt(), loss=KL.binary_crossentropy, metrics=metrics)
    return fused, plain


# ---- 1. hook sequence, logs, and the unchanged step ---------------------------------------------------------------------------
def test_hook_sequence_and_logs_match_on_both_paths(dev, monkeypatch):
    from handyrec_b200 import keras_lite as KL

    n = 3 * BS + 100  # a partial last batch
    x, y = _deepfm_data(n)
    xv, yv = _deepfm_data(300, seed=5)
    fused, plain = _compiled_pair(monkeypatch, lambda: KL.Adam(0.01), metrics=["AUC"])
    _pin_units(fused)
    recs = []
    for m in (fused, plain):
        r = _Recorder()
        h = m.fit(x, y, batch_size=BS, epochs=2, validation_data=(xv, yv), callbacks=[r])
        recs.append((r, h))
    (rf, hf), (rp, hp) = recs
    assert rf.events == rp.events
    assert [e[0] for e in rf.events[:3]] == ["train_begin", "epoch_begin", "batch_begin"]
    assert rf.events[-1][0] == "train_end"
    assert ("epoch_end", 0, ("auc", "loss", "val_auc", "val_loss")) in rf.events
    assert ("batch_end", 0, ("auc", "loss")) in rf.events and ("test_batch_end", 1, ("auc", "loss")) in rf.events
    # batch-end losses are the running sample-weighted mean of the step losses; the epoch's last one is the epoch loss
    sizes = [BS, BS, BS, 100]
    steps = fused.last_losses
    run = [np.dot(steps[: i + 1], sizes[: i + 1]) / sum(sizes[: i + 1]) for i in range(4)]
    np.testing.assert_allclose(rf.batch_losses[4:], run, rtol=1e-12)
    assert rf.batch_losses[7] == pytest.approx(hf.history["loss"][1], rel=1e-12)
    np.testing.assert_allclose(rp.batch_losses, rf.batch_losses, rtol=2e-4)
    for k in hf.history:  # val_loss: the layer path averages its validation batches, the fused path its rows (as before)
        if k != "val_loss":
            np.testing.assert_allclose(hp.history[k], hf.history[k], rtol=2e-3)
    assert [dict(d) for d in rf.epoch_logs] == [{k: v[e] for k, v in hf.history.items()} for e in range(2)]
    assert hf.epoch == [0, 1] and hf.params["epochs"] == 2 and hf.model is fused


def test_batch_hooks_leave_the_step_unchanged(dev, monkeypatch):
    """The per-step read-back changes when the host waits, not what the GPU computes: same launches, same bits."""
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.engine import launch_count

    x, y = _deepfm_data(4 * BS)
    runs = []
    for cbs in (None, [_Recorder()], [_C().TerminateOnNaN()]):
        m = _model(0)
        m.dense_table_max_rows = SMALL
        m.compile(optimizer=KL.Adam(0.01), loss=KL.binary_crossentropy)
        _pin_units(m)
        c0 = launch_count()
        h = m.fit(x, y, batch_size=BS, epochs=2, callbacks=cbs)
        torch.cuda.synchronize()
        runs.append((launch_count() - c0, h.history, _weights(m)))
    for launches, hist, w in runs[1:]:
        assert launches == runs[0][0] and hist == runs[0][1]
        for k in w:
            assert torch.equal(w[k], runs[0][2][k]), k


# ---- 2. epoch-level callbacks: same launches, same weights as rates set by hand --------------------------------------------------
def test_epoch_callbacks_keep_launches_and_equal_rates_set_by_hand(dev, monkeypatch, tmp_path):
    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.engine import launch_count

    C = _C()
    x, y = _deepfm_data(4 * BS)
    xv, yv = _deepfm_data(300, seed=5)
    epochs = 3
    m = _model(0)
    m.dense_table_max_rows = SMALL
    m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    eng = _pin_units(m)
    # min_delta 10: no epoch after the first improves, so the rate is cut at the end of epochs 1 and 2
    cbs = [C.EarlyStopping(patience=10), C.ModelCheckpoint(str(tmp_path / "best"), save_best_only=True, save_weights_only=True),
           C.ReduceLROnPlateau(factor=0.5, patience=0, min_delta=10.0), C.CSVLogger(str(tmp_path / "log.csv"))]
    c0 = launch_count()
    h = m.fit(x, y, batch_size=BS, epochs=epochs, validation_data=(xv, yv), callbacks=cbs)
    torch.cuda.synchronize()
    with_cbs = launch_count() - c0
    assert m._fused.engine is eng and m.optimizer.iterations == 4 * epochs and eng.step_count == 4 * epochs
    lr0 = float(np.float32(0.02))
    assert h.history["lr"] == [lr0, lr0, float(np.float32(lr0 * 0.5))]
    assert os.path.exists(tmp_path / "best" / "manifest.json") and len(open(tmp_path / "log.csv").read().splitlines()) == 4

    ref = _model(0)
    ref.dense_table_max_rows = SMALL
    ref.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    reng = _pin_units(ref)
    rates = [0.02, 0.02, float(np.float32(lr0 * 0.5))]
    c0 = launch_count()
    for e in range(epochs):
        if e and rates[e] != rates[e - 1]:  # the callback left epoch 1 at the compiled float 0.02
            ref._set_learning_rate(rates[e])
        ref.fit(x, y, batch_size=BS, validation_data=(xv, yv))
    torch.cuda.synchronize()
    assert launch_count() - c0 == with_cbs
    assert ref._fused.engine is reng
    wa, wb = _weights(m), _weights(ref)
    for k in wa:
        assert torch.equal(wa[k], wb[k]), k


# ---- 3. learning-rate callbacks on the fused path: no rebuild, slots kept --------------------------------------------------------
@pytest.mark.parametrize("kind", ["scheduler", "plateau"])
def test_lr_callbacks_keep_the_engine_and_match_the_layer_path(dev, monkeypatch, kind):
    from handyrec_b200 import keras_lite as KL

    C = _C()
    x, y = _deepfm_data(3 * BS)
    fused, plain = _compiled_pair(monkeypatch, lambda: KL.Adam(0.02))
    eng = _pin_units(fused)
    m_slot = eng.opt_m
    epochs = 3
    hs = []
    for m in (fused, plain):
        cb = (C.LearningRateScheduler(lambda e, lr: lr * 0.5 if e else lr) if kind == "scheduler"
              else C.ReduceLROnPlateau(monitor="loss", factor=0.5, patience=0, min_delta=10.0))
        hs.append(m.fit(x, y, batch_size=BS, epochs=epochs, callbacks=[cb]))
    assert fused._fused.engine is eng and eng.opt_m is m_slot and float(m_slot.abs().max()) > 0
    assert fused.optimizer.iterations == plain.optimizer.iterations == 3 * epochs and eng.step_count == 3 * epochs
    assert hs[0].history["lr"] == hs[1].history["lr"] and len(set(hs[0].history["lr"])) == 3 - (kind == "plateau")
    assert eng.lr == hs[0].history["lr"][-1]  # the rate of the last epoch (ReduceLROnPlateau cuts after it)
    # a reset of Adam's moments at a rate change would move the fused weights far beyond this
    wf, wp = _weights(fused), _weights(plain)
    for k in wf:
        close(wf[k], wp[k], 1e-3)


# ---- 4. EarlyStopping(restore_best_weights=True) ------------------------------------------------------------------------------
@pytest.mark.parametrize("fuse", [True, False])
def test_early_stopping_restores_the_best_epoch(dev, monkeypatch, fuse):
    from handyrec_b200 import keras_lite as KL

    C = _C()
    x, y = _deepfm_data(3 * BS)
    m = _model(0)
    m.fuse = fuse
    m.dense_table_max_rows = SMALL
    m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    if fuse:
        _pin_units(m)
    score = [1.0, 0.5, 0.7, 0.8, 0.9, 0.1]

    def scripted(epoch, logs):
        logs["score"] = score[epoch]

    rec = _Recorder(batch_hooks=False)
    es = C.EarlyStopping(monitor="score", patience=2, restore_best_weights=True)
    h = m.fit(x, y, batch_size=BS, epochs=6, callbacks=[C.LambdaCallback(on_epoch_end=scripted), rec, es])
    assert len(h.history["loss"]) == 4 and es.stopped_epoch == 3 and m.optimizer.iterations == 12
    best = rec.weights[1]
    got = m.get_weights()
    assert len(got) == len(best) and all(np.array_equal(a, b) for a, b in zip(got, best))
    assert not all(np.array_equal(a, b) for a, b in zip(rec.weights[3], best))
    # the restored weights are the ones the model now runs: the same predictions as a layer-path model given them
    p = m.predict(x, batch_size=BS)
    other = _model(1)
    other.fuse = False
    other.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    other.set_weights(best)
    close(p, other.predict(x, batch_size=BS), 1e-5)
    if fuse:  # and the engine trains on from them: a fit continues from the restored weights, slots kept
        eng = m._fused.engine
        w_eng = eng.get_dense_weights(0)[0].numpy()
        dense0 = next(w for w in best if w.shape == tuple(w_eng.shape))
        assert np.array_equal(w_eng, dense0)
        m.fit(x, y, batch_size=BS)
        assert m._fused.engine is eng and m.optimizer.iterations == 15


# ---- 5. ModelCheckpoint + load_weights (the reference's Quickstart flow) ------------------------------------------------------------
def test_model_checkpoint_quickstart_flow(dev, monkeypatch, tmp_path):
    from handyrec_b200 import keras_lite as KL

    C = _C()
    x, y = _deepfm_data(3 * BS)
    xv, yv = _deepfm_data(300, seed=5)
    m = _model(0)
    m.dense_table_max_rows = SMALL
    m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    path = str(tmp_path / "ckpt")
    every = C.ModelCheckpoint(str(tmp_path / "ep{epoch:02d}"), save_weights_only=True)
    m.fit(x, y, batch_size=BS, epochs=2, validation_data=(xv, yv),
          callbacks=[C.ModelCheckpoint(path, save_best_only=True, save_weights_only=True, monitor="val_loss"), every])
    assert os.path.isdir(tmp_path / "ep01") and os.path.isdir(tmp_path / "ep02")
    fresh = _model(7)
    fresh.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    fresh.load_weights(str(tmp_path / "ep02"))
    close(fresh.predict(xv, batch_size=BS), m.predict(xv, batch_size=BS), 1e-5)
    fresh.load_weights(path)  # the best epoch's weights load too
    assert len(fresh.get_weights()) == len(m.get_weights())


def _fit_steps(k, x, y):
    """A fused model from seed 0 after k steps of plain fits over x (4 batches an epoch; a split fit continues the same engine)."""
    from handyrec_b200 import keras_lite as KL

    m = _model(0)
    m.dense_table_max_rows = SMALL
    m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    _pin_units(m)
    epochs, rest = divmod(k, 4)
    if epochs:
        m.fit(x, y, batch_size=BS, epochs=epochs)
    if rest:
        m.fit({n: v[: rest * BS] for n, v in x.items()}, y[: rest * BS], batch_size=BS)
    return m


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(u, v) for u, v in zip(a, b))


def test_model_checkpoint_every_n_batches_on_the_fused_path(dev, tmp_path):
    """ModelCheckpoint(save_freq=2) saves twice an epoch from inside the fused engine's epoch, next to a batch callback that reads
    the weights at every batch: every checkpoint holds the weights of the step it was written after (dense and FM weights
    included), and after the fit the layers hold the final ones."""
    from handyrec_b200 import keras_lite as KL

    C = _C()
    x, y = _deepfm_data(4 * BS)
    ck = tmp_path / "ck"
    ck.mkdir()
    path = str(ck / "e{epoch}_{loss:.12f}")

    class Seen(C.Callback):
        def __init__(self):
            super().__init__()
            self.at, self.epoch = [], 0

        def on_epoch_begin(self, epoch, logs=None):
            self.epoch = epoch

        def on_train_batch_end(self, batch, logs=None):
            self.at.append((path.format(epoch=self.epoch + 1, **logs), self.model.get_weights()))

    m = _model(0)
    m.dense_table_max_rows = SMALL
    m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    _pin_units(m)
    seen = Seen()
    m.fit(x, y, batch_size=BS, epochs=2, callbacks=[C.ModelCheckpoint(path, save_freq=2, save_weights_only=True), seen])
    assert len(seen.at) == 8
    step_of = {p: i + 1 for i, (p, _) in enumerate(seen.at)}
    saved = sorted(os.listdir(ck))
    assert sorted(step_of[str(ck / f)] for f in saved) == [2, 4, 6, 8]
    for f in saved:
        k = step_of[str(ck / f)]
        want = _fit_steps(k, x, y).get_weights()
        fresh = _model(7)
        fresh.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
        fresh.load_weights(str(ck / f))
        assert _same(fresh.get_weights(), want), k
        assert _same(seen.at[k - 1][1], want), k
    final = _fit_steps(8, x, y).get_weights()
    assert _same(m.get_weights(), final)
    eng = m._fused.engine
    for i, d in enumerate(m._fused._dense_layers()):
        w, b = eng.get_dense_weights(i)
        assert torch.equal(w, d.kernel.detach().cpu()) and torch.equal(b, d.bias.detach().cpu())
    m.save_weights(str(tmp_path / "end"))
    fresh = _model(7)
    fresh.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    fresh.load_weights(str(tmp_path / "end"))
    assert _same(fresh.get_weights(), final)


# ---- 6. TerminateOnNaN ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fuse", [True, False])
def test_terminate_on_nan_stops_after_the_first_nan_batch(dev, monkeypatch, fuse):
    from handyrec_b200 import keras_lite as KL

    x, y = _deepfm_data(4 * BS)
    y = y.copy()
    y[BS + 3] = np.nan  # batch 1: a NaN label makes that batch's loss NaN
    m = _model(0)
    m.fuse = fuse
    m.dense_table_max_rows = SMALL
    m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy)
    rec = _Recorder()
    h = m.fit(x, y, batch_size=BS, epochs=3, callbacks=[_C().TerminateOnNaN(), rec])
    assert m.optimizer.iterations == 2 and m.stop_training
    assert len(h.history["loss"]) == 1 and np.isnan(h.history["loss"][0])
    assert [e[1] for e in rec.events if e[0] == "batch_end"] == [0, 1]
    if fuse:
        assert len(m.last_losses) == 2 and m._fused.engine.step_count == 2


# ---- 7. the sharded engine on 2 emulated ranks --------------------------------------------------------------------------------
def test_sharded_ranks_take_identical_decisions(dev, monkeypatch, tmp_path):
    import torch.distributed as dist

    from handyrec_b200 import keras_lite as KL
    from handyrec_b200.sharded import shard_rows
    from tests import shard_helpers as H
    from tests.test_gpu_sharded import _run_threads

    C = _C()
    world = 2

    class Comm(H.ThreadComm):
        group = None

        def alloc_tables(self, vocabs, dim, device, replicate_max_rows=0):
            rows = [v if v <= replicate_max_rows else shard_rows(v, self.rank, self.N) for v in vocabs]
            return [torch.zeros(r, dim, device=device) for r in rows], None

    # every rank builds its model from the same seed, so the weights rank 0 would broadcast are already everywhere
    monkeypatch.setattr(dist, "broadcast", lambda *a, **k: None)
    def make_models():
        shared = Comm.Shared(world)
        out = []
        for r in range(world):
            m = _model(0)
            m.dense_table_max_rows = SMALL  # movie_id (50 rows) is row-sharded, the other tables replicated
            m.compile(optimizer=KL.Adam(0.02), loss=KL.binary_crossentropy, distribute=Comm(shared, r))
            out.append(m)
        return out

    models = make_models()
    sizes = [2 * BS + 40, 2 * BS + 90]  # ranks with different sample counts weight the global means
    data = [_deepfm_data(sizes[r], seed=10 + r) for r in range(world)]
    val = [_deepfm_data(200 + 50 * r, seed=20 + r) for r in range(world)]
    ck = str(tmp_path / "best")
    out = [None] * world

    def rank_fn(r):
        rec = _Recorder(batch_hooks=False)
        es = C.EarlyStopping(patience=1, min_delta=1e-4)
        mc = C.ModelCheckpoint(ck, save_best_only=True, save_weights_only=True)
        h = models[r].fit(*data[r], batch_size=BS, epochs=4, validation_data=val[r], callbacks=[rec, es, mc])
        out[r] = (rec, es, mc, h)

    _run_threads(world, rank_fn)
    (r0, es0, mc0, h0), (r1, es1, mc1, h1) = out
    assert r0.epoch_logs == r1.epoch_logs  # the same global logs on every rank
    assert es0.stopped_epoch == es1.stopped_epoch and es0.best == es1.best and mc0.best == mc1.best
    assert len(h0.history["loss"]) == len(h1.history["loss"]) == len(r0.epoch_logs)
    nv = [len(v[1]) for v in val]
    for e, logs in enumerate(r0.epoch_logs):
        # history keeps each rank's own values; the callbacks saw their sample-count-weighted means
        want = (h0.history["loss"][e] * sizes[0] + h1.history["loss"][e] * sizes[1]) / sum(sizes)
        assert logs["loss"] == pytest.approx(want, rel=1e-12)
        want = (h0.history["val_loss"][e] * nv[0] + h1.history["val_loss"][e] * nv[1]) / sum(nv)
        assert logs["val_loss"] == pytest.approx(want, rel=1e-12)
    assert h0.history["loss"] != h1.history["loss"]
    # and they are the values a fit without callbacks records (same epochs, fresh models from the same seed)
    plain, hist = make_models(), [None] * world

    def plain_fn(r):
        hist[r] = plain[r].fit(*data[r], batch_size=BS, epochs=len(h0.history["loss"]), validation_data=val[r]).history

    _run_threads(world, plain_fn)
    for r, h in enumerate((h0, h1)):
        assert list(hist[r]) == list(h.history)
        for k in h.history:
            np.testing.assert_allclose(h.history[k], hist[r][k], rtol=1e-6)
    # the per-rank checkpoint of the best epoch round-trips: each rank reads back its own rows
    vl = [d["val_loss"] for d in r0.epoch_logs]
    best = int(np.argmin(vl))
    names = sorted(os.listdir(ck))
    assert "manifest.rank0of2.json" in names and "manifest.rank1of2.json" in names
    for r in range(world):
        models[r].load_weights(ck)
        got, want = models[r].get_weights(), out[r][0].weights[best]
        assert all(np.array_equal(a, b) for a, b in zip(got, want))
