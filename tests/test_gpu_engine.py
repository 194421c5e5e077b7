"""GPU: one fused DeepFM train step (engine) == oracle forward + autograd + the same optimiser rule."""
from collections import OrderedDict

import numpy as np
import pytest
import torch

import oracle
from tests.test_gpu_parity import close, rand_ids, rnd

pytestmark = pytest.mark.gpu


def _setup(dev, B, D, n_dense, hidden, optimizer, seq=True, dense_int=False):
    from handyrec_b200.engine import DeepFMEngine

    vocabs = [7, 50, 1000] + ([23] if seq else [])
    tables = [rnd(v, D, seed=10 + i, scale=0.05) for i, v in enumerate(vocabs)]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 1, "none")] + ([(3, 5, "mean"), (1, 3, "mean")] if seq else [])
    g = torch.Generator().manual_seed(B)
    cols = [torch.randint(0, vocabs[t], (B, 1), generator=g, dtype=torch.int32) for t in (0, 1, 2)]
    if seq:
        cols += [rand_ids(B, 5, vocabs[3], seed=1), rand_ids(B, 3, vocabs[1], seed=2)]
    ids = torch.cat(cols, 1)
    dense = torch.randint(0, 5, (B, n_dense), generator=g, dtype=torch.int32) if dense_int else rnd(B, n_dense, seed=3)
    label = (torch.rand(B, generator=g) < 0.3).float()
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer=optimizer, lr=0.05)
    return eng, tables, fields, ids, dense, label


def _oracle_step(eng, tables, fields, ids, dense, label, B, hidden):
    leaf = [t.clone().requires_grad_(True) for t in tables]
    p = oracle.DNNParams(eng.K0, hidden)
    for i in range(len(eng.units)):
        w, b = eng.get_dense_weights(i)
        p.W.append(w.requires_grad_(True))
        p.b.append(b.requires_grad_(True))
    fm_w = eng.fm_w.cpu().reshape(-1, 1).clone().requires_grad_(True)
    fm_w0 = eng.fm_w0.cpu().clone().requires_grad_(True)
    sparse, seqs, col = OrderedDict(), OrderedDict(), 0
    for f, (ti, L, pool) in enumerate(fields):
        if L == 1 and pool == "none":
            sparse[f"f{f}"] = (leaf[ti], ids[:, col : col + 1], False)
        else:
            seqs[f"f{f}"] = (leaf[ti], ids[:, col : col + L])
        col += L
    embds = oracle.group_embedding_lookup(sparse, seqs, "mean")  # looked up twice in the reference: same values
    logit = oracle.deepfm_forward([dense], embds, embds, p, fm_w, fm_w0, return_logit=True)
    loss = oracle.bce_from_logits(logit[:, 0], label)
    loss.backward()
    return leaf, p, fm_w, fm_w0, logit, loss


@pytest.mark.parametrize("B,D,n_dense,hidden,seq,dense_int", [(1024, 8, 3, (32, 16, 1), True, False), (2048, 16, 13, (64, 8, 1), False, False), (33, 8, 3, (8, 1), True, False), (257, 16, 13, (32, 16, 1), False, False), (64, 8, 1, (4, 1), True, True),
                                                              (1000, 16, 13, (64, 8, 1), False, False), (4100, 8, 3, (32, 16, 1), True, False)])
def test_engine_sgd_step_matches_oracle(dev, B, D, n_dense, hidden, seq, dense_int):
    eng, tables, fields, ids, dense, label = _setup(dev, B, D, n_dense, hidden, "sgd", seq, dense_int)
    assert eng.use_tc == (B >= 512 and B % 4 == 0)  # B = 1000, 4100: the batch is the weight gradients' reduction, a partial k-block
    leaf, p, fm_w, fm_w0, logit, loss = _oracle_step(eng, tables, fields, ids, dense, label, B, hidden)
    prob = eng.predict_on_device(ids.to(dev), dense.to(dev))
    close(prob, torch.sigmoid(logit[:, 0]), 1e-5)
    eng.train_step_on_device(ids.to(dev), dense.to(dev), label.to(dev))
    close(eng.loss_sum / B, loss.detach().reshape(1), 1e-5)
    for i in range(len(eng.units)):
        dw, db = eng.get_dense_grads(i)
        close(dw, p.W[i].grad, 1e-4)
        close(db, p.b[i].grad, 1e-4)
        w, b = eng.get_dense_weights(i)
        close(w, p.W[i].detach() - 0.05 * p.W[i].grad, 1e-4)
    close(eng.d_fm[: eng.D], fm_w.grad[:, 0], 1e-4)
    close(eng.d_fm[eng.D :], fm_w0.grad, 1e-4)
    for t, (dt, lf) in enumerate(zip(eng.tables, leaf)):
        close(dt, tables[t] - 0.05 * lf.grad, 1e-4)


def test_engine_adam_and_host_api(dev):
    B, D, n_dense, hidden = 128, 8, 2, (8, 1)
    eng, tables, fields, ids, dense, label = _setup(dev, B, D, n_dense, hidden, "adam")
    leaf, p, fm_w, fm_w0, logit, loss = _oracle_step(eng, tables, fields, ids, dense, label, B, hidden)
    got = eng.train_on_batch(ids.pin_memory(), dense.pin_memory(), label.pin_memory())
    assert abs(got - float(loss.detach())) <= 1e-5 * max(1.0, abs(float(loss.detach())))
    lr_t = 0.05 * np.sqrt(1 - 0.999) / (1 - 0.9)
    for i in range(len(eng.units)):
        g = p.W[i].grad
        want = p.W[i].detach() - lr_t * (0.1 * g) / ((0.001 * g * g).sqrt() + 1e-7)
        close(eng.get_dense_weights(i)[0], want, 2e-4)
    for t, lf in enumerate(leaf):
        g = lf.grad
        want = tables[t] - lr_t * (0.1 * g) / ((0.001 * g * g).sqrt() + 1e-7)
        close(eng.tables[t], want, 2e-4)
    # a second step runs and the loss goes down on the same batch
    l2 = eng.train_on_batch(ids.pin_memory(), dense.pin_memory(), label.pin_memory())
    assert l2 < got
    pr = eng.predict(ids.pin_memory(), dense.pin_memory())
    assert pr.shape == (B, 1) and float(pr.min()) > 0 and float(pr.max()) < 1


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
def test_engine_dense_updated_tables(dev, optimizer):
    """Tables <= dense_table_max_rows take the dense (Keras) optimiser step -- moment decay and l2_embd on EVERY row --
    while larger tables keep the touched-rows-only update.  Two steps on different batches tell the two apart."""
    from handyrec_b200.engine import DeepFMEngine

    B, D, n_dense, hidden, lr, l2 = 64, 8, 2, (8, 1), 0.05, 0.01
    vocabs = [7, 50, 1000]
    tables = [rnd(v, D, seed=20 + i, scale=0.05) for i, v in enumerate(vocabs)]
    fields = [(0, 1, "none"), (1, 1, "none"), (2, 1, "none")]
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer=optimizer, lr=lr, l2_embd=l2,
                       dense_table_max_rows=50)
    assert eng.dense_tables == [0, 1]
    m = [torch.zeros_like(t) for t in tables]
    v = [torch.zeros_like(t) for t in tables]
    cur = [t.clone() for t in tables]
    for step in (1, 2):
        g = torch.Generator().manual_seed(100 + step)
        ids = torch.cat([torch.randint(0, vv, (B, 1), generator=g, dtype=torch.int32) for vv in vocabs], 1)
        dense, label = rnd(B, n_dense, seed=step), (torch.rand(B, generator=g) < 0.3).float()
        leaf, *_ = _oracle_step(eng, cur, fields, ids, dense, label, B, hidden)
        eng.train_step_on_device(ids.to(dev), dense.to(dev), label.to(dev))
        lr_t = lr * np.sqrt(1 - 0.999 ** step) / (1 - 0.9 ** step)
        for t in range(3):
            touched = torch.zeros(vocabs[t], dtype=torch.bool)
            touched[ids[:, t].long()] = True
            rows = torch.ones_like(touched) if t in eng.dense_tables else touched
            gt = (leaf[t].grad + 2 * l2 * cur[t]) * rows[:, None]
            if optimizer == "sgd":
                cur[t] = cur[t] - lr * gt
            else:
                m_new, v_new = 0.9 * m[t] + 0.1 * gt, 0.999 * v[t] + 0.001 * gt * gt
                m[t] = torch.where(rows[:, None], m_new, m[t])
                v[t] = torch.where(rows[:, None], v_new, v[t])
                cur[t] = torch.where(rows[:, None], cur[t] - lr_t * m[t] / (v[t].sqrt() + 1e-7), cur[t])
            close(eng.tables[t], cur[t], 2e-4)
        cur = [t_.cpu().clone() for t_ in eng.tables]  # the next oracle step starts from the engine's state


def test_engine_rejects_bad_configs(dev):
    from handyrec_b200.engine import DeepFMEngine

    t = [torch.zeros(10, 8, device=dev)]
    with pytest.raises(ValueError):  # models/ranking/context_aware/DeepFM.py:59-60
        DeepFMEngine(t, [(0, 1, "none")], 0, (8, 4))
    with pytest.raises(ValueError):
        DeepFMEngine([torch.zeros(10, 8, device=dev), torch.zeros(10, 16, device=dev)], [(0, 1, "none"), (1, 1, "none")], 0, (8, 1))


def test_fit_batches_equals_blocking_calls(dev):
    B, D, n_dense, hidden = 96, 8, 2, (8, 1)
    eng_a, tables, fields, ids, dense, label = _setup(dev, B, D, n_dense, hidden, "sgd")
    eng_b, *_ = _setup(dev, B, D, n_dense, hidden, "sgd")
    g = torch.Generator().manual_seed(9)
    batches = []
    for t in range(5):
        perm = torch.randperm(B, generator=g)
        batches.append((ids[perm].contiguous().pin_memory(), dense[perm].contiguous().pin_memory(), label[perm].contiguous().pin_memory()))
    want = [eng_a.train_on_batch(*b) for b in batches]
    got = eng_b.fit_batches(batches)
    assert len(got) == 5 and all(abs(a - b) <= 1e-6 * max(1.0, abs(a)) for a, b in zip(want, got))
    for ta, tb in zip(eng_a.tables, eng_b.tables):
        assert torch.equal(ta, tb)
    assert torch.equal(eng_a.params, eng_b.params)


@pytest.mark.parametrize("optimizer", ["sgd", "adam"])
def test_engine_step_at_bench_configuration(dev, optimizer):
    """ONE step of the exact bench.py configuration -- B = 65536, 26 plain fields, D = 16, 13 dense features, DNN 429-256-128-1
    (K0 = 429 -> the CTA-pair tcgen05 GEMMs, the fused logit layer, the sort-free embedding backward with dense-updated small
    tables next to in-place large ones) -- against the oracle end to end: probabilities, loss, every dense gradient, the FM
    gradient and every table.  Vocabularies are capped at 200 000 rows so that the CPU oracle's dense autograd fits."""
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
    lr = 1000.0 if optimizer == "sgd" else 1e-3  # SGD: a large step makes the tiny (1/B-scaled) row gradients visible in fp32
    eng = DeepFMEngine([t.clone().to(dev) for t in tables], fields, n_dense, hidden, "relu", batch_size=B, optimizer=optimizer, lr=lr,
                       dense_table_max_rows=131072)
    assert eng.use_tc and len(eng.dense_tables) == 17
    torch.set_num_threads(max(1, torch.get_num_threads()))
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
    close(eng.d_fm[eng.D :], fm_w0.grad, 1e-4)
    # relu'(z) is discontinuous at z = 0: among the 53 M hidden pre-activations of this batch a handful lie within rounding distance
    # of 0, where the CPU and the GPU legitimately disagree on the sign and that sample's gradient differs by one hidden unit's
    # share (~1 %).  Those samples are found in the oracle's forward and their rows are left out of the row-wise comparison.
    with torch.no_grad():
        embds = [tables[t][ids[:, t].long()] for t in range(len(vocabs))]
        x = torch.cat([dense] + embds, 1)
        amb = torch.zeros(B, dtype=torch.bool)
        for i in range(len(eng.units) - 1):
            z = x @ p.W[i].detach() + p.b[i].detach()
            amb |= (z.abs() < 2e-6 * z.abs().max()).any(1)
            x = torch.relu(z)
    assert int(amb.sum()) < B // 20
    lr_t = lr * np.sqrt(1 - 0.999) / (1 - 0.9)
    for t, lf in enumerate(leaf):
        gr = lf.grad
        got = eng.tables[t].cpu()
        touched = torch.zeros(vocabs[t], dtype=torch.bool)
        touched[ids[:, t].long()] = True
        clean = torch.ones(vocabs[t], dtype=torch.bool)
        clean[ids[amb, t].long()] = False
        if optimizer == "sgd":
            close(((tables[t] - got) / lr)[clean], gr[clean], 1e-4)  # the row gradients themselves (dense-updated and in-place tables alike)
        else:
            # |g| ~ 1e-7 here (1/B-scaled), i.e. next to eps = 1e-7: the step is ~linear in g and well conditioned
            want = tables[t] - lr_t * (0.1 * gr) / ((0.001 * gr * gr).sqrt() + 1e-7)
            close(got[clean], want[clean], 2e-4)
        assert torch.equal(got[~touched], tables[t][~touched])
