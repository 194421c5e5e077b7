"""GPU: the DIN training path against float64 references -- the attention glue kernels, the grouped-bias tcgen05 GEMM of the
local-activation MLP's first layer, LAUFirstLayerFn on its own, and one whole DIN train step at the benchmark's shape.

Copies and single fp32 operations are compared bit for bit; sums against float64 with the project's bar (`close`: 1e-5 for
forward values, 1e-4 for gradients, relative to max |ref|)."""
import math
from collections import OrderedDict

import numpy as np
import pytest
import torch

import oracle
from oracle import layers_ref
from tests.test_gpu_models import _dnn_params
from tests.test_gpu_parity import FWD_TOL, GRAD_TOL, close, rand_ids, rnd

pytestmark = pytest.mark.gpu

SENTINEL = -12345.5  # written into pad columns that a kernel must leave alone


def _abi():
    from handyrec_b200 import _lib
    from handyrec_b200 import kernels as K

    return _lib, K


# ------------------------------------------------------------------------------------------------
# the element-wise glue of the LAU training path (lau.cu), called as autograd_ops.LAUFirstLayerFn calls it
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [4, 32, 128])
@pytest.mark.parametrize("U", [16, 20, 128, 512])
def test_lau_split_weights_and_merge_wgrads(dev, D, U):
    """split: wq = Wa + Wc, wp = [Wb - Wc; Wd], wpt = wp^T; merge: dW = [dwq; dwp_k; dwq - dwp_k; dwp_m].  Single fp32 operations and
    copies: bit-exact.  W and dW are column slices of wider buffers (ldw > U): the split never reads the pad columns (NaN there)
    and the merge never writes them."""
    _lib, K = _abi()
    ldw = U + 12
    Wbuf = torch.full((4 * D, ldw), float("nan"))
    Wbuf[:, :U] = rnd(4 * D, U, seed=D + U)
    W = Wbuf[:, :U]
    # every device input is held by a name until its kernel is queued: a temporary's memory would go to the next allocation
    Wdev = Wbuf.to(dev)
    wq, wp, wpt = torch.empty(D, U, device=dev), torch.empty(2 * D, U, device=dev), torch.empty(U, 2 * D, device=dev)
    _lib.call("hrb_lau_split_weights", K._p(Wdev), ldw, D, U, K._p(wq), K._p(wp), K._p(wpt), K._stream())
    Wa, Wb, Wc, Wd = W.split(D)
    assert torch.equal(wq.cpu(), Wa + Wc)
    assert torch.equal(wp.cpu(), torch.cat([Wb - Wc, Wd]))
    assert torch.equal(wpt.cpu(), torch.cat([Wb - Wc, Wd]).t())
    dwq, dwp = rnd(D, U, seed=1), rnd(2 * D, U, seed=2)
    dwqd, dwpd = dwq.to(dev), dwp.to(dev)
    dW = torch.full((4 * D, ldw), SENTINEL, device=dev)
    _lib.call("hrb_lau_merge_wgrads", K._p(dwqd), K._p(dwpd), D, U, K._p(dW), ldw, K._stream())
    got = dW.cpu()
    assert torch.equal(got[:, :U], torch.cat([dwq, dwp[:D], dwq - dwp[:D], dwp[D:]]))
    assert bool((got[:, U:] == SENTINEL).all())


@pytest.mark.parametrize("B,T,D", [(37, 50, 32), (5, 1, 4), (9, 257, 128), (300, 3, 36)])
def test_lau_pack_fwd_bwd(dev, B, T, D):
    """A'[b*T+t] = [k | q*k] (bit-exact); dk = dA'[:, :D] + dA'[:, D:]*q and dq (+)= sum_t dA'[:, D:]*k against float64, with and
    without accumulation into dq (NaN in dq when not accumulating: it must be overwritten, never read); fixed order: two runs
    give the same bits."""
    _lib, K = _abi()
    q, k = rnd(B, D, seed=1), rnd(B, T, D, seed=2)
    qd, kd = q.to(dev), k.to(dev)
    A = torch.empty(B * T, 2 * D, device=dev)
    _lib.call("hrb_lau_pack_fwd", K._p(qd), K._p(kd), B, T, D, K._p(A), K._stream())
    assert torch.equal(A.cpu(), torch.cat([k, q[:, None] * k], -1).reshape(B * T, 2 * D))
    dA = rnd(B * T, 2 * D, seed=3)
    dAd = dA.to(dev)
    q64, k64, dA64 = q.double(), k.double(), dA.double().reshape(B, T, 2 * D)
    want_dk = dA64[..., :D] + dA64[..., D:] * q64[:, None]
    want_dq = (dA64[..., D:] * k64).sum(1)
    base = rnd(B, D, seed=4)
    for accumulate in (0, 1):
        outs = []
        for _ in range(2):
            dq = base.to(dev) if accumulate else torch.full((B, D), float("nan"), device=dev)  # a fresh buffer each run
            dk = torch.empty(B, T, D, device=dev)
            _lib.call("hrb_lau_pack_bwd", K._p(qd), K._p(kd), K._p(dAd), B, T, D, accumulate, K._p(dq), K._p(dk), K._stream())
            outs.append((dq, dk))
        (dq, dk), (dq2, dk2) = outs
        close(dk, want_dk, GRAD_TOL)
        close(dq, want_dq + (base.double() if accumulate else 0.0), GRAD_TOL)
        assert torch.equal(dq, dq2) and torch.equal(dk, dk2)


@pytest.mark.parametrize("T", [1, 50, 257])
@pytest.mark.parametrize("n,ldx", [(20, 28), (128, 132), (512, 512)])
def test_group_sum(dev, T, n, ldx):
    """out[g] = sum_{t<T} x[g*T+t, :n] from a row pitch ldx >= n (the pad columns hold NaN and must not be read); fixed order."""
    _lib, K = _abi()
    groups = 67
    x = torch.full((groups * T, ldx), float("nan"))
    x[:, :n] = rnd(groups * T, n, seed=T + n)
    xd = x.to(dev)
    outs = []
    for _ in range(2):
        out = torch.empty(groups, n, device=dev)
        _lib.call("hrb_group_sum", K._p(xd), ldx, groups, T, n, K._p(out), K._stream())
        outs.append(out)
    close(outs[0], x[:, :n].double().reshape(groups, T, n).sum(1), GRAD_TOL)
    assert torch.equal(outs[0], outs[1])
    _lib.call("hrb_group_sum", K._p(xd), ldx, 0, T, n, K._p(outs[0]), K._stream())  # no groups: nothing to do


# ------------------------------------------------------------------------------------------------
# the attention glue of the materialised path (layers_misc.cu): [q,k,q-k,q*k], the key mask, the weighted key sum
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 50, 200])
@pytest.mark.parametrize("D", [4, 32, 36, 128])
def test_attention_glue_kernels(dev, T, D):
    from handyrec_b200.autograd_ops import AttInputFn, AttPoolFn, MaskScoresFn

    B = 37
    q, k = rnd(B, D, seed=1), rnd(B, T, D, seed=2)
    ids = rand_ids(B, T, 1000, seed=T + D)
    ids[0] = 0  # an all-padding history
    mask = ids != 0
    # [q, k, q-k, q*k]: copies and one fp32 operation each -> bit-exact; its backward against float64
    qd, kd = q.to(dev).requires_grad_(True), k.to(dev).requires_grad_(True)
    att = AttInputFn.apply(qd, kd)
    qe = q[:, None].expand(B, T, D)
    assert torch.equal(att.detach().cpu(), torch.cat([qe, k, qe - k, qe * k], -1))
    g = rnd(B, T, 4 * D, seed=3)
    att.backward(g.to(dev))
    q64, k64 = q.double().requires_grad_(True), k.double().requires_grad_(True)
    qe64 = q64[:, None].expand(B, T, D)
    (torch.cat([qe64, k64, qe64 - k64, qe64 * k64], -1) * g.double()).sum().backward()
    close(qd.grad, q64.grad, GRAD_TOL)
    close(kd.grad, k64.grad, GRAD_TOL)
    # mask: forward and backward are the same select, exact
    s = rnd(B, T, seed=4).to(dev).requires_grad_(True)
    ms = MaskScoresFn.apply(s, mask.to(dev))
    assert torch.equal(ms.detach().cpu(), torch.where(mask, s.detach().cpu(), torch.zeros(())))
    gs = rnd(B, T, seed=5)
    ms.backward(gs.to(dev))
    assert torch.equal(s.grad.cpu(), torch.where(mask, gs, torch.zeros(())))
    # pooled[b] = sum_t s[b,t] k[b,t]: forward and ds against float64, dk = s*g is one fp32 product -> exact
    sc = ms.detach().reshape(B, 1, T).clone().requires_grad_(True)
    kd2 = k.to(dev).requires_grad_(True)
    pooled = AttPoolFn.apply(sc, kd2)
    s64 = sc.detach().cpu().double().requires_grad_(True)
    k64 = k.double().requires_grad_(True)
    want = oracle.din_attention_pool(s64, k64)
    close(pooled, want, FWD_TOL)
    assert float(pooled[0].abs().max()) == 0.0  # every score of the all-padding row is 0
    gp = rnd(B, 1, D, seed=6)
    pooled.backward(gp.to(dev))
    want.backward(gp.double())
    close(sc.grad, s64.grad, GRAD_TOL)
    assert torch.equal(kd2.grad.cpu(), sc.detach().cpu().reshape(B, T, 1) * gp)


def test_attention_glue_kernels_empty_batch(dev):
    from handyrec_b200.autograd_ops import AttInputFn, AttPoolFn, MaskScoresFn

    T, D = 50, 32
    q = torch.zeros(0, D, device=dev, requires_grad=True)
    k = torch.zeros(0, T, D, device=dev, requires_grad=True)
    att = AttInputFn.apply(q, k)
    assert att.shape == (0, T, 4 * D)
    att.sum().backward()
    s = torch.zeros(0, T, device=dev, requires_grad=True)
    ms = MaskScoresFn.apply(s, torch.zeros(0, T, dtype=torch.bool, device=dev))
    pooled = AttPoolFn.apply(ms.reshape(0, 1, T), k)
    assert ms.shape == (0, T) and pooled.shape == (0, 1, D)
    pooled.sum().backward()
    assert s.grad.shape == (0, T) and k.grad.shape == (0, T, D)


# ------------------------------------------------------------------------------------------------
# hrb_dense_fwd_t_grouped: y = act(x . wt^T + group_bias[m / group_rows])
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,Kd,N,T,act", [
    (512, 16, 16, 1, "relu"), (512, 64, 20, 3, "sigmoid"), (512, 256, 128, 128, "tanh"),
    (4100, 256, 512, 129, "tanh"), (4100, 64, 128, 50, None), (4100, 16, 512, 256, "linear"),
    (50000, 16, 20, 257, "relu"), (50000, 64, 128, 50, "sigmoid"), (50000, 256, 16, 256, "tanh"),
    (204800, 64, 128, 50, "relu"), (204800, 256, 20, 257, "sigmoid"),
])
def test_dense_fwd_t_grouped(dev, M, Kd, N, T, act):
    """Group sizes that straddle the 128- and 256-row tiles (129, 257, a last group cut short by M), reductions shorter than one
    32-wide k-block (16), N not a multiple of the 32-column epilogue sub-tile (20), strided group biases and outputs (the output's
    pad columns are left alone)."""
    _lib, K = _abi()
    G = (M + T - 1) // T
    x = rnd(M, Kd, seed=1)
    wt = rnd(N, Kd, seed=2) / math.sqrt(Kd)
    ldgb, ldy = N + 4, (N + 3) // 4 * 4 + 8
    gb = torch.full((G, ldgb), float("nan"))
    gb[:, :N] = rnd(G, N, seed=3, scale=0.5)
    xd, wtd, gbd = x.to(dev), wt.to(dev), gb.to(dev)
    y = torch.full((M, ldy), SENTINEL, device=dev)
    _lib.call("hrb_dense_fwd_t_grouped", K._p(xd), Kd, K._p(wtd), Kd, K._p(gbd), ldgb, T, M, Kd, N, _lib.ACT[act], K._p(y), ldy, K._stream())
    want = oracle.activation(act, x.double() @ wt.double().t() + gb[:, :N].double().repeat_interleave(T, 0)[:M])
    got = y.cpu()
    close(got[:, :N], want, FWD_TOL)
    assert bool((got[:, N:] == SENTINEL).all())


def test_dense_fwd_t_grouped_rejects_short_inputs(dev):
    """Fewer than 512 rows are not a tensor-core shape: the call is refused (no silent fall-back)."""
    _lib, K = _abi()
    M, Kd, N = 511, 64, 32
    x, wt, gb, y = (torch.zeros(r, c, device=dev) for r, c in ((M, Kd), (N, Kd), (M, N), (M, N)))
    with pytest.raises(_lib.HrbError) as e:
        _lib.call("hrb_dense_fwd_t_grouped", K._p(x), Kd, K._p(wt), Kd, K._p(gb), N, 1, M, Kd, N, 0, K._p(y), N, K._stream())
    assert e.value.status == _lib.HRB_UNSUPPORTED


# ------------------------------------------------------------------------------------------------
# LAUFirstLayerFn on its own: widths and a missing bias that the LocalActivationUnit layer never passes it
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,U,act,bias", [(32, 16, "relu", False), (8, 20, "sigmoid", True), (32, 256, None, False), (16, 20, "tanh", False)])
def test_lau_first_layer_fn(dev, D, U, act, bias):
    """act([q, k, q-k, q*k] . W + b) without the (B,T,4D) tensor == the materialised input through a float64 Dense; every
    gradient against float64 autograd; forward and backward twice give the same bits."""
    from handyrec_b200.autograd_ops import LAUFirstLayerFn

    B, T = 100, 50
    q, k = rnd(B, D, seed=1, scale=0.5), rnd(B, T, D, seed=2, scale=0.5)
    W = rnd(4 * D, U, seed=3) / math.sqrt(4 * D)
    b = rnd(U, seed=4, scale=0.1) if bias else None
    g = rnd(B, T, U, seed=5)
    q64, k64, W64 = q.double().requires_grad_(True), k.double().requires_grad_(True), W.double().requires_grad_(True)
    b64 = b.double().requires_grad_(True) if bias else None
    qe = q64[:, None].expand(B, T, D)
    want = oracle.activation(act, oracle.dense(torch.cat([qe, k64, qe - k64, qe * k64], -1), W64, b64))
    (want * g.double()).sum().backward()

    def run():
        leaves = [t.to(dev).requires_grad_(True) for t in (q, k, W)] + ([b.to(dev).requires_grad_(True)] if bias else [])
        y = LAUFirstLayerFn.apply(*leaves[:3], leaves[3] if bias else None, act)
        (y * g.to(dev)).sum().backward()
        return y.detach(), [t.grad for t in leaves]

    y, grads = run()
    close(y, want, FWD_TOL)
    for got, ref in zip(grads, [q64, k64, W64] + ([b64] if bias else [])):
        close(got, ref.grad, GRAD_TOL)
    y2, grads2 = run()
    assert torch.equal(y, y2) and all(torch.equal(a, c) for a, c in zip(grads, grads2))


# ------------------------------------------------------------------------------------------------
# one DIN train step at the benchmark's shape (bench_models.build_din / din_data): B = 4096, T = 50, D = 32
# ------------------------------------------------------------------------------------------------
SPARSE = ["user_id", "gender", "occupation", "zip", "age", "movie_id", "year"]


def _float64(p):
    """A DNNParams of float32 leaves as float64 leaves (same values)."""
    p.W = [w.detach().double().requires_grad_(True) for w in p.W]
    p.b = [b.detach().double().requires_grad_(True) for b in p.b]
    p.dice_alpha = [a.detach().double().requires_grad_(True) if a is not None else None for a in p.dice_alpha]
    p.dice_mean = [m.double() if m is not None else None for m in p.dice_mean]
    p.dice_var = [v.double() if v is not None else None for v in p.dice_var]
    return p


def din_oracle_step(x, y, tables, p_lau, p_dnn):
    """bench_models.build_din restated on the oracle (float64 leaves in `tables` / the DNNParams): the loss after backward, and
    the Dice batch statistics (mean, biased variance) in call order -- the LAU's Dice layers, then the tower's."""
    stats = []

    def dice(v, alpha, mm, mv, training=False, eps=1e-9):
        red = tuple(range(v.dim() - 1))
        stats.append((v.detach().mean(red), v.detach().var(red, unbiased=False)))
        return orig(v, alpha, mm, mv, training, eps)

    orig, layers_ref.dice = layers_ref.dice, dice
    try:
        sparse = OrderedDict((n, (tables[n], torch.from_numpy(x[n]), n == "movie_id")) for n in SPARSE)
        seqs = OrderedDict((("genres", (tables["genre_id"], torch.from_numpy(x["genres"]))),))
        other = oracle.group_embedding_lookup(sparse, seqs, "mean")
        keys, kmask = oracle.squeeze_mask(*oracle.custom_embedding(tables["movie_id"], torch.from_numpy(x["hist_movie"]), True))
        q, _ = oracle.custom_embedding(tables["movie_id"], torch.from_numpy(x["movie_id"]), True)
        att = oracle.local_activation_unit(q, keys, kmask, p_lau, act="dice", training=True)
        logit = oracle.dnn(oracle.concat([], other + [oracle.din_attention_pool(att, keys)]), p_dnn, act="dice", output_activation=None,
                           training=True)
    finally:
        layers_ref.dice = orig
    loss = oracle.bce_from_logits(logit[:, 0], torch.from_numpy(y).double())
    loss.backward()
    return float(loss.detach()), stats


def _din_parts(m):
    from handyrec_b200.layers import LocalActivationUnit
    from handyrec_b200.layers.activation import Dice
    from handyrec_b200.layers.core import Dense
    from handyrec_b200.layers.tools import CustomEmbedding

    lau = [l for l in m._all_layers() if isinstance(l, LocalActivationUnit)][0].dnn
    tower = [l for l in m.layers if type(l).__name__ == "DNN"][0]
    tables = {l.name[len("embd_"):]: l for l in m._all_layers() if isinstance(l, CustomEmbedding)}
    denses = [l for d in (lau, tower) for l in d.layers if isinstance(l, Dense)]
    dices = [l for d in (lau, tower) for l in d.layers if isinstance(l, Dice)]
    return lau, tower, tables, denses, dices


@pytest.mark.parametrize("opt", ["sgd", "adam"])
@pytest.mark.parametrize("B,item_vocab", [(4096, None), (1000, None), (4096, 200_000)])
def test_din_train_step_at_bench_shape(dev, opt, B, item_vocab):
    """bench.py --workload din, one step on the layer face (LAUFirstLayerFn over B*T rows, the tensor-core Dense tower, Dice over
    204 800 rows, the attention glue) against float64 autograd of the oracle: the loss, every table, Dense kernel and bias, every
    Dice alpha, and Dice's batch and moving statistics.  B = 1000 is the last partial batch of a DIN fit (50 000 LAU rows, a
    partial k-block in every weight gradient); item_vocab = 200 000 puts the movie table on the touched-rows update path with
    Zipf-distributed histories.  SGD uses a large lr so that (old - new) / lr is the gradient itself; Adam (the benchmark's
    optimiser) is compared with Keras' formula."""
    import bench_models
    from handyrec_b200 import keras_lite as KL

    torch.manual_seed(0)
    vocab = {} if item_vocab is None else {"item_vocab": item_vocab}
    m = bench_models.build_din(**vocab)
    x, y = bench_models.din_data(B, **vocab)
    lau, tower, tables, denses, dices = _din_parts(m)
    assert len(dices) == 5 and tables["movie_id"].embeddings.shape[0] == (item_vocab or bench_models.ML["movie_id"][0])
    for d in denses:
        d.bias.data.normal_(0, 0.1)
    for d in dices:
        d.alphas.data.uniform_(-0.3, 0.3)
        d.moving_mean.data.uniform_(-0.2, 0.2)
        d.moving_variance.data.uniform_(0.5, 1.5)
    lr = 1000.0 if opt == "sgd" else 1e-3
    m.compile(optimizer=KL.SGD(lr=lr) if opt == "sgd" else KL.Adam(learning_rate=lr), loss=KL.binary_crossentropy)

    leaf = {n: l.embeddings.detach().cpu().double().requires_grad_(True) for n, l in tables.items()}
    p_lau = _float64(_dnn_params(lau, 4 * 32, (32, 1)))
    p_dnn = _float64(_dnn_params(tower, 188, (64, 32, 1)))
    old = {"t_" + n: l.embeddings.detach().cpu().clone() for n, l in tables.items()}
    old.update({f"W{i}": d.kernel.detach().cpu().clone() for i, d in enumerate(denses)})
    old.update({f"b{i}": d.bias.detach().cpu().clone() for i, d in enumerate(denses)})
    old.update({f"a{i}": d.alphas.detach().cpu().clone() for i, d in enumerate(dices)})
    moving = [(d.moving_mean.detach().cpu().double(), d.moving_variance.detach().cpu().double()) for d in dices]

    torch.set_num_threads(max(1, torch.get_num_threads()))
    loss, want_stats = din_oracle_step(x, y, leaf, p_lau, p_dnn)
    ref = {"t_" + n: t.grad for n, t in leaf.items()}
    ref.update({f"W{i}": w.grad for i, w in enumerate(p_lau.W + p_dnn.W)})
    ref.update({f"b{i}": b.grad for i, b in enumerate(p_lau.b + p_dnn.b)})
    ref.update({f"a{i}": a.grad for i, a in enumerate([a for a in p_lau.dice_alpha + p_dnn.dice_alpha if a is not None])})

    batch_stats = []  # the Dice layers' batch statistics, read as the step commits them to the moving averages
    for d in dices:
        commit = d._commit_moving_stats
        d._commit_moving_stats = lambda d=d, commit=commit: (batch_stats.append(tuple(t.cpu() for t in d._pending)), commit())
    got_loss = m.train_on_batch(x, y)
    assert abs(got_loss - loss) < 1e-5 * max(1.0, abs(loss))

    new = {"t_" + n: l.embeddings.detach().cpu() for n, l in tables.items()}
    new.update({f"W{i}": d.kernel.detach().cpu() for i, d in enumerate(denses)})
    new.update({f"b{i}": d.bias.detach().cpu() for i, d in enumerate(denses)})
    new.update({f"a{i}": d.alphas.detach().cpu() for i, d in enumerate(dices)})
    assert set(new) == set(ref)
    lr_t = lr * np.sqrt(1 - 0.999) / (1 - 0.9)
    for name in sorted(ref):
        g = ref[name]
        if opt == "sgd":
            close((old[name].double() - new[name].double()) / lr, g, GRAD_TOL)
        else:
            # where |g| is within float32 rounding of 0 its sign, and so the direction of Adam's step, is not determined: left out
            amb = (g.abs() < 1e-6 * float(g.abs().max())) & (g != 0)
            assert int(amb.sum()) <= max(2, g.numel() // 100), (name, int(amb.sum()), g.numel())
            want = old[name].double() - lr_t * (0.1 * g) / ((0.001 * g * g).sqrt() + 1e-7)
            close(new[name][~amb], want[~amb], 2e-4)
    if item_vocab is not None:  # the touched-rows update leaves every row no position gathered exactly as it was
        t = "t_movie_id"
        assert torch.equal(new[t][ref[t].abs().sum(1) == 0], old[t][ref[t].abs().sum(1) == 0])

    assert len(batch_stats) == len(want_stats) == 5
    for d, (bm, bv), (wm, wv), (mm, mv) in zip(dices, batch_stats, want_stats, moving):
        close(bm, wm, GRAD_TOL)
        close(bv, wv, GRAD_TOL)
        close(d.moving_mean, 0.99 * mm + 0.01 * wm, FWD_TOL)
        close(d.moving_variance, 0.99 * mv + 0.01 * wv, FWD_TOL)
