"""GPU: the tcgen05 3xTF32 GEMM path against float64 references (fp32-parity tolerances)."""
import numpy as np
import pytest
import torch

import oracle
from tests.test_gpu_parity import close, rnd

pytestmark = pytest.mark.gpu


def K():
    from handyrec_b200 import kernels

    return kernels


@pytest.mark.parametrize("M,Kd,N,act", [(1024, 432, 429, "relu"), (4096, 432, 256, "relu"), (512, 256, 128, None), (2048, 128, 32, "sigmoid"), (1000, 64, 100, "tanh"), (65536, 432, 429, "relu")])
def test_dense_fwd_t(dev, M, Kd, N, act):
    k = K()
    x = rnd(M, Kd, seed=1)
    W = rnd(Kd, N, seed=2) / np.sqrt(Kd)
    b = rnd(N, seed=3, scale=0.1)
    want = oracle.activation(act, x.double() @ W.double() + b.double()).float()
    ld = (N + 3) // 4 * 4
    out = torch.zeros(M, ld, device=dev)
    out_t = torch.zeros(N, M, device=dev)
    wt = W.t().contiguous().to(dev)
    k.dense_fwd_t(x.to(dev), wt, b.to(dev), act, out=out[:, :N], out_t=out_t)
    close(out[:, :N], want, 1e-5)
    close(out_t, want.t(), 1e-5)
    if ld > N:
        assert float(out[:, N:].abs().max()) == 0.0
    # element-wise relative error of the error-compensated product is fp32-like
    err = (out[:, :N].cpu().double() - want.double()).abs().max().item()
    assert err < 2e-6 * float(want.abs().max()) * np.sqrt(Kd)


@pytest.mark.parametrize("M,Kd,N", [(2048, 432, 429), (1024, 256, 128), (4096, 128, 256), (1000, 256, 128), (4100, 64, 20)])
def test_dense_bwd_x_t(dev, M, Kd, N):
    k = K()
    a_prev = torch.relu(rnd(M, Kd, seed=1))
    W = rnd(Kd, N, seed=2) / 20
    dz = rnd(M, N, seed=3)
    want = ((dz.double() @ W.double().T) * (a_prev > 0)).float()
    ldk, ldn = (Kd + 3) // 4 * 4, (N + 3) // 4 * 4
    Wd = torch.zeros(Kd, ldn, device=dev)
    Wd[:, :N] = W.to(dev)
    dzd = torch.zeros(M, ldn, device=dev)
    dzd[:, :N] = dz.to(dev)
    ap = torch.zeros(M, ldk, device=dev)
    ap[:, :Kd] = a_prev.to(dev)
    out = torch.zeros(M, ldk, device=dev)
    out_t = torch.zeros(Kd, M, device=dev)
    k.dense_bwd_x_t(dzd[:, :N], Wd[:, :N], a_prev=ap[:, :Kd], act_prev="relu", out=out[:, :Kd], out_t=out_t)
    close(out[:, :Kd], want, 1e-4)
    close(out_t, want.t(), 1e-4)
    # no activation gradient
    out2 = k.dense_bwd_x_t(dzd[:, :N], Wd[:, :N])
    close(out2, (dz.double() @ W.double().T).float(), 1e-4)


@pytest.mark.parametrize("M,Kd,N", [(65536, 432, 429), (4096, 256, 128), (2048, 128, 32), (1024, 40, 16), (1000, 128, 64), (50000, 64, 128)])
def test_dense_bwd_w_t(dev, M, Kd, N):
    k = K()
    x = rnd(M, Kd, seed=1)
    dz = rnd(M, N, seed=2)
    want_w = (x.double().T @ dz.double()).float()
    want_b = dz.double().sum(0).float()
    xt = k.transpose(x.to(dev))
    dzt = k.transpose(dz.to(dev))
    assert torch.equal(xt.cpu(), x.t().contiguous())
    dw, db = k.dense_bwd_w_t(xt, dzt, dz.to(dev))
    close(dw, want_w, 1e-4)
    close(db, want_b, 1e-4)
    assert torch.equal(dw, k.dense_bwd_w_t(xt, dzt, dz.to(dev))[0])  # deterministic


@pytest.mark.parametrize("M,Kd,N", [(65536, 432, 429), (4096, 256, 128), (2048, 132, 32), (1024, 40, 16), (1000, 64, 128), (50000, 128, 20)])
def test_dense_bwd_w_untransposed_x(dev, M, Kd, N):
    """The weight gradient from x as stored: the kernel transposes the tile on its way into tensor memory."""
    k = K()
    x = rnd(M, Kd, seed=3)
    dz = rnd(M, N, seed=4)
    want_w = (x.double().T @ dz.double()).float()
    want_b = dz.double().sum(0).float()
    dzt = k.transpose(dz.to(dev))
    dw, db = k.dense_bwd_w_xn(x.to(dev), dzt)
    close(dw, want_w, 1e-4)
    close(db, want_b, 1e-4)
    assert torch.equal(dw, k.dense_bwd_w_xn(x.to(dev), dzt)[0])  # deterministic


def test_transpose_odd_shapes(dev):
    k = K()
    for r, c in ((1, 1), (33, 65), (1000, 13), (5, 432)):
        x = rnd(r, c, seed=r)
        assert torch.equal(k.transpose(x.to(dev)).cpu(), x.t().contiguous())


@pytest.mark.parametrize("M,Kd,act", [(65536, 128, "relu"), (1000, 36, "sigmoid"), (33, 8, None), (4096, 132, "relu"), (2050, 256, "relu"), (777, 188, None)])
def test_dense1_logit_layer(dev, M, Kd, act):
    k = K()
    ld = (Kd + 3) // 4 * 4
    xa = oracle.activation(act, rnd(M, Kd, seed=1)).requires_grad_(False)
    xbuf = torch.zeros(M, ld)
    xbuf[:, :Kd] = xa
    w = rnd(Kd, seed=2) / np.sqrt(Kd)
    b = torch.tensor([0.3])
    dy = rnd(M, seed=3)
    xd = xbuf.to(dev)
    wd = torch.zeros(ld, device=dev)
    wd[:Kd] = w.to(dev)
    y = k.dense1_fwd(xd[:, :Kd], wd, b.to(dev))
    close(y[:, 0], (xa.double() @ w.double() + 0.3).float(), 1e-5)
    dz, dzt, dw, db = k.dense1_bwd(xd[:, :Kd], wd, dy.to(dev), act_prev=act, want_t=True)
    if act == "relu":
        g = (xa > 0).double()
    elif act == "sigmoid":
        g = (xa * (1 - xa)).double()
    else:
        g = torch.ones_like(xa).double()
    want = dy.double()[:, None] * w.double()[None, :] * g
    close(dz, want.float(), 1e-4)
    close(dzt, want.float().t(), 1e-4)
    close(dw, (xa.double().T @ dy.double()).float(), 1e-4)
    close(db, dy.double().sum().float().reshape(1), 1e-4)


def test_relu_sign_mask_round_trip(dev):
    """The forward's relu sign bits drive the activation-gradient epilogue exactly like re-reading the activations."""
    k = K()
    M, Kd, N = 2048, 128, 429
    x = rnd(M, Kd, seed=1).to(dev)
    wt = (rnd(N, Kd, seed=2) / 10).to(dev)
    ldn = (N + 3) // 4 * 4
    a = torch.zeros(M, ldn, device=dev)
    mask = torch.zeros(M, (N + 31) // 32, device=dev, dtype=torch.int32)
    k.dense_fwd_t(x, wt, None, "relu", out=a[:, :N], relu_mask=mask)
    bits = (mask.cpu().numpy().astype(np.uint32)[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1
    assert np.array_equal(bits.reshape(M, -1)[:, :N].astype(bool), (a[:, :N] > 0).cpu().numpy())
    # layer above: dz (M, 64) through w (N, 64) back to (M, N), masked by relu'(a)
    dz = rnd(M, 64, seed=3).to(dev)
    w = (rnd(N, 64, seed=4) / 8).to(dev)
    ref = k.dense_bwd_x_t(dz, w, a_prev=a[:, :N], act_prev="relu", out=torch.zeros(M, ldn, device=dev)[:, :N])
    got = k.dense_bwd_x_t(dz, w, act_prev="relu", relu_mask=mask, out=torch.zeros(M, ldn, device=dev)[:, :N])
    assert torch.equal(ref, got)
