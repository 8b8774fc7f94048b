"""Pooling and cross-map response norm at the AlexNet layer sizes (batch 128), every element against float64.

References, in torch float64 on the [N, C, H, W] view of the cudamat layout (image index n + N*(x + W*(y + H*c))):
  AvgPool / AvgPoolUndo   avg_pool2d without the padding in the count (each window divides by its clipped size) and its
                          adjoint (each window spreads g / size over its clipped pixels);
  MaxPoolUndo             every pixel EQUAL to its window's maximum receives that window's gradient (ties duplicate it, as
                          the reference's `==` test does; torch's own max-pool backward picks one), summed over the windows
                          through unfold / fold; quantised inputs make ties common;
  ResponseNormCrossMap    y_j = x_j (1 + a S_j)^-b, S_j = sum of x_i^2 over the window of channel j ([j - k/2, j - k/2 + k),
                          or j's block of k when blocked, clipped to the channels) — the formula of test_gpu_net._torch_net;
  ...Undo                 its exact gradient: dy_j D_j^-b - 2ab x_j sum_{i : j in window(i)} dy_i x_i D_i^(-b-1).
The check is ratio = max |ours - ref| / (mag + tiny), mag = the same expression on absolute values, as in
test_gpu_conv_fp64.py.  Thresholds: fp32 arithmetic of a few terms for pooling; the response norm raises to a power with
__powf, like the reference's GPU build; both are about 10x the worst ratio measured on a B200."""
import numpy as np
import pytest
import torch

import fp64_conv_ref as R
from convnet_b200.abi import GetConvDesc, num_modules

pytestmark = pytest.mark.gpu

ALEX_POOL = {"pool1": (110, 96), "pool2": (27, 256), "pool5": (12, 512)}      # image size, channels; 3x3 stride 2 pad 1
ALEX_RNORM = {"rnorm1": (55, 96, 24), "rnorm2": (14, 256, 64)}                # image size, channels, window
ALPHA, BETA = 5e-4, 0.75
N = 128
TOL_POOL = 2e-6        # measured on a B200: <= 1.8e-7 (avg-pool undo)
TOL_RNORM = 2e-5       # measured on a B200: <= 1.8e-6 (rnorm1 undo)


@pytest.fixture(scope="module")
def env():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from convnet_b200 import conv_gemm as cg
    from convnet_b200 import lib
    from convnet_b200.matrix import CUDAMatrix
    lib.load()

    class E:
        pass
    e = E()
    e.torch, e.cg, e.M = torch, cg, CUDAMatrix

    def nan(rows, cols, sh):
        m = CUDAMatrix(rows, cols, sh)
        m.fill_(float("nan"))
        return m
    e.nan = nan
    yield e
    torch.cuda.empty_cache()


def _nchw(t, W, C):
    return t.double().view(C, W, W, N).permute(3, 0, 1, 2)


def _flat(t):                      # [N, C, H, W] -> cudamat order
    return t.permute(1, 2, 3, 0).reshape(-1)


@pytest.mark.parametrize("layer", list(ALEX_POOL))
def test_pool_layers_vs_float64(env, layer):
    torch, Fn = env.torch, env.torch.nn.functional
    W, C = ALEX_POOL[layer]
    mod = num_modules(W, 3, 2, 1)
    d = GetConvDesc(C, C, 3, 3, 2, 2, 1, 1)
    ish, psh = (N, W, W, C), (N, mod, mod, C)
    g = torch.Generator(device="cuda").manual_seed(31)
    x = env.M(N, W * W * C, ish)
    x.storage.copy_(torch.round(torch.randn(x.storage.numel(), device="cuda", generator=g) * 2) / 2)   # ties
    gr = env.M(N, mod * mod * C, psh); gr.storage.normal_(generator=g)
    xd, gd = _nchw(x.storage, W, C), _nchw(gr.storage, mod, C)
    res = {}
    # AvgPool
    out = env.nan(N, mod * mod * C, psh); env.cg.AvgPool(x, out, d)
    ref = _flat(Fn.avg_pool2d(xd, 3, 2, 1, count_include_pad=False))
    mag = _flat(Fn.avg_pool2d(xd.abs(), 3, 2, 1, count_include_pad=False))
    res["AvgPool"] = R.ratio(out.storage, ref, mag)[0]
    # AvgPoolUndo: the adjoint of the average
    out = env.nan(N, W * W * C, ish); env.cg.AvgPoolUndo(gr, out, d)
    res["AvgPoolUndo"] = []
    for gg in (gd, gd.abs()):
        x0 = torch.zeros_like(xd, requires_grad=True)
        (dx,) = torch.autograd.grad(Fn.avg_pool2d(x0, 3, 2, 1, count_include_pad=False), x0, gg)
        res["AvgPoolUndo"].append(_flat(dx))
    res["AvgPoolUndo"] = R.ratio(out.storage, *res["AvgPoolUndo"])[0]
    # MaxPool (exact) and MaxPoolUndo with every tied maximum receiving the gradient
    mx = env.nan(N, mod * mod * C, psh); env.cg.MaxPool(x, mx, d)
    xp = Fn.pad(xd, (1, 1, 1, 1), value=float("-inf"))
    cols = Fn.unfold(xp.reshape(N * C, 1, W + 2, W + 2), 3, stride=2)           # [N*C, 9, mod*mod]
    top = cols.max(dim=1, keepdim=True).values
    assert torch.equal(_flat(top.view(N, C, mod, mod)), mx.storage.double())
    tie = (cols == top).double()
    gcol = gd.reshape(N * C, 1, mod * mod)
    fold = lambda v: _flat(Fn.fold(v, (W + 2, W + 2), 3, stride=2).view(N, C, W + 2, W + 2)[:, :, 1:-1, 1:-1])
    ref, mag = fold(tie * gcol), fold(tie * gcol.abs())
    assert (tie.sum(dim=1) > 1).any()                                            # the inputs do produce ties
    out = env.nan(N, W * W * C, ish); env.cg.MaxPoolUndo(x, gr, mx, out, d)
    res["MaxPoolUndo"] = R.ratio(out.storage, ref, mag)[0]
    print(layer, res)
    assert all(q < TOL_POOL for q in res.values()), res


def _window_sums(v, k, blocked, adjoint):
    """per channel j (dim 1 of [N, C, ...]): sum of v over window(j), or with adjoint over {i : j in window(i)}"""
    C = v.shape[1]
    j = np.arange(C)
    if blocked:
        lo, hi = (j // k) * k, (j // k) * k + k
    elif adjoint:
        lo, hi = j - k + k // 2 + 1, j + k // 2 + 1
    else:
        lo, hi = j - k // 2, j - k // 2 + k
    lo, hi = np.clip(lo, 0, C), np.clip(hi, 0, C)
    cs = v.new_zeros((v.shape[0], C + 1) + tuple(v.shape[2:]))
    cs[:, 1:] = v.cumsum(dim=1)
    hi_t, lo_t = torch.as_tensor(hi, device=v.device), torch.as_tensor(lo, device=v.device)
    return cs.index_select(1, hi_t) - cs.index_select(1, lo_t)


@pytest.mark.parametrize("blocked", [False, True])
@pytest.mark.parametrize("layer", list(ALEX_RNORM))
def test_rnorm_layers_vs_float64(env, layer, blocked):
    torch = env.torch
    W, C, k = ALEX_RNORM[layer]
    ish = (N, W, W, C)
    g = torch.Generator(device="cuda").manual_seed(37)
    x = env.M(N, W * W * C, ish); x.storage.normal_(generator=g).mul_(4.0)      # a S of order 1: the power matters
    dy = env.M(N, W * W * C, ish); dy.storage.normal_(generator=g)
    xd, dyd = _nchw(x.storage, W, C), _nchw(dy.storage, W, C)
    D = 1 + ALPHA * _window_sums(xd * xd, k, blocked, False)
    res = {}
    out = env.nan(N, W * W * C, ish); env.cg.ResponseNormCrossMap(x, out, k, ALPHA, BETA, blocked)
    y = xd * D ** -BETA
    res["fwd"] = R.ratio(out.storage, _flat(y), _flat(y.abs()))[0]
    out = env.nan(N, W * W * C, ish); env.cg.ResponseNormCrossMapUndo(dy, x, out, k, ALPHA, BETA, blocked)
    t = dyd * xd * D ** (-BETA - 1)
    ref = dyd * D ** -BETA - 2 * ALPHA * BETA * xd * _window_sums(t, k, blocked, True)
    mag = dyd.abs() * D ** -BETA + 2 * ALPHA * BETA * xd.abs() * _window_sums(t.abs(), k, blocked, True)
    res["undo"] = R.ratio(out.storage, _flat(ref), _flat(mag))[0]
    print(layer, blocked, res)
    assert all(q < TOL_RNORM for q in res.values()), res
