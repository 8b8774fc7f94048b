"""The float64 conv reference (fp64_conv_ref.py) against the C oracle, before it is trusted at training sizes.

Fed the same fp32 operands, the two differ only by the oracle's fp32 accumulation, so every element must agree to a
small multiple of 2^-24 relative to `mag` (the same op on |operands|): an indexing, padding, stride, sub-range, frame or
scaleTargets mistake in either is off by a whole term, orders of magnitude more.  Measured worst ratio over these
cases: 5.0e-7 (x86-64 CPU); the bar is 4e-6."""
import numpy as np
import pytest
import torch

import fp64_conv_ref as R
from cases import F, GOLDEN_3D, Z, geo3d, load_golden
from convnet_b200.abi import GetConvDesc, num_modules
from test_gpu_parity import CONV_CASES

TOL = 4e-6
BATCH_CAP = 16                       # the oracle is a plain loop nest: batch cut down, geometry kept


def _case(shape, seed=5):
    N, W, H, Cin, Cout, ky, kx, sy, sx, py, px = shape
    N = min(N, BATCH_CAP)
    modY, modX = num_modules(H, ky, sy, py), num_modules(W, kx, sx, px)
    d = GetConvDesc(Cin, Cout, ky, kx, sy, sx, py, px)
    ish, fsh, tsh = (N, W, H, Cin), (Cout, kx, ky, Cin), (N, modX, modY, Cout)
    r = np.random.RandomState(seed)
    x = F(r.randn(N, W * H * Cin))
    w = F(r.randn(Cout, kx * ky * Cin) / np.sqrt(kx * ky * Cin))
    dy = F(r.randn(N, modX * modY * Cout))
    return d, ish, fsh, tsh, x, w, dy


def _check(ref_mag, oracle_out):
    ref, mag = ref_mag
    q, i = R.ratio(torch.from_numpy(oracle_out.ravel(order="F").copy()), ref, mag)
    assert q < TOL, (q, i)
    return q


def _all_ops(oracle, d, ish, fsh, tsh, x, w, dy, st, r):
    """convUp / convDown / convOutp with scaleTargets = st over a random init, scaleOutput != 1 for wgrad"""
    N = ish[0]
    init = F(r.randn(*dy.shape)); out = init.copy(order="F")
    oracle.convUp(x, w, out, ish, fsh, tsh, d, st)
    _check(R.conv_up(x, w, d, ish, fsh, tsh, st, init=init), out)
    init = F(r.randn(*x.shape)); out = init.copy(order="F")
    oracle.convDown(dy, w, out, tsh, fsh, ish, d, st)
    _check(R.conv_down(dy, w, d, tsh, fsh, ish, st, init=init), out)
    init = F(r.randn(*w.shape)); out = init.copy(order="F")
    oracle.convOutp(x, dy, out, ish, tsh, fsh, d, st, 1.0 / N)
    _check(R.conv_outp(x, dy, d, ish, tsh, fsh, st, 1.0 / N, init=init), out)


@pytest.mark.parametrize("case", sorted(CONV_CASES))
def test_reference_matches_oracle_2d(oracle, case):
    d, ish, fsh, tsh, x, w, dy = _case(CONV_CASES[case])
    _all_ops(oracle, d, ish, fsh, tsh, x, w, dy, 0.0, np.random.RandomState(1))


@pytest.mark.parametrize("st", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("shape", [(8, 9, 8, 12, 20, 3, 2, 2, 1, 1, 0),      # kx != ky, sx != sy, px != py
                                   (4, 10, 10, 4, 8, 2, 2, 3, 3, 0, 0),      # stride > kernel: pixels without taps
                                   (8, 11, 11, 16, 24, 5, 5, 2, 2, 1, 1)])   # conv2-like 4 stride phases
def test_reference_scale_targets(oracle, shape, st):
    d, ish, fsh, tsh, x, w, dy = _case(shape)
    _all_ops(oracle, d, ish, fsh, tsh, x, w, dy, st, np.random.RandomState(2))


@pytest.mark.parametrize("st", [0.0, 0.5, 1.0])
def test_reference_channel_subranges(oracle, st):
    N, W, H, Cin, Cout = 8, 8, 7, 24, 32
    d = GetConvDesc(Cin, Cout, 3, 3, 1, 2, 1, 0, input_channel_begin=8, input_channel_end=24,
                    output_channel_begin=16, output_channel_end=32)
    modX, modY = num_modules(W, 3, 2, 0), num_modules(H, 3, 1, 1)
    ish, fsh, tsh = (N, W, H, Cin), (16, 3, 3, 16), (N, modX, modY, Cout)
    r = np.random.RandomState(3)
    x, w, dy = F(r.randn(N, W * H * Cin)), F(r.randn(16, 9 * 16) / 12), F(r.randn(N, modX * modY * Cout))
    _all_ops(oracle, d, ish, fsh, tsh, x, w, dy, st, r)


@pytest.mark.parametrize("name", GOLDEN_3D)
def test_reference_matches_oracle_3d(oracle, name):
    g = load_golden(name)
    d, pd, ish, fsh, tsh, psh = geo3d(g)
    x, w, dy = g["images"], g["filters"], g["derivs"]
    r = np.random.RandomState(4)
    for st in (0.0, 1.0):
        init = F(r.randn(*dy.shape)); out = init.copy(order="F")
        oracle.convUp3D(x, w, out, ish, fsh, tsh, d, st)
        _check(R.conv_up(x, w, d, ish, fsh, tsh, st, init=init), out)
        init = F(r.randn(*x.shape)); out = init.copy(order="F")
        oracle.convDown3D(dy, w, out, tsh, fsh, ish, d, st)
        _check(R.conv_down(dy, w, d, tsh, fsh, ish, st, init=init), out)
        init = F(r.randn(*w.shape)); out = init.copy(order="F")
        oracle.convOutp3D(x, dy, out, ish, tsh, fsh, d, st, 0.25)
        _check(R.conv_outp(x, dy, d, ish, tsh, fsh, st, 0.25, init=init), out)


def test_ratio_sees_one_missing_term(oracle):
    """the metric itself: one product left out of one element of the oracle's result is caught"""
    d, ish, fsh, tsh, x, w, dy = _case((8, 6, 6, 16, 8, 3, 3, 1, 1, 1, 1))
    out = Z(*dy.shape); oracle.convUp(x, w, out, ish, fsh, tsh, d)
    ref, mag = R.conv_up(x, w, d, ish, fsh, tsh)
    assert R.ratio(torch.from_numpy(out.ravel(order="F").copy()), ref, mag)[0] < TOL
    # element (n = 3, module (2, 2), o = 5) without the product of tap (1, 1), channel 7
    n, mx, my, o, tx, ty, c = 3, 2, 2, 5, 1, 1, 7
    X, Y = mx + tx - 1, my + ty - 1
    out[n, mx + 6 * my + 36 * o] -= x[n, X + 6 * (Y + 6 * c)] * w[o, tx + 3 * (ty + 3 * c)]
    q, i = R.ratio(torch.from_numpy(out.ravel(order="F").copy()), ref, mag)
    assert q > 100 * TOL and i == n + 8 * (mx + 6 * my + 36 * o)


@pytest.mark.parametrize("mode", ["bf16", "tf32_rne", "tf32_trunc"])
def test_operand_emulation(mode):
    x = torch.tensor([1.0, 1 + 2 ** -9, 1 + 3 * 2 ** -9, 1 + 2 ** -11 + 2 ** -20, -(1 + 2 ** -11 + 2 ** -20), 3e-39],
                     dtype=torch.float32)
    got = R.emulate(x, mode)
    if mode == "bf16":        # 8 mantissa bits (7 stored), ties to even
        want = [1.0, 1.0, 1 + 2 ** -7, 1.0, -1.0, float(torch.tensor(3e-39).to(torch.bfloat16))]
    elif mode == "tf32_rne":  # 11 mantissa bits (10 stored)
        want = [1.0, 1 + 2 ** -9, 1 + 3 * 2 ** -9, 1 + 2 ** -10, -(1 + 2 ** -10), None]
    else:
        want = [1.0, 1 + 2 ** -9, 1 + 3 * 2 ** -9, 1.0, -1.0, None]
    for g_, w_ in zip(got.tolist(), want):
        if w_ is not None:
            assert g_ == w_, (got, want)
