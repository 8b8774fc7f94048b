"""BASELINE-size parity on the GPU against the REFERENCE'S OWN CUDA KERNELS.

The reference side is cudamat/cudamat_conv_gemm.cu + cudamat_conv3d_gemm.cu compiled unmodified for sm_100
(oracle/Makefile -> oracle/_ref/libcudamat_conv_gemm_ref.so); what it computed is stored in tests/golden/ref_cuda.npz
(tests/golden_ref.py: seeded samples, and a digest of every output that must match bit for bit), recorded on a B200 with
CONVNET_B200_RECORD_GOLDEN=1, which runs the reference live.  Every layer of net A
(examples/imagenet/CLS_net_20140801232522.pbtxt, SURVEY.md Appendix B) at batch 128 (BASELINE config 2) and 256
(config 3), and the cfg4 C3D conv1a / conv2a shapes at batch 32, runs on identical seeded inputs (the CUDA generator):
fprop / dgrad / wgrad, pool1/2/5 (+undo), rnorm1/2 (+undo).

Metric and tolerances are the ones of tests/test_gpu_parity.py: Diff = max|a-b| / mean|a+b| (py/test_conv.py:382-385);
fp32 mode 1e-4 (the reference's own bar), tf32 5e-3, bf16 2.5e-2; max-pool values bit-exact; pool-undo / rnorm 1e-4, rnorm
undo 2e-4.  The measured numbers are written to gpurun_out/ref_cuda_parity.json (copied to profiles/ by hand).
"""
import json
import os
import zlib

import numpy as np
import pytest

import golden_ref
import ref_cuda_lib
from convnet_b200.abi import GetConvDesc, num_modules

pytestmark = pytest.mark.gpu

TOL = {"fp32": 1e-4, "tf32": 5e-3, "bf16": 2.5e-2}
TOL_MEM = 1e-4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_RESULTS = {}


@pytest.fixture(scope="module")
def env():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    if golden_ref.RECORD and not ref_cuda_lib.available():
        pytest.fail("recording needs oracle/_ref/libcudamat_conv_gemm_ref.so: run `make -C oracle` where the reference exists")
    from convnet_b200 import conv_gemm as cg
    from convnet_b200 import lib
    from convnet_b200.matrix import CUDAMatrix
    lib.load()

    class E:
        pass
    e = E()
    e.torch, e.lib, e.ours, e.M = torch, lib, cg.gemm, CUDAMatrix
    store = golden_ref.RefStore("ref_cuda")
    ref_api = ref_cuda_lib.binding() if golden_ref.RECORD else None

    def rand(rows, cols, s4, gen, scale=1.0, uniform=False):
        m = CUDAMatrix(rows, cols, s4)
        if uniform:
            m.storage.uniform_(generator=gen)
        else:
            m.storage.normal_(generator=gen)
        if scale != 1.0:
            m.storage.mul_(scale)
        return m

    def nan(rows, cols, s4):
        m = CUDAMatrix(rows, cols, s4)
        m.fill_(float("nan"))
        return m
    e.rand, e.nan = rand, nan

    def ref(key, rows, cols, s4, call, init=None, exact=False):
        """the reference's result of call(api, target) on a zero (or `init`) target: live when recording, else stored"""
        def compute():
            m = CUDAMatrix(rows, cols, s4)
            if init is not None:
                m.storage.copy_(init.storage)
            call(ref_api, m)
            torch.cuda.synchronize()
            return m.storage
        return store.reference(key, compute, exact)
    e.ref = ref

    def diff(a, b):
        a = a.storage
        assert torch.isfinite(a).all()
        if not isinstance(b, golden_ref.Stored):
            assert torch.isfinite(b).all()
        return golden_ref.diff(a, b)
    e.diff = diff
    e.equal = lambda a, b: golden_ref.equal(a.storage, b)
    yield e
    store.save()
    lib.set_precision("tf32")
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "ref_cuda_parity.json"), "w") as f:
        json.dump(_RESULTS, f, indent=1, sort_keys=True)


# name: W, H, Cin, Cout, ky, kx, sy, sx, py, px        (net A, SURVEY.md Appendix B)
ALEX_CONV = {
    "conv1": (224, 224, 3, 96, 7, 7, 2, 2, 1, 1),
    "conv2": (55, 55, 96, 256, 5, 5, 2, 2, 1, 1),
    "nin2_1": (27, 27, 256, 256, 1, 1, 1, 1, 0, 0),
    "conv3": (14, 14, 256, 384, 3, 3, 1, 1, 1, 1),
    "nin3_1": (14, 14, 384, 768, 1, 1, 1, 1, 0, 0),
    "conv4": (14, 14, 768, 384, 3, 3, 1, 1, 1, 1),
    "nin4_1": (14, 14, 384, 768, 1, 1, 1, 1, 0, 0),
    "nin4_2": (14, 14, 768, 384, 1, 1, 1, 1, 0, 0),
    "conv5": (14, 14, 384, 512, 3, 3, 1, 1, 0, 0),
    "nin5_1": (12, 12, 512, 1024, 1, 1, 1, 1, 0, 0),
    "nin5_2": (12, 12, 1024, 512, 1, 1, 1, 1, 0, 0),
    "fc6": (1, 1, 18432, 4096, 1, 1, 1, 1, 0, 0),         # FC as a 1x1 conv on a 1x1 image (host/edge.cc FCEdge)
    "fc7": (1, 1, 4096, 4096, 1, 1, 1, 1, 0, 0),
    "fc8": (1, 1, 4096, 1000, 1, 1, 1, 1, 0, 0),
}


@pytest.mark.parametrize("N", [128, 256])
@pytest.mark.parametrize("layer", list(ALEX_CONV))
def test_alexnet_conv_layers(env, layer, N):
    torch = env.torch
    W, H, Cin, Cout, ky, kx, sy, sx, py, px = ALEX_CONV[layer]
    modY, modX = num_modules(H, ky, sy, py), num_modules(W, kx, sx, px)
    d = GetConvDesc(Cin, Cout, ky, kx, sy, sx, py, px)
    ish, fsh, tsh = (N, W, H, Cin), (Cout, kx, ky, Cin), (N, modX, modY, Cout)
    K = kx * ky * Cin
    g = torch.Generator(device="cuda").manual_seed(zlib.crc32(("%s_%d" % (layer, N)).encode()) & 0xFFFF)
    x = env.rand(N, W * H * Cin, ish, g)
    w = env.rand(Cout, K, fsh, g, scale=1.0 / np.sqrt(K))
    dv = env.rand(N, modX * modY * Cout, tsh, g)
    # the reference, once
    key = "%s_b%d/" % (layer, N)
    r_up = env.ref(key + "fprop", N, modX * modY * Cout, tsh, lambda api, t: api.convUp(x, w, t, d, 0))
    r_dn = env.ref(key + "dgrad", N, W * H * Cin, ish, lambda api, t: api.convDown(dv, w, t, d, 0))
    r_dw = env.ref(key + "wgrad", Cout, K, fsh, lambda api, t: api.convOutp(x, dv, t, d, 0, 1.0 / N))
    for mode in ("fp32", "tf32", "bf16"):
        env.lib.set_precision(mode)
        out = env.nan(N, modX * modY * Cout, tsh); env.ours.convUp(x, w, out, d, 0); p_up = env.lib.last_conv_path()
        d_up = env.diff(out, r_up)
        out = env.nan(N, W * H * Cin, ish); env.ours.convDown(dv, w, out, d, 0); p_dn = env.lib.last_conv_path()
        d_dn = env.diff(out, r_dn)
        out = env.nan(Cout, K, fsh); env.ours.convOutp(x, dv, out, d, 0, 1.0 / N); p_dw = env.lib.last_conv_path()
        d_dw = env.diff(out, r_dw)
        _RESULTS["%s_b%d_%s" % (layer, N, mode)] = {"fprop": d_up, "dgrad": d_dn, "wgrad": d_dw,
                                                    "paths": [p_up, p_dn, p_dw]}
        # a call that the tensor path declines runs on the fp32 CUDA-core kernels and must then meet the fp32 bar
        for name, dd, path in (("fprop", d_up, p_up), ("dgrad", d_dn, p_dn), ("wgrad", d_dw, p_dw)):
            tol = TOL["fp32"] if path == "cuda-core-fp32" else TOL[mode]
            assert dd < tol, (layer, N, mode, name, path, dd)


@pytest.mark.parametrize("N", [128, 256])
def test_alexnet_conv_accumulate(env, N):
    """scaleTargets = 1 at BASELINE size (conv3, all three ops) against the reference's kWriteRowsMult / Sgemm beta path."""
    torch = env.torch
    W, H, Cin, Cout, ky, kx, sy, sx, py, px = ALEX_CONV["conv3"]
    d = GetConvDesc(Cin, Cout, ky, kx, sy, sx, py, px)
    ish, fsh, tsh = (N, W, H, Cin), (Cout, kx, ky, Cin), (N, 14, 14, Cout)
    K = kx * ky * Cin
    g = torch.Generator(device="cuda").manual_seed(77 + N)
    x, w, dv = env.rand(N, W * H * Cin, ish, g), env.rand(Cout, K, fsh, g, 1.0 / np.sqrt(K)), env.rand(N, 196 * Cout, tsh, g)
    i_up, i_dn, i_dw = env.rand(N, 196 * Cout, tsh, g), env.rand(N, W * H * Cin, ish, g), env.rand(Cout, K, fsh, g)

    def run(api):
        a = env.M(N, 196 * Cout, tsh); a.storage.copy_(i_up.storage); api.convUp(x, w, a, d, 1)
        b = env.M(N, W * H * Cin, ish); b.storage.copy_(i_dn.storage); api.convDown(dv, w, b, d, 1)
        c = env.M(Cout, K, fsh); c.storage.copy_(i_dw.storage); api.convOutp(x, dv, c, d, 1, 0.5)
        return a, b, c
    key = "conv3_accum_b%d/" % N
    ref = (env.ref(key + "fprop", N, 196 * Cout, tsh, lambda api, t: api.convUp(x, w, t, d, 1), init=i_up),
           env.ref(key + "dgrad", N, W * H * Cin, ish, lambda api, t: api.convDown(dv, w, t, d, 1), init=i_dn),
           env.ref(key + "wgrad", Cout, K, fsh, lambda api, t: api.convOutp(x, dv, t, d, 1, 0.5), init=i_dw))
    for mode in ("fp32", "tf32", "bf16"):
        env.lib.set_precision(mode)
        for name, a, b in zip(("fprop", "dgrad", "wgrad"), run(env.ours), ref):
            dd = env.diff(a, b)
            _RESULTS.setdefault("conv3_accum_b%d_%s" % (N, mode), {})[name] = dd
            assert dd < TOL[mode], (mode, name, dd)


ALEX_POOL = {"pool1": (110, 96), "pool2": (27, 256), "pool5": (12, 512)}      # image size, channels; 3x3 stride 2 pad 1


@pytest.mark.parametrize("N", [128, 256])
@pytest.mark.parametrize("layer", list(ALEX_POOL))
def test_alexnet_pool_layers(env, layer, N):
    torch = env.torch
    W, C = ALEX_POOL[layer]
    mod = num_modules(W, 3, 2, 1)
    d = GetConvDesc(C, C, 3, 3, 2, 2, 1, 1)
    ish, psh = (N, W, W, C), (N, mod, mod, C)
    g = torch.Generator(device="cuda").manual_seed(5 + N)
    x = env.rand(N, W * W * C, ish, g)
    gr = env.rand(N, mod * mod * C, psh, g)
    res = {}
    key = "%s_b%d/" % (layer, N)
    r_mx = env.ref(key + "max", N, mod * mod * C, psh, lambda api, t: api.MaxPool(x, t, d), exact=True)
    o_mx = env.nan(N, mod * mod * C, psh); env.ours.MaxPool(x, o_mx, d)
    assert env.equal(o_mx, r_mx), "max-pool values must be bit-exact"
    r_av = env.ref(key + "avg", N, mod * mod * C, psh, lambda api, t: api.AvgPool(x, t, d))
    o_av = env.nan(N, mod * mod * C, psh); env.ours.AvgPool(x, o_av, d)
    res["avg"] = env.diff(o_av, r_av)
    for st in (0, 1):
        init = env.rand(N, W * W * C, ish, g)
        r = env.ref(key + "max_undo_st%d" % st, N, W * W * C, ish,
                    lambda api, t: api.MaxPoolUndo(x, gr, env.M(N, mod * mod * C, psh, storage=r_mx), t, d, st), init=init)
        o = env.M(N, W * W * C, ish); o.storage.copy_(init.storage if st else torch.full_like(init.storage, float("nan")))
        env.ours.MaxPoolUndo(x, gr, o_mx, o, d, st)
        res["max_undo_st%d" % st] = env.diff(o, r)
        r = env.ref(key + "avg_undo_st%d" % st, N, W * W * C, ish, lambda api, t: api.AvgPoolUndo(gr, t, d, st), init=init)
        o = env.M(N, W * W * C, ish); o.storage.copy_(init.storage if st else torch.full_like(init.storage, float("nan")))
        env.ours.AvgPoolUndo(gr, o, d, st)
        res["avg_undo_st%d" % st] = env.diff(o, r)
    _RESULTS["%s_b%d" % (layer, N)] = res
    for k, v in res.items():
        assert v < TOL_MEM, (layer, N, k, v)


ALEX_RNORM = {"rnorm1": (55, 96, 24), "rnorm2": (14, 256, 64)}      # image size, channels, window (frac 0.25)


@pytest.mark.parametrize("N", [128, 256])
@pytest.mark.parametrize("layer", list(ALEX_RNORM))
def test_alexnet_rnorm_layers(env, layer, N):
    torch = env.torch
    W, C, k = ALEX_RNORM[layer]
    ish = (N, W, W, C)
    g = torch.Generator(device="cuda").manual_seed(9 + N)
    x, dy = env.rand(N, W * W * C, ish, g), env.rand(N, W * W * C, ish, g)
    res = {}
    for blocked in (False, True):
        key = "%s_b%d/blocked%d_" % (layer, N, blocked)
        r = env.ref(key + "fwd", N, W * W * C, ish, lambda api, t: api.ResponseNormCrossMap(x, t, k, 5e-4, 0.75, blocked))
        o = env.nan(N, W * W * C, ish); env.ours.ResponseNormCrossMap(x, o, k, 5e-4, 0.75, blocked)
        res["fwd_blocked%d" % blocked] = env.diff(o, r)
        r = env.ref(key + "undo", N, W * W * C, ish,
                    lambda api, t: api.ResponseNormCrossMapUndo(dy, x, t, k, 5e-4, 0.75, blocked))
        o = env.nan(N, W * W * C, ish); env.ours.ResponseNormCrossMapUndo(dy, x, o, k, 5e-4, 0.75, blocked)
        res["undo_blocked%d" % blocked] = env.diff(o, r)
    _RESULTS["%s_b%d" % (layer, N)] = res
    for kk, v in res.items():
        assert v < (2 * TOL_MEM if kk.startswith("undo") else TOL_MEM), (layer, N, kk, v)


# BASELINE config 4 (SURVEY.md 8(d)): clips of 16 frames 112x112x3, batch 32, 3x3x3 kernels, pad y/x 1, pad t 0
C3D_CONV = {
    # name: W, Cin, T, Cout
    "conv1a": (112, 3, 16, 64),
    "conv2a": (56, 64, 14, 128),
}


@pytest.mark.parametrize("layer", list(C3D_CONV))
def test_c3d_conv_layers(env, layer):
    torch = env.torch
    N = 32
    W, Cin, T, Cout = C3D_CONV[layer]
    kt, To = 3, T - 2
    d = GetConvDesc(Cin, Cout, 3, 3, 1, 1, 1, 1, kernel_size_t=kt, stride_t=1, padding_t=0)
    ish, fsh, tsh = (N, W, W, Cin * T), (Cout, 3, 3, Cin * kt), (N, W, W, Cout * To)
    K = 9 * Cin * kt
    g = torch.Generator(device="cuda").manual_seed(31)
    x = env.rand(N, W * W * Cin * T, ish, g)
    w = env.rand(Cout, K, fsh, g, scale=1.0 / np.sqrt(K))
    dv = env.rand(N, W * W * Cout * To, tsh, g)
    key = "c3d_%s_b%d/" % (layer, N)
    r_up = env.ref(key + "fprop", N, W * W * Cout * To, tsh, lambda api, t: api.convUp3D(x, w, t, d, 0))
    r_dn = env.ref(key + "dgrad", N, W * W * Cin * T, ish, lambda api, t: api.convDown3D(dv, w, t, d, 0))
    r_dw = env.ref(key + "wgrad", Cout, K, fsh, lambda api, t: api.convOutp3D(x, dv, t, d, 0, 1.0 / N))
    for mode in ("fp32", "tf32", "bf16"):
        env.lib.set_precision(mode)
        out = env.nan(N, W * W * Cout * To, tsh); env.ours.convUp3D(x, w, out, d, 0); p_up = env.lib.last_conv_path()
        d_up = env.diff(out, r_up)
        out = env.nan(N, W * W * Cin * T, ish); env.ours.convDown3D(dv, w, out, d, 0); p_dn = env.lib.last_conv_path()
        d_dn = env.diff(out, r_dn)
        out = env.nan(Cout, K, fsh); env.ours.convOutp3D(x, dv, out, d, 0, 1.0 / N); p_dw = env.lib.last_conv_path()
        d_dw = env.diff(out, r_dw)
        _RESULTS["c3d_%s_b%d_%s" % (layer, N, mode)] = {"fprop": d_up, "dgrad": d_dn, "wgrad": d_dw,
                                                        "paths": [p_up, p_dn, p_dw]}
        for name, dd, path in (("fprop", d_up, p_up), ("dgrad", d_dn, p_dn), ("wgrad", d_dw, p_dw)):
            tol = TOL["fp32"] if path == "cuda-core-fp32" else TOL[mode]
            assert dd < tol, (layer, mode, name, path, dd)


def test_c3d_pool_layer(env):
    """cfg4's 2x2x2 max-pool (kernel_size_t / stride_t through kPool, cudamat_conv_gemm.cu:153-200) at batch 32."""
    torch = env.torch
    N, W, C, T = 32, 56, 128, 12
    d = GetConvDesc(C, C, 2, 2, 2, 2, 0, 0, kernel_size_t=2, stride_t=2, padding_t=0)
    ish, psh = (N, W, W, C * T), (N, W // 2, W // 2, C * (T // 2))
    g = torch.Generator(device="cuda").manual_seed(3)
    x = env.rand(N, W * W * C * T, ish, g)
    gr = env.rand(N, (W // 2) ** 2 * C * (T // 2), psh, g)
    r_mx = env.ref("c3d_pool2_b32/max", gr.rows, gr.cols, psh, lambda api, t: api.MaxPool(x, t, d), exact=True)
    o_mx = env.nan(gr.rows, gr.cols, psh); env.ours.MaxPool(x, o_mx, d)
    assert env.equal(o_mx, r_mx)
    r = env.ref("c3d_pool2_b32/max_undo", x.rows, x.cols, ish,
                lambda api, t: api.MaxPoolUndo(x, gr, env.M(gr.rows, gr.cols, psh, storage=r_mx), t, d, 0))
    o = env.nan(x.rows, x.cols, ish); env.ours.MaxPoolUndo(x, gr, o_mx, o, d, 0)
    dd = env.diff(o, r)
    _RESULTS["c3d_pool2_b32"] = {"max_undo": dd}
    assert dd < TOL_MEM
