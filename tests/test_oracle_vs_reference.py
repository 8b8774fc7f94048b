"""Pin oracle/conv_oracle.c (CPU, no GPU) against
  (a) the golden vectors produced by the reference's py/conv_cpu.py (tools/gen_golden.py), and
  (b) the reference's compiled CPU library (eigenmat/cpumat_conv.cc built into oracle/_ref/libeigenmat_ref.so), whose
      results are stored in tests/golden/ref_eigenmat.npz (tests/golden_ref.py).
Metric and tolerance are the reference's own: Diff < 1e-4 (py/test_conv.py:382-392)."""
import numpy as np
import pytest

import golden_ref
from cases import F, GOLDEN_2D, GOLDEN_3D, Z, geo2d, geo3d, load_golden
from oracle_lib import Diff, RefLib

TOL = 1e-4


@pytest.mark.parametrize("name", GOLDEN_2D)
def test_oracle_conv2d_vs_python_reference(oracle, name):
    g = load_golden(name)
    d, pd, ish, fsh, tsh, psh = geo2d(g)
    N = g["N"]
    out = Z(N, g["convUp"].shape[1]); oracle.convUp(g["images"], g["filters"], out, ish, fsh, tsh, d)
    assert Diff(out, g["convUp"]) < TOL
    out = Z(N, g["convDown"].shape[1]); oracle.convDown(g["derivs"], g["filters"], out, tsh, fsh, ish, d)
    assert Diff(out, g["convDown"]) < TOL
    out = Z(*g["convOutp"].shape); oracle.convOutp(g["images"], g["derivs"], out, ish, tsh, fsh, d)
    assert Diff(out, g["convOutp"]) < TOL
    # partial sums (ABI-2 target layout)
    chunks = g["convOutpPartial"].shape[1] // g["convOutp"].shape[1]
    out = Z(*g["convOutpPartial"].shape)
    oracle.convOutpPartial(g["images"], g["derivs"], out, ish, tsh,
                           (g["Cout"], g["kx"], g["ky"], g["Cin"] * chunks), d, g["psy"], g["psx"])
    assert Diff(out, g["convOutpPartial"]) < TOL


@pytest.mark.parametrize("name", GOLDEN_2D)
def test_oracle_pool2d_vs_python_reference(oracle, name):
    g = load_golden(name)
    d, pd, ish, fsh, tsh, psh = geo2d(g)
    N = g["N"]
    mx = Z(N, g["maxPool"].shape[1]); oracle.pool(True, g["pool_images"], mx, ish, psh, pd)
    assert np.array_equal(mx, g["maxPool"])          # max values are exact
    av = Z(N, g["avgPool"].shape[1]); oracle.pool(False, g["pool_images"], av, ish, psh, pd)
    assert Diff(av, g["avgPool"]) < TOL
    out = Z(N, g["maxPoolUndo"].shape[1])
    oracle.maxPoolUndo(g["pool_images"], g["pool_derivs"], mx, out, ish, psh, pd)
    assert Diff(out, g["maxPoolUndo"]) < TOL
    out = Z(N, g["avgPoolUndo"].shape[1]); oracle.avgPoolUndo(g["pool_derivs"], out, psh, ish, pd)
    assert Diff(out, g["avgPoolUndo"]) < TOL


@pytest.mark.parametrize("name", GOLDEN_2D)
@pytest.mark.parametrize("blocked", [False, True])
def test_oracle_rnorm_vs_python_reference(oracle, name, blocked):
    g = load_golden(name)
    tag = "_blocked" if blocked else ""
    out = Z(*g["images"].shape)
    oracle.rnorm(g["images"], out, g["Cin"], g["sizeF"], g["add_scale"], g["pow_scale"], blocked)
    assert Diff(out, g["rnorm" + tag]) < TOL
    out = Z(*g["images"].shape)
    oracle.rnormUndo(g["rnorm_derivs"], g["images"], out, g["Cin"], g["sizeF"], g["add_scale"],
                     g["pow_scale"], blocked)
    assert Diff(out, g["rnormUndo" + tag]) < TOL


@pytest.mark.parametrize("name", GOLDEN_3D)
def test_oracle_3d_vs_python_reference(oracle, name):
    g = load_golden(name)
    d, pd, ish, fsh, tsh, psh = geo3d(g)
    N = g["N"]
    out = Z(N, g["convUp3D"].shape[1]); oracle.convUp3D(g["images"], g["filters"], out, ish, fsh, tsh, d)
    assert Diff(out, g["convUp3D"]) < TOL
    out = Z(N, g["convDown3D"].shape[1]); oracle.convDown3D(g["derivs"], g["filters"], out, tsh, fsh, ish, d)
    assert Diff(out, g["convDown3D"]) < TOL
    out = Z(*g["convOutp3D"].shape); oracle.convOutp3D(g["images"], g["derivs"], out, ish, tsh, fsh, d)
    assert Diff(out, g["convOutp3D"]) < TOL
    mx = Z(N, g["maxPool3D"].shape[1]); oracle.pool(True, g["pool_images"], mx, ish, psh, pd)
    assert np.array_equal(mx, g["maxPool3D"])
    av = Z(N, g["avgPool3D"].shape[1]); oracle.pool(False, g["pool_images"], av, ish, psh, pd)
    assert Diff(av, g["avgPool3D"]) < TOL
    out = Z(N, g["maxPool3DUndo"].shape[1])
    oracle.maxPoolUndo(g["pool_images"], g["pool_derivs"], mx, out, ish, psh, pd)
    assert Diff(out, g["maxPool3DUndo"]) < TOL
    out = Z(N, g["avgPool3DUndo"].shape[1]); oracle.avgPoolUndo(g["pool_derivs"], out, psh, ish, pd)
    assert Diff(out, g["avgPool3DUndo"]) < TOL


# ---- (b) the reference's compiled CPU library ------------------------------------------------
@pytest.fixture(scope="module")
def reflib():
    """(stored results, live library): the library only while recording (tests/golden_ref.py)"""
    store = golden_ref.RefStore("ref_eigenmat")
    if golden_ref.RECORD and not RefLib.available():
        pytest.fail("recording needs oracle/_ref/libeigenmat_ref.so: run `make -C oracle` where the reference exists")
    yield store, RefLib() if golden_ref.RECORD else None
    store.save()


def _reference(reflib, key, init, run, exact=True):
    """what run(library, target) leaves in a copy of `init` (live when recording, else stored)"""
    store, lib = reflib

    def live():
        b = init.copy(order="F")
        run(lib, b)
        return b
    return store.reference(key, live, exact)


CONV_SHAPES = [
    # N, W, H, Cin, Cout, ky, kx, sy, sx, py, px
    (16, 12, 12, 32, 64, 3, 3, 2, 2, 1, 1),      # py/test_conv.py 2-D geometry
    (6, 9, 7, 3, 10, 3, 2, 1, 2, 1, 0),
    (4, 15, 15, 3, 8, 7, 7, 2, 2, 1, 1),         # conv1-like
    (8, 6, 6, 16, 16, 1, 1, 1, 1, 0, 0),         # 1x1 (ConvOneToOne / FC shape)
    (3, 11, 11, 5, 7, 4, 4, 1, 1, 0, 0),         # mnist-conv 4x4 p0
]


@pytest.mark.parametrize("shape", CONV_SHAPES)
@pytest.mark.parametrize("scaleTargets", [0.0, 1.0])
def test_oracle_conv_bit_exact_vs_compiled_reference(oracle, reflib, shape, scaleTargets):
    from convnet_b200.abi import GetConvDesc, num_modules
    N, W, H, Cin, Cout, ky, kx, sy, sx, py, px = shape
    modY, modX = num_modules(H, ky, sy, py), num_modules(W, kx, sx, px)
    d = GetConvDesc(Cin, Cout, ky, kx, sy, sx, py, px)
    ish, fsh, tsh = (N, W, H, Cin), (Cout, kx, ky, Cin), (N, modX, modY, Cout)
    r = np.random.RandomState(7)
    images, filters = F(r.randn(N, W * H * Cin)), F(r.randn(Cout, kx * ky * Cin))
    derivs = F(r.randn(N, modX * modY * Cout))
    for op, args, oshape in (
            ("convUp", (images, filters, ish, fsh, tsh), (N, modX * modY * Cout)),
            ("convDown", (derivs, filters, tsh, fsh, ish), (N, W * H * Cin)),
            ("convOutp", (images, derivs, ish, tsh, fsh), (Cout, kx * ky * Cin))):
        init = F(r.randn(*oshape))
        a = init.copy(order="F")
        getattr(oracle, op)(args[0], args[1], a, *args[2:], d, scaleTargets, 0.5)
        key = "conv_%s_st%g/%s" % ("x".join(map(str, shape)), scaleTargets, op)
        b = _reference(reflib, key, init, lambda lib, b: getattr(lib, op)(args[0], args[1], b, *args[2:], d, scaleTargets, 0.5))
        assert golden_ref.equal(a, b), (op, golden_ref.diff(a, b))


def test_oracle_channel_subrange_vs_compiled_reference(oracle, reflib):
    from convnet_b200.abi import GetConvDesc
    N, W, H, Cin, Cout = 4, 8, 8, 12, 16
    d = GetConvDesc(Cin, Cout, 3, 3, 1, 1, 1, 1, input_channel_begin=4, input_channel_end=10,
                    output_channel_begin=8, output_channel_end=16)
    ish, fsh, tsh = (N, W, H, Cin), (8, 3, 3, 6), (N, 8, 8, Cout)
    r = np.random.RandomState(3)
    images, filters, derivs = F(r.randn(N, W * H * Cin)), F(r.randn(8, 9 * 6)), F(r.randn(N, 64 * Cout))
    for op, args, oshape in (("convUp", (images, filters, ish, fsh, tsh), (N, 64 * Cout)),
                             ("convDown", (derivs, filters, tsh, fsh, ish), (N, 64 * Cin)),
                             ("convOutp", (images, derivs, ish, tsh, fsh), (8, 54))):
        init = F(r.randn(*oshape))
        a = init.copy(order="F")
        getattr(oracle, op)(args[0], args[1], a, *args[2:], d, 1.0, 1.0)
        b = _reference(reflib, "channel_subrange/" + op, init,
                       lambda lib, b: getattr(lib, op)(args[0], args[1], b, *args[2:], d, 1.0, 1.0))
        assert golden_ref.equal(a, b), op


@pytest.mark.parametrize("F_sizeF", [(32, 8), (96, 24), (7, 3), (16, 16)])
@pytest.mark.parametrize("blocked", [False, True])
def test_oracle_rnorm_bit_exact_vs_compiled_reference(oracle, reflib, F_sizeF, blocked):
    nf, sizeF = F_sizeF
    r = np.random.RandomState(11)
    x, dy = F(r.randn(6, 5 * 5 * nf)), F(r.randn(6, 5 * 5 * nf))
    key = "rnorm_%d_%d_blocked%d/" % (nf, sizeF, blocked)
    a = Z(*x.shape)
    oracle.rnorm(x, a, nf, sizeF, 0.005, 0.75, blocked)
    b = _reference(reflib, key + "fwd", Z(*x.shape), lambda lib, b: lib.rnorm(x, b, nf, sizeF, 0.005, 0.75, blocked),
                   exact=False)
    assert golden_ref.diff(a, b) < 1e-6
    oracle.rnormUndo(dy, x, a, nf, sizeF, 0.005, 0.75, blocked)
    b = _reference(reflib, key + "undo", Z(*x.shape),
                   lambda lib, b: lib.rnormUndo(dy, x, b, nf, sizeF, 0.005, 0.75, blocked), exact=False)
    assert golden_ref.diff(a, b) < 1e-6
