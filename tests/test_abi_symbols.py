"""CPU-only: the C-ABI library builds for sm_100a, loads without a GPU, and exports every symbol
that include/*.h declares (no compute calls)."""
import ctypes as ct
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADERS = ["convnet_b200_conv_gemm.h", "convnet_b200_conv.h", "convnet_b200_ext.h"]
# the reference's two symbol sets (cudamat/cudamat_conv_gemm.cuh:36-138, cudamat/cudamat_conv.cuh:8-78)
ABI1 = ("convUpGemm convDownGemm convOutpGemm convInnerpGemm localUpGemm localDownGemm localOutpGemm MaxPoolGemm "
        "MaxPoolUndoGemm MaxPoolRpropGemm AvgPoolGemm AvgPoolUndoGemm UpSampleGemm DownSampleGemm "
        "ResponseNormCrossMapGemm ResponseNormCrossMapUndoGemm ResponseNormCrossMapRpropGemm Scale convUp3DGemm "
        "convDown3DGemm convOutp3DGemm ResponseNormCrossMap3DGemm ResponseNormCrossMap3DUndoGemm").split()
ABI2 = ("SetupTexture convUp localUp convDown localDown convOutp localOutp ResponseNormCrossMap "
        "ResponseNormCrossMapUndo ResponseNorm ResponseNormUndo ContrastNorm ContrastNormUndo MaxPool AvgPool "
        "MaxPoolUndo AvgPoolUndo UpSample DownSample RGBToYUV").split()


def declared_functions():
    names = []
    for h in HEADERS:
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names += re.findall(r"^\s*(?:void\*?|int|unsigned long long)\s+\*?(\w+)\s*\(", src, flags=re.M)
    return names


@pytest.fixture(scope="module")
def libpath():
    from convnet_b200 import build
    return build.build()


def test_headers_declare_both_reference_symbol_sets():
    decl = set(declared_functions())
    assert set(ABI1) <= decl and set(ABI2) <= decl


def test_library_exports_every_declared_symbol(libpath):
    lib = ct.CDLL(libpath)          # loads with no GPU and no libcuda (cudart static, driver API resolved lazily)
    for name in declared_functions():
        assert hasattr(lib, name), name
    for alias in ("libcudamat_conv_gemm.so", "libcudamat_conv.so"):     # names the reference Makefile:72-77 links
        assert os.path.exists(os.path.join(os.path.dirname(libpath), alias))


def test_ctypes_signatures_cover_every_declared_symbol(libpath):
    from convnet_b200 import lib
    assert set(lib.SIGNATURES) == set(declared_functions())
    L = lib.load()
    assert L.convnet_b200_version() >= 100
    assert L.convnet_b200_get_conv_precision() in (0, 1, 2)
    assert L.convnet_b200_last_conv_path() == -1
    assert L.convnet_b200_last_conv_kernel() == -1


def test_abi_struct_sizes_match_reference_layout():
    from convnet_b200.abi import ConvDesc, Shape4D, cudamat
    assert (ct.sizeof(cudamat), ct.sizeof(Shape4D), ct.sizeof(ConvDesc)) == (48, 16, 64)
    assert cudamat.data_device.offset == 8 and cudamat.size.offset == 24 and cudamat.tex_obj.offset == 40


def test_sass_is_sm100a(libpath):
    out = subprocess.run(["cuobjdump", "-lelf", libpath], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from convnet_b200 import lib
    monkeypatch.setattr(lib, "_lib", None)
    monkeypatch.setattr(lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        lib.load()
