"""Link-level drop-in proof: a C++ translation unit that includes the reference's OWN headers
(cudamat/cudamat_conv_gemm.cuh, cudamat/cudamat_conv.cuh) links against the product under the library names the
reference's Makefile uses (`-lcudamat_conv_gemm -lcudamat_conv`, Makefile:72-77), and — on the GPU — computes
the right numbers through both symbol sets.  The reference's headers are used where CONVNET_REFERENCE names its source
tree; elsewhere the same program is compiled against the project's own declarations (include/), which must declare
every function of both symbol sets exactly as the reference's headers do: same type, same (C) linkage, same struct
sizes.  What the reference's headers declare is stored in tests/golden/ref_abi_facts.json (drop_in/abi_facts.cc);
CONVNET_B200_RECORD_GOLDEN=1 with CONVNET_REFERENCE set re-records it."""
import json
import os
import subprocess

import pytest

import golden_ref
from convnet_b200.build import DROP_IN_BIN as BIN
from convnet_b200.build import ROOT, build, build_drop_in, reference_headers

FACTS_SRC = os.path.join(ROOT, "tests", "drop_in", "abi_facts.cc")
FACTS_GOLDEN = os.path.join(golden_ref.GOLDEN, "ref_abi_facts.json")


def abi_facts(ref_headers, out_dir):
    """(printed facts, undefined symbols of the ABI) of drop_in/abi_facts.cc compiled against `ref_headers` (the
    reference's) or, when None, the project's headers, and linked against the product"""
    libdir = os.path.dirname(build())
    exe = os.path.join(str(out_dir), "abi_facts_%s" % ("reference" if ref_headers else "own"))
    headers = ["-I" + ref_headers] if ref_headers else ["-DDROP_IN_OWN_HEADERS", "-I" + os.path.join(ROOT, "include")]
    subprocess.run(["g++", "-O1", "-std=c++14"] + headers + ["-I/usr/local/cuda/include", FACTS_SRC, "-o", exe,
                    "-L" + libdir, "-lcudamat_conv_gemm", "-L/usr/local/cuda/lib64", "-lcudart", "-Wl,--no-undefined",
                    "-Wl,-rpath," + libdir, "-Wl,-rpath,/usr/local/cuda/lib64"], check=True)
    printed = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines()
    names = [l.split()[0] for l in printed if not l.startswith("sizeof")]
    syms = subprocess.run(["nm", "-D", "--undefined-only", exe], capture_output=True, text=True, check=True).stdout
    undefined = sorted({l.split()[-1].split("@")[0] for l in syms.splitlines() if any(n in l for n in names)})
    return {"declarations": printed, "undefined_symbols": undefined}


def test_reference_headers_compile_and_link_against_the_product(tmp_path):
    ref = reference_headers()
    for b, name in zip(build_drop_in(ref), ("libcudamat_conv_gemm.so", "libcudamat_conv.so")):
        out = subprocess.run(["ldd", b], capture_output=True, text=True).stdout
        line = [l for l in out.splitlines() if name in l]
        assert line and os.path.join("convnet_b200", "lib") in line[0], out
        # every reference prototype the program calls resolved to the product (-Wl,--no-undefined made the link fail otherwise)
        syms = subprocess.run(["nm", "-D", "--undefined-only", b], capture_output=True, text=True).stdout
        for s in ("convUpGemm", "convUp", "MaxPoolGemm", "MaxPool", "SetupTexture"):
            assert (" U %s\n" % s) in syms or (" U %s@" % s) in syms, (s, syms)
    # the project's declarations of both symbol sets are the reference's: live where its headers are at hand, else stored
    if ref:
        want = abi_facts(ref, tmp_path)
        if golden_ref.RECORD:
            with open(FACTS_GOLDEN, "w") as f:
                json.dump(want, f, indent=1)
                f.write("\n")
    else:
        with open(FACTS_GOLDEN) as f:
            want = json.load(f)
    assert len(want["declarations"]) == 46 and len(want["undefined_symbols"]) == 43, want
    assert abi_facts(None, tmp_path) == want


@pytest.mark.gpu
def test_drop_in_binary_runs_on_the_gpu():
    for alias in ("cudamat_conv_gemm", "cudamat_conv"):
        b = BIN + "_" + alias
        if not os.path.exists(b):
            pytest.fail("%s was not built (run __graft_entry__.build())" % b)
        r = subprocess.run([b], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and "DROP-IN OK" in r.stdout, (r.returncode, r.stdout, r.stderr)
