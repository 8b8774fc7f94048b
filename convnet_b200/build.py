"""Build convnet_b200/lib/libconvnet_b200.so in-tree with nvcc for sm_100a.

One shared object exports both reference symbol sets (ABI-1 `*Gemm`, ABI-2) plus the
extension API.  cudart is linked statically and the driver API (cuTensorMapEncodeTiled)
is resolved at run time through cudaGetDriverEntryPoint, so the library loads on a
machine without libcuda (the CPU-only build/test container).
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libconvnet_b200.so")
SOURCES = ["abi.cu", "ext.cu", "stage.cu", "conv_simt.cu", "conv_tc.cu", "pool.cu", "rnorm.cu", "elementwise.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
         "-ccbin", "g++"]
# no --use_fast_math: softmax / cross-entropy / avg-pool division / the fp32 conv path are IEEE-compliant; the kernels
# that want the fast intrinsics call them by name (rnorm: __powf, like the reference's --use_fast_math build)


def _stamp():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                h.update(f.encode())
                h.update(open(os.path.join(root, f), "rb").read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    stamp_file = os.path.join(LIBDIR, ".stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== nvcc %s ==\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-cudart", "static", "-ccbin", "g++"]
    subprocess.run(cmd, check=True)
    for alias in ("libcudamat_conv_gemm.so", "libcudamat_conv.so"):   # the names reference/Makefile:72-77 links
        dst = os.path.join(LIBDIR, alias)
        if os.path.lexists(dst):
            os.remove(dst)
        os.symlink("libconvnet_b200.so", dst)
    open(stamp_file, "w").write(stamp)
    return LIB


HOST = os.path.join(HERE, "host")
HOST_LIB = os.path.join(LIBDIR, "libconvnet_b200_host.so")
HOST_SOURCES = ["matrix.cc", "edge.cc", "convnet.cc", "models.cc", "data.cc", "capi.cc"]


def build_host(force=False):
    """host C++ (Matrix / Edge / ConvNet / GradChecker / DataParallelSync) -> libconvnet_b200_host.so"""
    build(force=False)
    h = hashlib.sha256()
    for f in sorted(os.listdir(HOST)):
        h.update(open(os.path.join(HOST, f), "rb").read())
    h.update(open(os.path.join(LIBDIR, ".stamp")).read().encode())
    stamp_file = os.path.join(LIBDIR, ".stamp_host")
    if not force and os.path.exists(HOST_LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == h.hexdigest():
        return HOST_LIB
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-I/usr/local/cuda/include",
           "-o", HOST_LIB] + [os.path.join(HOST, f) for f in HOST_SOURCES] + [
           "-L" + LIBDIR, "-lconvnet_b200", "-Wl,-rpath,$ORIGIN", "-L/usr/local/cuda/lib64", "-lcudart_static",
           "-ldl", "-lrt", "-lpthread"]
    subprocess.run(cmd, check=True)
    open(stamp_file, "w").write(h.hexdigest())
    return HOST_LIB


ROOT = os.path.dirname(HERE)
DROP_IN_SRC = os.path.join(ROOT, "tests", "drop_in", "link_drop_in.cc")
DROP_IN_BIN = os.path.join(ROOT, "tests", "drop_in", "_build", "link_drop_in")


def reference_headers():
    """the reference's cudamat/ header directory, when CONVNET_REFERENCE names the reference's source tree"""
    ref = os.environ.get("CONVNET_REFERENCE")
    return os.path.join(ref, "cudamat") if ref and os.path.isdir(os.path.join(ref, "cudamat")) else None


def build_drop_in(ref_headers=None):
    """the link-level drop-in program (tests/drop_in), twice: linked with -lcudamat_conv_gemm only and with
    -lcudamat_conv only (both names are aliases of the one product library, so either must resolve BOTH symbol sets the
    program calls); rpath points at convnet_b200/lib relative to the binary.  It is compiled against the reference's own
    headers from `ref_headers` when given, else against the project's declarations of the same two ABIs (include/)."""
    libdir = os.path.dirname(build())
    os.makedirs(os.path.dirname(DROP_IN_BIN), exist_ok=True)
    headers = ["-I" + ref_headers] if ref_headers else ["-DDROP_IN_OWN_HEADERS", "-I" + os.path.join(ROOT, "include")]
    outs = []
    for alias in ("cudamat_conv_gemm", "cudamat_conv"):
        out = DROP_IN_BIN + "_" + alias
        cmd = ["g++", "-O1", "-std=c++14"] + headers + ["-I/usr/local/cuda/include", DROP_IN_SRC, "-o", out,
               "-L" + libdir, "-l" + alias, "-L/usr/local/cuda/lib64", "-lcudart",
               "-Wl,--no-undefined", "-Wl,-rpath,$ORIGIN/../../../convnet_b200/lib", "-Wl,-rpath,/usr/local/cuda/lib64"]
        subprocess.run(cmd, check=True)
        outs.append(out)
    return outs


if __name__ == "__main__":
    build_host(force="--force" in sys.argv)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
