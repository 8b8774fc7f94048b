"""Load libconvnet_b200.so and declare the C ABI (include/*.h) for ctypes.

There is NO fallback: if the shared library is missing this raises, so a GPU run can
never silently take a CPU / PyTorch path.
"""
import ctypes as ct
import os

from .abi import ConvDesc, Shape4D, cudamat

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libconvnet_b200.so")

MP = ct.POINTER(cudamat)
SP = ct.POINTER(Shape4D)
F, I, B = ct.c_float, ct.c_int, ct.c_bool
FP = ct.c_void_p          # raw device pointers for the cnb_* helpers

# name -> argtypes; every symbol declared in include/*.h (tests/test_abi_symbols.py checks the headers against this)
SIGNATURES = {
    # ---- ABI-1: include/convnet_b200_conv_gemm.h
    "convUpGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "convDownGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "convOutpGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F, F],
    "convInnerpGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F, F],
    "localUpGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "localDownGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "localOutpGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F, F],
    "MaxPoolGemm": [MP, MP, SP, SP, ConvDesc, F, F],
    "AvgPoolGemm": [MP, MP, SP, SP, ConvDesc, F, F],
    "MaxPoolUndoGemm": [MP, MP, MP, MP, SP, SP, ConvDesc, F],
    "MaxPoolRpropGemm": [MP, MP, MP, MP, SP, SP, ConvDesc, F],
    "AvgPoolUndoGemm": [MP, MP, SP, SP, ConvDesc, F],
    "UpSampleGemm": [MP, MP, SP, SP, I, F],
    "DownSampleGemm": [MP, MP, SP, SP, I],
    "ResponseNormCrossMapGemm": [MP, MP, I, I, F, F, B],
    "ResponseNormCrossMapUndoGemm": [MP, MP, MP, I, I, F, F, B],
    "ResponseNormCrossMapRpropGemm": [MP, MP, MP, I, I, F, F, B],
    "Scale": [MP, F],
    "convUp3DGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "convDown3DGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "convOutp3DGemm": [MP, MP, MP, SP, SP, SP, ConvDesc, F, F],
    "ResponseNormCrossMap3DGemm": [MP, MP, I, I, F, F, B, I],
    "ResponseNormCrossMap3DUndoGemm": [MP, MP, MP, I, I, F, F, B, I],
    # ---- ABI-2: include/convnet_b200_conv.h
    "SetupTexture": [MP],
    "convUp": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "localUp": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "convDown": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "localDown": [MP, MP, MP, SP, SP, SP, ConvDesc, F],
    "convOutp": [MP, MP, MP, SP, SP, SP, ConvDesc, I, I, F, F],
    "localOutp": [MP, MP, MP, SP, SP, SP, ConvDesc, F, F],
    "ResponseNormCrossMap": [MP, MP, I, I, F, F, B],
    "ResponseNormCrossMapUndo": [MP, MP, MP, MP, I, I, F, F, B],
    "ResponseNorm": [MP, MP, MP, I, I, F, F],
    "ResponseNormUndo": [MP, MP, MP, MP, MP, I, I, F, F],
    "ContrastNorm": [MP, MP, MP, MP, I, I, F, F],
    "ContrastNormUndo": [MP, MP, MP, MP, MP, I, I, F, F],
    "MaxPool": [MP, MP, SP, SP, ConvDesc],
    "AvgPool": [MP, MP, SP, SP, ConvDesc],
    "MaxPoolUndo": [MP, MP, MP, MP, SP, SP, ConvDesc, F],
    "AvgPoolUndo": [MP, MP, SP, SP, ConvDesc, F],
    "UpSample": [MP, MP, SP, SP, I, F],
    "DownSample": [MP, MP, SP, SP, I],
    "RGBToYUV": [MP, MP],
    # ---- extensions: include/convnet_b200_ext.h
    "convnet_b200_version": [],
    "convnet_b200_set_stream": [ct.c_void_p],
    "convnet_b200_get_stream": [],
    "convnet_b200_set_conv_precision": [I],
    "convnet_b200_get_conv_precision": [],
    "convnet_b200_last_conv_path": [],
    "convnet_b200_last_conv_kernel": [],
    "convnet_b200_launch_count": [],
    "convnet_b200_fuse_next": [FP, I, FP],
    "convnet_b200_bf16_stage": [FP, ct.c_longlong],
    "convnet_b200_bf16_ensure": [FP, ct.c_longlong],
    "convnet_b200_bf16_is_staged": [FP, ct.c_longlong],
    "convnet_b200_emit_bf16_next": [],
    "convnet_b200_reserve_sms": [I],
    "convnet_b200_pool_cache_next": [],
    "convnet_b200_prestage_next": [],
    "convnet_b200_extract_patches": [MP, MP, MP, MP, MP, I, I, I, I],
    "convnet_b200_fuse_next_dropout": [ct.c_float, ct.c_float, ct.c_ulonglong],
    "convnet_b200_fuse_next_scale": [F],
    "convnet_b200_fuse_next_bias_grad": [FP, F, F],
    "convnet_b200_bf16_invalidate": [FP],
    "convnet_b200_reset_launch_count": [],
    "convnet_b200_release_workspace": [],
    "cnb_add_channel_bias": [FP, FP, ct.c_longlong, I],
    "cnb_add_channel_bias_relu": [FP, FP, ct.c_longlong, I],
    "cnb_channel_bias_grad": [FP, FP, ct.c_longlong, I, F, F],
    "cnb_relu": [FP, ct.c_longlong],
    "cnb_relu_deriv": [FP, FP, ct.c_longlong],
    "cnb_sgd_momentum": [FP, FP, FP, ct.c_longlong, F, F, F],
    "cnb_sgd_momentum_multi": [ct.c_void_p, I],
    "cnb_dropout": [FP, FP, ct.c_longlong, F, F, ct.c_ulonglong],
    "cnb_mult": [FP, FP, ct.c_longlong],
    "cnb_softmax": [FP, I, I],
    "cnb_softmax_ce_deriv": [FP, FP, FP, FP, I, I],
    "cnb_sum": [FP, FP, I],
}
RESTYPES = {
    "convnet_b200_version": I, "convnet_b200_get_stream": ct.c_void_p,
    "convnet_b200_get_conv_precision": I, "convnet_b200_last_conv_path": I, "convnet_b200_last_conv_kernel": I,
    "convnet_b200_bf16_is_staged": I,
    "convnet_b200_launch_count": ct.c_ulonglong, "convnet_b200_extract_patches": I,
}

_lib = None


def load():
    """Return the loaded CDLL; raise if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "convnet_b200: %s is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        lib = ct.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)     # AttributeError if the symbol is not exported
            fn.argtypes = args
            fn.restype = RESTYPES.get(name)
        _lib = lib
    return _lib


PRECISION = {"fp32": 0, "tf32": 1, "bf16": 2}
PATH_NAME = {-1: "none", 0: "cuda-core-fp32", 1: "tcgen05-tf32", 2: "tcgen05-bf16"}


def set_precision(mode):
    load().convnet_b200_set_conv_precision(PRECISION[mode] if isinstance(mode, str) else int(mode))


def last_conv_path():
    return PATH_NAME[load().convnet_b200_last_conv_path()]


KERNEL_BITS = {"lean": 1, "pair": 2, "xmode": 4, "split": 8, "dgrad_as_fprop": 16, "a_merged": 32, "b_merged": 64}


def last_conv_kernel():
    """the variant the last conv call ran (convnet_b200_last_conv_kernel): the set of KERNEL_BITS names plus the number
    of stride phases of a dgrad-as-fprop call, or None before the first call"""
    v = load().convnet_b200_last_conv_kernel()
    if v < 0:
        return None
    return {name for name, bit in KERNEL_BITS.items() if v & bit}, v >> 8
