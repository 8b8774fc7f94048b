"""Every tensor-core conv variant, element by element, against float64 at the shapes of the training step.

How a conv call runs is decided by its shape and mode (csrc/conv_tc.cu): the general tcgen05 kernel or the lean one, single
CTA or CTA pair, x-mode for RGB inputs, split-K with reduce_split, wgrad reduction splits, dgrad as a stride-1 fprop per
stride phase, the 3-D frame loop, and the CUDA-core fp32 kernels.  Each case below exists for one or more of these and
asserts, through convnet_b200_last_conv_kernel and convnet_b200_last_conv_path, that it reaches them.

Every output element is compared with fp64_conv_ref at the operands the kernel multiplies (bf16 / tf32 conversion
emulated), so what may remain is the kernel's fp32 accumulation, measured relative to `mag` (the op on |operands|):
    ratio = max_i |ours_i - ref_i| / mag_i
Outputs start NaN-poisoned (scaleTargets = 0) or hold a random init; every element must be finite.  Negative controls
take the fp64 contribution of one K slice of 16 terms over one 128-row block out of the kernel's result and require the
check to fail, so the thresholds are known to see a dropped tile, phase or border row.

Setting CONVNET_B200_PARITY_JSON=<path> writes the measured ratio and variant of every case / op / mode there.
"""
import json
import os
import zlib

import numpy as np
import pytest

import fp64_conv_ref as R
from convnet_b200.abi import GetConvDesc, num_modules

pytestmark = pytest.mark.gpu

MODES = ("fp32", "tf32", "bf16")
# max ratio per path: about 10x the worst ratio measured on a B200 over every case below (fp32 5.1e-7, tf32 2.0e-6,
# bf16 1.05e-6), and at least 18x below the weakest negative control (3.6e-4: conv2 wgrad, K = 93312 reduction terms)
THRESH = {"cuda-core-fp32": 5e-6, "tcgen05-tf32": 2e-5, "tcgen05-bf16": 1e-5}
# tcgen05 kind::tf32 TRUNCATES fp32 operands to 10 mantissa bits: emulated that way the worst tf32 ratio is 2.0e-6,
# rounded to nearest even it is 1.0e-3 (B200, DESIGN.md).  Both are recorded for tf32 calls; the check uses truncation.
TF32_OPERANDS = ("tf32_trunc", "tf32_rne")
TF32_EMULATION = "tf32_trunc"
OPERANDS = {"cuda-core-fp32": "fp32", "tcgen05-tf32": TF32_EMULATION, "tcgen05-bf16": "bf16"}
PATH = {"fp32": "cuda-core-fp32", "tf32": "tcgen05-tf32", "bf16": "tcgen05-bf16", "simt": "cuda-core-fp32"}

_RESULTS = []


@pytest.fixture(scope="module")
def env():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from convnet_b200 import conv_gemm as cg
    from convnet_b200 import lib
    from convnet_b200.matrix import CUDAMatrix
    L = lib.load()

    class E:
        pass
    e = E()
    e.torch, e.cg, e.lib, e.L, e.M = torch, cg, lib, L, CUDAMatrix
    e.sms = torch.cuda.get_device_properties(0).multi_processor_count
    yield e
    L.convnet_b200_bf16_invalidate(None)
    lib.set_precision("fp32")
    path = os.environ.get("CONVNET_B200_PARITY_JSON")
    if path:
        with open(path, "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "thresholds": THRESH, "results": _RESULTS}, f, indent=1)


class Case:
    """shape = (N, W, H, Cin, Cout, ky, kx, sy, sx, py, px); expect[op][mode] = "path=<mode> +bit -bit phases=n"
    (bits: lib.KERNEL_BITS); unspecified: the mode's own path.  fp32 mode always expects the CUDA-core kernels."""

    def __init__(self, name, shape, why, expect=None, T=1, kt=1, st=(0.0, 0.0, 0.0), so_outp=None, sub=None,
                 stage_weights=False, modes=MODES, control=False):
        self.name, self.shape, self.why, self.expect = name, shape, why, expect or {}
        self.T, self.kt, self.st, self.so_outp, self.sub = T, kt, st, so_outp, sub
        self.stage_weights, self.modes, self.control = stage_weights, modes, control


# AlexNet (CLS_net_20140801232522) layers: conv1 224->110 k7s2p1, conv2 55->27 k5s2p1, conv3/4 14 k3p1, conv5 14->12 k3p0,
# 1x1 nin layers, fc6 18432->4096, fc8 4096->1000.  num_sms() / 2 CTA-pair slots (74 on a B200) decide pair mode.
CASES = [
    Case("conv1_b128", (128, 224, 224, 3, 96, 7, 7, 2, 2, 1, 1), "tf32 x-mode lean fprop + wgrad; dgrad on CUDA cores",
         {"up": {"tf32": "+lean +xmode", "bf16": "path=tf32 +lean +xmode"},
          "down": {"tf32": "path=simt", "bf16": "path=simt"},
          "outp": {"tf32": "+lean +xmode", "bf16": "path=tf32 +lean +xmode"}}),
    Case("conv2_b128", (128, 55, 55, 96, 256, 5, 5, 2, 2, 1, 1), "lean pair fprop; 4-phase dgrad-as-fprop (28/27); lean wgrad + splits",
         {"up": {"tf32": "+pair -lean", "bf16": "+lean +pair +a_merged +b_merged"},
          "down": {"tf32": "-dgrad_as_fprop", "bf16": "+dgrad_as_fprop +lean +pair phases=4"},
          "outp": {"bf16": "+lean +split"}}, control=True),
    Case("nin2_b128", (128, 27, 27, 256, 256, 1, 1, 1, 1, 0, 0), "1x1 nin layer",
         {"up": {"bf16": "+lean +pair"}, "down": {"bf16": "+dgrad_as_fprop phases=1"}, "outp": {"bf16": "+lean"}}),
    Case("conv3_b128", (128, 14, 14, 256, 384, 3, 3, 1, 1, 1, 1), "conv3; wgrad with 3 o-tiles (no pair)",
         {"up": {"bf16": "+lean +pair"}, "down": {"bf16": "+dgrad_as_fprop phases=1"}, "outp": {"bf16": "+lean -pair"}}),
    Case("conv3_b256", (256, 14, 14, 256, 384, 3, 3, 1, 1, 1, 1), "conv3 at batch 256",
         {"up": {"bf16": "+lean +pair"}, "down": {"bf16": "+dgrad_as_fprop phases=1"}, "outp": {"bf16": "+lean -pair"}}),
    Case("conv4_b128", (128, 14, 14, 768, 384, 3, 3, 1, 1, 1, 1), "conv4",
         {"up": {"bf16": "+lean +pair"}, "down": {"bf16": "+dgrad_as_fprop phases=1"}, "outp": {"bf16": "+lean -pair"}},
         control=True),
    Case("conv4_b256", (256, 14, 14, 768, 384, 3, 3, 1, 1, 1, 1), "conv4 at batch 256",
         {"up": {"bf16": "+lean +pair"}, "down": {"bf16": "+dgrad_as_fprop phases=1"}, "outp": {"bf16": "+lean"}}),
    Case("conv5_b128", (128, 14, 14, 384, 512, 3, 3, 1, 1, 0, 0), "conv5, no padding",
         {"up": {"bf16": "+lean +pair"}, "down": {"bf16": "+dgrad_as_fprop phases=1"}, "outp": {"bf16": "+lean"}}),
    Case("fc6_b128", (128, 1, 1, 18432, 4096, 1, 1, 1, 1, 0, 0), "split-K fprop + dgrad; bf16 without staged weights -> tf32",
         {"up": {"tf32": "+split", "bf16": "path=tf32 +split"}, "down": {"tf32": "+split", "bf16": "path=tf32 +split"},
          "outp": {"tf32": "-split", "bf16": "+lean"}}, control=True),
    Case("fc6_b128_staged", (128, 1, 1, 18432, 4096, 1, 1, 1, 1, 0, 0), "fc6 with staged bf16 weights: bf16 split-K",
         {"up": {"bf16": "+split"}, "down": {"bf16": "+split"}, "outp": {"bf16": "+lean"}},
         stage_weights=True, modes=("bf16",)),
    Case("fc8_b128", (128, 1, 1, 4096, 1000, 1, 1, 1, 1, 0, 0), "Cout = 1000, not a multiple of 32",
         {"up": {"tf32": "+split", "bf16": "path=tf32 +split"}, "down": {"tf32": "+split", "bf16": "path=tf32 +split"},
          "outp": {"bf16": "+lean"}}),
    # edges
    Case("n136", (136, 14, 14, 256, 384, 3, 3, 1, 1, 1, 1), "N % 128 != 0: bf16 general kernel, unmerged A",
         {"up": {"bf16": "-lean -a_merged"}, "down": {"bf16": "-dgrad_as_fprop -a_merged"}, "outp": {"bf16": "-lean"}}),
    Case("n132", (132, 14, 14, 256, 384, 3, 3, 1, 1, 1, 1), "N % 8 != 0: bf16 declines, tf32 runs",
         {"up": {"bf16": "path=tf32"}, "down": {"bf16": "path=tf32"}, "outp": {"bf16": "path=tf32"}}),
    Case("conv1_n96", (96, 224, 224, 3, 96, 7, 7, 2, 2, 1, 1), "conv1-like at N = 96: general x-mode",
         {"up": {"tf32": "+xmode -lean", "bf16": "path=tf32 +xmode -lean"},
          "down": {"tf32": "path=simt", "bf16": "path=simt"},
          "outp": {"tf32": "+xmode -lean", "bf16": "path=tf32 +xmode -lean"}}),
    Case("cout96", (128, 27, 27, 64, 96, 5, 5, 2, 2, 1, 1), "Cout = 96: lean fprop without the merged B map",
         {"up": {"bf16": "+lean -b_merged"}, "down": {"bf16": "+dgrad_as_fprop phases=4"}}),
    Case("cin48", (128, 14, 14, 48, 128, 3, 3, 1, 1, 1, 1), "Cin = 48: no dgrad-as-fprop, no lean wgrad",
         {"down": {"bf16": "-dgrad_as_fprop"}, "outp": {"bf16": "-lean"}}),
    Case("pair_below", None, "fprop one pair tile below num_sms/2: single CTA", {"up": {"bf16": "+lean -pair"}}),
    Case("pair_at", None, "fprop at num_sms/2 pair tiles: CTA pair", {"up": {"bf16": "+lean +pair"}}),
    Case("rect", (128, 20, 17, 64, 128, 5, 3, 2, 1, 2, 1), "kx != ky, sx != sy, px != py",
         {"down": {"bf16": "+dgrad_as_fprop phases=2"}}),
    Case("stride_gt_kernel", (128, 16, 16, 64, 64, 2, 2, 3, 3, 0, 0), "phases without taps: dgrad falls back",
         {"down": {"bf16": "-dgrad_as_fprop"}}),
    # accumulation at a pair-mode shape: fprop / dgrad leave the lean paths, wgrad keeps the lean kernel with splits
    Case("conv2_accumulate", (128, 55, 55, 96, 256, 5, 5, 2, 2, 1, 1), "scaleTargets 0.5 / 1, wgrad scaleOutput 1/N",
         {"up": {"bf16": "-lean +pair"}, "down": {"bf16": "-dgrad_as_fprop"}, "outp": {"bf16": "+lean +split"}},
         st=(0.5, 1.0, 1.0), so_outp="1/N"),
    Case("subrange_b128", (128, 14, 14, 256, 384, 3, 3, 1, 1, 1, 1), "input channels [64, 256), output [128, 384)",
         st=(1.0, 0.5, 0.0), sub=(64, 256, 128, 384)),
    # 3-D (C3D conv1a / conv2a, batch 32): frames outermost in the channel axis, per-frame dgrad launches
    Case("c3d_conv1a", (32, 112, 112, 3, 64, 3, 3, 1, 1, 1, 1), "3-D conv1a", {}, T=16, kt=3),
    Case("c3d_conv2a", (32, 56, 56, 64, 128, 3, 3, 1, 1, 1, 1), "3-D conv2a", {}, T=14, kt=3),
]
BY_NAME = {c.name: c for c in CASES}


def _shape(env, case):
    if case.name.startswith("pair_"):
        half = env.sms // 2                 # 1x1, N = 128, Cout = 256 (one n-tile): pair tiles = modules / 2
        modules = 2 * half - (2 if case.name == "pair_below" else 0)
        return (128, modules, 1, 64, 256, 1, 1, 1, 1, 0, 0)
    return case.shape


def _expect(case, op, mode):
    spec = "path=simt" if mode == "fp32" else case.expect.get(op, {}).get(mode, "")
    path, need, absent, phases = PATH[mode], set(), set(), None
    for tok in spec.split():
        if tok.startswith("path="):
            path = PATH[tok[5:]]
        elif tok.startswith("phases="):
            phases = int(tok[7:])
        elif tok[0] == "+":
            need.add(tok[1:])
        elif tok[0] == "-":
            absent.add(tok[1:])
    return path, need, absent, phases


def _variant_errors(env, case, op, mode):
    path, need, absent, phases = _expect(case, op, mode)
    got_path = env.lib.last_conv_path()
    bits, got_phases = env.lib.last_conv_kernel()
    errs = []
    if got_path != path:
        errs.append("path %s, expected %s" % (got_path, path))
    if got_path == "cuda-core-fp32" and bits:
        errs.append("CUDA-core path with kernel bits %s" % sorted(bits))
    if need - bits or absent & bits:
        errs.append("bits %s, expected %s and not %s" % (sorted(bits), sorted(need), sorted(absent)))
    if phases is not None and got_phases != phases:
        errs.append("%d phases, expected %d" % (got_phases, phases))
    return errs, got_path, sorted(bits), got_phases


class Problem:
    """the tensors of one case on the GPU (fp32), in the cudamat layout"""

    def __init__(self, env, case):
        torch = env.torch
        N, W, H, Cin, Cout, ky, kx, sy, sx, py, px = _shape(env, case)
        T, kt = case.T, case.kt
        modY, modX = num_modules(H, ky, sy, py), num_modules(W, kx, sx, px)
        modT = T - kt + 1
        if case.sub:
            c0, c1, o0, o1 = case.sub
            self.d = GetConvDesc(Cin, Cout, ky, kx, sy, sx, py, px, input_channel_begin=c0, input_channel_end=c1,
                                 output_channel_begin=o0, output_channel_end=o1)
            ci, co = c1 - c0, o1 - o0
        else:
            self.d = GetConvDesc(Cin, Cout, ky, kx, sy, sx, py, px, kernel_size_t=kt)
            ci, co = Cin, Cout
        self.three_d = T > 1
        self.N, self.K = N, kx * ky * ci * kt
        self.ish, self.fsh, self.tsh = (N, W, H, Cin * T), (co, kx, ky, ci * kt), (N, modX, modY, Cout * modT)
        self.geo = dict(N=N, W=W, H=H, Cin=Cin, Cout=Cout, kx=kx, ky=ky, sx=sx, sy=sy, px=px, py=py, modX=modX,
                        modY=modY, T=T, kt=kt, co=co, ci=ci)
        g = torch.Generator(device="cuda").manual_seed(zlib.crc32(case.name.encode()))
        M = env.M
        self.x = M(N, W * H * Cin * T, self.ish); self.x.storage.normal_(generator=g)
        self.w = M(co, self.K, self.fsh); self.w.storage.normal_(generator=g).mul_(1.0 / np.sqrt(self.K))
        self.dy = M(N, modX * modY * Cout * modT, self.tsh); self.dy.storage.normal_(generator=g)
        self.g = g

    def target(self, env, rows, cols, sh, st):
        """NaN-poisoned target (scaleTargets = 0) or one holding a random init; returns (matrix, init or None)"""
        m = env.M(rows, cols, sh)
        if st == 0:
            m.fill_(float("nan"))
            return m, None
        m.storage.normal_(generator=self.g)
        return m, m.storage.clone()


def _run_op(env, pb, op, st, so):
    """run one op of the library; returns (output matrix, init)"""
    cg, d = env.cg, pb.d
    three = pb.three_d
    if op == "up":
        out, init = pb.target(env, pb.N, pb.tsh[1] * pb.tsh[2] * pb.tsh[3], pb.tsh, st)
        (cg.convUp3D if three else cg.convUp)(pb.x, pb.w, out, d, st)
    elif op == "down":
        out, init = pb.target(env, pb.N, pb.ish[1] * pb.ish[2] * pb.ish[3], pb.ish, st)
        (cg.convDown3D if three else cg.convDown)(pb.dy, pb.w, out, d, st)
    else:
        out, init = pb.target(env, pb.fsh[0], pb.K, pb.fsh, st)
        (cg.convOutp3D if three else cg.convOutp)(pb.x, pb.dy, out, d, st, so)
    return out, init


def _reference(pb, op, st, so, init, operands, x=None, w=None, dy=None):
    x = pb.x.storage if x is None else x
    w = pb.w.storage if w is None else w
    dy = pb.dy.storage if dy is None else dy
    if op == "up":
        return R.conv_up(x, w, pb.d, pb.ish, pb.fsh, pb.tsh, st, so, init=init, operands=operands)
    if op == "down":
        return R.conv_down(dy, w, pb.d, pb.tsh, pb.fsh, pb.ish, st, so, init=init, operands=operands)
    return R.conv_outp(x, dy, pb.d, pb.ish, pb.tsh, pb.fsh, st, so, init=init, operands=operands)


def _check_against_reference(pb, op, st, so, out, init, path):
    """(ratio, operand emulation, ratios per tf32 emulation or None, (ref, mag))"""
    emu = OPERANDS[path]
    ref_mag = _reference(pb, op, st, so, init, emu)
    q = R.ratio(out.storage, *ref_mag)[0]
    if path != "tcgen05-tf32":
        return q, emu, None, ref_mag
    per = {emu: q}
    for other in TF32_OPERANDS:
        if other != emu:
            ref, mag = _reference(pb, op, st, so, init, other)
            per[other] = R.ratio(out.storage, ref, mag)[0]
            del ref, mag
    return q, emu, per, ref_mag


def _control(env, pb, op, st, so, out, ref_mag, operands):
    """subtract the fp64 contribution of one K slice of 16 terms over one 128-row block from the kernel's result;
    returns the ratio of the doctored result"""
    torch = env.torch
    G = pb.geo
    N, kx, ky, ci, co = G["N"], G["kx"], G["ky"], G["ci"], G["co"]
    mx, my = min(1, G["modX"] - 1), min(1, G["modY"] - 1)
    tx, ty = kx // 2, ky // 2
    m0 = mx + G["modX"] * my
    modules = G["modX"] * G["modY"]
    rows = min(128, N)
    if op == "up":        # K = (tap, channel): tap (tx, ty) x channels [0, 16) ; rows = 128 images at module m0
        wm = torch.zeros_like(pb.w.storage)
        wm.view(ci, ky, kx, co)[:16, ty, tx, :] = pb.w.storage.view(ci, ky, kx, co)[:16, ty, tx, :]
        part, _ = _reference(pb, op, 0.0, so, None, operands, w=wm)
        keep = torch.zeros_like(part, dtype=torch.bool)
        keep.view(co, modules, N)[:, m0, :rows] = True
    elif op == "down":    # K = (tap, output channel): tap (tx, ty) x outputs [0, 16) ; rows = 128 images at one input pixel
        wm = torch.zeros_like(pb.w.storage)
        wm.view(ci, ky, kx, co)[:, ty, tx, :16] = pb.w.storage.view(ci, ky, kx, co)[:, ty, tx, :16]
        part, _ = _reference(pb, op, 0.0, so, None, operands, w=wm)
        X, Y = mx * G["sx"] - G["px"] + tx, my * G["sy"] - G["py"] + ty
        keep = torch.zeros_like(part, dtype=torch.bool)
        keep.view(G["Cin"], G["H"], G["W"], N)[:, Y, X, :rows] = True
    else:                 # K = (image, module): images [0, 16) at module m0 ; rows = output channels [0, 128)
        dym = torch.zeros_like(pb.dy.storage)
        v, s = dym.view(G["Cout"], modules, N), pb.dy.storage.view(G["Cout"], modules, N)
        v[:, m0, :16] = s[:, m0, :16]
        part, _ = _reference(pb, op, 0.0, so, None, operands, dy=dym)
        keep = torch.zeros_like(part, dtype=torch.bool)
        keep.view(ci * ky * kx, co)[:, :min(128, co)] = True
    doctored = out.storage[:part.numel()].double() - torch.where(keep, part, torch.zeros_like(part))
    return R.ratio(doctored, *ref_mag)[0]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_conv_variant_vs_float64(env, name, mode):
    case = BY_NAME[name]
    if mode not in case.modes:
        pytest.skip("the case exists for %s only" % "/".join(case.modes))
    torch, L = env.torch, env.L
    env.lib.set_precision(mode)
    L.convnet_b200_bf16_invalidate(None)
    pb = Problem(env, case)
    errors = []
    try:
        if case.stage_weights:
            L.convnet_b200_bf16_stage(pb.w.ptr, pb.w.storage.numel())
        for op, st in zip(("up", "down", "outp"), case.st):
            so = 1.0 / pb.N if (op == "outp" and case.so_outp == "1/N") else 1.0
            out, init = _run_op(env, pb, op, st, so)
            torch.cuda.synchronize()
            verr, path, bits, phases = _variant_errors(env, case, op, mode)
            q, emu, per, ref_mag = _check_against_reference(pb, op, st, so, out, init, path)
            rec = dict(case=name, op=op, mode=mode, path=path, bits=bits, phases=phases, ratio=q, operands=emu,
                       K=pb.K, why=case.why)
            if per:
                rec["tf32_ratios"] = per
            if case.control and path in THRESH:
                rec["control_ratio"] = qc = _control(env, pb, op, st, so, out, ref_mag, emu)
                if not qc > THRESH[path]:
                    errors.append("%s: negative control ratio %.3g does not exceed the threshold %.3g" % (op, qc, THRESH[path]))
            _RESULTS.append(rec)
            errors += ["%s: %s" % (op, e) for e in verr]
            if not q < THRESH.get(path, 0):
                errors.append("%s: ratio %.3g >= %.3g (%s, %s)" % (op, q, THRESH.get(path, 0), path, emu))
            del out, init, ref_mag
    finally:
        L.convnet_b200_bf16_invalidate(None)
        del pb
        torch.cuda.empty_cache()
    assert not errors, "\n".join(errors)


@pytest.mark.parametrize("mode", MODES)
def test_fused_epilogues_vs_float64(env, mode):
    """conv2 geometry (lean pair fprop, 4-phase dgrad-as-fprop in bf16): bias + ReLU fused into fprop, the ReLU' mask
    fused into the stride-2 dgrad (each phase writes its own pixels), and in bf16 the bf16 twin of the output, which must
    equal the round-to-nearest-even of the fp32 output bit for bit."""
    torch, L, cg = env.torch, env.L, env.cg
    env.lib.set_precision(mode)
    L.convnet_b200_bf16_invalidate(None)
    case = BY_NAME["conv2_b128"]
    pb = Problem(env, case)
    try:
        G = pb.geo
        bias = torch.randn(G["Cout"], device="cuda", generator=pb.g)
        out, _ = pb.target(env, pb.N, pb.tsh[1] * pb.tsh[2] * pb.tsh[3], pb.tsh, 0.0)
        L.convnet_b200_fuse_next(bias.data_ptr(), 1, None)
        if mode == "bf16":
            L.convnet_b200_emit_bf16_next()
        cg.convUp(pb.x, pb.w, out, pb.d)
        torch.cuda.synchronize()
        verr, path, bits, _ = _variant_errors(env, case, "up", mode)
        assert not verr, verr
        pre, mag = _reference(pb, "up", 0.0, 1.0, None, OPERANDS[path])
        b = bias.double().view(G["Cout"], 1).expand(G["Cout"], pb.N * G["modX"] * G["modY"]).reshape(-1)
        pre, mag = pre + b, mag + b.abs()
        ambiguous = pre.abs() <= THRESH[path] * mag      # the clamp there is decided by the accumulation's rounding
        q = R.ratio(out.storage, pre.clamp(min=0), mag, skip=ambiguous)[0]
        _RESULTS.append(dict(case="conv2_bias_relu", op="up", mode=mode, path=path, bits=bits, ratio=q))
        assert q < THRESH[path], q
        if mode == "bf16":                                  # the twin, read through a 1x1 identity conv (one exact term)
            C, n_out = G["Cout"], out.storage.numel()
            assert L.convnet_b200_bf16_is_staged(out.ptr, n_out) == 1
            eye = env.M(C, C, (C, 1, 1, C)); eye.storage.copy_(torch.eye(C, device="cuda").reshape(-1))
            d1 = GetConvDesc(C, C, 1, 1, 1, 1, 0, 0)
            sh = (pb.N, G["modX"], G["modY"], C)
            twin = env.M(pb.N, G["modX"] * G["modY"] * C, sh); twin.fill_(float("nan"))
            cg.convUp(out, eye, twin, d1)
            assert env.lib.last_conv_path() == "tcgen05-bf16"
            want = out.storage.to(torch.bfloat16).float()
            assert torch.equal(twin.storage, want), int((twin.storage != want).sum())
        # dgrad with the ReLU' mask of the layer below
        state = torch.randn(pb.ish[1] * pb.ish[2] * pb.ish[3] * pb.N, device="cuda", generator=pb.g)
        dn, _ = pb.target(env, pb.N, pb.ish[1] * pb.ish[2] * pb.ish[3], pb.ish, 0.0)
        L.convnet_b200_fuse_next(None, 0, state.data_ptr())
        cg.convDown(pb.dy, pb.w, dn, pb.d)
        torch.cuda.synchronize()
        verr, path, bits, phases = _variant_errors(env, case, "down", mode)
        assert not verr, verr
        ref, mag = _reference(pb, "down", 0.0, 1.0, None, OPERANDS[path])
        ref = torch.where(state.double() > 0, ref, torch.zeros_like(ref))
        q = R.ratio(dn.storage, ref, mag)[0]
        _RESULTS.append(dict(case="conv2_relu_mask", op="down", mode=mode, path=path, bits=bits, phases=phases, ratio=q))
        assert q < THRESH[path], q
    finally:
        L.convnet_b200_bf16_invalidate(None)
        del pb
        torch.cuda.empty_cache()


def test_dgrad_banks_follow_weights_written_outside_the_library(env):
    """bf16 dgrad-as-fprop derives per-phase filter banks from the weights.  A caller that updates its weights with its own
    code (the original project's trainer: its own optimizer, then ConvDown with scale_targets = 0) must get the dgrad
    of the NEW weights from the next call, without any invalidation call in between."""
    torch, L, cg = env.torch, env.L, env.cg
    env.lib.set_precision("bf16")
    L.convnet_b200_bf16_invalidate(None)
    pb = Problem(env, BY_NAME["conv2_b128"])
    try:
        for step in range(2):
            if step:
                pb.w.storage.copy_(torch.randn(pb.w.storage.numel(), device="cuda", generator=pb.g) / np.sqrt(pb.K))
            out, _ = pb.target(env, pb.N, pb.ish[1] * pb.ish[2] * pb.ish[3], pb.ish, 0.0)
            cg.convDown(pb.dy, pb.w, out, pb.d, 0)
            torch.cuda.synchronize()
            bits, phases = env.lib.last_conv_kernel()
            assert "dgrad_as_fprop" in bits and phases == 4
            ref, mag = _reference(pb, "down", 0.0, 1.0, None, "bf16")
            q = R.ratio(out.storage, ref, mag)[0]
            assert q < THRESH["tcgen05-bf16"], (step, q)
    finally:
        L.convnet_b200_bf16_invalidate(None)
        del pb
        torch.cuda.empty_cache()

