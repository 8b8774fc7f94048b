"""Float64 reference of the conv ops in the cudamat layout (torch, CPU or CUDA).

    conv_up(images, filters, d, ish, fsh, tsh, ...)      convUp / convUp3D
    conv_down(derivs, filters, d, dsh, fsh, tsh, ...)    convDown / convDown3D
    conv_outp(images, derivs, d, ish, dsh, tsh, ...)     convOutp / convOutp3D

Arguments follow oracle_lib.Oracle: tensors are flat (a CUDAMatrix's storage, or a Fortran-ordered numpy matrix), shapes
are the Shape4D tuples, `d` is a ConvDesc.  The layout is that of csrc/geom.h and oracle/conv_oracle.c:
    image   [n + N*(x + W*(y + H*(c + C*t)))]        (3-D: frames outermost in the channel axis)
    filter  [o + Cout*(tx + kx*(ty + ky*(c + Cin*dt)))]
    module m = (mx, my) reads the window starting at (mx*sx - px, my*sy - py); mod counts come from the target shape.
Channel sub-ranges of the descriptor (2-D): fprop reads input channels [cin0, cin1) and writes output channels
[cout0, cout1), leaving the rest of the target as it was; dgrad scales the WHOLE target by scaleTargets first, as the
reference does; wgrad reads both sub-ranges.

Each op returns (ref, mag), float64, flat in the layout of the target: ref is the exact result of the operands as the
kernel sees them, mag the same op applied to |operands| plus |scaleTargets * init|.  `operands` says how the kernel
converts its fp32 operands (see emulate): with the conversion emulated, what remains between a correct kernel and `ref`
is the rounding of its fp32 accumulation, which is bounded relative to `mag`; ratio() measures it.
"""
import numpy as np
import torch
import torch.nn.functional as Fn

OPERAND_MODES = ("fp32", "bf16", "tf32_rne", "tf32_trunc")


def flat(a, device=None):
    """a 1-D float32 torch tensor with the elements of `a` in cudamat order"""
    if isinstance(a, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float32).ravel(order="F")))
    else:
        t = a.reshape(-1)
    return t if device is None else t.to(device)


def emulate(t, mode):
    """fp32 operand values as the kernel multiplies them, as float64.
    fp32: as given (CUDA-core fp32 FMA).  bf16: round to nearest even to 8 mantissa bits (__float2bfloat16_rn, which is
    also what torch's conversion does).  tf32_rne / tf32_trunc: 10 mantissa bits, rounded to nearest even / truncated."""
    t = t.to(torch.float32)
    if mode == "fp32":
        pass
    elif mode == "bf16":
        t = t.to(torch.bfloat16).to(torch.float32)
    elif mode in ("tf32_rne", "tf32_trunc"):
        u = t.contiguous().view(torch.int32)
        if mode == "tf32_rne":
            u = u + (0xFFF + ((u >> 13) & 1))
        t = (u & ~0x1FFF).view(torch.float32)
    else:
        raise ValueError(mode)
    return t.to(torch.float64)


class _Geo:
    def __init__(self, d, ish, osh):
        """ish: the image-side Shape4D, osh: the output (module) side"""
        self.N, self.W, self.H = ish[0], ish[1], ish[2]
        self.CinT, self.CoutT = d.num_input_channels, d.num_output_channels
        self.cin0, self.cout0 = d.input_channel_begin, d.output_channel_begin
        self.Cin = (d.input_channel_end or self.CinT) - self.cin0
        self.Cout = (d.output_channel_end or self.CoutT) - self.cout0
        self.kx, self.ky, self.kt = d.kernel_size_x, d.kernel_size_y, max(d.kernel_size_t, 1)
        self.sx, self.sy, self.st = d.stride_x, d.stride_y, max(d.stride_t, 1)
        self.px, self.py = -d.padding_x, -d.padding_y
        assert d.padding_t == 0 and self.px >= 0 and self.py >= 0
        assert ish[3] % self.CinT == 0 and osh[3] % self.CoutT == 0 and osh[0] == self.N
        self.T, self.modT = ish[3] // self.CinT, osh[3] // self.CoutT
        self.modX, self.modY = osh[1], osh[2]
        if self.T > 1 or self.kt > 1:
            assert self.Cin == self.CinT and self.Cout == self.CoutT, "3-D: channel sub-ranges are not supported"
        self.img_n = self.N * self.W * self.H * self.CinT * self.T
        self.out_n = self.N * self.modX * self.modY * self.CoutT * self.modT
        self.flt_n = self.Cout * self.kx * self.ky * self.Cin * self.kt

    # flat cudamat tensors <-> conv3d's (N, C, D, H, W)
    def images(self, x):
        return x.view(self.T, self.CinT, self.H, self.W, self.N).permute(4, 1, 0, 2, 3)[:, self.cin0:self.cin0 + self.Cin]

    def outputs(self, y):
        return y.view(self.modT, self.CoutT, self.modY, self.modX, self.N).permute(4, 1, 0, 2, 3)[
            :, self.cout0:self.cout0 + self.Cout]

    def filters(self, w):
        return w.view(self.kt, self.Cin, self.ky, self.kx, self.Cout).permute(4, 1, 0, 2, 3)

    def forward(self, x, w):
        """x: (N, Cin, T, H, W), w: (Cout, Cin, kt, ky, kx) -> (N, Cout, modT, modY, modX)"""
        rx = max(0, (self.modX - 1) * self.sx + self.kx - self.px - self.W)
        ry = max(0, (self.modY - 1) * self.sy + self.ky - self.py - self.H)
        x = Fn.pad(x, (self.px, rx, self.py, ry))
        if self.T == 1 and self.kt == 1:                      # 2-D: conv2d, which every backend has in float64
            y = Fn.conv2d(x[:, :, 0], w[:, :, 0], stride=(self.sy, self.sx)).unsqueeze(2)
        else:
            y = Fn.conv3d(x, w, stride=(self.st, self.sy, self.sx))
        assert y.shape[2] >= self.modT and y.shape[3] >= self.modY and y.shape[4] >= self.modX, (y.shape, self.modX)
        return y[:, :, :self.modT, :self.modY, :self.modX]


def _f64(a, n, mode, device):
    t = flat(a, device)
    assert t.numel() >= n, (t.numel(), n)
    return emulate(t[:n], mode)


def _init(init, n, device):
    return torch.zeros(n, dtype=torch.float64, device=device) if init is None else flat(init, device)[:n].double()


def conv_up(images, filters, d, ish, fsh, tsh, scaleTargets=0.0, scaleOutput=1.0, init=None, operands="fp32",
            device=None):
    g = _Geo(d, ish, tsh)
    assert tuple(fsh) == (g.Cout, g.kx, g.ky, g.Cin * g.kt), (fsh, g.Cout, g.Cin)
    x, w = _f64(images, g.img_n, operands, device), _f64(filters, g.flt_n, operands, device)
    t0 = _init(init, g.out_n, x.device)
    res = []
    for xx, ww, s, so, base in ((x, w, scaleTargets, scaleOutput, t0),
                                (x.abs(), w.abs(), abs(scaleTargets), abs(scaleOutput), t0.abs())):
        y = so * g.forward(g.images(xx), g.filters(ww))
        out = base.clone()                                   # channels outside the output sub-range stay as they were
        g.outputs(out).copy_(y if s == 0 else s * g.outputs(base) + y)
        res.append(out)
    return res[0], res[1]


def conv_down(derivs, filters, d, dsh, fsh, tsh, scaleTargets=0.0, scaleOutput=1.0, init=None, operands="fp32",
              device=None):
    g = _Geo(d, tsh, dsh)
    assert tuple(fsh) == (g.Cout, g.kx, g.ky, g.Cin * g.kt), (fsh, g.Cout, g.Cin)
    dy, w = _f64(derivs, g.out_n, operands, device), _f64(filters, g.flt_n, operands, device)
    t0 = _init(init, g.img_n, dy.device)
    res = []
    for yy, ww, s, so, base in ((dy, w, scaleTargets, scaleOutput, t0),
                                (dy.abs(), w.abs(), abs(scaleTargets), abs(scaleOutput), t0.abs())):
        x0 = torch.zeros_like(g.images(base), requires_grad=True)
        (gx,) = torch.autograd.grad(g.forward(x0, g.filters(ww)), x0, g.outputs(yy))
        out = s * base if s != 0 else torch.zeros_like(base)   # the WHOLE target is scaled (cpumat_conv.cc:304-307)
        g.images(out).add_(so * gx)
        res.append(out)
    return res[0], res[1]


def conv_outp(images, derivs, d, ish, dsh, tsh, scaleTargets=0.0, scaleOutput=1.0, init=None, operands="fp32",
              device=None):
    g = _Geo(d, ish, dsh)
    assert tuple(tsh) == (g.Cout, g.kx, g.ky, g.Cin * g.kt), (tsh, g.Cout, g.Cin)
    x, dy = _f64(images, g.img_n, operands, device), _f64(derivs, g.out_n, operands, device)
    t0 = _init(init, g.flt_n, x.device)
    res = []
    for xx, yy, s, so, base in ((x, dy, scaleTargets, scaleOutput, t0),
                                (x.abs(), dy.abs(), abs(scaleTargets), abs(scaleOutput), t0.abs())):
        w0 = torch.zeros_like(g.filters(base), requires_grad=True)
        (gw,) = torch.autograd.grad(g.forward(g.images(xx), w0), w0, g.outputs(yy))
        out = s * base if s != 0 else torch.zeros_like(base)
        g.filters(out).add_(so * gw)
        res.append(out)
    return res[0], res[1]


def ratio(ours, ref, mag, skip=None):
    """(max_i |ours_i - ref_i| / (mag_i + tiny), argmax i) over every element; non-finite values of `ours` count as
    infinitely wrong.  `skip`: boolean mask of elements left out (e.g. a fused ReLU's clamp decided by rounding)."""
    o = flat(ours, ref.device).double()
    r = (o - ref).abs() / (mag + torch.finfo(torch.float64).tiny)
    r = torch.where(torch.isfinite(o), r, torch.full_like(r, float("inf")))
    if skip is not None:
        r = torch.where(skip, torch.zeros_like(r), r)
    i = int(torch.argmax(r))
    return float(r[i]), i
