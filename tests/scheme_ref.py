"""Float64 emulation of the tensor-core split-precision schemes (CPU): one statement of the operand planes and of the partial
products each scheme sums, so that a kernel can be compared with its own scheme instead of only with the exact result.

TEST INFRASTRUCTURE (imports oracle/).  Used by tests/test_scheme_ref.py (CPU), tests/test_gpu_schemes.py (B200) and
tests/precision_study.py.

Planes (kernels.cuh, cgvc_quant4; simt_kernels.cu, pad_split / st4_quant; tc_gemm.cu, prep_weights_*):
    bf16x3   hi = bf16(x), lo = bf16(x - hi)                      products hi*hi + hi*lo + lo*hi
    f16f8    q16 = fp16(x), q8hi = e4m3(sat(q16 * S_hi)), q8lo = e4m3(sat((x - q16) * S_lo))
             products q16*q16 + q8hi_a*q8lo_b + q8lo_a*q8hi_b, every plane divided back by its scale
             activations and gradients (S_hi, S_lo) = (1, 2^12), weights (2^3, 2^15); sat = clamp(+-448) (__NV_SATFINITE)
    fp16     q16 only (the `wgrad_f16` weight gradient of an F16F8 engine)
Every plane function returns its parts already divided back, so that the sum of the partial products is the emulated value.
"""
from __future__ import annotations

import contextlib

import torch

from oracle import cyclegan_oracle as O

F64 = torch.float64
E4 = torch.float8_e4m3fn
E4_MAX = 448.0
ROLE_SCALES = {"act": (1.0, 4096.0), "weight": (8.0, 32768.0)}      # CGVC_Q_ACT_SHI/SLO, CGVC_Q_W_SHI/SLO
# broken versions of the schemes, each emulated the way a kernel with that defect would compute
MUTANTS = {
    "bf16x3": ("no_lo_hi",),
    "f16f8": ("no_a8hi_b8lo", "no_a8lo_b8hi", "fp16_only", "act_lo_scale_half"),
}


def rn(x, dt):
    """round to dt (nearest even) and back to float64"""
    return x.to(dt).to(F64)


def e4m3(x):
    """saturating e4m3 (what __nv_cvt_float2_to_fp8x2(..., __NV_SATFINITE, __NV_E4M3) stores), as float64"""
    return rn(x.clamp(-E4_MAX, E4_MAX), E4)


def planes_bf16x3(x):
    """(hi, lo): hi = bf16(x), lo = bf16(x - hi)"""
    x = x.to(F64)
    h = rn(x, torch.bfloat16)
    return h, rn(x - h, torch.bfloat16)


def planes_fp16(x):
    return rn(x.to(F64), torch.float16)


def planes_f16f8(x, role, lo_write_scale=None):
    """(q16, q8hi, q8lo), the e4m3 planes divided back by their scales.  role: "act" (activations and gradients) or "weight".
    lo_write_scale: the scale the lo plane is written with, if not the one it is read back with (a defective plane writer)."""
    s_hi, s_lo = ROLE_SCALES[role]
    x = x.to(F64)
    h = rn(x, torch.float16)
    return h, e4m3(h * s_hi) / s_hi, e4m3((x - h) * (lo_write_scale or s_lo)) / s_lo


def terms(a, b, scheme, roles=("act", "weight"), mutant=None):
    """(A part, B part) pairs whose products the scheme sums.  roles: the F16F8 roles of a and b -- forward (act, weight), data
    gradient (gradient = act, weight), weight gradient (act, gradient = act)."""
    if scheme == "exact":
        return [(a, b)]
    if scheme == "bf16x3":
        (ah, al), (bh, bl) = planes_bf16x3(a), planes_bf16x3(b)
        t = [(ah, bh), (ah, bl), (al, bh)]
        if mutant == "no_lo_hi":
            t.pop(2)
        return t
    if scheme in ("f16f8", "f16f8_w16"):
        if scheme == "f16f8_w16" or mutant == "fp16_only":
            return [(planes_fp16(a), planes_fp16(b))]
        half = lambda r: ROLE_SCALES[r][1] / 2 if (mutant == "act_lo_scale_half" and r == "act") else None
        a16, a8h, a8l = planes_f16f8(a, roles[0], half(roles[0]))
        b16, b8h, b8l = planes_f16f8(b, roles[1], half(roles[1]))
        t = [(a16, b16), (a8h, b8l), (a8l, b8h)]
        if mutant == "no_a8hi_b8lo":
            t.pop(1)
        elif mutant == "no_a8lo_b8hi":
            t.pop(2)
        return t
    raise ValueError(scheme)


def bilinear(fn, a, b, scheme, roles, mutant=None):
    out = None
    for x, y in terms(a, b, scheme, roles, mutant):
        t = fn(x, y)
        out = t if out is None else out + t
    return out


# ---- single convolutions: channels-last, TF SAME, the argument order of cgvc_conv_forward / cgvc_conv_backward ----------------
def _fwd(x, w, sh, sw):
    return O.conv2d_same(x, w, None, (sh, sw))


def _dgrad(xshape, sh, sw):
    def f(g, w):
        x0 = torch.zeros(xshape, dtype=F64, requires_grad=True)
        return torch.autograd.grad(O.conv2d_same(x0, w, None, (sh, sw)), x0, g)[0]
    return f


def _wgrad(wshape, sh, sw):
    def f(x, g):
        w0 = torch.zeros(wshape, dtype=F64, requires_grad=True)
        return torch.autograd.grad(O.conv2d_same(x, w0, None, (sh, sw)), w0, g)[0]
    return f


def emulate_conv_fwd(x, w, dy, B, H, W, Cin, kh, kw, Cout, sh, sw, scheme, mutant=None):
    """y = conv(x, w) without bias, [B, Hy, Wy, Cout] (dy unused: the common signature of the three)"""
    x, w = x.to(F64).reshape(B, H, W, Cin), w.to(F64).reshape(kh, kw, Cin, Cout)
    s = "f16f8" if scheme == "f16f8_w16" else scheme
    with torch.no_grad():
        return bilinear(lambda a, b: _fwd(a, b, sh, sw), x, w, s, ("act", "weight"), mutant)


def emulate_conv_dgrad(x, w, dy, B, H, W, Cin, kh, kw, Cout, sh, sw, scheme, mutant=None):
    """dx = d<dy, conv(x, w)>/dx, [B, H, W, Cin]; the gradient takes the activation-role planes"""
    w = w.to(F64).reshape(kh, kw, Cin, Cout)
    s = "f16f8" if scheme == "f16f8_w16" else scheme
    return bilinear(_dgrad((B, H, W, Cin), sh, sw), dy.to(F64), w, s, ("act", "weight"), mutant)


def emulate_conv_wgrad(x, w, dy, B, H, W, Cin, kh, kw, Cout, sh, sw, scheme, mutant=None):
    """dw = d<dy, conv(x, w)>/dw, [kh, kw, Cin, Cout]; both operands take the activation-role planes (f16f8_w16: fp16 planes alone)"""
    x = x.to(F64).reshape(B, H, W, Cin)
    return bilinear(_wgrad((kh, kw, Cin, Cout), sh, sw), x, dy.to(F64), scheme, ("act", "act"), mutant)


def emulate_conv_f32(x, w, dy, B, H, W, Cin, kh, kw, Cout, sh, sw, scheme):
    """the float32 accumulation floor: the scheme's rounded operands, each partial product through a float32 convolution and
    the partial products summed in float32.  Returns (y, dx, dw)."""
    x = x.to(F64).reshape(B, H, W, Cin); w = w.to(F64).reshape(kh, kw, Cin, Cout); dy = dy.to(F64)
    f32 = torch.float32
    fw = lambda a, b: _fwd(a.to(f32), b.to(f32), sh, sw)

    def dg(g, ww):
        x0 = torch.zeros((B, H, W, Cin), dtype=f32, requires_grad=True)
        return torch.autograd.grad(O.conv2d_same(x0, ww.to(f32), None, (sh, sw)), x0, g.to(f32))[0]

    def wg(xx, g):
        w0 = torch.zeros((kh, kw, Cin, Cout), dtype=f32, requires_grad=True)
        return torch.autograd.grad(O.conv2d_same(xx.to(f32), w0, None, (sh, sw)), w0, g.to(f32))[0]
    sf = "f16f8" if scheme == "f16f8_w16" else scheme
    with torch.no_grad():
        y = bilinear(fw, x, w, sf, ("act", "weight"))
    dx = bilinear(dg, dy, w, sf, ("act", "weight"))
    dw = bilinear(wg, x, dy, scheme, ("act", "act"))
    return y.to(F64), dx.to(F64), dw.to(F64)


# ---- whole model: the oracle with every tensor-core convolution replaced by the scheme ------------------------------------
class _EmuConv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, nd, stride, cfg):
        ctx.save_for_backward(x, w); ctx.nd = nd; ctx.stride = stride; ctx.cfg = cfg
        conv = torch.nn.functional.conv1d if nd == 1 else torch.nn.functional.conv2d
        return bilinear(lambda a, b: conv(a, b, None, stride=stride), x.detach(), w.detach(), cfg["fwd"], ("act", "weight"), cfg["mutant"])

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        nd, stride, cfg = ctx.nd, ctx.stride, ctx.cfg
        G = torch.nn.grad
        gi = (lambda g, ww: G.conv1d_input(x.shape, ww, g, stride=stride)) if nd == 1 else (lambda g, ww: G.conv2d_input(x.shape, ww, g, stride=stride))
        gw = (lambda xx, g: G.conv1d_weight(xx, w.shape, g, stride=stride)) if nd == 1 else (lambda xx, g: G.conv2d_weight(xx, w.shape, g, stride=stride))
        ls = cfg["loss_scale"]
        g = gy.contiguous() * ls             # the engine's gradients carry the loss scale where they are split into planes
        dx = bilinear(gi, g, w.detach(), cfg["dgrad"], ("act", "weight"), cfg["mutant"]) / ls
        dw = bilinear(gw, x.detach(), g, cfg["wgrad"], ("act", "act"), cfg["mutant"]) / ls
        return dx, dw, None, None, None


@contextlib.contextmanager
def emulated_oracle(scheme, loss_scale=1.0, wgrad16=False, mutant=None):
    """O.conv1d_same / O.conv2d_same replaced by the scheme inside the block.  Convolutions with one input channel (the
    discriminator's input layer, which the engine runs in float32 SIMT) stay exact; so does the dense head (not a convolution)."""
    cfg = {"fwd": scheme, "dgrad": scheme, "wgrad": "f16f8_w16" if (scheme == "f16f8" and wgrad16) else scheme,
           "loss_scale": loss_scale if scheme == "f16f8" else 1.0, "mutant": mutant}
    orig1, orig2 = O.conv1d_same, O.conv2d_same

    def conv1d_same(x, kernel, bias, stride=1):
        k = kernel.shape[0]
        pl, pr = O.same_pad(x.shape[1], k, stride)
        xt = torch.nn.functional.pad(x.transpose(1, 2), (pl, pr))
        y = _EmuConv.apply(xt.contiguous(), kernel.permute(2, 1, 0).contiguous(), 1, stride, cfg) + bias.view(1, -1, 1)
        return y.transpose(1, 2)

    def conv2d_same(x, kernel, bias, strides):
        if kernel.shape[2] == 1:
            return orig2(x, kernel, bias, strides)
        kh, kw = kernel.shape[0], kernel.shape[1]
        pt, pb = O.same_pad(x.shape[1], kh, strides[0])
        pl, pr = O.same_pad(x.shape[2], kw, strides[1])
        xt = torch.nn.functional.pad(x.permute(0, 3, 1, 2), (pl, pr, pt, pb))
        y = _EmuConv.apply(xt.contiguous(), kernel.permute(3, 2, 0, 1).contiguous(), 2, tuple(strides), cfg) + bias.view(1, -1, 1, 1)
        return y.permute(0, 2, 3, 1)

    O.conv1d_same, O.conv2d_same = conv1d_same, conv2d_same
    try:
        yield
    finally:
        O.conv1d_same, O.conv2d_same = orig1, orig2


def rel_l2(a, b):
    a = torch.as_tensor(a, dtype=F64).reshape(-1); b = torch.as_tensor(b, dtype=F64).reshape(-1)
    n = float(b.norm())
    return float((a - b).norm()) / n if n > 0 else float((a - b).norm())
