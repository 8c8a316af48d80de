#!/usr/bin/env python
"""Offline numerical study (CPU, float64 emulation): which split-precision schemes for the tensor-core products stay
inside the 1e-3 parity budget (BASELINE.json north_star), and what they cost in tcgen05 MMA issue slots.

TEST INFRASTRUCTURE (imports oracle/): run by hand, results quoted in DESIGN.md section 10.  Nothing in the product
imports this.

Every convolution of the oracle graph (forward, data gradient, weight gradient) is replaced by an emulation of

    D = sum over the scheme's MMA terms of  q_a(A_part) * q_b(B_part)      (exact products, float64 accumulation)

where the parts are the hi / lo splits the kernels keep as planes in HBM.  Cost unit: one bf16/fp16 MMA of the tile = 1,
one fp8 (kind::f8f6f4) MMA = 0.5, one tf32 MMA = 2.

    python tests/precision_study.py [--batch 1] [--schemes bf16x3,bf16_f8,...]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import cyclegan_oracle as O  # noqa: E402
from scheme_ref import F64, planes_bf16x3, planes_f16f8, rn  # noqa: E402  (the engine's plane definitions, stated once)


def q_tf32(x):
    """round-to-nearest-even to 10 explicit mantissa bits (what a pre-rounded TF32 operand holds)."""
    xi = x.to(torch.float32).view(torch.int32)
    r = ((xi >> 13) & 1) + 0x0FFF
    return ((xi + r) & ~0x1FFF).view(torch.float32).to(F64)


def pow2_scale(x, target_max):
    """per-tensor power-of-two scale s with max|x*s| <= target_max (what a dynamic per-tensor amax would give)."""
    m = float(x.abs().max())
    if m == 0.0:
        return 1.0
    import math
    return 2.0 ** math.floor(math.log2(target_max / m))


def q8(x, dt, target):
    s = pow2_scale(x, target)
    return rn((x * s).clamp(-target, target), dt) / s


E4, E5 = torch.float8_e4m3fn, torch.float8_e5m2


def split(x, hi_dt):
    h = rn(x, hi_dt)
    return h, x - h


LOSS_SCALE = 1.0      # fp16_f8_train: every upstream gradient is multiplied by this before it is split into planes (and the result divided)


def _q_act(x):
    """activation-role planes: q16, e4m3(q16), e4m3(lo * 2^12) -> (hi16, hi8, lo8 already divided back)"""
    return planes_f16f8(x, "act")


def _q_w(x):
    """weight-role planes: q16, e4m3(q16 * 2^3), e4m3(lo * 2^15)"""
    return planes_f16f8(x, "weight")


def terms(a, b, scheme, role="fwd"):
    """list of (A_part, B_part) pairs whose products are summed; a, b float64."""
    if scheme in ("fp16_f8_train", "fp16_f8_train_w16"):
        # whole-step variant (DESIGN.md 10, round-2 item 2).  Activations AND gradients use the activation-role scales (1, 2^12), weights
        # (2^3, 2^15): forward and data gradient fold 2^15 out of the accumulator, the weight gradient (activation x gradient) 2^12.
        # role: fwd = (activation, weight), dgrad = (gradient, weight), wgrad = (activation, gradient)
        ah, ah8, al8 = _q_act(a)
        bh, bh8, bl8 = _q_act(b) if role == "wgrad" else _q_w(b)
        if role == "wgrad" and scheme == "fp16_f8_train_w16":     # weight gradients are leaves of the graph: one fp16 MMA, no cross terms
            return [(ah, bh)]
        return [(ah, bh), (ah8, bl8), (al8, bh8)]
    if scheme == "exact":
        return [(a, b)]
    if scheme == "bf16":
        return [(rn(a, torch.bfloat16), rn(b, torch.bfloat16))]
    if scheme == "fp16":
        return [(rn(a, torch.float16), rn(b, torch.float16))]
    if scheme == "tf32":
        return [(q_tf32(a), q_tf32(b))]
    if scheme == "bf16x3":                       # the engine's current mode: hi*hi + hi*lo + lo*hi, lo kept in bf16
        (ah, al), (bh, bl) = planes_bf16x3(a), planes_bf16x3(b)
        return [(ah, bh), (ah, bl), (al, bh)]
    if scheme == "fp16x2":                       # A exact to 22 bits, B rounded to fp16: (ah+al)*bh
        ah, al = split(a, torch.float16); bh = rn(b, torch.float16)
        return [(ah, bh), (rn(al, torch.float16), bh)]
    if scheme in ("bf16_f8", "fp16_f8", "bf16_f8e5", "fp16_f8e5"):
        # hi*hi in 16 bit (1 unit) + the two cross terms in fp8 (0.5 unit each); per-tensor power-of-two scales
        hi_dt = torch.bfloat16 if scheme.startswith("bf16") else torch.float16
        lo_dt = E5 if scheme.endswith("e5") else E4
        tgt = 57344.0 if lo_dt is E5 else 448.0
        ah, al = split(a, hi_dt); bh, bl = split(b, hi_dt)
        return [(ah, bh), (q8(ah, E4, 448.0), q8(bl, lo_dt, tgt)), (q8(al, lo_dt, tgt), q8(bh, E4, 448.0))]
    if scheme == "fp16_f8_static":
        # the forward-pass variant sketched in DESIGN.md 10: STATIC power-of-two scales (no amax pass):
        #   a_hi8 = e4m3(a_hi), b_lo8 = e4m3(b_lo * 2^15);  a_lo8 = e4m3(a_lo * 2^12), b_hi8 = e4m3(b_hi * 2^3); both products * 2^-15
        ah, ah8, al8 = _q_act(a)
        bh, bh8, bl8 = _q_w(b)
        return [(ah, bh), (ah8, bl8), (al8, bh8)]
    raise ValueError(scheme)


COST = {"exact": None, "bf16": 1, "fp16": 1, "tf32": 2, "bf16x3": 3, "fp16x2": 2, "bf16_f8": 2, "fp16_f8": 2, "bf16_f8e5": 2, "fp16_f8e5": 2, "fp16_f8_static": 2, "fp16_f8_train": 2, "fp16_f8_train_w16": 1.75}
SCHEME = "exact"


def bilinear(fn, a, b, role="fwd"):
    a, b = a.detach(), b.detach()
    back = 1.0
    if SCHEME.startswith("fp16_f8_train") and role != "fwd":       # global loss scaling: the gradient operand is a (dgrad) or b (wgrad)
        if role == "dgrad":
            a = a * LOSS_SCALE
        else:
            b = b * LOSS_SCALE
        back = 1.0 / LOSS_SCALE
    out = None
    for (x, y) in (terms(a, b, SCHEME, role) if SCHEME.startswith("fp16_f8_train") else terms(a, b, SCHEME)):
        t = fn(x, y)
        out = t if out is None else out + t
    return out * back if back != 1.0 else out


class EmuConv(torch.autograd.Function):
    """y = conv(x, w) (+ bias outside); forward, dgrad and wgrad each evaluated with the scheme's split products."""

    @staticmethod
    def forward(ctx, x, w, nd, stride):
        ctx.save_for_backward(x, w); ctx.nd = nd; ctx.stride = stride
        conv = F.conv1d if nd == 1 else F.conv2d
        return bilinear(lambda a, b: conv(a, b, None, stride=stride), x, w)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        nd, stride = ctx.nd, ctx.stride
        if nd == 1:
            gi = lambda g, ww: torch.nn.grad.conv1d_input(x.shape, ww, g, stride=stride)
            gw = lambda xx, g: torch.nn.grad.conv1d_weight(xx, w.shape, g, stride=stride)
        else:
            gi = lambda g, ww: torch.nn.grad.conv2d_input(x.shape, ww, g, stride=stride)
            gw = lambda xx, g: torch.nn.grad.conv2d_weight(xx, w.shape, g, stride=stride)
        gy = gy.contiguous()
        return bilinear(gi, gy, w, "dgrad"), bilinear(gw, x, gy, "wgrad"), None, None


def conv1d_same(x, kernel, bias, stride=1):
    k = kernel.shape[0]
    pl, pr = O.same_pad(x.shape[1], k, stride)
    xt = F.pad(x.transpose(1, 2), (pl, pr))
    y = EmuConv.apply(xt.contiguous(), kernel.permute(2, 1, 0).contiguous(), 1, stride) + bias.view(1, -1, 1)
    return y.transpose(1, 2)


def conv2d_same(x, kernel, bias, strides):
    kh, kw = kernel.shape[0], kernel.shape[1]
    pt, pb = O.same_pad(x.shape[1], kh, strides[0])
    pl, pr = O.same_pad(x.shape[2], kw, strides[1])
    xt = F.pad(x.permute(0, 3, 1, 2), (pl, pr, pt, pb))
    y = EmuConv.apply(xt.contiguous(), kernel.permute(3, 2, 0, 1).contiguous(), 2, tuple(strides)) + bias.view(1, -1, 1, 1)
    return y.permute(0, 2, 3, 1)


def rel(a, b):
    d = float((a - b).norm()); n = float(b.norm())
    return d / n if n > 0 else d


FORWARD_ONLY = False


def run(scheme, A, B, P):
    global SCHEME
    SCHEME = scheme
    taps = {}
    with torch.no_grad():
        y = O.generator_forward(A, P, "generator_A2B", taps)
        if FORWARD_ONLY:
            y2 = O.generator_forward(y, P, "generator_B2A")          # a cycle pass: 58 convolutions deep
            return {"gen_out": y, "taps": taps, "cycle_out": y2}
    L, G, gA, gB = O.gradients(A, B, P, 10.0, 5.0)
    return {"gen_out": y, "taps": taps, "L": L, "G": G}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--schemes", default="bf16x3,fp16_f8,bf16_f8,fp16_f8e5,fp16x2,tf32,fp16,bf16")
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--loss-scales", default="", help="for fp16_f8_train: comma-separated log2 loss scales to sweep (the scheme is run once per value)")
    ap.add_argument("--forward-only", action="store_true", help="generator forward (and the taps) only: for schemes that only make sense on the forward pass")
    a = ap.parse_args()
    global FORWARD_ONLY
    FORWARD_ONLY = a.forward_only
    if a.threads:
        torch.set_num_threads(a.threads)
    P = O.init_params(seed=3, dtype=F64, perturb_affine=True)
    A, B = O.synthetic_batch(seed=5, batch=a.batch, frames=128, dtype=F64)
    orig = (O.conv1d_same, O.conv2d_same)
    ref = run("exact", A, B, P)                               # stock oracle convolutions, float64
    O.conv1d_same, O.conv2d_same = conv1d_same, conv2d_same
    chk = run("exact", A, B, P)                               # the emulation harness itself must be exact
    if FORWARD_ONLY:
        for sname in a.schemes.split(","):
            r = run(sname, A, B, P)
            print(json.dumps({"scheme": sname, "mma_units": COST[sname], "gen_h1": rel(r["taps"]["h1_glu"], ref["taps"]["h1_glu"]),
                              "gen_r6": rel(r["taps"]["r6"], ref["taps"]["r6"]), "gen_out": rel(r["gen_out"], ref["gen_out"]),
                              "cycle_out": rel(r["cycle_out"], ref["cycle_out"])}))
        O.conv1d_same, O.conv2d_same = orig
        return
    print("harness self-check (exact scheme vs stock oracle): gen_out %.1e, worst grad %.1e" %
          (rel(chk["gen_out"], ref["gen_out"]), max(rel(chk["G"][k], ref["G"][k]) for k in ref["G"] if float(ref["G"][k].norm()) > 1e-12)))
    rows = []
    global LOSS_SCALE
    jobs = []
    for s in a.schemes.split(","):
        if s.startswith("fp16_f8_train") and a.loss_scales:
            jobs += [(s, 2.0 ** int(k)) for k in a.loss_scales.split(",")]
        else:
            jobs.append((s, 1.0))
    for s, ls in jobs:
        LOSS_SCALE = ls
        r = run(s, A, B, P)
        # gradient tensors that are analytically zero (conv bias in front of an instance norm) are skipped
        gerr = {k: rel(r["G"][k], ref["G"][k]) for k in ref["G"] if float(ref["G"][k].norm()) > 1e-9 * max(1.0, float(ref["G"][k].numel()) ** 0.5)}
        worst = max(gerr, key=gerr.get)
        lerr = max(abs(float(r["L"][k]) - float(ref["L"][k])) / abs(float(ref["L"][k])) for k in ref["L"])
        nonfinite = sum(int(not torch.isfinite(r["G"][k]).all()) for k in r["G"])
        row = {"scheme": s if ls == 1.0 else "%s@L=2^%d" % (s, round(math.log2(ls))), "nonfinite_grad_tensors": nonfinite, "mma_units": COST[s], "gen_h1": rel(r["taps"]["h1_glu"], ref["taps"]["h1_glu"]),
               "gen_r6": rel(r["taps"]["r6"], ref["taps"]["r6"]), "gen_out": rel(r["gen_out"], ref["gen_out"]), "loss_worst": lerr,
               "grad_worst": gerr[worst], "grad_worst_name": worst,
               "grad_median": sorted(gerr.values())[len(gerr) // 2]}
        rows.append(row)
        print(json.dumps(row))
    O.conv1d_same, O.conv2d_same = orig
    return rows


if __name__ == "__main__":
    main()
