"""CPU: the float64 emulation of the tensor-core schemes (tests/scheme_ref.py) pinned before any kernel is held to it --
hand-worked plane values, the exact scheme against the oracle, and the margins that make the GPU bounds of
tests/test_gpu_schemes.py meaningful (every broken version of a scheme far outside the float32 accumulation floor)."""
import math

import pytest
import torch

import scheme_ref as S
from test_gpu_schemes import CASES, SWEEP_CASES, case_data, emulate, mutant_distances

F64 = torch.float64

# activation role: x -> (q16, e4m3 hi plane, lo part, represented value q16 + lo), all divided back
ACT_LITERALS = [
    (1 + 2 ** -11, 1.0, 1.0, 2 ** -11, 1 + 2 ** -11),                    # fp16 tie to even; the lo plane keeps x exactly
    (1 + 3 * 2 ** -11, 1 + 2 ** -9, 1.0, -2 ** -11, 1 + 3 * 2 ** -11),     # tie rounds up to the even neighbour; negative lo
    (1 + 17 * 2 ** -16, 1.0, 1.0, 2 ** -12, 1 + 2 ** -12),                 # lo x 4096 = 1.0625: an e4m3 tie, to 1.0
    (500.0, 500.0, 448.0, 0.0, 500.0),                                     # hi plane saturates at 448
    (256.125, 256.0, 256.0, 448 / 4096, 256.109375),                       # lo x 4096 = 512 saturates at 448
    (1 + 3 * 2 ** -23, 1.0, 1.0, 2 ** -21, 1 + 2 ** -21),                  # lo x 4096 = 0.75 * 2^-9: e4m3 subnormal, to 2^-9
    (3 * 2 ** -26, 2 ** -24, 0.0, -0.0, 2 ** -24),                         # fp16 subnormal 2^-24; lo underflows to -0
]


@pytest.mark.parametrize("lit", ACT_LITERALS, ids=[repr(l[0]) for l in ACT_LITERALS])
def test_activation_plane_literals(lit):
    x, q16, hi8, lo8, rep = lit
    assert torch.tensor(x, dtype=torch.float32).double().item() == x          # every literal is a float32
    h, a8h, a8l = (float(t) for t in S.planes_f16f8(torch.tensor([x], dtype=F64), "act"))
    assert (h, a8h, a8l) == (q16, hi8, lo8)
    assert math.copysign(1.0, a8l) == math.copysign(1.0, lo8)
    assert h + a8l == rep
    for sign in (-1.0,):                                                       # the planes are odd functions of x
        hn, a8hn, a8ln = (float(t) for t in S.planes_f16f8(torch.tensor([sign * x], dtype=F64), "act"))
        assert (hn, a8hn, a8ln) == (-q16, -hi8, -lo8)


def test_weight_plane_literals():
    h, w8h, w8l = (float(t) for t in S.planes_f16f8(torch.tensor([60.0], dtype=F64), "weight"))
    assert (h, w8h, w8l) == (60.0, 56.0, 0.0)             # hi plane e4m3(60 * 2^3 = 480) saturates at 448, i.e. 56
    h, w8h, w8l = (float(t) for t in S.planes_f16f8(torch.tensor([1 + 2 ** -12], dtype=F64), "weight"))
    assert (h, w8h, w8l) == (1.0, 1.0, 2 ** -12)          # lo x 2^15 = 8, exact in e4m3
    h, lo = (float(t) for t in S.planes_bf16x3(torch.tensor([1 + 2 ** -8], dtype=F64)))
    assert (h, lo) == (1.0, 2 ** -8)                      # bf16 tie to even (down); the lo plane keeps the rest
    h, lo = (float(t) for t in S.planes_bf16x3(torch.tensor([1 + 3 * 2 ** -8], dtype=F64)))
    assert (h, lo) == (1 + 2 ** -6, -2 ** -8)             # bf16 tie to even (up); negative lo
    h, lo = (float(t) for t in S.planes_bf16x3(torch.tensor([1 + 2 ** -8 + 2 ** -20], dtype=F64)))
    assert (h, lo) == (1 + 2 ** -7, -2 ** -8)             # the lo plane is bf16 too: x - hi = -2^-8 + 2^-20 loses its last bit


def test_split_is_exact_in_float32():
    """q16 + (x - q16) == x for float32 x inside the fp16 range (the lo plane is formed in float32 without rounding), and the
    same for the bf16 hi part"""
    g = torch.Generator().manual_seed(0)
    x = (torch.randn(200000, generator=g, dtype=F64) * torch.pow(2.0, torch.randint(-30, 15, (200000,), generator=g).double())).float()
    x = x[x.abs() < 65504]
    for dt in (torch.float16, torch.bfloat16):
        h = x.to(dt).float()
        assert torch.equal(h + (x - h), x)
        assert torch.equal((x - h).double(), x.double() - h.double())


@pytest.mark.parametrize("case", [c for c in CASES if c[0] in ("G.h1", "G.d1", "D.d1", "D.d3", "raggedM")], ids=lambda c: c[0])
def test_exact_scheme_reproduces_oracle(case):
    from oracle import cyclegan_oracle as O
    name, B, H, W, Cin, kh, kw, Cout, sh, sw = case
    x, w, b, dy = case_data(case)
    xr, wr = x.double().requires_grad_(True), w.double().requires_grad_(True)
    y = O.conv2d_same(xr, wr, None, (sh, sw))
    y.backward(dy.double())
    ey, edx, edw = emulate(case, x, w, dy, "exact")
    assert S.rel_l2(ey, y.detach()) < 1e-12 and S.rel_l2(edx, xr.grad) < 1e-12 and S.rel_l2(edw, wr.grad) < 1e-12


def _floor(case, x, w, dy, scheme):
    ref = emulate(case, x, w, dy, scheme)
    f32 = S.emulate_conv_f32(x, w, dy, *case[1:], scheme)
    return ref, {k: S.rel_l2(a, r) for k, a, r in zip(("y", "dx", "dw"), f32, ref)}


# how far outside the float32 floor each broken scheme must sit.  A dropped product (or both cross terms) 100x; the lo plane
# written at half its scale is half a cross term wrong, and at the deepest contractions (G.o1 K = 3840, D.d3 K = 9216, where
# the float32 floor is 1.1e-6 / 1.5e-6) it sits 68-70x out: 50x for it.
MARGIN = {"act_lo_scale_half": 50.0}


@pytest.mark.parametrize("scheme", ["bf16x3", "f16f8", "f16f8_w16"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_mutants_are_far_outside_the_float32_floor(case, scheme):
    """every broken version of the scheme far outside the same rounded operands through float32 accumulation (the floor a
    kernel's MMAs can reach): a GPU bound at a few times the floor tells them apart"""
    x, w, b, dy = case_data(case)
    ref, floor = _floor(case, x, w, dy, scheme)
    dist = mutant_distances(case, x, w, dy, scheme, ref)
    for k in ("y", "dx", "dw"):
        m = min(dist[k].values())
        print("%-9s %-9s %-2s float32 floor %.1e  nearest mutant %.1e (%s, %.0fx)" % (case[0], scheme, k, floor[k], m, min(dist[k], key=dist[k].get), m / floor[k]))
        for name, d in dist[k].items():
            assert d >= MARGIN.get(name, 100.0) * floor[k], (k, name, floor[k], dist[k])


def test_f16f8_window():
    """the magnitude window the product relies on: with inputs (x and dy) scaled by 2^-8 ... 2^7 and weights at the glorot scale
    the F16F8 scheme stays within 5e-5 of exact on G.res_h1, forward and data gradient.  The weight gradient multiplies two
    scaled operands, whose lo planes both reach the e4m3 subnormals: its window is one binade narrower at the bottom (6.4e-5
    at 2^-8)."""
    case = [c for c in SWEEP_CASES if c[0] == "G.res_h1"][0]
    x, w, b, dy = case_data(case)
    rows = []
    for k in range(-8, 8):
        s = 2.0 ** k
        got = emulate(case, x * s, w, dy * s, "f16f8")
        ex = emulate(case, x * s, w, dy * s, "exact")
        e = [S.rel_l2(a, r) for a, r in zip(got, ex)]
        rows.append((k, e))
        assert e[0] < 5e-5 and e[1] < 5e-5, (k, e)
        if k >= -7:
            assert e[2] < 5e-5, (k, e)
    print("f16f8 vs exact (y, dx, dw) at inputs 2^k:", ["%d: %.1e %.1e %.1e" % (k, *e) for k, e in rows])
