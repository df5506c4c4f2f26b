"""conv_transpose2d (ConvTranspose2d k4 s2 p1, no bias) over the whole domain the library accepts, against fp64 torch
autograd with a per-element gate: padded M / N tiles, partial main-term chunks, every wgrad slice count the plan
produces, exponents far outside O(1), the memory contract of the cdr_deconv_train_* entry points, layouts, streams,
CUDA graphs and non-finite inputs.  test_gpu_deconv_train.py covers the three CDRNet decoder layers."""
import ctypes as C
import functools

import pytest
import torch
import torch.nn.functional as F

import train_conv_checks as checks
from train_conv_checks import SENTINEL, Region, bits_equal, f32_region, graph_replay, on_side_stream

pytestmark = pytest.mark.gpu


def slices(n, cin, cout, h):
    """The number of K slices of the weight gradient: M = Cin over the x pixels, N = Cout, 16 taps."""
    return checks.wgrad_slices(n * h * h, cin, cout, 16)


# (N, Cin, Cout, H, wgrad slices): padded N and M tiles (Cin or Cout % 128 == 64), partial kSplitChunk chunks (K-block
# counts not a multiple of 8), half-full last pixel tiles, and every slice count from 1 to 32, some ending mid-image
TABLE = [
    (1, 64, 64, 8, 1),         # 64-pixel M tile, padded N in every GEMM, padded wgrad M, 4 forward K blocks
    (3, 192, 320, 16, 1),      # chunk of 8 + 4, Cout % 128 = 64
    (7, 320, 64, 16, 1),       # 20 forward K blocks, padded N
    (33, 64, 128, 8, 1),       # odd K-block count, last pixel tile half full
    (2, 1088, 64, 8, 1),       # 68 forward K blocks
    (8, 128, 128, 16, 2),
    (5, 128, 192, 32, 4),      # slice boundaries mid-image
    (32, 64, 128, 16, 8),
    (16, 64, 64, 32, 16),
    (32, 64, 64, 32, 32),      # the largest slice count the plan produces
]

WORST = {"y": 0.0, "dx": 0.0, "dw": 0.0}     # largest (|got - ref| - 2^-126) / m seen by the gated tests, per pass
_report_worst = checks.report_worst(WORST, __name__)
gate = functools.partial(checks.gate, worst=WORST)


def inputs(n, cin, cout, h, seed=0, ex=0, ew=0, edy=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n, cin, h, h), device="cuda", generator=g) * 2.0 ** ex
    w = torch.randn((cin, cout, 4, 4), device="cuda", generator=g) * ((1.0 / (cin * 4) ** 0.5) * 2.0 ** ew)
    dy = torch.randn((n, cout, 2 * h, 2 * h), device="cuda", generator=g) * 2.0 ** edy
    return x, w, dy


def ours(pkg, x, w, dy, need=(True, True)):
    x = x.detach().requires_grad_(need[0])
    w = w.detach().requires_grad_(need[1])
    y = pkg.conv_transpose2d(x, w)
    grads = torch.autograd.grad(y, [t for t, r in ((x, need[0]), (w, need[1])) if r], dy)
    return (y.detach(), *grads)


def reference(x, w, dy):
    """fp64 autograd of F.conv_transpose2d -> (y, dx, dW), and the same on |x|, |w|, |dy| -> their magnitudes m."""
    out = []
    for f in (lambda t: t, torch.abs):
        x64 = f(x.detach().double()).requires_grad_(True)
        w64 = f(w.detach().double()).requires_grad_(True)
        y64 = F.conv_transpose2d(x64, w64, stride=2, padding=1)
        dx64, dw64 = torch.autograd.grad(y64, (x64, w64), f(dy.detach().double()))
        out.append((y64.detach(), dx64, dw64))
    return out


def check_all(pkg, x, w, dy, label, max_gate=True):
    (y, dx, dw), ((ry, rdx, rdw), (my, mdx, mdw)) = ours(pkg, x, w, dy), reference(x, w, dy)
    r = {k: gate(k, a, b, m, max_gate) for k, a, b, m in (("y", y, ry, my), ("dx", dx, rdx, mdx), ("dw", dw, rdw, mdw))}
    print(f"\n{label}: " + ", ".join(f"{k} {v[0]:.2e}/m {v[1]:.2e}/max" for k, v in r.items()))
    return y, dx, dw


@pytest.mark.parametrize("n,cin,cout,h,s", TABLE)
def test_shape_table(cuda_pkg, n, cin, cout, h, s):
    assert slices(n, cin, cout, h) == s
    check_all(cuda_pkg, *inputs(n, cin, cout, h, seed=n + cin + cout + h), f"N={n} {cin}->{cout} {h}x{h} slices={s}")


# (e_x, e_w, e_dy): x, w and dy times 2^e.  Every fp64 reference output stays in the normal fp32 range, while the
# amax of one operand falls below 2^-114, where an uncapped 2^(13 - ilogb(amax)) scale overflows to +Inf.
EXPONENTS = [(-120, 0, 0), (0, 0, -120), (0, -118, 0), (-60, 0, -60), (100, 0, -100), (0, 0, 100)]
SWEEP_SHAPES = [(2, 256, 256, 16), (3, 192, 320, 16)]     # decoder.deconv2, and a padded shape of the table


@pytest.mark.parametrize("n,cin,cout,h", SWEEP_SHAPES)
@pytest.mark.parametrize("ex,ew,edy", EXPONENTS)
def test_exponent_sweep(cuda_pkg, n, cin, cout, h, ex, ew, edy):
    x, w, dy = inputs(n, cin, cout, h, seed=5, ex=ex, ew=ew, edy=edy)
    check_all(cuda_pkg, x, w, dy, f"N={n} {cin}->{cout} {h}x{h} 2^({ex}, {ew}, {edy})")


@pytest.mark.parametrize("n,cin,cout,h", SWEEP_SHAPES)
def test_subnormal_input(cuda_pkg, n, cin, cout, h):
    """Every x value subnormal (|x| in [2^-135, 2^-134)), dy times 2^100 so that dW = sum x dy is a normal float; y
    is below the fp32 normal range and only has to be near zero."""
    x, w, dy = inputs(n, cin, cout, h, seed=6, edy=100)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.sign(x) * (1 + torch.rand(x.shape, device="cuda", generator=g)) * 2.0 ** -135
    assert bool(((x != 0) & (x.abs() < 2.0 ** -126)).all())
    check_all(cuda_pkg, x, w, dy, f"N={n} {cin}->{cout} {h}x{h} subnormal x", max_gate=False)


# ---- memory contract of the C ABI: exact byte counts, guard bytes around every buffer, stale workspace contents ----
def _abi_run(pkg, x, w, dy, fill, gen):
    """forward, full backward, dx-only and dW-only backward through the C ABI, every buffer guarded."""
    L = pkg._lib.lib()
    n, cin, h, _ = x.shape
    cout = w.shape[1]
    sb, wb = C.c_size_t(), C.c_size_t()
    pkg._lib.check(L.cdr_deconv_train_workspace_bytes(n, cin, cout, h, h, C.byref(sb), C.byref(wb)))
    st = pkg._lib.current_stream_ptr()
    ptr = pkg._lib.ptr
    saved, ws = Region(sb.value, fill, gen), Region(wb.value, fill, gen)
    ry, y = f32_region((n, cout, 2 * h, 2 * h))
    pkg._lib.check(L.cdr_deconv_train_forward(ptr(x), ptr(w), n, cin, cout, h, h, ptr(y), ptr(saved.inner), sb.value,
                                              ptr(ws.inner), wb.value, st))
    regions, outs = [saved, ws, ry], {"y": y}
    for tag, want_dx, want_dw in (("", True, True), ("_xonly", True, False), ("_wonly", False, True)):
        ws_b = Region(wb.value, fill, gen)
        rdx, dx = f32_region((n, cin, h, h)) if want_dx else (None, None)
        rdw, dw = f32_region((cin, cout, 4, 4)) if want_dw else (None, None)
        pkg._lib.check(L.cdr_deconv_train_backward(ptr(saved.inner), ptr(w), ptr(dy), n, cin, cout, h, h, ptr(dx),
                                                   ptr(dw), ptr(ws_b.inner), wb.value, st))
        regions += [r for r in (ws_b, rdx, rdw) if r is not None]
        if want_dx:
            outs["dx" + tag] = dx
        if want_dw:
            outs["dw" + tag] = dw
    assert all(r.guards_intact() for r in regions), "a write landed outside its buffer"
    for k, t in outs.items():
        assert not bool((t.view(torch.int32) == SENTINEL * 0x01010101).any()), f"{k}: elements never written"
    return {k: t.clone() for k, t in outs.items()}


@pytest.mark.parametrize("n,cin,cout,h", [(1, 64, 64, 8), (5, 128, 192, 32), (3, 192, 320, 16)])
def test_memory_contract(cuda_pkg, n, cin, cout, h):
    x, w, dy = inputs(n, cin, cout, h, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(12)
    runs = [_abi_run(cuda_pkg, x, w, dy, fill, gen) for fill in (0x00, 0xFF, "random")]
    for k in runs[0]:
        assert all(bits_equal(runs[0][k], r[k]) for r in runs[1:]), f"{k} depends on stale workspace contents"
    a = runs[0]
    assert bits_equal(a["dx_xonly"], a["dx"]) and bits_equal(a["dw_wonly"], a["dw"])
    y, dx, dw = ours(cuda_pkg, x, w, dy)                 # the autograd op is the same computation
    assert bits_equal(y, a["y"]) and bits_equal(dx, a["dx"]) and bits_equal(dw, a["dw"])
    (ry, rdx, rdw), (my, mdx, mdw) = reference(x, w, dy)
    gate("y", a["y"], ry, my), gate("dx", a["dx"], rdx, mdx), gate("dw", a["dw"], rdw, mdw)


# ---- layouts, streams, CUDA graphs ----
LAYOUT_SHAPE = (5, 128, 192, 32)


def test_layouts_give_the_same_bits(cuda_pkg):
    n, cin, cout, h = LAYOUT_SHAPE
    x, w, dy = inputs(n, cin, cout, h, seed=21)
    base = ours(cuda_pkg, x, w, dy)
    x_cl, dy_cl = x.to(memory_format=torch.channels_last), dy.to(memory_format=torch.channels_last)
    w_nc = w.transpose(0, 1).contiguous().transpose(0, 1)          # (Cin, Cout, 4, 4) view with Cout outermost
    assert not x_cl.is_contiguous() and not dy_cl.is_contiguous() and not w_nc.is_contiguous()
    # contiguous views 4 bytes past an aligned address, as x[1:] of a larger buffer gives
    x_off, dy_off = (torch.empty(t.numel() + 1, device="cuda")[1:].view(t.shape).copy_(t) for t in (x, dy))
    assert x_off.is_contiguous() and x_off.data_ptr() % 16 == 4 and dy_off.data_ptr() % 16 == 4
    for xs, ws, dys in ((x_cl, w_nc, dy_cl), (x_off, w, dy_off)):
        got = ours(cuda_pkg, xs, ws, dys)
        assert all(bits_equal(a.contiguous(), b.contiguous()) for a, b in zip(base, got))


def test_side_stream_gives_the_same_bits(cuda_pkg):
    n, cin, cout, h = LAYOUT_SHAPE
    x, w, dy = inputs(n, cin, cout, h, seed=22)
    base = ours(cuda_pkg, x, w, dy)
    got = on_side_stream(ours, cuda_pkg, x, w, dy)
    assert all(bits_equal(a, b) for a, b in zip(base, got))


def test_cuda_graph_replay_equals_eager(cuda_pkg):
    n, cin, cout, h = LAYOUT_SHAPE
    x, w, dy = inputs(n, cin, cout, h, seed=23)
    sx, sw, sdy = x.clone().requires_grad_(True), w.clone().requires_grad_(True), dy.clone()

    def step():
        y = cuda_pkg.conv_transpose2d(sx, sw)
        return (y.detach(), *torch.autograd.grad(y, (sx, sw), sdy))
    x2, w2, dy2 = inputs(n, cin, cout, h, seed=24)
    static_out = graph_replay(step, (sx, sw, sdy), (x2, w2, dy2))
    eager = ours(cuda_pkg, x2, w2, dy2)
    assert all(bits_equal(a, b) for a, b in zip(static_out, eager))


# ---- non-finite inputs: a diverging run is never reported finite ----
@pytest.mark.parametrize("where,value,pixel", [("x", float("nan"), (3, 5)), ("x", float("nan"), (0, 0)),
                                               ("dy", float("nan"), (6, 9)), ("x", float("inf"), (3, 5))])
def test_non_finite_inputs(cuda_pkg, where, value, pixel):
    n, cin, cout, h = 2, 128, 192, 16
    x, w, dy = inputs(n, cin, cout, h, seed=31)
    (x if where == "x" else dy)[1, 7, pixel[0], pixel[1]] = value
    (y, dx, dw), ((ry, rdx, rdw), (my, mdx, mdw)) = ours(cuda_pkg, x, w, dy), reference(x, w, dy)
    assert not bool(torch.isfinite(ry).all() and torch.isfinite(rdx).all() and torch.isfinite(rdw).all())
    # y and dx: non-finite exactly where the reference is, and the finite elements inside the gate
    for name, got, ref, mag in (("y", y, ry, my), ("dx", dx, rdx, mdx)):
        gate(name, got, ref, mag, max_gate=False)
        assert torch.equal(torch.isfinite(got), torch.isfinite(ref)), name
    # dW: every non-finite reference element non-finite; the finite elements of both inside the gate.  dW may have
    # more: a NaN pixel meets the zero fill of its out-of-image taps as NaN * 0.  (On a B200 with torch 2.11 there
    # were none: the fp64 reference's own zero padding poisons the same taps, so the sets are equal.)
    both = torch.isfinite(dw) & torch.isfinite(rdw)
    assert not bool(torch.isfinite(dw[~torch.isfinite(rdw)]).any())
    gate("dw", dw[both], rdw[both], mdw[both], max_gate=False)
    extra = int((~torch.isfinite(dw) & torch.isfinite(rdw)).sum())
    print(f"\n{value} in {where} at {pixel}: non-finite y {int((~torch.isfinite(y)).sum())}, dx "
          f"{int((~torch.isfinite(dx)).sum())}, dW {int((~torch.isfinite(dw)).sum())} "
          f"(reference {int((~torch.isfinite(rdw)).sum())}, extra {extra})")
