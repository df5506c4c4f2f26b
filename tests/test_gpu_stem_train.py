"""The encoder's stem in training: stem_conv (the 7x7 stride-2 pad-3 conv, forward and weight gradient) against fp64
torch autograd with the per-element gate of the other training convolutions, over its whole domain (shapes, every kind
of wgrad slice plan, exponents, the memory contract of cdr_stem_train_*, layouts, streams, CUDA graphs, non-finite
inputs); max_pool3x3 bit for bit against torch's CUDA max-pool, forward and backward; and ResNet.forward_train /
CDRNet with the stem on the library against fp64."""
import copy
import ctypes as C
import functools

import pytest
import torch
import torch.nn.functional as F

import train_conv_checks as checks
from fast_3d_human_pose_estimation_b200 import synth
from train_conv_checks import SENTINEL, Region, bits_equal, f32_region, graph_replay, on_side_stream

pytestmark = pytest.mark.gpu

TARGET_SLICES = 2 * 148


def slices(n, h, w):
    """Python mirror of the stem's wgrad slice rule (csrc/stem.cu: stem_train_plan): K chunks of 2 output rows x 32
    output columns, ceil(chunks / 296) chunks per slice."""
    chunks = n * (h // 4) * (w // 64)
    cps = -(-chunks // TARGET_SLICES)
    return -(-chunks // cps)


# (N, H, W, slices): one chunk per slice (slices = chunks), several per slice with a ragged last slice, slices that end
# mid-image, H != W both ways, the B = 64 stem shape
TABLE = [
    (1, 256, 256, 256),      # one chunk per slice
    (2, 256, 256, 256),      # two per slice
    (64, 256, 256, 293),     # the B = 64 view: 56 chunks per slice, the last one 32
    (5, 256, 256, 256),      # 5 chunks per slice, 256 per image: slices end mid-image
    (19, 128, 128, 244),     # 5 per slice, a last slice of 1 chunk
    (1, 128, 256, 128),      # H != W
    (1, 256, 64, 64),        # W = 64, the narrowest image
    (3, 64, 128, 96),
    (3, 256, 192, 288),      # W = 192: three 32-column chunks per output row
    (1, 16, 64, 4),          # the smallest image
]

WORST = {"y": 0.0, "dw": 0.0}
_report_worst = checks.report_worst(WORST, __name__)
gate = functools.partial(checks.gate, worst=WORST)


def inputs(n, h, w, seed=0, ex=0, ew=0, edy=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n, 3, h, w), device="cuda", generator=g) * 2.0 ** ex
    wt = torch.randn((64, 3, 7, 7), device="cuda", generator=g) * ((1.0 / 147 ** 0.5) * 2.0 ** ew)
    dy = torch.randn((n, 64, h // 2, w // 2), device="cuda", generator=g) * 2.0 ** edy
    return x, wt, dy


def ours(pkg, x, w, dy):
    w = w.detach().requires_grad_(True)
    y = pkg.stem_conv(x.detach(), w)
    (dw,) = torch.autograd.grad(y, (w,), dy)
    return y.detach(), dw


def reference(x, w, dy):
    """fp64 autograd of F.conv2d -> (y, dW), and the same on |x|, |w|, |dy| -> their magnitudes m."""
    out = []
    for f in (lambda t: t, torch.abs):
        w64 = f(w.detach().double()).requires_grad_(True)
        y64 = F.conv2d(f(x.detach().double()), w64, stride=2, padding=3)
        (dw64,) = torch.autograd.grad(y64, (w64,), f(dy.detach().double()))
        out.append((y64.detach(), dw64))
    return out


def check_all(pkg, x, w, dy, label, max_gate=True):
    got, (ref, mag) = ours(pkg, x, w, dy), reference(x, w, dy)
    r = {k: gate(k, got[i], ref[i], mag[i], max_gate) for i, k in enumerate(("y", "dw"))}
    print(f"\n{label}: " + ", ".join(f"{k} {v[0]:.2e}/m {v[1]:.2e}/max" for k, v in r.items()))
    return got


@pytest.mark.parametrize("n,h,w,sl", TABLE)
def test_shape_table(cuda_pkg, n, h, w, sl):
    assert slices(n, h, w) == sl
    check_all(cuda_pkg, *inputs(n, h, w, seed=n + h + w), f"N={n} {h}x{w} slices={sl}")


# (e_x, e_w, e_dy): x, w and dy times 2^e.  An amax below 2^-114 is where an uncapped 2^(13 - ilogb(amax)) scale
# overflows to +Inf.
EXPONENTS = [(-120, 0, 0), (100, 0, 0), (0, -120, 0), (0, 100, 0), (0, 0, -120), (0, 0, 100)]


@pytest.mark.parametrize("ex,ew,edy", EXPONENTS)
def test_exponent_sweep(cuda_pkg, ex, ew, edy):
    check_all(cuda_pkg, *inputs(2, 64, 128, seed=5, ex=ex, ew=ew, edy=edy), f"2^({ex}, {ew}, {edy})")


def test_subnormal_input(cuda_pkg):
    """Every x value subnormal (|x| in [2^-135, 2^-134)), dy times 2^100 so that dW = sum x dy is a normal float; y
    is below the fp32 normal range and only has to be near zero."""
    x, wt, dy = inputs(2, 64, 128, seed=6, edy=100)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.sign(x) * (1 + torch.rand(x.shape, device="cuda", generator=g)) * 2.0 ** -135
    assert bool(((x != 0) & (x.abs() < 2.0 ** -126)).all())
    check_all(cuda_pkg, x, wt, dy, "subnormal x", max_gate=False)


# ---- memory contract of the C ABI ----
def _abi_run(pkg, x, w, dy, fill, gen):
    """forward and backward through the C ABI, every buffer guarded and exactly as large as reported"""
    L = pkg._lib.lib()
    n, _, h, wd = x.shape
    sb, wb = C.c_size_t(), C.c_size_t()
    pkg._lib.check(L.cdr_stem_train_workspace_bytes(n, 3, 64, h, wd, C.byref(sb), C.byref(wb)))
    st = pkg._lib.current_stream_ptr()
    ptr = pkg._lib.ptr
    saved, ws, ws_b = Region(sb.value, fill, gen), Region(wb.value, fill, gen), Region(wb.value, fill, gen)
    ry, y = f32_region((n, 64, h // 2, wd // 2))
    rdw, dw = f32_region((64, 3, 7, 7))
    pkg._lib.check(L.cdr_stem_train_forward(ptr(x), ptr(w), n, 3, 64, h, wd, ptr(y), ptr(saved.inner), sb.value,
                                            ptr(ws.inner), wb.value, st))
    pkg._lib.check(L.cdr_stem_train_backward(ptr(saved.inner), ptr(w), ptr(dy), n, 3, 64, h, wd, None, ptr(dw),
                                             ptr(ws_b.inner), wb.value, st))
    assert L.cdr_stem_train_backward(ptr(saved.inner), ptr(w), ptr(dy), n, 3, 64, h, wd, ptr(dw), ptr(dw),
                                     ptr(ws_b.inner), wb.value, st) == 1           # a data gradient is refused
    assert b"dx must be NULL" in L.cdr_last_error()
    assert L.cdr_stem_train_forward(ptr(x), ptr(w), n, 3, 64, h, wd, ptr(y), ptr(saved.inner), sb.value - 1,
                                    ptr(ws.inner), wb.value, st) == 3              # saved one byte short
    assert L.cdr_stem_train_backward(ptr(saved.inner), ptr(w), ptr(dy), n, 3, 64, h, wd, None, ptr(dw),
                                     ptr(ws_b.inner), wb.value - 1, st) == 3       # the backward's workspace, one byte short
    assert all(r.guards_intact() for r in (saved, ws, ws_b, ry, rdw)), "a write landed outside its buffer"
    outs = {"y": y, "dw": dw}
    for k, t in outs.items():
        assert not bool((t.view(torch.int32) == SENTINEL * 0x01010101).any()), f"{k}: elements never written"
    return {k: t.clone() for k, t in outs.items()}


@pytest.mark.parametrize("n,h,w", [(1, 16, 64), (3, 64, 128), (2, 256, 256)])
def test_memory_contract(cuda_pkg, n, h, w):
    x, wt, dy = inputs(n, h, w, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(12)
    runs = [_abi_run(cuda_pkg, x, wt, dy, fill, gen) for fill in (0x00, 0xFF, "random")]
    for k in runs[0]:
        assert all(bits_equal(runs[0][k], r[k]) for r in runs[1:]), f"{k} depends on stale buffer contents"
    got = ours(cuda_pkg, x, wt, dy)                       # the autograd op is the same computation
    assert bits_equal(got[0], runs[0]["y"]) and bits_equal(got[1], runs[0]["dw"])
    ref, mag = reference(x, wt, dy)
    for i, k in enumerate(("y", "dw")):
        gate(k, runs[0][k], ref[i], mag[i])


# ---- layouts, streams, CUDA graphs, repeated backward ----
SHAPE = (4, 64, 128)


def test_layouts_give_the_same_bits(cuda_pkg):
    x, w, dy = inputs(*SHAPE, seed=21)
    base = ours(cuda_pkg, x, w, dy)
    x_cl, dy_cl = x.to(memory_format=torch.channels_last), dy.to(memory_format=torch.channels_last)
    w_nc = torch.cat([w, w], 3)[:, :, :, :7]                  # a non-contiguous weight
    buf = torch.empty(x.numel() + 1, device="cuda")
    x_off = buf[1:].view(x.shape)                             # a view 4 bytes past a 16-byte boundary
    x_off.copy_(x)
    assert x_off.data_ptr() % 16 != 0
    assert not x_cl.is_contiguous() and not dy_cl.is_contiguous() and not w_nc.is_contiguous()
    for xs, ws, dys in ((x_cl, w, dy_cl), (x, w_nc, dy), (x_off, w, dy)):
        got = ours(cuda_pkg, xs, ws, dys)
        assert all(bits_equal(a, g.contiguous()) for a, g in zip(base, got))


def test_side_stream_gives_the_same_bits(cuda_pkg):
    x, w, dy = inputs(*SHAPE, seed=22)
    base = ours(cuda_pkg, x, w, dy)
    got = on_side_stream(ours, cuda_pkg, x, w, dy)
    assert all(bits_equal(a, g) for a, g in zip(base, got))


def test_cuda_graph_replay_equals_eager(cuda_pkg):
    x, w, dy = inputs(*SHAPE, seed=23)
    sx, sw, sdy = x.clone(), w.clone().requires_grad_(True), dy.clone()

    def step():
        y = cuda_pkg.stem_conv(sx, sw)
        return (y.detach(), *torch.autograd.grad(y, (sw,), sdy))
    x2, w2, dy2 = inputs(*SHAPE, seed=24)
    static_out = graph_replay(step, (sx, sw, sdy), (x2, w2, dy2))
    eager = ours(cuda_pkg, x2, w2, dy2)
    assert all(bits_equal(a, e) for a, e in zip(static_out, eager))


def test_two_backward_calls_and_zero_dy(cuda_pkg):
    x, w, _ = inputs(*SHAPE, seed=25)
    w = w.requires_grad_(True)
    y = cuda_pkg.stem_conv(x, w)
    (zero,) = torch.autograd.grad(y, (w,), torch.zeros_like(y), retain_graph=True)
    assert bool((zero == 0).all())                            # exact zeros
    dy = torch.randn_like(y)
    first = torch.autograd.grad(y, (w,), dy, retain_graph=True)
    second = torch.autograd.grad(y, (w,), dy)
    assert bits_equal(first[0], second[0])


# ---- non-finite inputs: a diverging run is never reported finite ----
def _y_wider(x, n_out_w):
    """Where y may be non-finite although the reference is not: the forward's K axis is laid out as 7 rows of 22 (21
    taps x channels + one padding slot), and the padding slot, whose weight is zero, reads channel 0 of the input column
    just right of the window, 2 ox + 4, in each of its 7 rows (except for the last column of a 16-column tile, where
    the patch ends).  A non-finite value there times the zero weight is NaN."""
    bad = ~torch.isfinite(x[:, 0].double())                                   # (n, H, W)
    n, h, w = bad.shape
    shifted = torch.zeros_like(bad)
    shifted[:, :, :w - 4] = bad[:, :, 4:]                                     # shifted[.., ix'] = bad[.., ix' + 4]
    rows = F.max_pool2d(shifted.double().unsqueeze(1), (7, 1), stride=1, padding=(3, 0)) > 0   # any of rows iy-3..iy+3
    wider = rows[:, :, ::2, ::2]                                              # (n, 1, H/2, W/2): ix' = 2 ox
    wider[..., 15::16] = False
    return wider.expand(n, 64, h // 2, n_out_w)


@pytest.mark.parametrize("where,value", [("x", float("nan")), ("x", float("inf")), ("x", float("-inf")),
                                         ("dy", float("nan")), ("dy", float("-inf"))])
def test_non_finite_inputs(cuda_pkg, where, value):
    """dW is non-finite exactly where the reference is.  y is non-finite wherever the reference is, and elsewhere only
    in the set _y_wider describes (a non-finite x in channel 0, 4 columns right of a window)."""
    x, w, dy = inputs(2, 64, 128, seed=31)
    t = x if where == "x" else dy
    for c, iy, ix in ((0, 9, 20), (1, 30, 51), (2, 0, 0), (0, 40, 127)):
        t[1, c, iy % t.shape[2], ix % t.shape[3]] = value
    got, (ref, mag) = ours(cuda_pkg, x, w, dy), reference(x, w, dy)
    assert not all(bool(torch.isfinite(r).all()) for r in ref)
    wider = _y_wider(x, got[0].shape[3])
    bad_y, ref_bad_y = ~torch.isfinite(got[0]), ~torch.isfinite(ref[0])
    assert bool((bad_y >= ref_bad_y).all()) and bool((bad_y <= (ref_bad_y | wider)).all())
    gate("y", got[0], ref[0], mag[0], max_gate=False, nonfinite=wider)
    assert torch.equal(torch.isfinite(got[1]), torch.isfinite(ref[1]))
    gate("dw", got[1], ref[1], mag[1], max_gate=False)


def test_argument_errors(cuda_pkg):
    x, w, _ = inputs(1, 16, 64)
    with pytest.raises(ValueError, match="requires grad"):
        cuda_pkg.stem_conv(x.clone().requires_grad_(True), w)
    for xs, ws in (((1, 4, 16, 64), (64, 4, 7, 7)),       # Cin = 4
                   ((1, 3, 16, 64), (32, 3, 7, 7)),       # Cout = 32
                   ((1, 3, 16, 64), (64, 3, 5, 5)),       # 5x5
                   ((1, 3, 24, 64), (64, 3, 7, 7)),       # H % 16
                   ((1, 3, 16, 96), (64, 3, 7, 7))):      # W % 64
        with pytest.raises(ValueError, match="expected|unsupported"):
            cuda_pkg.stem_conv(torch.zeros(xs, device="cuda"), torch.zeros(ws, device="cuda"))
    with pytest.raises(ValueError, match="float32"):
        cuda_pkg.stem_conv(x.double(), w.double())
    with pytest.raises(ValueError, match="CUDA"):
        cuda_pkg.stem_conv(x.cpu(), w)


# ---- max_pool3x3: torch's CUDA max-pool, bit for bit ----
def _pool_case(kind, shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, device="cuda", generator=g)
    if kind == "relu":
        x = x.clamp_min(0)                                    # about half exact zeros: all-zero windows
    elif kind == "ties":
        x = torch.randint(1, 4, shape, device="cuda", generator=g).float()     # repeated positive values
    elif kind == "nonfinite":
        r = torch.rand(shape, device="cuda", generator=g)
        x = torch.where(r < 0.05, float("nan"), x)
        x = torch.where((r >= 0.05) & (r < 0.1), float("inf"), x)
        x = torch.where((r >= 0.1) & (r < 0.15), float("-inf"), x)
    return x


def _pool_both(pkg, x, dy_seed):
    xr, xo = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    yr, yo = F.max_pool2d(xr, 3, 2, 1), pkg.max_pool3x3(xo)
    g = torch.Generator(device="cuda").manual_seed(dy_seed)
    dy = torch.randn(yr.shape, device="cuda", generator=g)
    yr.backward(dy)
    yo.backward(dy)
    return (yr.detach(), xr.grad), (yo.detach(), xo.grad)


POOL_SHAPES = [(2, 3, 17, 23), (1, 1, 1, 1), (2, 2, 1, 5), (2, 2, 2, 2), (1, 4, 5, 1), (3, 5, 2, 7), (2, 8, 33, 64),
               (1, 2, 128, 129)]


@pytest.mark.parametrize("kind", ["random", "relu", "ties", "nonfinite"])
@pytest.mark.parametrize("shape", POOL_SHAPES)
def test_max_pool_bits(cuda_pkg, kind, shape):
    (yr, dxr), (yo, dxo) = _pool_both(cuda_pkg, _pool_case(kind, shape, sum(shape)), 1)
    assert bits_equal(yo, yr), "y"
    assert bits_equal(dxo, dxr), "dx"


@pytest.mark.parametrize("kind", ["random", "relu"])
def test_max_pool_stem_shape(cuda_pkg, kind):
    (yr, dxr), (yo, dxo) = _pool_both(cuda_pkg, _pool_case(kind, (64, 64, 128, 128), 3), 4)
    assert bits_equal(yo, yr) and bits_equal(dxo, dxr)


@pytest.mark.parametrize("shape", [(2, 3, 17, 23), (1, 2, 16, 16)])
def test_max_pool_memory_contract(cuda_pkg, shape):
    """y, argmax (n*c*ho*wo bytes) and dx in guarded buffers of exactly their size, argmax pre-filled two ways"""
    L = cuda_pkg._lib.lib()
    ptr, st = cuda_pkg._lib.ptr, cuda_pkg._lib.current_stream_ptr()
    n, c, h, w = shape
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    x = _pool_case("ties", shape, 9)
    dy = torch.randn((n, c, ho, wo), device="cuda")
    (yr, dxr), _ = _pool_both(cuda_pkg, x, 0)
    for fill in (0x00, 0xFF):
        ra = Region(n * c * ho * wo, fill)
        ry, y = f32_region((n, c, ho, wo))
        rdx, dx = f32_region(shape)
        cuda_pkg._lib.check(L.cdr_maxpool3x3_train_forward(ptr(x), n, c, h, w, ptr(y), ptr(ra.inner), st))
        cuda_pkg._lib.check(L.cdr_maxpool3x3_train_backward(ptr(ra.inner), ptr(dy), n, c, h, w, ptr(dx), st))
        assert all(r.guards_intact() for r in (ra, ry, rdx))
        assert bits_equal(y, yr)
        xr = x.clone().requires_grad_(True)
        F.max_pool2d(xr, 3, 2, 1).backward(dy)
        assert bits_equal(dx, xr.grad)
        assert int(ra.inner.max()) <= 8


def test_max_pool_side_stream_and_graph(cuda_pkg):
    x = _pool_case("ties", (4, 8, 32, 32), 13)
    dy = torch.randn((4, 8, 16, 16), device="cuda")

    def run(xin, dyin):
        xo = xin.detach().requires_grad_(True)
        y = cuda_pkg.max_pool3x3(xo)
        return (y.detach(), *torch.autograd.grad(y, (xo,), dyin))
    base = run(x, dy)
    assert all(bits_equal(a, b) for a, b in zip(base, on_side_stream(run, x, dy)))
    sx, sdy = x.clone().requires_grad_(True), dy.clone()

    def step():
        y = cuda_pkg.max_pool3x3(sx)
        return (y.detach(), *torch.autograd.grad(y, (sx,), sdy))
    x2, dy2 = _pool_case("relu", (4, 8, 32, 32), 14), torch.randn((4, 8, 16, 16), device="cuda")
    static_out = graph_replay(step, (sx, sdy), (x2, dy2))
    assert all(bits_equal(a, b) for a, b in zip(static_out, run(x2, dy2)))


# ---- ResNet.forward_train / CDRNet with the stem on the library ----
def _encoder(cuda_pkg):
    torch.manual_seed(0)
    return cuda_pkg.ResNet(synth.make_cfg(50, 19)).cuda().train()


def _all_convs(enc):
    return {n: c for n, c in enc.named_modules() if isinstance(c, torch.nn.Conv2d)}


def test_stem_on_library_calls_no_torch_stem(cuda_pkg, monkeypatch):
    enc = _encoder(cuda_pkg)
    x = synth.make_images(2, seed=1)[0].cuda()

    def boom(*a, **k):
        raise AssertionError("a torch conv / pool module or F.max_pool2d was called")
    for c in _all_convs(enc).values():
        c.forward = boom
    enc.maxpool.forward = boom
    monkeypatch.setattr(F, "max_pool2d", boom)
    y = enc.forward_train(x, stem_on_library=True)
    assert y.shape == (2, 2048, 8, 8) and bool(torch.isfinite(y).all())
    y.square().mean().backward()
    for name, p in enc.named_parameters():
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name


def _stats(m):
    return {n: b.detach().double().clone() for n, b in m.named_buffers() if n.endswith(("running_mean", "running_var"))}


def test_encoder_training_step_vs_fp64(cuda_pkg):
    """One training forward + backward of a ResNet-50 encoder (2 images of 256 x 256) with everything on the library,
    and with its stem on torch (TF32 off), both against the fp64 encoder: the library must be as close to fp64 as the
    torch-stem encoder is, within a factor of 2, in the output, every conv weight gradient (conv1 included) and every
    BatchNorm running statistic (bn1 included)."""
    enc = _encoder(cuda_pkg)
    x = synth.make_images(2, seed=1)[0].cuda()
    up = torch.randn((2, 2048, 8, 8), device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))

    def run(model, xin, upstream, stem=None):
        model.zero_grad()
        y = model(xin) if stem is None else model.forward_train(xin, stem_on_library=stem)
        (y * upstream).sum().backward()
        return y.detach().double(), {n: c.weight.grad.double() for n, c in _all_convs(model).items()}, _stats(model)
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        lib = run(copy.deepcopy(enc), x, up, True)
        tst = run(copy.deepcopy(enc), x, up, False)
        ref = run(copy.deepcopy(enc).double(), x.double(), up.double())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    rel = lambda a, b: float((a - b).norm() / b.norm())     # noqa: E731
    assert "conv1" in ref[1] and "bn1.running_mean" in ref[2]
    e = [(rel(r[0], ref[0]), max(rel(r[1][n], ref[1][n]) for n in ref[1]), max(rel(r[2][n], ref[2][n]) for n in ref[2]),
          rel(r[1]["conv1"], ref[1]["conv1"])) for r in (lib, tst)]
    print("\nvs fp64, stem on library / on torch: output %.2e / %.2e, worst conv weight gradient %.2e / %.2e, worst "
          "running stat %.2e / %.2e, conv1 gradient %.2e / %.2e" % tuple(v for pair in zip(*e) for v in pair))
    for name, a, b in zip(("output", "gradient", "running stat", "conv1 gradient"), *e):
        assert a <= 2 * b + 1e-7, (name, a, b)


def _model(cuda_pkg, stem):
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), trainable=True, train_encoder_on_library=True, train_stem_on_library=stem)
    with torch.no_grad():
        m.decoder.final_layer.weight.mul_(10.0)      # train-mode BN keeps activations O(1): peaky heat-maps need gain
    return m.cuda().train()


def _inputs(b):
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    targets = [torch.from_numpy(gt["gt2d_l"]).float().cuda(), torch.from_numpy(gt["gt2d_r"]).float().cuda()]
    return imgs, Ps, targets


def test_training_step_vs_fp64(cuda_pkg):
    """One training step of CDRNet(trainable=True, train_encoder_on_library=True, train_stem_on_library=True) and of the
    same model with its stem on torch (TF32 off), against the same network in fp64 (torch modules, the oracle's
    operators): within a factor of 2 of the torch-stem model's distance in the joints, the loss, every encoder conv
    weight gradient (conv1 included) and every encoder running statistic (bn1 included)."""
    from oracle import cdr_oracle as O
    lib_m, tst_m = _model(cuda_pkg, True), _model(cuda_pkg, False)
    tst_m.load_state_dict(lib_m.state_dict())
    imgs, Ps, targets = _inputs(2)
    mse = lambda kps, tg: sum(((kps[v] - tg[v]) ** 2).mean() for v in range(2))      # noqa: E731

    def step(model):
        model.zero_grad()
        kps, _ = model(imgs, Ps)
        loss = mse(kps, targets)
        loss.backward()
        return ([k.detach().double() for k in kps], float(loss),
                {n: c.weight.grad.double() for n, c in _all_convs(model.encoder).items()}, _stats(model.encoder))
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        lib, tst = step(lib_m), step(tst_m)
        m64 = copy.deepcopy(_model(cuda_pkg, False)).double()
        feats = [m64.encoder(x.double()) for x in imgs]
        pinv = [torch.linalg.pinv(p.double()) for p in Ps]
        z = torch.cat([O.ftl(m64.CF.conv_layer1(feats[v]), pinv[v]) for v in range(2)], 1)
        f = m64.CF.conv_layer2(z)
        kps64 = []
        for v in range(2):
            o = m64.CF.out_layer[v](O.ftl(f, Ps[v].double()))
            d = m64.decoder
            h = d.final_layer(d.deconv3(d.deconv2(d.deconv1(o))))
            kps64.append(O.process_heatmap(h) * (256 / h.shape[2]))
        loss64 = mse(kps64, [t.double() for t in targets])
        loss64.backward()
        ref = ([k.detach() for k in kps64], float(loss64),
               {n: c.weight.grad for n, c in _all_convs(m64.encoder).items()}, _stats(m64.encoder))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    rel = lambda a, b: float((a - b).norm() / b.norm())     # noqa: E731
    assert "conv1" in ref[2] and "bn1.running_var" in ref[3]

    def errs(r):
        return (max(float((a - b).abs().max()) for a, b in zip(r[0], ref[0])), abs(r[1] - ref[1]) / abs(ref[1]),
                max(rel(r[2][n], ref[2][n]) for n in ref[2]), max(rel(r[3][n], ref[3][n]) for n in ref[3]))
    e_l, e_t = errs(lib), errs(tst)
    print("\nvs fp64, stem on library / on torch: joints %.2e / %.2e px, loss %.2e / %.2e, worst encoder weight "
          "gradient %.2e / %.2e, worst running stat %.2e / %.2e" % tuple(v for pair in zip(e_l, e_t) for v in pair))
    for name, a, b in zip(("joints", "loss", "gradient", "running stat"), e_l, e_t):
        assert a <= 2 * b + 1e-7, (name, a, b)


def test_stem_flag_needs_the_encoder_flag(cuda_pkg):
    with pytest.raises(ValueError, match="train_encoder_on_library"):
        cuda_pkg.CDRNet(synth.make_cfg(50, 19), trainable=True, train_stem_on_library=True)
