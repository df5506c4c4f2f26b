"""conv1x1 (a 1x1 Conv2d with optional bias) in training, over the whole domain the library accepts, against fp64 torch
autograd with a per-element gate: every 1x1 conv of the CDRNet head, the fusion block at other widths, channel counts
that are not multiples of 64, a partial last pixel tile, every wgrad slice count the plan produces, exponents far
outside O(1), the memory contract of the cdr_conv1x1_train_* entry points, layouts, streams, CUDA graphs, non-finite
inputs, and forward_train on it."""
import copy
import ctypes as C
import functools

import pytest
import torch
import torch.nn.functional as F

import train_conv_checks as checks
from fast_3d_human_pose_estimation_b200 import synth
from train_conv_checks import GATE_C, SENTINEL, TINY, Region, bits_equal, f32_region, graph_replay, on_side_stream

pytestmark = pytest.mark.gpu

def slices(n, cin, cout, h, w):
    """The number of K slices of the weight gradient: M = Cout over the pixels, N = Cin, 1 tap."""
    return checks.wgrad_slices(n * h * w, cout, cin, 1)


# (N, Cin, Cout, H, W, bias): the head's layers at the default widths (fusion_hid_ch1 = 300)
HEAD = [(2048, 300, 8, 8), (800, 400, 8, 8), (400, 400, 8, 8), (300, 2048, 8, 8), (256, 19, 64, 64)]
# the fusion block at fusion_hid_ch1 = 12, 36, 600 (fusion_hid_ch2 = 4/3 of it): conv_layer1, conv_layer2[0] and [3],
# out_layer
FUSION = [s for h1 in (12, 36, 600) for s in ((2048, h1), (8 * h1 // 3, 4 * h1 // 3), (4 * h1 // 3, 4 * h1 // 3),
                                               (h1, 2048))]
# (N, Cin, Cout, H, W, slices): channels = 1 and 63 (mod 64), a half-full last 128-pixel tile, and every wgrad slice
# count the plan produces (1 .. 512)
TABLE = [
    (1, 1, 1, 8, 8, 1),          # 64 pixels: a half-full 128-pixel tile, one channel in and out
    (3, 65, 127, 8, 8, 1),       # 192 pixels: the last tile half full
    (2, 127, 65, 16, 4, 1),      # H != W
    (5, 63, 1, 8, 16, 1),
    (2, 1025, 191, 8, 8, 1),     # 17 forward K blocks: a partial kSplitChunk chunk
    (2, 16, 16, 32, 32, 2),
    (4, 16, 16, 32, 32, 4),
    (3, 129, 129, 32, 32, 2),    # 1.5 images per slice: a slice ends mid-image; padded M and N tiles in wgrad
    (8, 16, 16, 32, 32, 8),
    (16, 16, 16, 32, 32, 16),
    (32, 16, 16, 32, 32, 32),
    (64, 16, 16, 32, 32, 64),
    (128, 16, 16, 32, 32, 128),
    (256, 16, 16, 32, 32, 256),
    (512, 16, 16, 32, 32, 512),  # the largest slice count the plan produces
    (7, 3, 5, 24, 24, 1),        # H*W = 576: a K slice of 64 pixels ends mid-row
]

WORST = {"y": 0.0, "dx": 0.0, "dw": 0.0, "db": 0.0}
_report_worst = checks.report_worst(WORST, __name__)
gate = functools.partial(checks.gate, worst=WORST)


def inputs(n, cin, cout, h, w, seed=0, ex=0, ew=0, edy=0, bias=True):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n, cin, h, w), device="cuda", generator=g) * 2.0 ** ex
    wt = torch.randn((cout, cin, 1, 1), device="cuda", generator=g) * ((1.0 / cin ** 0.5) * 2.0 ** ew)
    b = torch.randn((cout,), device="cuda", generator=g) * 2.0 ** (ex + ew) if bias else None
    dy = torch.randn((n, cout, h, w), device="cuda", generator=g) * 2.0 ** edy
    return x, wt, b, dy


def ours(pkg, x, w, b, dy, need=(True, True, True)):
    x = x.detach().requires_grad_(need[0])
    w = w.detach().requires_grad_(need[1])
    b = None if b is None else b.detach().requires_grad_(need[2])
    y = pkg.conv1x1(x, w, b)
    wanted = [t for t, r in ((x, need[0]), (w, need[1]), (b, need[2])) if r and t is not None]
    return (y.detach(), *torch.autograd.grad(y, wanted, dy))


def reference(x, w, b, dy):
    """fp64 autograd of F.conv2d -> (y, dx, dW, db), and the same on |x|, |w|, |b|, |dy| -> their magnitudes m."""
    out = []
    for f in (lambda t: t, torch.abs):
        x64 = f(x.detach().double()).requires_grad_(True)
        w64 = f(w.detach().double()).requires_grad_(True)
        b64 = f(b.detach().double()) if b is not None else None
        y64 = F.conv2d(x64, w64, b64)
        dy64 = f(dy.detach().double())
        dx64, dw64 = torch.autograd.grad(y64, (x64, w64), dy64)
        out.append((y64.detach(), dx64, dw64, dy64.sum((0, 2, 3))))
    return out


def check_all(pkg, x, w, b, dy, label, max_gate=True):
    got, (ref, mag) = ours(pkg, x, w, b, dy), reference(x, w, b, dy)
    names = ("y", "dx", "dw", "db") if b is not None else ("y", "dx", "dw")
    r = {k: gate(k, got[i], ref[i], mag[i], max_gate) for i, k in enumerate(names)}
    print(f"\n{label}: " + ", ".join(f"{k} {v[0]:.2e}/m {v[1]:.2e}/max" for k, v in r.items()))
    return got


@pytest.mark.parametrize("n", [1, 2, 64])
@pytest.mark.parametrize("cin,cout,h,w", HEAD)
def test_head_layers(cuda_pkg, cin, cout, h, w, n):
    check_all(cuda_pkg, *inputs(n, cin, cout, h, w, seed=cin + cout + n), f"N={n} {cin}->{cout} {h}x{w}")


@pytest.mark.parametrize("cin,cout", FUSION)
def test_fusion_widths(cuda_pkg, cin, cout):
    check_all(cuda_pkg, *inputs(2, cin, cout, 8, 8, seed=cin * 7 + cout), f"N=2 {cin}->{cout} 8x8")


@pytest.mark.parametrize("n,cin,cout,h,w,s", TABLE)
def test_shape_table(cuda_pkg, n, cin, cout, h, w, s):
    assert slices(n, cin, cout, h, w) == s
    check_all(cuda_pkg, *inputs(n, cin, cout, h, w, seed=n + cin + cout + h), f"N={n} {cin}->{cout} {h}x{w} slices={s}")


def test_without_bias(cuda_pkg):
    x, w, _, dy = inputs(3, 65, 127, 8, 8, seed=3, bias=False)
    y, dx, dw = check_all(cuda_pkg, x, w, None, dy, "N=3 65->127 8x8 no bias")
    y0 = cuda_pkg.conv1x1(x, w, torch.zeros(127, device="cuda"))
    assert torch.equal(y, y0)


# (e_x, e_w, e_dy): x, w and dy times 2^e (the bias follows x*w).  An amax below 2^-114 is where an uncapped
# 2^(13 - ilogb(amax)) scale overflows to +Inf.
EXPONENTS = [(-120, 0, 0), (100, 0, 0), (0, -120, 0), (0, 100, 0), (0, 0, -120), (0, 0, 100)]
SWEEP_SHAPES = [(2, 800, 400, 8, 8), (3, 65, 127, 8, 8)]


@pytest.mark.parametrize("n,cin,cout,h,w", SWEEP_SHAPES)
@pytest.mark.parametrize("ex,ew,edy", EXPONENTS)
def test_exponent_sweep(cuda_pkg, n, cin, cout, h, w, ex, ew, edy):
    x, wt, b, dy = inputs(n, cin, cout, h, w, seed=5, ex=ex, ew=ew, edy=edy)
    check_all(cuda_pkg, x, wt, b, dy, f"N={n} {cin}->{cout} 2^({ex}, {ew}, {edy})")


@pytest.mark.parametrize("n,cin,cout,h,w", SWEEP_SHAPES)
def test_subnormal_input(cuda_pkg, n, cin, cout, h, w):
    """Every x value subnormal (|x| in [2^-135, 2^-134)), dy times 2^100 so that dW = sum x dy is a normal float; y
    is below the fp32 normal range and only has to be near zero."""
    x, wt, _, dy = inputs(n, cin, cout, h, w, seed=6, edy=100, bias=False)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.sign(x) * (1 + torch.rand(x.shape, device="cuda", generator=g)) * 2.0 ** -135
    assert bool(((x != 0) & (x.abs() < 2.0 ** -126)).all())
    check_all(cuda_pkg, x, wt, None, dy, f"N={n} {cin}->{cout} subnormal x", max_gate=False)


# ---- memory contract of the C ABI: exact byte counts, guard bytes around every buffer, stale workspace contents ----
def _abi_run(pkg, x, w, b, dy, fill, gen):
    """forward, then full, dx-only, dW-only and db-only backward through the C ABI, every buffer guarded."""
    L = pkg._lib.lib()
    n, cin, h, wd = x.shape
    cout = w.shape[0]
    sb, wb = C.c_size_t(), C.c_size_t()
    pkg._lib.check(L.cdr_conv1x1_train_workspace_bytes(n, cin, cout, h, wd, C.byref(sb), C.byref(wb)))
    st = pkg._lib.current_stream_ptr()
    ptr = pkg._lib.ptr
    saved, ws = Region(sb.value, fill, gen), Region(wb.value, fill, gen)
    ry, y = f32_region((n, cout, h, wd))
    pkg._lib.check(L.cdr_conv1x1_train_forward(ptr(x), ptr(w), ptr(b), n, cin, cout, h, wd, ptr(y), ptr(saved.inner),
                                               sb.value, ptr(ws.inner), wb.value, st))
    regions, outs = [saved, ws, ry], {"y": y}
    for tag, want in (("", "xwb"), ("_xonly", "x"), ("_wonly", "w"), ("_bonly", "b")):
        ws_b = Region(wb.value, fill, gen)
        rdx, dx = f32_region((n, cin, h, wd)) if "x" in want else (None, None)
        rdw, dw = f32_region((cout, cin, 1, 1)) if "w" in want else (None, None)
        rdb, db = f32_region((cout,)) if "b" in want else (None, None)
        pkg._lib.check(L.cdr_conv1x1_train_backward(ptr(saved.inner), ptr(w), ptr(dy), n, cin, cout, h, wd, ptr(dx),
                                                    ptr(dw), ptr(db), ptr(ws_b.inner), wb.value, st))
        regions += [r for r in (ws_b, rdx, rdw, rdb) if r is not None]
        for k, t in (("dx", dx), ("dw", dw), ("db", db)):
            if t is not None:
                outs[k + tag] = t
    assert all(r.guards_intact() for r in regions), "a write landed outside its buffer"
    for k, t in outs.items():
        assert not bool((t.view(torch.int32) == SENTINEL * 0x01010101).any()), f"{k}: elements never written"
    return {k: t.clone() for k, t in outs.items()}


@pytest.mark.parametrize("n,cin,cout,h,w", [(1, 1, 1, 8, 8), (3, 65, 127, 8, 8), (2, 300, 19, 16, 16),
                                            (4, 127, 300, 8, 8)])
def test_memory_contract(cuda_pkg, n, cin, cout, h, w):
    x, wt, b, dy = inputs(n, cin, cout, h, w, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(12)
    runs = [_abi_run(cuda_pkg, x, wt, b, dy, fill, gen) for fill in (0x00, 0xFF, "random")]
    for k in runs[0]:
        assert all(bits_equal(runs[0][k], r[k]) for r in runs[1:]), f"{k} depends on stale workspace contents"
    a = runs[0]
    assert bits_equal(a["dx_xonly"], a["dx"]) and bits_equal(a["dw_wonly"], a["dw"])
    assert bits_equal(a["db_bonly"], a["db"])
    got = ours(cuda_pkg, x, wt, b, dy)                   # the autograd op is the same computation
    assert all(bits_equal(g, a[k]) for g, k in zip(got, ("y", "dx", "dw", "db")))
    ref, mag = reference(x, wt, b, dy)
    for i, k in enumerate(("y", "dx", "dw", "db")):
        gate(k, a[k], ref[i], mag[i])


def test_needs_input_grad_each_alone(cuda_pkg):
    x, w, b, dy = inputs(3, 65, 127, 8, 8, seed=13)
    full = ours(cuda_pkg, x, w, b, dy)
    for i, need in enumerate(((True, False, False), (False, True, False), (False, False, True))):
        (g,) = ours(cuda_pkg, x, w, b, dy, need)[1:]
        assert bits_equal(g, full[1 + i])


# ---- layouts, streams, CUDA graphs, repeated backward ----
LAYOUT_SHAPE = (4, 127, 300, 8, 8)


def test_layouts_give_the_same_bits(cuda_pkg):
    x, w, b, dy = inputs(*LAYOUT_SHAPE, seed=21)
    base = ours(cuda_pkg, x, w, b, dy)
    x_cl, dy_cl = x.to(memory_format=torch.channels_last), dy.to(memory_format=torch.channels_last)
    w_cl = w.to(memory_format=torch.channels_last)
    b_nc = torch.stack([b, b], 1)[:, 0]                           # stride 2
    x_nc = torch.cat([x, x], 3)[:, :, :, :x.shape[3]]            # a non-contiguous slice
    assert not x_cl.is_contiguous() and not dy_cl.is_contiguous() and not b_nc.is_contiguous()
    assert not x_nc.is_contiguous()
    for xs, ws, bs, dys in ((x_cl, w_cl, b_nc, dy_cl), (x_nc, w, b, dy)):
        got = ours(cuda_pkg, xs, ws, bs, dys)
        assert all(bits_equal(a.contiguous(), g.contiguous()) for a, g in zip(base, got))


def test_side_stream_gives_the_same_bits(cuda_pkg):
    x, w, b, dy = inputs(*LAYOUT_SHAPE, seed=22)
    base = ours(cuda_pkg, x, w, b, dy)
    got = on_side_stream(ours, cuda_pkg, x, w, b, dy)
    assert all(bits_equal(a, g) for a, g in zip(base, got))


def test_cuda_graph_replay_equals_eager(cuda_pkg):
    x, w, b, dy = inputs(*LAYOUT_SHAPE, seed=23)
    sx, sw, sb = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    sdy = dy.clone()

    def step():
        y = cuda_pkg.conv1x1(sx, sw, sb)
        return (y.detach(), *torch.autograd.grad(y, (sx, sw, sb), sdy))
    x2, w2, b2, dy2 = inputs(*LAYOUT_SHAPE, seed=24)
    static_out = graph_replay(step, (sx, sw, sb, sdy), (x2, w2, b2, dy2))
    eager = ours(cuda_pkg, x2, w2, b2, dy2)
    assert all(bits_equal(a, e) for a, e in zip(static_out, eager))


def test_two_backward_calls_and_zero_dy(cuda_pkg):
    x, w, b, _ = inputs(*LAYOUT_SHAPE, seed=25)
    x, w, b = x.requires_grad_(True), w.requires_grad_(True), b.requires_grad_(True)
    y = cuda_pkg.conv1x1(x, w, b)
    zero = torch.autograd.grad(y, (x, w, b), torch.zeros_like(y), retain_graph=True)
    assert all(bool((g == 0).all()) for g in zero)                 # exact zeros, no NaN from the pad columns
    dy = torch.randn_like(y)
    first = torch.autograd.grad(y, (x, w, b), dy, retain_graph=True)
    second = torch.autograd.grad(y, (x, w, b), dy)
    assert all(bits_equal(a, c) for a, c in zip(first, second))


# ---- non-finite inputs: a diverging run is never reported finite ----
@pytest.mark.parametrize("where,value", [("x", float("nan")), ("x", float("inf")), ("dy", float("nan")),
                                         ("dy", float("-inf"))])
def test_non_finite_inputs(cuda_pkg, where, value):
    x, w, b, dy = inputs(2, 65, 127, 8, 8, seed=31)
    (x if where == "x" else dy)[1, 7, 3, 5] = value
    got, (ref, mag) = ours(cuda_pkg, x, w, b, dy), reference(x, w, b, dy)
    assert not all(bool(torch.isfinite(r).all()) for r in ref)
    for i, k in enumerate(("y", "dx", "dw", "db")):
        gate(k, got[i], ref[i], mag[i], max_gate=False)
        assert torch.equal(torch.isfinite(got[i]), torch.isfinite(ref[i])), k


# ---- forward_train ----
def _model(cuda_pkg):
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), trainable=True)
    with torch.no_grad():
        m.decoder.final_layer.weight.mul_(10.0)      # train-mode BN keeps activations O(1): peaky heat-maps need gain
        m.decoder.final_layer.bias.normal_(0.0, 0.01)
    return m.cuda().train()


def _inputs(b):
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    targets = [torch.from_numpy(gt["gt2d_l"]).float().cuda(), torch.from_numpy(gt["gt2d_r"]).float().cuda()]
    return imgs, Ps, targets, torch.from_numpy(gt["vis"]).float().cuda()


def _head_convs(m):
    """name -> Conv2d of every 1x1 conv of the head"""
    cf = m.CF
    convs = {"CF.conv_layer1.0": cf.conv_layer1[0], "CF.conv_layer2.0": cf.conv_layer2[0],
             "CF.conv_layer2.3": cf.conv_layer2[3], "decoder.final_layer": m.decoder.final_layer}
    for v in range(len(cf.out_layer)):
        convs[f"CF.out_layer.{v}.0"] = cf.out_layer[v][0]
    return convs


def test_forward_train_does_not_call_the_conv_modules(cuda_pkg):
    m = _model(cuda_pkg)
    imgs, Ps, targets, vis = _inputs(2)

    def boom(*a, **k):
        raise AssertionError("head Conv2d module called")
    convs = _head_convs(m)
    for c in convs.values():
        c.forward = boom
    kps, xyz = m(imgs, Ps)
    loss = sum(cuda_pkg.MPJPELoss(True)(kps[v], targets[v], vis) for v in range(2))
    loss.backward()
    assert bool(torch.isfinite(xyz).all())
    for name, c in convs.items():
        assert c.weight.grad is not None and bool(torch.isfinite(c.weight.grad).all()), name
        assert c.bias.grad is not None and bool(torch.isfinite(c.bias.grad).all()), name


def test_training_step_vs_torch_conv2d(cuda_pkg, monkeypatch):
    """One training step of the same model with the head's 1x1 convs on libcdrhead and on cuDNN (fp32, TF32 off)."""
    from fast_3d_human_pose_estimation_b200 import autograd as AG
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ours_m = _model(cuda_pkg)
        theirs = copy.deepcopy(ours_m)
        imgs, Ps, targets, vis = _inputs(2)

        def step(model):
            model.zero_grad()
            kps, _ = model(imgs, Ps)
            loss = sum(cuda_pkg.MPJPELoss(True)(kps[v], targets[v], vis) for v in range(2))
            loss.backward()
            return [k.detach() for k in kps], float(loss)
        heat_grads = []                     # dL/dheat of both views, as final_layer's backward receives it
        lib_conv1x1 = AG.conv1x1

        def spy(x, w, b=None):
            y = lib_conv1x1(x, w, b)
            if w is ours_m.decoder.final_layer.weight:
                y.register_hook(lambda g: heat_grads.append(g.detach().double()))
            return y
        with monkeypatch.context() as mp:
            mp.setattr(AG, "conv1x1", spy)
            k_o, l_o = step(ours_m)
        with monkeypatch.context() as mp:
            mp.setattr(AG, "conv1x1", lambda x, w, b=None: F.conv2d(x, w, b))
            k_t, l_t = step(theirs)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    d2 = max(float((a - b).abs().max()) for a, b in zip(k_o, k_t))
    print(f"\n2D joints {d2:.2e} px, loss {l_o:.8f} vs {l_t:.8f}")
    assert d2 <= 1e-3
    assert abs(l_o - l_t) <= 1e-5 * abs(l_t)
    co, ct = _head_convs(ours_m), _head_convs(theirs)

    def compare(name, a, b):
        a, b = a.double().flatten(), b.double().flatten()
        cos, ratio = float(torch.dot(a, b) / (a.norm() * b.norm())), float(a.norm() / b.norm())
        print(f"{name}: cosine {cos:.7f}, norm ratio {ratio:.7f}")
        assert cos >= 0.9999 and abs(ratio - 1) <= 1e-3, name
    for name in co:
        compare(name + ".weight", co[name].weight.grad, ct[name].weight.grad)
    # decoder.final_layer feeds soft_argmax_2d, a softmax over each heat-map: a constant added to one map changes
    # nothing, so the true gradient of final_layer.bias is the sum over the map of dL/dheat = 0, and both sides return
    # rounding noise whose direction means nothing.  Checked instead: our bias gradient equals the fp64 sum of the
    # heat-map gradient the op received, inside the per-element gate, and that sum is zero up to rounding.
    assert len(heat_grads) == 2
    ref = sum(g.sum((0, 2, 3)) for g in heat_grads)
    mag = sum(g.abs().sum((0, 2, 3)) for g in heat_grads)
    gb = co["decoder.final_layer"].bias.grad.double()
    print(f"decoder.final_layer.bias: max |grad| {float(gb.abs().max()):.3e}, max |fp64 sum| {float(ref.abs().max()):.3e}"
          f", min sum |dL/dheat| {float(mag.min()):.3e}")
    assert bool((gb - ref).abs().le(GATE_C * mag + TINY).all())
    assert bool(ref.abs().le(1e-5 * mag).all())
    assert bool(torch.isfinite(ct["decoder.final_layer"].bias.grad).all())
    # a conv bias in front of a train-mode BatchNorm has a true gradient of 0 as well: only its finiteness and size are
    # checked, against the weight gradient of the same layer
    for name in co:
        if name == "decoder.final_layer":
            continue
        gb, gw = co[name].bias.grad, co[name].weight.grad
        assert bool(torch.isfinite(gb).all()), name
        small = float(gb.abs().max()) <= 1e-3 * float(gw.abs().max())
        print(f"{name}.bias: max |grad| {float(gb.abs().max()):.3e} (weight {float(gw.abs().max()):.3e})")
        assert small, name
