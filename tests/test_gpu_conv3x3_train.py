"""conv3x3 (a 3x3 pad-1 Conv2d without bias, stride 1 or 2) in training, over the whole domain the library accepts,
against fp64 torch autograd with a per-element gate: every distinct 3x3 conv of ResNet-50/101/152 at 256 x 256 inputs,
every wgrad slice count the plan produces, exponents far outside O(1), the memory contract of the
cdr_conv3x3_train_* entry points, layouts, streams, CUDA graphs, non-finite inputs, and ResNet.forward_train, the
encoder's Bottleneck blocks on it."""
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

def slices(n, cin, cout, h, w, s):
    """The number of K slices of the weight gradient: M = Cout over the output pixels, N = Cin, 9 taps; h x w is the
    input map."""
    return checks.wgrad_slices(n * (h // s) * (w // s), cout, cin, 9)


# (C, input H = W, stride): every distinct 3x3 conv of ResNet-50/101/152 at 256 x 256 images (conv2 of each block;
# the first block of layer2..4 carries the stride)
RESNET = [(64, 64, 1), (128, 32, 1), (256, 16, 1), (512, 8, 1), (128, 64, 2), (256, 32, 2), (512, 16, 2)]
# (N, Cin, Cout, h, w, stride, slices): every wgrad slice count the plan produces (1 .. 64), slices that end mid-image,
# half-full last 128-pixel tiles, H != W, padded N tiles, the widest channel counts
TABLE = [
    (1, 64, 64, 8, 8, 1, 1),         # 64 output pixels: a half-full 128-pixel tile
    (3, 192, 64, 4, 16, 1, 1),       # H*W = 64 with H != W, an odd N: the last tile half full; a padded wgrad N tile
    (2, 128, 128, 16, 8, 1, 1),      # H*W = 128, W = 8
    (2, 64, 64, 16, 64, 1, 2),       # W = 64, H = 16
    (3, 64, 128, 32, 32, 1, 2),      # 1.5 images per slice: a slice ends mid-image
    (3, 64, 64, 64, 64, 2, 2),       # the same at stride 2
    (4, 64, 64, 32, 32, 1, 4),
    (8, 64, 64, 32, 32, 1, 8),
    (16, 64, 64, 64, 64, 2, 16),
    (32, 64, 64, 32, 32, 1, 32),
    (64, 64, 64, 32, 32, 1, 64),     # the largest slice count the plan produces
    (1, 2048, 64, 8, 8, 1, 1),       # forward K = 9 * 2048
    (2, 64, 2048, 16, 16, 2, 1),     # dgrad K at stride 2 = 4 * 2048 per phase
    (2, 192, 320, 16, 16, 2, 1),     # Cin, Cout not multiples of 128: padded M and N tiles
]

WORST = {"y": 0.0, "dx": 0.0, "dw": 0.0}
_report_worst = checks.report_worst(WORST, __name__)
gate = functools.partial(checks.gate, worst=WORST)


def inputs(n, cin, cout, h, w, s, seed=0, ex=0, ew=0, edy=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n, cin, h, w), device="cuda", generator=g) * 2.0 ** ex
    wt = torch.randn((cout, cin, 3, 3), device="cuda", generator=g) * ((1.0 / (9 * cin) ** 0.5) * 2.0 ** ew)
    dy = torch.randn((n, cout, h // s, w // s), device="cuda", generator=g) * 2.0 ** edy
    return x, wt, dy, s


def ours(pkg, x, w, dy, s, need=(True, True)):
    x = x.detach().requires_grad_(need[0])
    w = w.detach().requires_grad_(need[1])
    y = pkg.conv3x3(x, w, s)
    wanted = [t for t, r in ((x, need[0]), (w, need[1])) if r]
    return (y.detach(), *torch.autograd.grad(y, wanted, dy))


def reference(x, w, dy, s):
    """fp64 autograd of F.conv2d -> (y, dx, dW), and the same on |x|, |w|, |dy| -> their magnitudes m."""
    out = []
    for f in (lambda t: t, torch.abs):
        x64 = f(x.detach().double()).requires_grad_(True)
        w64 = f(w.detach().double()).requires_grad_(True)
        y64 = F.conv2d(x64, w64, stride=s, padding=1)
        dy64 = f(dy.detach().double())
        dx64, dw64 = torch.autograd.grad(y64, (x64, w64), dy64)
        out.append((y64.detach(), dx64, dw64))
    return out


def check_all(pkg, x, w, dy, s, label, max_gate=True):
    got, (ref, mag) = ours(pkg, x, w, dy, s), reference(x, w, dy, s)
    r = {k: gate(k, got[i], ref[i], mag[i], max_gate) for i, k in enumerate(("y", "dx", "dw"))}
    print(f"\n{label}: " + ", ".join(f"{k} {v[0]:.2e}/m {v[1]:.2e}/max" for k, v in r.items()))
    return got


@pytest.mark.parametrize("n", [1, 2, 64])
@pytest.mark.parametrize("c,h,s", RESNET)
def test_resnet_layers(cuda_pkg, c, h, s, n):
    check_all(cuda_pkg, *inputs(n, c, c, h, h, s, seed=c + h + s + n), f"N={n} {c}->{c} {h}x{h} stride {s}")


@pytest.mark.parametrize("n,cin,cout,h,w,s,sl", TABLE)
def test_shape_table(cuda_pkg, n, cin, cout, h, w, s, sl):
    assert slices(n, cin, cout, h, w, s) == sl
    check_all(cuda_pkg, *inputs(n, cin, cout, h, w, s, seed=n + cin + cout + h + s),
              f"N={n} {cin}->{cout} {h}x{w} stride {s} slices={sl}")


# (e_x, e_w, e_dy): x, w and dy times 2^e.  An amax below 2^-114 is where an uncapped 2^(13 - ilogb(amax)) scale
# overflows to +Inf.
EXPONENTS = [(-120, 0, 0), (100, 0, 0), (0, -120, 0), (0, 100, 0), (0, 0, -120), (0, 0, 100)]
SWEEP_SHAPES = [(2, 128, 128, 16, 16, 1), (2, 128, 128, 32, 32, 2)]


@pytest.mark.parametrize("n,cin,cout,h,w,s", SWEEP_SHAPES)
@pytest.mark.parametrize("ex,ew,edy", EXPONENTS)
def test_exponent_sweep(cuda_pkg, n, cin, cout, h, w, s, ex, ew, edy):
    x, wt, dy, _ = inputs(n, cin, cout, h, w, s, seed=5, ex=ex, ew=ew, edy=edy)
    check_all(cuda_pkg, x, wt, dy, s, f"N={n} {cin}->{cout} stride {s} 2^({ex}, {ew}, {edy})")


@pytest.mark.parametrize("n,cin,cout,h,w,s", SWEEP_SHAPES)
def test_subnormal_input(cuda_pkg, n, cin, cout, h, w, s):
    """Every x value subnormal (|x| in [2^-135, 2^-134)), dy times 2^100 so that dW = sum x dy is a normal float; y
    is below the fp32 normal range and only has to be near zero."""
    x, wt, dy, _ = inputs(n, cin, cout, h, w, s, seed=6, edy=100)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.sign(x) * (1 + torch.rand(x.shape, device="cuda", generator=g)) * 2.0 ** -135
    assert bool(((x != 0) & (x.abs() < 2.0 ** -126)).all())
    check_all(cuda_pkg, x, wt, dy, s, f"N={n} {cin}->{cout} stride {s} subnormal x", max_gate=False)


# ---- memory contract of the C ABI: exact byte counts, guard bytes around every buffer, stale workspace contents ----
def _abi_run(pkg, x, w, dy, s, fill, gen):
    """forward, then full, dx-only and dW-only backward through the C ABI, every buffer guarded."""
    L = pkg._lib.lib()
    n, cin, h, wd = x.shape
    cout = w.shape[0]
    sb, wb = C.c_size_t(), C.c_size_t()
    pkg._lib.check(L.cdr_conv3x3_train_workspace_bytes(n, cin, cout, h, wd, s, C.byref(sb), C.byref(wb)))
    st = pkg._lib.current_stream_ptr()
    ptr = pkg._lib.ptr
    saved, ws = Region(sb.value, fill, gen), Region(wb.value, fill, gen)
    ry, y = f32_region((n, cout, h // s, wd // s))
    pkg._lib.check(L.cdr_conv3x3_train_forward(ptr(x), ptr(w), n, cin, cout, h, wd, s, ptr(y), ptr(saved.inner),
                                               sb.value, ptr(ws.inner), wb.value, st))
    regions, outs = [saved, ws, ry], {"y": y}
    for tag, want in (("", "xw"), ("_xonly", "x"), ("_wonly", "w")):
        ws_b = Region(wb.value, fill, gen)
        rdx, dx = f32_region((n, cin, h, wd)) if "x" in want else (None, None)
        rdw, dw = f32_region((cout, cin, 3, 3)) if "w" in want else (None, None)
        pkg._lib.check(L.cdr_conv3x3_train_backward(ptr(saved.inner), ptr(w), ptr(dy), n, cin, cout, h, wd, s, ptr(dx),
                                                    ptr(dw), ptr(ws_b.inner), wb.value, st))
        regions += [r for r in (ws_b, rdx, rdw) if r is not None]
        for k, t in (("dx", dx), ("dw", dw)):
            if t is not None:
                outs[k + tag] = t
    assert all(r.guards_intact() for r in regions), "a write landed outside its buffer"
    for k, t in outs.items():
        assert not bool((t.view(torch.int32) == SENTINEL * 0x01010101).any()), f"{k}: elements never written"
    return {k: t.clone() for k, t in outs.items()}


@pytest.mark.parametrize("n,cin,cout,h,w,s", [(1, 64, 64, 8, 8, 1), (3, 192, 64, 4, 16, 1), (2, 128, 192, 16, 16, 2),
                                              (3, 64, 128, 32, 32, 1)])
def test_memory_contract(cuda_pkg, n, cin, cout, h, w, s):
    x, wt, dy, _ = inputs(n, cin, cout, h, w, s, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(12)
    runs = [_abi_run(cuda_pkg, x, wt, dy, s, fill, gen) for fill in (0x00, 0xFF, "random")]
    for k in runs[0]:
        assert all(bits_equal(runs[0][k], r[k]) for r in runs[1:]), f"{k} depends on stale workspace contents"
    a = runs[0]
    assert bits_equal(a["dx_xonly"], a["dx"]) and bits_equal(a["dw_wonly"], a["dw"])
    got = ours(cuda_pkg, x, wt, dy, s)                   # the autograd op is the same computation
    assert all(bits_equal(g, a[k]) for g, k in zip(got, ("y", "dx", "dw")))
    ref, mag = reference(x, wt, dy, s)
    for i, k in enumerate(("y", "dx", "dw")):
        gate(k, a[k], ref[i], mag[i])


@pytest.mark.parametrize("s", [1, 2])
def test_needs_input_grad_each_alone(cuda_pkg, s):
    x, w, dy, _ = inputs(3, 64, 128, 16, 16, s, seed=13)
    full = ours(cuda_pkg, x, w, dy, s)
    for i, need in enumerate(((True, False), (False, True))):
        (g,) = ours(cuda_pkg, x, w, dy, s, need)[1:]
        assert bits_equal(g, full[1 + i])


# ---- layouts, streams, CUDA graphs, repeated backward ----
LAYOUT_SHAPES = [(4, 128, 64, 16, 16, 1), (4, 64, 128, 32, 32, 2)]


@pytest.mark.parametrize("shape", LAYOUT_SHAPES)
def test_layouts_give_the_same_bits(cuda_pkg, shape):
    x, w, dy, s = inputs(*shape, seed=21)
    base = ours(cuda_pkg, x, w, dy, s)
    x_cl, dy_cl = x.to(memory_format=torch.channels_last), dy.to(memory_format=torch.channels_last)
    w_cl = w.to(memory_format=torch.channels_last)
    x_nc = torch.cat([x, x], 3)[:, :, :, :x.shape[3]]            # a non-contiguous slice
    assert not x_cl.is_contiguous() and not dy_cl.is_contiguous() and not w_cl.is_contiguous()
    assert not x_nc.is_contiguous()
    for xs, ws, dys in ((x_cl, w_cl, dy_cl), (x_nc, w, dy)):
        got = ours(cuda_pkg, xs, ws, dys, s)
        assert all(bits_equal(a.contiguous(), g.contiguous()) for a, g in zip(base, got))


@pytest.mark.parametrize("shape", LAYOUT_SHAPES)
def test_side_stream_gives_the_same_bits(cuda_pkg, shape):
    x, w, dy, s = inputs(*shape, seed=22)
    base = ours(cuda_pkg, x, w, dy, s)
    got = on_side_stream(ours, cuda_pkg, x, w, dy, s)
    assert all(bits_equal(a, g) for a, g in zip(base, got))


@pytest.mark.parametrize("shape", LAYOUT_SHAPES)
def test_cuda_graph_replay_equals_eager(cuda_pkg, shape):
    x, w, dy, s = inputs(*shape, seed=23)
    sx, sw, sdy = x.clone().requires_grad_(True), w.clone().requires_grad_(True), dy.clone()

    def step():
        y = cuda_pkg.conv3x3(sx, sw, s)
        return (y.detach(), *torch.autograd.grad(y, (sx, sw), sdy))
    x2, w2, dy2, _ = inputs(*shape, seed=24)
    static_out = graph_replay(step, (sx, sw, sdy), (x2, w2, dy2))
    eager = ours(cuda_pkg, x2, w2, dy2, s)
    assert all(bits_equal(a, e) for a, e in zip(static_out, eager))


@pytest.mark.parametrize("shape", LAYOUT_SHAPES)
def test_two_backward_calls_and_zero_dy(cuda_pkg, shape):
    x, w, _, s = inputs(*shape, seed=25)
    x, w = x.requires_grad_(True), w.requires_grad_(True)
    y = cuda_pkg.conv3x3(x, w, s)
    zero = torch.autograd.grad(y, (x, w), torch.zeros_like(y), retain_graph=True)
    assert all(bool((g == 0).all()) for g in zero)                 # exact zeros
    dy = torch.randn_like(y)
    first = torch.autograd.grad(y, (x, w), dy, retain_graph=True)
    second = torch.autograd.grad(y, (x, w), dy)
    assert all(bits_equal(a, c) for a, c in zip(first, second))


# ---- non-finite inputs: a diverging run is never reported finite ----
@pytest.mark.parametrize("s", [1, 2])
@pytest.mark.parametrize("where,value", [("x", float("nan")), ("x", float("inf")), ("dy", float("nan")),
                                         ("dy", float("-inf"))])
def test_non_finite_inputs(cuda_pkg, where, value, s):
    """Non-finite exactly where the reference is, except one case: at stride 2 dx is a transposed conv with the
    weight zero-padded to 4x4, so a non-finite dy element also reaches the dx row and column just past its 3x3
    footprint (Inf or NaN times the zero taps).  There dx may be non-finite where the reference is finite."""
    x, w, dy, _ = inputs(2, 64, 128, 16, 16, s, seed=31)
    (x if where == "x" else dy)[1, 7, 3, 5] = value
    got, (ref, mag) = ours(cuda_pkg, x, w, dy, s), reference(x, w, dy, s)
    assert not all(bool(torch.isfinite(r).all()) for r in ref)
    for i, k in enumerate(("y", "dx", "dw")):
        wider = None
        if k == "dx" and s == 2:
            w4 = F.pad(w.double(), (0, 1, 0, 1))
            wider = ~torch.isfinite(F.conv_transpose2d(dy.double(), w4, stride=2, padding=1))
            assert torch.equal(~torch.isfinite(got[i]), wider | ~torch.isfinite(ref[i])), k
        else:
            assert torch.equal(torch.isfinite(got[i]), torch.isfinite(ref[i])), k
        gate(k, got[i], ref[i], mag[i], max_gate=False, nonfinite=wider)


# ---- ResNet.forward_train: the encoder's bottleneck blocks on the library ----
def _encoder(cuda_pkg):
    torch.manual_seed(0)
    return cuda_pkg.ResNet(synth.make_cfg(50, 19)).cuda().train()


def _encoder_convs(enc):
    """name -> Conv2d of every encoder conv but the stem's"""
    return {n: c for n, c in enc.named_modules() if isinstance(c, torch.nn.Conv2d) and n != "conv1"}


def test_encoder_forward_train_does_not_call_the_conv_modules(cuda_pkg):
    enc = _encoder(cuda_pkg)
    x = synth.make_images(2, seed=1)[0].cuda()

    def boom(*a, **k):
        raise AssertionError("encoder Conv2d module called")
    convs = _encoder_convs(enc)
    assert len(convs) == 16 * 3 + 4
    for c in convs.values():
        c.forward = boom
    y = enc.forward_train(x)
    assert y.shape == (2, 2048, 8, 8) and bool(torch.isfinite(y).all())
    y.square().mean().backward()
    for name, p in enc.named_parameters():
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name


def test_encoder_training_step_vs_fp64(cuda_pkg, monkeypatch):
    """One training forward + backward of a ResNet-50 encoder (train-mode BatchNorm, 2 images of 256 x 256): the library
    (ResNet.forward_train) and the same blocks with their convs on cuDNN (TF32 off), both against the fp64 encoder (the
    torch modules' own forward in fp64).  A random-init ResNet-50 in train mode amplifies fp32 rounding through 16
    BatchNorm'd blocks, so the two fp32 paths are not compared with each other: the library must be as close to fp64 as
    cuDNN's fp32 is, within a factor of 2, for the output, every conv weight gradient and every BatchNorm running
    statistic."""
    from fast_3d_human_pose_estimation_b200 import encoder as E
    enc = _encoder(cuda_pkg)
    x = synth.make_images(2, seed=1)[0].cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    up = torch.randn((2, 2048, 8, 8), device="cuda", generator=g)

    def run(model, xin, upstream, train=True):
        model.zero_grad()
        y = model.forward_train(xin) if train else model(xin)
        (y * upstream).sum().backward()
        convs = _encoder_convs(model)
        stats = {n: b.detach().double().clone() for n, b in model.named_buffers() if n.endswith(("running_mean", "running_var"))}
        return y.detach().double(), {n: c.weight.grad.double() for n, c in convs.items()}, stats
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ours = run(copy.deepcopy(enc), x, up)
        with monkeypatch.context() as mp:
            mp.setattr(E, "_conv1x1", lambda t, w: F.conv2d(t, w))
            mp.setattr(E, "_conv3x3", lambda t, w, s: F.conv2d(t, w, stride=s, padding=1))
            theirs = run(copy.deepcopy(enc), x, up)
        ref = run(copy.deepcopy(enc).double(), x.double(), up.double(), train=False)    # torch modules in fp64
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    rel = lambda a, b: float((a - b).norm() / b.norm())     # noqa: E731
    y_o, y_t = rel(ours[0], ref[0]), rel(theirs[0], ref[0])
    g_o = max(rel(ours[1][n], ref[1][n]) for n in ref[1])
    g_t = max(rel(theirs[1][n], ref[1][n]) for n in ref[1])
    s_o = max(rel(ours[2][n], ref[2][n]) for n in ref[2])
    s_t = max(rel(theirs[2][n], ref[2][n]) for n in ref[2])
    cos = min(float(torch.dot(ours[1][n].flatten(), ref[1][n].flatten()) / (ours[1][n].norm() * ref[1][n].norm()))
              for n in ref[1])
    print(f"\nvs fp64, library / cuDNN fp32: output {y_o:.2e} / {y_t:.2e}, worst conv weight gradient {g_o:.2e} / "
          f"{g_t:.2e}, worst BatchNorm running stat {s_o:.2e} / {s_t:.2e}; library's worst gradient cosine {cos:.8f}")
    assert y_o <= 2 * y_t + 1e-7 and g_o <= 2 * g_t + 1e-7 and s_o <= 2 * s_t + 1e-7


# ---- CDRNet.forward_train: the encoder trains on the library ----
def _model(cuda_pkg):
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), trainable=True, train_encoder_on_library=True)
    with torch.no_grad():
        m.decoder.final_layer.weight.mul_(10.0)      # train-mode BN keeps activations O(1): peaky heat-maps need gain
    return m.cuda().train()


def _inputs(b):
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    targets = [torch.from_numpy(gt["gt2d_l"]).float().cuda(), torch.from_numpy(gt["gt2d_r"]).float().cuda()]
    return imgs, Ps, targets, torch.from_numpy(gt["vis"]).float().cuda()


def test_forward_train_does_not_call_the_encoder_conv_modules(cuda_pkg):
    m = _model(cuda_pkg)
    imgs, Ps, targets, vis = _inputs(2)

    def boom(*a, **k):
        raise AssertionError("encoder Conv2d module called")
    convs = _encoder_convs(m.encoder)
    assert len(convs) == 16 * 3 + 4
    for c in convs.values():
        c.forward = boom
    kps, xyz = m(imgs, Ps)
    loss = sum(cuda_pkg.MPJPELoss(True)(kps[v], targets[v], vis) for v in range(2))
    loss.backward()
    assert bool(torch.isfinite(xyz).all())
    for name, p in m.encoder.named_parameters():
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name


def _pure_torch_kps(m, feats, Ps):
    """the head of forward_train with the oracle's pure-torch operators (models/cdrnet.py:224-268) on given features"""
    from oracle import cdr_oracle as O
    pinv = [torch.linalg.pinv(p) for p in Ps]
    z = torch.cat([O.ftl(m.CF.conv_layer1(feats[v]), pinv[v]) for v in range(2)], 1)
    f = m.CF.conv_layer2(z)
    kps = []
    for v in range(2):
        o = m.CF.out_layer[v](O.ftl(f, Ps[v]))
        d = m.decoder
        h = d.final_layer(d.deconv3(d.deconv2(d.deconv1(o))))
        kps.append(O.process_heatmap(h) * (256 / h.shape[2]))
    return kps


def _mse(kps, targets):
    return sum(((kps[v] - targets[v]) ** 2).mean() for v in range(2))


def test_training_step_vs_fp64(cuda_pkg, monkeypatch):
    """One training step of CDRNet(trainable=True, train_encoder_on_library=True), and of the same model with the
    encoder's convs on cuDNN (TF32 off), both against the same network in fp64 (torch modules, the oracle's operators).
    A random-init ResNet-50 in train mode amplifies fp32 rounding through its BatchNorms, so the two fp32 models are not
    gated against each other: the library model must be as close to fp64 as the cuDNN-encoder model is, within a factor
    of 2, in the 2D joints, the loss, every encoder conv weight gradient and every encoder BatchNorm running statistic."""
    from fast_3d_human_pose_estimation_b200 import encoder as E
    m = _model(cuda_pkg)
    imgs, Ps, targets, _ = _inputs(2)

    def step(model):
        model.zero_grad()
        kps, _ = model(imgs, Ps)
        loss = _mse(kps, targets)
        loss.backward()
        enc = model.encoder
        return ([k.detach().double() for k in kps], float(loss),
                {n: c.weight.grad.double() for n, c in _encoder_convs(enc).items()},
                {n: b.double() for n, b in enc.named_buffers() if n.endswith(("running_mean", "running_var"))})
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ours = step(copy.deepcopy(m))
        with monkeypatch.context() as mp:
            mp.setattr(E, "_conv1x1", lambda t, w: F.conv2d(t, w))
            mp.setattr(E, "_conv3x3", lambda t, w, s: F.conv2d(t, w, stride=s, padding=1))
            theirs = step(copy.deepcopy(m))
        m64 = copy.deepcopy(m).double()
        feats = [m64.encoder(x.double()) for x in imgs]
        kps64 = _pure_torch_kps(m64, feats, [p.double() for p in Ps])
        loss64 = _mse(kps64, [t.double() for t in targets])
        loss64.backward()
        ref = ([k.detach() for k in kps64], float(loss64),
               {n: c.weight.grad for n, c in _encoder_convs(m64.encoder).items()},
               {n: b for n, b in m64.encoder.named_buffers() if n.endswith(("running_mean", "running_var"))})
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    rel = lambda a, b: float((a - b).norm() / b.norm())     # noqa: E731

    def errs(r):
        return (max(float((a - b).abs().max()) for a, b in zip(r[0], ref[0])), abs(r[1] - ref[1]) / abs(ref[1]),
                max(rel(r[2][n], ref[2][n]) for n in ref[2]), max(rel(r[3][n], ref[3][n]) for n in ref[3]))
    e_o, e_t = errs(ours), errs(theirs)
    print("\nvs fp64, library / cuDNN-encoder model: joints %.2e / %.2e px, loss %.2e / %.2e, worst encoder weight "
          "gradient %.2e / %.2e, worst running stat %.2e / %.2e" % tuple(v for pair in zip(e_o, e_t) for v in pair))
    for name, a, b in zip(("joints", "loss", "gradient", "running stat"), e_o, e_t):
        assert a <= 2 * b + 1e-7, (name, a, b)


def test_head_gradients_on_library_features_match_fp64(cuda_pkg):
    """The head of forward_train on the library encoder's features against an fp64 head (torch modules, the oracle's
    operators) on the SAME features: every head weight gradient in direction and size.  This is what the library's
    features do to the head's arithmetic, apart from how they differ from cuDNN's."""
    m = _model(cuda_pkg)
    imgs, Ps, targets, _ = _inputs(2)
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            feats = [m.encoder.forward_train(x) for x in imgs]
        ours_m, m64 = copy.deepcopy(m), copy.deepcopy(m).double()
        it = iter([f.clone() for f in feats])
        ours_m.encoder.forward_train = lambda x: next(it)
        kps, _ = ours_m(imgs, Ps)
        _mse(kps, targets).backward()
        kps64 = _pure_torch_kps(m64, [f.double() for f in feats], [p.double() for p in Ps])
        _mse(kps64, [t.double() for t in targets]).backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    p64 = dict(m64.named_parameters())
    worst = (1.0, 0.0)
    for n, p in ours_m.named_parameters():
        if n.startswith(("CF.", "decoder.")) and p.dim() == 4:
            a, b = p.grad.double().flatten(), p64[n].grad.flatten()
            cos, ratio = float(torch.dot(a, b) / (a.norm() * b.norm())), float(a.norm() / b.norm())
            worst = (min(worst[0], cos), max(worst[1], abs(ratio - 1)))
            assert cos >= 0.9999 and abs(ratio - 1) <= 1e-3, (n, cos, ratio)
    print(f"\nhead weight gradients on library features vs fp64 head: worst cosine {worst[0]:.7f}, "
          f"worst |norm ratio - 1| {worst[1]:.2e}")
