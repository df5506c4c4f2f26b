"""The decoder's transposed convolutions in training: conv_transpose2d (ConvTranspose2d k4 s2 p1, no bias) forward, data
gradient and weight gradient on libcdrhead's f16x2 tensor-core GEMM against fp64 torch, and forward_train on it."""
import copy

import pytest
import torch
import torch.nn.functional as F

from fast_3d_human_pose_estimation_b200 import synth

pytestmark = pytest.mark.gpu

LAYERS = [(2048, 256, 8), (256, 256, 16), (256, 256, 32)]     # decoder.deconv{1,2,3}: Cin, Cout, input H = W
GATE = 2e-5                                                  # max error / max |reference| (the stage-tap gate)


def _err(got, want):
    return float((got.detach().double() - want.detach()).abs().max() / want.detach().abs().max().clamp_min(1e-300))


def _case(cuda_pkg, n, cin, cout, h, sx=1.0, sdy=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n, cin, h, h), device="cuda", generator=g) * sx
    w = torch.randn((cin, cout, 4, 4), device="cuda", generator=g) * (1.0 / (cin * 4) ** 0.5)
    dy = torch.randn((n, cout, 2 * h, 2 * h), device="cuda", generator=g) * sdy
    x.requires_grad_(True)
    w.requires_grad_(True)
    y = cuda_pkg.conv_transpose2d(x, w)
    dx, dw = torch.autograd.grad(y, (x, w), dy)
    x64 = x.detach().double().requires_grad_(True)
    w64 = w.detach().double().requires_grad_(True)
    y64 = F.conv_transpose2d(x64, w64, stride=2, padding=1)
    dx64, dw64 = torch.autograd.grad(y64, (x64, w64), dy.double())
    return {"y": _err(y, y64), "dx": _err(dx, dx64), "dw": _err(dw, dw64)}


@pytest.mark.parametrize("n", [1, 2, 64])
@pytest.mark.parametrize("cin,cout,h", LAYERS)
def test_forward_dgrad_wgrad_vs_fp64(cuda_pkg, cin, cout, h, n):
    errs = _case(cuda_pkg, n, cin, cout, h)
    print(f"\ndeconv {cin}->{cout} on {h}x{h}, N={n}: max err / max |ref| {errs}")
    assert all(e <= GATE for e in errs.values()), errs


@pytest.mark.parametrize("scale", [1e-5, 3e4])
@pytest.mark.parametrize("cin,cout,h", LAYERS)
def test_dynamic_range(cuda_pkg, cin, cout, h, scale):
    errs = _case(cuda_pkg, 2, cin, cout, h, sx=scale, sdy=scale, seed=1)
    print(f"\ndeconv {cin}->{cout} on {h}x{h}, x and dy x{scale:g}: {errs}")
    assert all(e <= GATE for e in errs.values()), errs


@pytest.mark.parametrize("cin,cout,h", LAYERS)
def test_zero_grad_and_determinism(cuda_pkg, cin, cout, h):
    n = 4
    x = torch.randn((n, cin, h, h), device="cuda", requires_grad=True)
    w = torch.randn((cin, cout, 4, 4), device="cuda", requires_grad=True)
    y = cuda_pkg.conv_transpose2d(x, w)
    dx0, dw0 = torch.autograd.grad(y, (x, w), torch.zeros_like(y), retain_graph=True)
    assert bool((dx0 == 0).all()) and bool((dw0 == 0).all())          # a dead ReLU: exact zeros, no NaN
    dy = torch.randn_like(y)
    a = torch.autograd.grad(y, (x, w), dy, retain_graph=True)
    b = torch.autograd.grad(y, (x, w), dy)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # needs_input_grad: the weight gradient alone, the data gradient alone
    (dw_only,) = torch.autograd.grad(cuda_pkg.conv_transpose2d(x.detach(), w), (w,), dy)
    (dx_only,) = torch.autograd.grad(cuda_pkg.conv_transpose2d(x, w.detach()), (x,), dy)
    assert torch.equal(dw_only, a[1]) and torch.equal(dx_only, a[0])


def _model(cuda_pkg):
    torch.manual_seed(0)
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), trainable=True)
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


def test_forward_train_does_not_call_the_deconv_modules(cuda_pkg):
    m = _model(cuda_pkg)
    imgs, Ps, targets, vis = _inputs(2)

    def boom(*a, **k):
        raise AssertionError("decoder ConvTranspose2d module called")
    for k in range(1, 4):
        getattr(m.decoder, f"deconv{k}")[0].forward = boom
    kps, xyz = m(imgs, Ps)
    loss = sum(cuda_pkg.MPJPELoss(True)(kps[v], targets[v], vis) for v in range(2))
    loss.backward()
    assert bool(torch.isfinite(xyz).all())
    assert all(bool(torch.isfinite(getattr(m.decoder, f"deconv{k}")[0].weight.grad).all()) for k in range(1, 4))


def test_training_step_vs_torch_convolutions(cuda_pkg, monkeypatch):
    """One training step of the same model with the decoder's convolutions on libcdrhead and on cuDNN (fp32, TF32 off)."""
    from fast_3d_human_pose_estimation_b200 import autograd as AG
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ours = _model(cuda_pkg)
        theirs = copy.deepcopy(ours)
        imgs, Ps, targets, vis = _inputs(2)

        def step(model):
            model.zero_grad()
            kps, _ = model(imgs, Ps)
            loss = sum(cuda_pkg.MPJPELoss(True)(kps[v], targets[v], vis) for v in range(2))
            loss.backward()
            return [k.detach() for k in kps], float(loss)
        k_o, l_o = step(ours)
        with monkeypatch.context() as mp:
            mp.setattr(AG, "conv_transpose2d", lambda x, w: F.conv_transpose2d(x, w, stride=2, padding=1))
            k_t, l_t = step(theirs)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    d2 = max(float((a - b).abs().max()) for a, b in zip(k_o, k_t))
    print(f"\n2D joints {d2:.2e} px, loss {l_o:.8f} vs {l_t:.8f}")
    assert d2 <= 1e-3
    assert abs(l_o - l_t) <= 1e-5 * abs(l_t)
    po, pt = dict(ours.named_parameters()), dict(theirs.named_parameters())
    for k in range(1, 4):
        n = f"decoder.deconv{k}.0.weight"
        a, b = po[n].grad.double().flatten(), pt[n].grad.double().flatten()
        cos, ratio = float(torch.dot(a, b) / (a.norm() * b.norm())), float(a.norm() / b.norm())
        print(f"{n}: cosine {cos:.7f}, norm ratio {ratio:.7f}")
        assert cos >= 0.9999 and abs(ratio - 1) <= 1e-3, n
    bo, bt = dict(ours.named_buffers()), dict(theirs.named_buffers())
    for n in bo:
        if n.startswith("decoder.") and n.endswith(("running_mean", "running_var")):
            err = float((bo[n].double() - bt[n].double()).abs().max() / bt[n].double().abs().max())
            assert err <= 1e-5, (n, err)
