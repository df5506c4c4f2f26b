"""SURVEY §8f rank 3, first slice: forward + backward of soft-argmax, DLT and FTL on libcdrhead.so against
torch autograd through the fp64 oracle (oracle/cdr_oracle.py restates models/cdrnet.py:45-56,120-179)."""
import json
import os

import numpy as np
import pytest
import torch

from fast_3d_human_pose_estimation_b200 import synth
from oracle import cdr_oracle as O

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("kind", ["randn3", "blob", "small"])
def test_softargmax_backward_vs_autograd(cuda_pkg, kind):
    g = torch.Generator().manual_seed(3)
    if kind == "randn3":
        h = 3 * torch.randn(3, 19, 64, 64, generator=g)
    elif kind == "blob":
        h = synth.blob_heatmaps(torch.rand(3, 19, 2, generator=g) * 63, seed=4)
    else:
        h = torch.randn(2, 5, 32, 48, generator=g) * 2          # ragged relative to the 64x64 fast path
    w = torch.randn(h.shape[0], h.shape[1], 2, generator=g)        # upstream gradient
    h64 = h.double().requires_grad_(True)
    kp64 = O.process_heatmap(h64) * 4.0
    (kp64 * w.double()).sum().backward()
    hd = h.cuda().requires_grad_(True)
    kp = cuda_pkg.soft_argmax_2d(hd, 4.0)
    (kp * w.cuda()).sum().backward()
    np.testing.assert_allclose(kp.detach().cpu().numpy(), kp64.detach().numpy(), rtol=0, atol=1e-4)
    assert hd.grad.shape == h.shape
    assert _rel(hd.grad.cpu().double(), h64.grad) < 2e-5
    # the gradient of a softmax-weighted mean sums to zero over each map
    assert float(hd.grad.sum((2, 3)).abs().max()) < 1e-4


def test_dlt_backward_vs_autograd(cuda_pkg):
    b, j = 6, 19
    cams = synth.make_cameras(b, seed=21)
    gt = synth.make_gt(cams, seed=22)
    rng = np.random.default_rng(5)
    kl = torch.from_numpy(gt["gt2d_l"] + rng.normal(0, 1.5, gt["gt2d_l"].shape)).float()   # near-consistent views
    kr = torch.from_numpy(gt["gt2d_r"] + rng.normal(0, 1.5, gt["gt2d_r"].shape)).float()
    Pl, Pr = torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])
    w = torch.randn(b, j, 3, generator=torch.Generator().manual_seed(6))
    # oracle in fp64 on the SAME fp32 inputs
    kl64, kr64 = kl.double().requires_grad_(True), kr.double().requires_grad_(True)
    projs = torch.stack([Pl.double(), Pr.double()], 1)
    x64 = torch.stack([O.dlt(projs, torch.stack([kl64[:, k], kr64[:, k]], 1)) for k in range(j)], 1)
    (x64 * w.double()).sum().backward()
    kld, krd = kl.cuda().requires_grad_(True), kr.cuda().requires_grad_(True)
    xyz = cuda_pkg.dlt(Pl.cuda(), Pr.cuda(), kld, krd)
    (xyz * w.cuda()).sum().backward()
    np.testing.assert_allclose(xyz.detach().cpu().numpy(), x64.detach().numpy(), rtol=0, atol=2e-3)   # mm, fp32 out
    for got, want in ((kld.grad, kl64.grad), (krd.grad, kr64.grad)):
        assert got.shape == want.shape
        assert _rel(got.cpu().double(), want) < 1e-4
    # finite differences through our own forward agree too (central, 0.05 px)
    eps = 0.05
    kp, km = kl.clone(), kl.clone()
    kp[0, 0, 0] += eps
    km[0, 0, 0] -= eps
    with torch.no_grad():
        fp = cuda_pkg.dlt(Pl.cuda(), Pr.cuda(), kp.cuda(), kr.cuda())
        fm = cuda_pkg.dlt(Pl.cuda(), Pr.cuda(), km.cuda(), kr.cuda())
    fd = float(((fp - fm).cpu() * w).sum() / (2 * eps))
    assert abs(fd - float(kld.grad[0, 0, 0])) < 2e-2 * max(1.0, abs(fd))


def test_ftl_autograd_nchw(cuda_pkg):
    b = 4
    g = torch.Generator().manual_seed(8)
    cams = synth.make_cameras(b, seed=23)
    P = torch.from_numpy(cams["P_l"])
    Pinv = torch.linalg.pinv(P.double()).float()
    for x, m in ((torch.randn(b, 300, 8, 8, generator=g), Pinv), (torch.randn(b, 400, 8, 8, generator=g), P)):
        w = torch.randn(b, m.shape[1] * (x.shape[1] // m.shape[2]), 8, 8, generator=g)
        x64 = x.double().requires_grad_(True)
        y64 = O.ftl(x64, m.double())
        (y64 * w.double()).sum().backward()
        xd = x.cuda().requires_grad_(True)
        y = cuda_pkg.ftl(xd, m.cuda())
        (y * w.cuda()).sum().backward()
        assert y.shape == y64.shape
        assert _rel(y.detach().cpu().double(), y64.detach()) < 1e-5
        assert _rel(xd.grad.cpu().double(), x64.grad) < 1e-5
    with pytest.raises(NotImplementedError):
        md = P.cuda().requires_grad_(True)
        cuda_pkg.ftl(torch.randn(b, 400, 8, 8).cuda().requires_grad_(True), md).sum().backward()


def test_differentiable_tail_end_to_end(cuda_pkg):
    """heat-maps -> 2D -> 3D -> MPJPE-style loss, gradient w.r.t. the logits, vs the fp64 oracle chain."""
    b, j = 2, 19
    cams = synth.make_cameras(b, seed=31)
    gt = synth.make_gt(cams, seed=32)
    hl = synth.blob_heatmaps(torch.from_numpy(gt["gt2d_l"] / 4.0).float(), seed=1)
    hr = synth.blob_heatmaps(torch.from_numpy(gt["gt2d_r"] / 4.0).float(), seed=2)
    Pl, Pr = torch.from_numpy(cams["P_l"]), torch.from_numpy(cams["P_r"])
    g3 = torch.from_numpy(gt["gt3d"])

    def loss_of(xyz, gt3):
        return torch.sqrt(((xyz - gt3) ** 2).sum(-1) + 1e-15).mean()          # models/loss.py:84-85 (MPJPELoss.cdist)

    hl64, hr64 = hl.double().requires_grad_(True), hr.double().requires_grad_(True)
    kl64, kr64 = O.process_heatmap(hl64) * 4.0, O.process_heatmap(hr64) * 4.0
    projs = torch.stack([Pl.double(), Pr.double()], 1)
    x64 = torch.stack([O.dlt(projs, torch.stack([kl64[:, k], kr64[:, k]], 1)) for k in range(j)], 1)
    l64 = loss_of(x64, g3)
    l64.backward()
    hld, hrd = hl.cuda().requires_grad_(True), hr.cuda().requires_grad_(True)
    xyz = cuda_pkg.dlt(Pl.cuda(), Pr.cuda(), cuda_pkg.soft_argmax_2d(hld, 4.0), cuda_pkg.soft_argmax_2d(hrd, 4.0))
    loss = loss_of(xyz, g3.float().cuda())
    loss.backward()
    assert abs(loss.item() - l64.item()) < 1e-2 * max(1.0, l64.item())
    for got, want in ((hld.grad, hl64.grad), (hrd.grad, hr64.grad)):
        assert _rel(got.cpu().double(), want) < 5e-3          # fp32 2D joints feed an ill-conditioned-at-times DLT


def test_forward_train_hybrid_matches_pure_torch_fp64(cuda_pkg):
    """CDRNet(trainable=True).train()(imgs, Ps): torch convs / train-mode BN + this library's ftl / soft-argmax / dlt
    (forward and backward) against the same modules in fp64 with the oracle's pure-torch operators."""
    import copy
    torch.manual_seed(0)
    b = 2
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False     # fp32 convs vs the fp64 copy
    try:
        _forward_train_case(cuda_pkg, copy, b)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def _forward_train_case(cuda_pkg, copy, b):
    m = cuda_pkg.CDRNet(synth.make_cfg(50, 19), trainable=True)
    with torch.no_grad():
        m.decoder.final_layer.weight.mul_(10.0)      # train-mode BN keeps activations O(1): peaky heat-maps need gain
    m = m.cuda().train()
    m64 = copy.deepcopy(m).double()
    imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
    cams = synth.make_cameras(b, seed=2)
    gt = synth.make_gt(cams, seed=3)
    Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
    g2 = [torch.from_numpy(gt["gt2d_l"]).cuda(), torch.from_numpy(gt["gt2d_r"]).cuda()]

    def pure_torch(mod, xs, projs):                      # models/cdrnet.py:224-268, operators from the oracle
        pinv = [torch.linalg.pinv(p) for p in projs]
        feats = [mod.encoder(x) for x in xs]
        z = torch.cat([O.ftl(mod.CF.conv_layer1(feats[v]), pinv[v]) for v in range(2)], 1)
        f = mod.CF.conv_layer2(z)
        kps = []
        for v in range(2):
            o = mod.CF.out_layer[v](O.ftl(f, projs[v]))
            d = mod.decoder
            h = d.final_layer(d.deconv3(d.deconv2(d.deconv1(o))))
            kps.append(O.process_heatmap(h) * (256 / h.shape[2]))
        return kps

    kps, xyz = m(imgs, Ps)
    assert xyz.shape == (b, 19, 3) and xyz.requires_grad and bool(torch.isfinite(xyz).all())
    loss = sum(((kps[v] - g2[v].float()) ** 2).mean() for v in range(2))
    loss.backward(retain_graph=True)
    names = ("decoder.final_layer.weight", "decoder.deconv1.0.weight", "CF.conv_layer2.3.weight",
             "CF.conv_layer1.0.weight", "CF.out_layer.1.0.weight", "encoder.layer4.2.conv3.weight")
    ours = {n: dict(m.named_parameters())[n].grad.detach().clone() for n in names}
    # forward against the fp64 copy of the network with the oracle's operators
    with torch.no_grad():
        kps64 = pure_torch(m64, [x.double() for x in imgs], [p.double() for p in Ps])
    loss64 = sum(((kps64[v] - g2[v]) ** 2).mean() for v in range(2))
    for v in range(2):
        assert float((kps[v].detach().double() - kps64[v]).abs().max()) < 0.2           # px: a whole fp32 ResNet-50 + head vs fp64
    assert abs(loss.item() - loss64.item()) < 1e-2 * loss64.item()
    # gradients against the SAME fp32 modules with the oracle's pure-torch operators (an fp64 network takes other
    # ReLU branches near zero, which is not what this test is about)
    m.zero_grad()
    kps_t = pure_torch(m, imgs, Ps)
    loss_t = sum(((kps_t[v] - g2[v].float()) ** 2).mean() for v in range(2))
    loss_t.backward()
    assert abs(loss.item() - loss_t.item()) < 1e-3 * abs(loss_t.item())
    report = {}
    for n in names:
        a, g_t = ours[n].double().flatten(), dict(m.named_parameters())[n].grad.double().flatten()
        report[n] = (float(torch.dot(a, g_t) / (a.norm() * g_t.norm())), float(a.norm() / g_t.norm()), _rel(a, g_t))
    print("\nforward_train gradients vs pure torch (cosine, norm ratio, max rel):", report)
    for n, (cos, ratio, _) in report.items():       # direction and size: train-mode BN backward cancels heavily, so
        assert cos > 0.995 and abs(ratio - 1) < 0.05, (n, report[n])    # element-wise ulps are not the criterion
    # the 3D branch reaches the parameters too (its operator-level gradient is checked above)
    m.zero_grad()
    xyz.abs().mean().backward()
    g = m.CF.conv_layer1[0].weight.grad
    assert g is not None and bool(torch.isfinite(g).all()) and float(g.abs().max()) > 0
    # and the opt-in is required
    with pytest.raises(RuntimeError, match="inference-only"):
        cuda_pkg.CDRNet(synth.make_cfg(50, 19)).cuda().train()(imgs, Ps)


class _OracleLosses:
    """The oracle's restatement of models/loss.py (pinned against the reference's modules by tests/test_oracle_golden.py),
    behind the reference's class names — used where the reference sources are absent."""

    @staticmethod
    def _mk(fn):
        class _L:
            def __init__(self, use_target_weight, *args):
                self.use, self.args = use_target_weight, args

            def __call__(self, output, target, target_weight):
                return fn(output, target, target_weight, self.use, *self.args)
        return _L

_OracleLosses.JointsMSELoss = _OracleLosses._mk(O.joints_mse_loss)
_OracleLosses.JointsMSESmoothLoss = _OracleLosses._mk(O.joints_mse_smooth_loss)
_OracleLosses.MPJPELoss = _OracleLosses._mk(O.mpjpe_loss)


def _ref_losses():
    """The reference's own loss modules where its sources are present, else the oracle's restatement."""
    from oracle import refload
    if refload.available():
        refload.load()
        import importlib
        return importlib.import_module("models.loss")
    return _OracleLosses


@pytest.mark.parametrize("name,args", [("MPJPELoss", ()), ("JointsMSESmoothLoss", ()), ("JointsMSESmoothLoss", (4.0,)),
                                       ("JointsMSELoss", ())])
@pytest.mark.parametrize("shape", [(8, 19, 3), (8, 19, 2), (1, 19, 3), (3, 5, 16, 16)])
@pytest.mark.parametrize("use_w", [True, False])
def test_losses_vs_reference_modules(cuda_pkg, name, args, shape, use_w):
    """SURVEY §8f rank 3: models/loss.py:5-98 on libcdrhead (forward and backward) against the UNMODIFIED reference
    modules evaluated in fp64 with torch autograd, on joints (B,J,D) as train_cdr.py:113-125 feeds them and on heat-maps
    (B,J,H,W) as train.py does."""
    ref = _ref_losses()
    if len(shape) == 4 and name != "JointsMSELoss":
        pytest.skip("only JointsMSELoss is applied to heat-maps in the reference")
    g = torch.Generator().manual_seed(sum(map(ord, name)) + sum(shape) + int(use_w))
    scale = 30.0 if name != "JointsMSELoss" else 1.0                  # mm-sized errors: both branches of the smooth loss
    pred = (torch.randn(shape, generator=g) * scale)
    tgt = (torch.randn(shape, generator=g) * scale)
    w = (torch.rand(shape[0], shape[1], 1, generator=g) > 0.2).float()
    up = torch.randn((), generator=g).abs() + 0.5                      # upstream gradient
    p64 = pred.double().requires_grad_(True)
    want = getattr(ref, name)(use_w, *args)(p64, tgt.double(), w.double())
    (want * up.double()).sum().backward()
    pd = pred.cuda().requires_grad_(True)
    got = getattr(cuda_pkg, name)(use_w, *args)(pd, tgt.cuda(), w.cuda())
    (got * up.cuda()).sum().backward()
    assert tuple(got.shape) == tuple(want.shape)
    np.testing.assert_allclose(got.detach().cpu().double().numpy(), want.detach().numpy(), rtol=2e-6)
    assert _rel(pd.grad.cpu().double(), p64.grad) < 2e-5
    # deterministic: the same bits on a second evaluation
    got2 = getattr(cuda_pkg, name)(use_w, *args)(pd, tgt.cuda(), w.cuda())
    assert torch.equal(got2, got)


@pytest.mark.parametrize("shape,relu", [((4, 300, 8, 8), True), ((6, 256, 32, 32), True), ((3, 64, 16, 16), False),
                                        ((2, 2048, 8, 8), True)])
def test_bn_train_vs_torch(cuda_pkg, shape, relu):
    """nn.BatchNorm2d in training mode (+ the ReLU that follows every BN of the head) on libcdrhead: outputs, running
    statistics and the gradients of x / weight / bias against torch's own module evaluated in fp64."""
    g = torch.Generator().manual_seed(11)
    x = torch.randn(shape, generator=g) * 2.0 + 0.3
    c = shape[1]
    bn = torch.nn.BatchNorm2d(c, momentum=0.1)
    bn.weight.data = 1.0 + 0.3 * torch.randn(c, generator=g)
    bn.bias.data = 0.2 * torch.randn(c, generator=g)
    bn.running_mean.data = 0.1 * torch.randn(c, generator=g)
    bn.running_var.data = 1.0 + 0.2 * torch.rand(c, generator=g)
    import copy
    ref = copy.deepcopy(bn).double().train()
    ours = copy.deepcopy(bn).cuda().train()
    up = torch.randn(shape, generator=g)
    x64 = x.double().requires_grad_(True)
    y64 = ref(x64)
    if relu:
        y64 = torch.relu(y64)
    (y64 * up.double()).sum().backward()
    xd = x.cuda().requires_grad_(True)
    y = cuda_pkg.batch_norm_train(xd, ours, relu=relu)
    (y * up.cuda()).sum().backward()
    assert _rel(y.detach().cpu().double(), y64.detach()) < 2e-6
    assert _rel(ours.running_mean.cpu().double(), ref.running_mean) < 1e-6
    assert _rel(ours.running_var.cpu().double(), ref.running_var) < 1e-6
    assert int(ours.num_batches_tracked) == int(ref.num_batches_tracked) == 1
    assert _rel(xd.grad.cpu().double(), x64.grad) < 2e-5
    assert _rel(ours.weight.grad.cpu().double(), ref.weight.grad) < 2e-5
    assert _rel(ours.bias.grad.cpu().double(), ref.bias.grad) < 2e-5
    with pytest.raises(RuntimeError):
        cuda_pkg.batch_norm_train(xd, ours.eval())


def test_training_step_vs_the_reference_model(cuda_pkg):
    """One training step of train_cdr.py (:105-127, warm-up branch: MPJPELoss on both views' 2D joints) — the UNMODIFIED
    reference CDRNet + its MPJPELoss in train mode on this GPU (fp32, TF32 off) against CDRNet(trainable=True) +
    this package's MPJPELoss: the head's BatchNorm / ReLU, pinv, FTL, soft-argmax, DLT and the loss run forward and
    backward on libcdrhead, the convolutions on cuDNN in both.  Loss, the script's grad_norm, the gradient direction of
    parameters all over the network and the BatchNorm running statistics after the step.  Where the reference's
    sources are absent: loss and grad_norm against the reference's recorded ones (tests/golden/reference_recorded.json)."""
    from oracle import refload
    live = refload.available()
    if live:
        ref = refload.load()
        import importlib
        ref_loss = importlib.import_module("models.loss")
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        b, cfg = 2, synth.make_cfg(50, 19)
        torch.manual_seed(0)
        ours = cuda_pkg.CDRNet(cfg, trainable=True)
        with torch.no_grad():
            ours.decoder.final_layer.weight.mul_(10.0)     # train-mode BN keeps activations O(1): peaky heat-maps need gain
        ours = ours.cuda().train()
        if live:
            theirs = ref.CDRNet(cfg)
            theirs.load_state_dict(ours.state_dict())
            theirs = theirs.cuda().train()
        imgs = [x.cuda() for x in synth.make_images(b, seed=1)]
        cams = synth.make_cameras(b, seed=2)
        gt = synth.make_gt(cams, seed=3)
        Ps = [torch.from_numpy(cams["P_l"]).cuda(), torch.from_numpy(cams["P_r"]).cuda()]
        targets = [torch.from_numpy(gt["gt2d_l"]).float().cuda(), torch.from_numpy(gt["gt2d_r"]).float().cuda()]
        weight = torch.from_numpy(gt["vis"]).float().cuda()

        def step(model, criterion):
            model.zero_grad()
            pred_2ds, pred_3ds = model(imgs, Ps)                                   # train_cdr.py:105
            loss = torch.zeros(1, device="cuda")
            for pred, target in zip(pred_2ds, targets):                           # :113-115
                loss = loss + criterion(pred, target, weight)
            loss.backward()                                                       # :127
            grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
            return float(loss), float(torch.norm(torch.cat([g.flatten() for g in grads.values()]))), grads, pred_3ds   # :129-130
        if not live:
            rec = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_recorded.json")))
            l_t, gn_t = rec["training_step"]["loss"], rec["training_step"]["grad_norm"]
            l_o, gn_o, g_o, xyz = step(ours, cuda_pkg.MPJPELoss(True))
            print(f"\ntraining step: loss {l_o:.6f} vs reference (recorded) {l_t}; grad_norm {gn_o:.6e} vs {gn_t:.6e}")
            assert abs(l_o - l_t) <= 1e-4 * abs(l_t)
            assert abs(gn_o - gn_t) <= 2e-2 * gn_t
            assert bool(torch.isfinite(xyz).all()) and all(bool(torch.isfinite(g).all()) for g in g_o.values())
            return
        l_t, gn_t, g_t, _ = step(theirs, ref_loss.MPJPELoss(True))
        l_o, gn_o, g_o, xyz = step(ours, cuda_pkg.MPJPELoss(True))
        print(f"\ntraining step: loss {l_o:.6f} vs reference {l_t:.6f}; grad_norm {gn_o:.6e} vs {gn_t:.6e}")
        assert abs(l_o - l_t) <= 1e-4 * abs(l_t)
        assert abs(gn_o - gn_t) <= 2e-2 * gn_t
        assert set(g_o) == set(g_t) and bool(torch.isfinite(xyz).all())
        worst = 1.0
        for n in ("decoder.final_layer.weight", "decoder.deconv1.0.weight", "decoder.deconv3.1.weight", "CF.conv_layer2.3.weight",
                  "CF.conv_layer1.1.bias", "CF.out_layer.1.0.weight", "encoder.layer4.2.conv3.weight", "encoder.conv1.weight"):
            a, w = g_o[n].double().flatten(), g_t[n].double().flatten()
            worst = min(worst, float(torch.dot(a, w) / (a.norm() * w.norm())))
        print(f"worst gradient cosine over 8 parameter tensors: {worst:.6f}")
        assert worst > 0.995
        for (n, bo), (_, bt) in zip(ours.named_buffers(), theirs.named_buffers()):
            if n.endswith(("running_mean", "running_var")) and n.startswith(("CF.", "decoder.")):
                assert _rel(bo.double(), bt.double()) < 1e-4, n
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
