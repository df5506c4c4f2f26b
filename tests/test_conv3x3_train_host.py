"""CPU: the argument checks of conv3x3 and of the cdr_conv3x3_train_* entry points, none of which may touch CUDA, the
identities the library's stride-2 and dgrad paths rest on, and the pieces of test_gpu_conv3x3_train.py that need no GPU:
its shape table against the wgrad slice plan, and the strictness of the
per-element gate it shares with the other training convolutions (train_conv_checks.py)."""
import ctypes as C
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

from train_conv_checks import GATE_C, f16_planes, gate


def _domain():
    """tests/test_gpu_conv3x3_train.py (its shape table and slice mirror), imported without a GPU."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_gpu_conv3x3_train.py")
    spec = importlib.util.spec_from_file_location("_conv3x3_train_domain", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _in_domain(n, cin, cout, h, w, s):
    ho, wo = h // s, w // s
    return (h % s == 0 and w % s == 0 and wo in (8, 16, 32, 64) and (ho * wo == 64 or ho * wo % 128 == 0)
            and n * ho * wo <= 1 << 22 and all(64 <= c <= 2048 and c % 64 == 0 for c in (cin, cout)))


def test_shape_table_covers_the_plan():
    """The GPU tables reach every wgrad slice count the plan produces (1 .. 64), at both strides, with a slice that ends
    mid-image and a half-full last 128-pixel tile."""
    D = _domain()
    assert all(D.slices(n, cin, cout, h, w, s) == sl for n, cin, cout, h, w, s, sl in D.TABLE)
    assert all(_in_domain(n, cin, cout, h, w, s) for n, cin, cout, h, w, s, _ in D.TABLE)
    produced = {D.slices(n, c, c2, h, h, s) for n in (1, 2, 3, 16, 64, 256, 1024, 4096) for c in (64, 128, 512, 2048)
                for c2 in (64, 320, 2048) for h in (8, 16, 32, 64, 128) for s in (1, 2)
                if _in_domain(n, c, c2, h, h, s)}
    assert produced <= {sl for *_, sl in D.TABLE} == {1 << i for i in range(7)}
    assert {s for *_, s, _ in D.TABLE} == {1, 2}
    assert any((n * (h // s) * (w // s)) % 128 == 64 for n, _, _, h, w, s, _ in D.TABLE)
    assert any((n * (h // s) * (w // s) // sl) % ((h // s) * (w // s)) for n, _, _, h, w, s, sl in D.TABLE)
    assert all(_in_domain(n, c, c, h, h, s) for c, h, s in D.RESNET for n in (1, 2, 64))


def test_slice_mirror_fits_the_reported_workspace(pkg):
    """The backward workspace holds the wgrad partials, [slices][9][Cout][round_up(Cin, 128)] fp32: a mirror that
    counted more slices than the library would not fit in what cdr_conv3x3_train_workspace_bytes reports."""
    D = _domain()
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    for n, cin, cout, h, wd, st, sl in D.TABLE:
        assert L.cdr_conv3x3_train_workspace_bytes(n, cin, cout, h, wd, st, C.byref(s), C.byref(w)) == 0
        assert w.value >= sl * 9 * cout * ((cin + 127) // 128 * 128) * 4
        assert s.value >= 2 * n * h * wd * cin * 2                      # x as fp16 hi / lo planes


def test_stride2_and_dgrad_identities_in_fp64():
    """The identities the library computes through: at stride 2 the data gradient is a k4 s2 p1 transposed conv with the
    weight zero-padded to 4x4 at index 3 and the weight gradient the 9 taps (ky, kx <= 2) of that transposed conv's
    weight gradient; at stride 1 the data gradient is a 3x3 conv of dy with W^T and the taps flipped; a 1x1 stride-2
    conv is a 1x1 conv of the stride-2 slice."""
    g = torch.Generator().manual_seed(0)
    n, ci, co, h = 2, 5, 7, 8
    w = torch.randn((co, ci, 3, 3), generator=g, dtype=torch.float64)
    w4 = F.pad(w, (0, 1, 0, 1))
    x = torch.randn((n, ci, 2 * h, 2 * h), generator=g, dtype=torch.float64, requires_grad=True)
    wr = w.clone().requires_grad_(True)
    y = F.conv2d(x, wr, stride=2, padding=1)
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    dx, dw = torch.autograd.grad(y, (x, wr), dy)
    torch.testing.assert_close(F.conv_transpose2d(dy, w4, stride=2, padding=1), dx, rtol=1e-12, atol=1e-12)
    w4r = w4.clone().requires_grad_(True)
    g4, = torch.autograd.grad(F.conv_transpose2d(dy, w4r, stride=2, padding=1), (w4r,), x.detach())
    torch.testing.assert_close(g4[:, :, :3, :3], dw, rtol=1e-12, atol=1e-12)
    x1 = torch.randn((n, ci, h, h), generator=g, dtype=torch.float64, requires_grad=True)
    y1 = F.conv2d(x1, w, padding=1)
    d1 = torch.randn(y1.shape, generator=g, dtype=torch.float64)
    dx1, = torch.autograd.grad(y1, (x1,), d1)
    torch.testing.assert_close(F.conv2d(d1, w.transpose(0, 1).flip(2, 3), padding=1), dx1, rtol=1e-12, atol=1e-12)
    w1 = torch.randn((co, ci, 1, 1), generator=g, dtype=torch.float64)
    torch.testing.assert_close(F.conv2d(x.detach(), w1, stride=2), F.conv2d(x.detach()[:, :, ::2, ::2], w1), rtol=0,
                               atol=0)


@pytest.mark.parametrize("s", [1, 2])
def test_per_element_gate_catches_a_lost_lo_plane(s):
    """With x through both planes the forward passes the per-element gate; with the hi plane alone (~2^-12 m) it
    fails.  So the gate's constant is tight enough to see the lo plane."""
    assert GATE_C <= 2.0 ** -14
    g = torch.Generator().manual_seed(0)
    x = torch.randn((2, 64, 16, 16), generator=g).double()        # fp32 values, held in fp64
    w = torch.randn((64, 64, 3, 3), generator=g).float().double()
    ref = F.conv2d(x, w, stride=s, padding=1)
    mag = F.conv2d(x.abs(), w.abs(), stride=s, padding=1)
    gate("y", F.conv2d(f16_planes(x, True), f16_planes(w, True), stride=s, padding=1), ref, mag)
    with pytest.raises(AssertionError, match="per-element gate"):
        gate("y", F.conv2d(f16_planes(x, False), f16_planes(w, True), stride=s, padding=1), ref, mag,
               max_gate=False)


def test_conv3x3_rejects_without_cuda(pkg, monkeypatch):
    import torch.cuda
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: pytest.fail("touched CUDA"))
    x = torch.zeros((2, 64, 16, 16))
    w = torch.zeros((128, 64, 3, 3))
    with pytest.raises(ValueError, match="CUDA"):
        pkg.conv3x3(x, w)                                             # CPU tensors
    with pytest.raises(ValueError, match="CUDA"):
        pkg.conv3x3(x, w, 2)
    with pytest.raises(ValueError, match="float32"):
        pkg.conv3x3(x.double(), w.double())
    with pytest.raises(ValueError, match="float32"):
        pkg.conv3x3(x, w.half())
    for xs, ws, s in (((2, 64, 16, 16), (128, 64, 1, 1), 1),          # not 3x3
                      ((2, 64, 16, 16), (128, 32, 3, 3), 1),          # Cin mismatch
                      ((2, 64, 16, 16), (128, 64, 3, 3), 3),          # stride 3
                      ((2, 64, 16, 16), (128, 64, 3, 3), 0),
                      ((2, 64, 16, 16), (128, 64, 3, 3), 1.0),        # not an int
                      ((2, 32, 16, 16), (128, 32, 3, 3), 1),          # Cin < 64
                      ((2, 96, 16, 16), (128, 96, 3, 3), 1),          # Cin not a multiple of 64
                      ((2, 64, 16, 16), (2112, 64, 3, 3), 1),         # Cout > 2048
                      ((2, 64, 16, 12), (128, 64, 3, 3), 1),          # W = 12 not a power of two
                      ((2, 64, 16, 4), (128, 64, 3, 3), 1),           # W = 4
                      ((2, 64, 16, 128), (128, 64, 3, 3), 1),         # W = 128
                      ((2, 64, 17, 16), (128, 64, 3, 3), 2),          # H not divisible by the stride
                      ((2, 64, 8, 16), (128, 64, 3, 3), 2),           # output 4 x 8: H*W = 32
                      ((2, 64, 24, 8), (128, 64, 3, 3), 1),           # H*W = 192: neither 64 nor a multiple of 128
                      ((1025, 64, 64, 64), (64, 64, 3, 3), 1),        # N*H*W > 2^22
                      ((64, 16, 16), (128, 64, 3, 3), 1)):            # not 4-D
        with pytest.raises(ValueError, match="expected|unsupported"):
            pkg.conv3x3(torch.zeros(xs), torch.zeros(ws), s)


def test_abi_validation_without_gpu(pkg):
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    assert L.cdr_conv3x3_train_workspace_bytes(64, 64, 64, 64, 64, 1, C.byref(s), C.byref(w)) == 0
    assert s.value >= 2 * 64 * 64 * 64 * 64 * 2 and w.value > 0
    assert L.cdr_conv3x3_train_workspace_bytes(64, 512, 512, 16, 16, 2, C.byref(s), C.byref(w)) == 0
    assert L.cdr_conv3x3_train_workspace_bytes(1, 2048, 2048, 8, 8, 1, C.byref(s), C.byref(w)) == 0
    for args in ((64, 64, 64, 64, 64, 3), (64, 64, 64, 64, 64, 0), (0, 64, 64, 8, 8, 1), (1, 0, 64, 8, 8, 1),
                 (1, 64, 0, 8, 8, 1), (1, 96, 64, 8, 8, 1), (1, 64, 2112, 8, 8, 1), (1, 64, 64, 12, 12, 1),
                 (1, 64, 64, 24, 8, 1), (1, 64, 64, 8, 16, 2), (1, 64, 64, 17, 16, 2), (1025, 64, 64, 64, 64, 1),
                 (1, 64, 64, 0, 64, 1), (1, 64, 64, 8, 128, 1)):
        assert L.cdr_conv3x3_train_workspace_bytes(*args, C.byref(s), C.byref(w)) == 1, args
        assert b"cdr_conv3x3_train_workspace_bytes" in L.cdr_last_error()
    assert L.cdr_conv3x3_train_workspace_bytes(1, 64, 64, 8, 8, 1, None, None) == 1
    assert L.cdr_conv3x3_train_forward(None, None, 1, 64, 64, 8, 8, 1, None, None, 0, None, 0, None) == 1
    assert b"cdr_conv3x3_train_forward" in L.cdr_last_error()
    assert L.cdr_conv3x3_train_backward(None, None, None, 1, 64, 64, 8, 8, 1, None, None, None, 0, None) == 1
    assert b"cdr_conv3x3_train_backward" in L.cdr_last_error()
    fake = C.c_void_p(1 << 20)                                        # never dereferenced: the shape check comes first
    assert L.cdr_conv3x3_train_forward(fake, fake, 1, 64, 64, 12, 12, 1, fake, fake, 1 << 30, fake, 1 << 30, None) == 1
    assert b"cdr_conv3x3_train_forward" in L.cdr_last_error()
    assert L.cdr_conv3x3_train_backward(fake, fake, fake, 1, 64, 64, 8, 8, 3, fake, None, fake, 1 << 30, None) == 1
    assert b"cdr_conv3x3_train_backward" in L.cdr_last_error()
    odd = C.c_void_p((1 << 20) + 4)                                   # misaligned: rejected before any CUDA call
    assert L.cdr_conv3x3_train_forward(odd, fake, 1, 64, 64, 8, 8, 1, fake, fake, 1 << 30, fake, 1 << 30, None) == 1
    assert L.cdr_conv3x3_train_forward(fake, fake, 1, 64, 64, 8, 8, 1, fake, fake, 16, fake, 1 << 30, None) == 3
    assert b"saved" in L.cdr_last_error()


def test_forward_train_binds_the_encoder_ops_at_import(pkg):
    """The encoder's training forward calls the ops bound when encoder.py loaded, so rebinding autograd.conv1x1 (as
    the head's training-step tests do) leaves the encoder where it is; and its bottleneck blocks go through them."""
    from fast_3d_human_pose_estimation_b200 import autograd as AG, encoder as E
    assert E._conv1x1 is AG.conv1x1 and E._conv3x3 is AG.conv3x3
    m = E.ResNet(type("Cfg", (), {"MODEL": type("M", (), {"NUM_LAYERS": 18})})())
    with pytest.raises(ValueError, match="Bottleneck"):
        m.forward_train(torch.zeros((1, 3, 256, 256)))
