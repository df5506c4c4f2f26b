"""CPU: the index algebra the transposed-convolution training kernels implement (gemm_tc.cu: kTapConv4s2 and the
MN-major weight-gradient tiles), in fp64 against torch autograd, and the argument checks of conv_transpose2d and of
the cdr_deconv_train_* entry points, none of which may touch CUDA.  Also the pieces of test_gpu_deconv_train_domain.py
that need no GPU: its shape table against the wgrad slice plan, and the strictness of the
per-element gate it shares with the other training convolutions (train_conv_checks.py)."""
import ctypes as C
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

from train_conv_checks import GATE_C, f16_planes, gate


def _shifted(t, dy, dx, h, w):
    """t[n, :, 2*iy + dy, 2*ix + dx] for iy < h, ix < w, zero outside t (the stride-2 box with hardware zero fill)."""
    n, c, H, W = t.shape
    out = torch.zeros((n, c, h, w), dtype=t.dtype)
    for iy in range(h):
        for ix in range(w):
            y, x = 2 * iy + dy, 2 * ix + dx
            if 0 <= y < H and 0 <= x < W:
                out[:, :, iy, ix] = t[:, :, y, x]
    return out


@pytest.fixture
def problem():
    g = torch.Generator().manual_seed(0)
    n, cin, cout, h = 2, 3, 5, 4
    x = torch.randn((n, cin, h, h), dtype=torch.float64, generator=g, requires_grad=True)
    w = torch.randn((cin, cout, 4, 4), dtype=torch.float64, generator=g, requires_grad=True)
    y = F.conv_transpose2d(x, w, stride=2, padding=1)
    dy = torch.randn(y.shape, dtype=torch.float64, generator=g)
    dx, dw = torch.autograd.grad(y, (x, w), dy)
    return x.detach(), w.detach(), dy, dx, dw


def test_dgrad_is_a_16_tap_stride_2_conv(problem):
    """dx[n,ci,iy,ix] = sum_{tap,co} dy[n,co,2iy-1+ky,2ix-1+kx] W[ci,co,ky,kx], tap = ky*4 + kx: the B operand
    [ci][tap*Cout + co] against the A rows of dy shifted by (tap/4 - 1, tap%4 - 1)."""
    x, w, dy, dx, _ = problem
    n, cin, h, _ = x.shape
    cout = w.shape[1]
    b = w.permute(0, 2, 3, 1).reshape(cin, 16 * cout)                  # packed [ci][tap*Cout + co]
    got = torch.zeros_like(dx)
    for tap in range(16):
        a = _shifted(dy, tap // 4 - 1, tap % 4 - 1, h, h)              # (n, cout, h, w)
        got += torch.einsum("nchw,ic->nihw", a, b[:, tap * cout:(tap + 1) * cout])
    assert torch.allclose(got, dx, rtol=1e-12, atol=1e-12)


def test_wgrad_is_16_per_tap_pixel_reductions(problem):
    """dW[ci,co,ky,kx] = sum over the pixels p = (n, iy, ix) of x[p, ci] * dy[n, 2iy-1+ky, 2ix-1+kx, co]: one GEMM
    per tap with M = Cin, N = Cout, K = pixels, K split into slices summed in order."""
    x, w, dy, _, dw = problem
    n, cin, h, _ = x.shape
    cout = w.shape[1]
    xr = x.permute(0, 2, 3, 1).reshape(-1, cin)                         # pixel-major rows, channels contiguous
    got = torch.zeros_like(dw)
    for tap in range(16):
        d = _shifted(dy, tap // 4 - 1, tap % 4 - 1, h, h).permute(0, 2, 3, 1).reshape(-1, cout)
        slices = [xr[k:k + 8].T @ d[k:k + 8] for k in range(0, xr.shape[0], 8)]
        got[:, :, tap // 4, tap % 4] = sum(slices)
    assert torch.allclose(got, dw, rtol=1e-12, atol=1e-12)


def _domain():
    """tests/test_gpu_deconv_train_domain.py (its shape table and slice mirror), imported without a GPU."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_gpu_deconv_train_domain.py")
    spec = importlib.util.spec_from_file_location("_deconv_train_domain", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_shape_table_covers_the_plan():
    """The GPU table reaches every wgrad slice count the plan produces, padded and unpadded channel tiles on both
    sides, partial kSplitChunk chunks of the forward (4*Cin/64 K blocks) and a slice that ends mid-image."""
    D = _domain()
    assert {s for *_, s in D.TABLE} == {1, 2, 4, 8, 16, 32}
    assert all(D.slices(n, cin, cout, h) == s for n, cin, cout, h, s in D.TABLE)
    assert {cin % 128 for _, cin, _, _, _ in D.TABLE} == {0, 64}
    assert {cout % 128 for _, _, cout, _, _ in D.TABLE} == {0, 64}
    assert any((4 * cin // 64) % 8 for _, cin, _, _, _ in D.TABLE)
    assert any((n * h * h) % (64 * s) == 0 and (n * h * h // s) % (h * h) for n, _, _, h, s in D.TABLE)
    # the mirror never grows past 32: the tile count of the smallest layer times 32 already fills two waves
    assert max(D.slices(n, 64, 64, h) for n in (1, 64, 1024, 4096) for h in (8, 16, 32)) == 32


def test_slice_mirror_fits_the_reported_workspace(pkg):
    """The backward workspace holds the wgrad partials, [slices][16 taps][Cin][round_up(Cout, 128)] fp32: a mirror
    that counted more slices than the library would not fit in what cdr_deconv_train_workspace_bytes reports."""
    D = _domain()
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    for n, cin, cout, h, sl in D.TABLE:
        assert L.cdr_deconv_train_workspace_bytes(n, cin, cout, h, h, C.byref(s), C.byref(w)) == 0
        assert w.value >= sl * 16 * cin * (cout + 127) // 128 * 128 * 4


def test_per_element_gate_catches_a_lost_lo_plane():
    """With x through both planes the forward passes the per-element gate; with the hi plane alone (~2^-12 m) it
    fails.  So the gate's constant is tight enough to see the lo plane, and c <= 2^-14."""
    assert GATE_C <= 2.0 ** -14
    g = torch.Generator().manual_seed(0)
    x = torch.randn((1, 4, 8, 8), generator=g).double()          # fp32 values, held in fp64
    w = torch.randn((4, 3, 4, 4), generator=g).float().double()
    ref = F.conv_transpose2d(x, w, stride=2, padding=1)
    mag = F.conv_transpose2d(x.abs(), w.abs(), stride=2, padding=1)
    gate("y", F.conv_transpose2d(f16_planes(x, True), w, stride=2, padding=1), ref, mag)
    with pytest.raises(AssertionError, match="per-element gate"):
        gate("y", F.conv_transpose2d(f16_planes(x, False), w, stride=2, padding=1), ref, mag, max_gate=False)


def test_conv_transpose2d_rejects_without_cuda(pkg, monkeypatch):
    import torch.cuda
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: pytest.fail("touched CUDA"))
    x = torch.zeros((2, 64, 8, 8))
    w = torch.zeros((64, 64, 4, 4))
    with pytest.raises(ValueError, match="CUDA"):
        pkg.conv_transpose2d(x, w)                                    # CPU tensors
    with pytest.raises(ValueError, match="float32"):
        pkg.conv_transpose2d(x.double(), w.double())
    with pytest.raises(ValueError, match="float32"):
        pkg.conv_transpose2d(x.half(), w)
    for xs, ws in (((2, 64, 8, 8), (64, 64, 3, 3)),                   # not 4x4
                   ((2, 64, 8, 8), (32, 64, 4, 4)),                   # Cin mismatch
                   ((2, 48, 8, 8), (48, 64, 4, 4)),                   # Cin not a multiple of 64
                   ((2, 64, 8, 8), (64, 40, 4, 4)),                   # Cout not a multiple of 64
                   ((2, 64, 12, 12), (64, 64, 4, 4)),                 # H not in {8, 16, 32}
                   ((2, 64, 8, 16), (64, 64, 4, 4)),                  # H != W
                   ((64, 8, 8), (64, 64, 4, 4))):                     # not 4-D
        with pytest.raises(ValueError, match="expected|unsupported"):
            pkg.conv_transpose2d(torch.zeros(xs), torch.zeros(ws))


def test_abi_validation_without_gpu(pkg):
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    assert L.cdr_deconv_train_workspace_bytes(64, 2048, 256, 8, 8, C.byref(s), C.byref(w)) == 0
    assert s.value >= 64 * 64 * 2048 * 4 and w.value > 0
    assert L.cdr_deconv_train_workspace_bytes(64, 2048, 256, 12, 12, C.byref(s), C.byref(w)) == 4
    assert L.cdr_deconv_train_workspace_bytes(64, 2000, 256, 8, 8, C.byref(s), C.byref(w)) == 4
    assert L.cdr_deconv_train_workspace_bytes(0, 2048, 256, 8, 8, C.byref(s), C.byref(w)) == 1
    assert L.cdr_deconv_train_workspace_bytes(1, 64, 64, 8, 8, None, None) == 1
    assert L.cdr_deconv_train_forward(None, None, 1, 64, 64, 8, 8, None, None, 0, None, 0, None) == 1
    assert b"cdr_deconv_train_forward" in L.cdr_last_error()
    assert L.cdr_deconv_train_backward(None, None, None, 1, 64, 64, 8, 8, None, None, None, 0, None) == 1
    fake = C.c_void_p(1 << 20)                                        # never dereferenced: the shape check comes first
    assert L.cdr_deconv_train_backward(fake, fake, fake, 1, 64, 64, 16, 8, None, fake, fake, 1 << 30, None) == 4
