"""CPU: the argument checks of conv1x1 and of the cdr_conv1x1_train_* entry points, none of which may touch CUDA, and the
pieces of test_gpu_conv1x1_train.py that need no GPU: its shape table against the wgrad slice plan, and the strictness
of the per-element gate it shares with the other training convolutions (train_conv_checks.py)."""
import ctypes as C
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

from train_conv_checks import GATE_C, f16_planes, gate


def _domain():
    """tests/test_gpu_conv1x1_train.py (its shape table and slice mirror), imported without a GPU."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_gpu_conv1x1_train.py")
    spec = importlib.util.spec_from_file_location("_conv1x1_train_domain", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_shape_table_covers_the_plan():
    """The GPU table reaches every wgrad slice count the plan produces (1 .. 512), channel counts = 1 and 63 (mod 64)
    on both sides, a half-full last 128-pixel tile and a slice that ends mid-image."""
    D = _domain()
    assert all(D.slices(n, cin, cout, h, w) == s for n, cin, cout, h, w, s in D.TABLE)
    produced = {D.slices(n, cin, cout, h, h) for n in (1, 2, 3, 16, 64, 256, 1024, 4096) for cin in (1, 300, 2048)
                for cout in (1, 19, 400) for h in (8, 16, 32, 64) if n * h * h <= 1 << 22}
    assert produced <= {s for *_, s in D.TABLE} == {1 << i for i in range(10)}
    assert max(D.slices((1 << 22) // (h * h), 1, 1, h, h) for h in (8, 64)) == 512
    assert {cin % 64 for _, cin, *_ in D.TABLE} >= {1, 63} and {cout % 64 for _, _, cout, *_ in D.TABLE} >= {1, 63}
    assert any((n * h * w) % 128 == 64 for n, _, _, h, w, _ in D.TABLE)
    assert any((n * h * w // s) % (h * w) for n, _, _, h, w, s in D.TABLE)


def test_slice_mirror_fits_the_reported_workspace(pkg):
    """The backward workspace holds the wgrad partials, [slices][Cout][round_up(Cin, 128)] fp32: a mirror that counted
    more slices than the library would not fit in what cdr_conv1x1_train_workspace_bytes reports."""
    D = _domain()
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    for n, cin, cout, h, wd, sl in D.TABLE:
        assert L.cdr_conv1x1_train_workspace_bytes(n, cin, cout, h, wd, C.byref(s), C.byref(w)) == 0
        assert w.value >= sl * cout * ((cin + 127) // 128 * 128) * 4
        assert s.value >= 2 * n * h * wd * ((cin + 63) // 64 * 64) * 2         # x as padded fp16 hi / lo planes


def test_per_element_gate_catches_a_lost_lo_plane():
    """With x through both planes the forward passes the per-element gate; with the hi plane alone (~2^-12 m) it
    fails.  So the gate's constant is tight enough to see the lo plane."""
    assert GATE_C <= 2.0 ** -14
    g = torch.Generator().manual_seed(0)
    x = torch.randn((2, 65, 8, 8), generator=g).double()        # fp32 values, held in fp64
    w = torch.randn((19, 65, 1, 1), generator=g).float().double()
    b = torch.randn((19,), generator=g).float().double()
    ref = F.conv2d(x, w, b)
    mag = F.conv2d(x.abs(), w.abs(), b.abs())
    gate("y", F.conv2d(f16_planes(x, True), w, b), ref, mag)
    with pytest.raises(AssertionError, match="per-element gate"):
        gate("y", F.conv2d(f16_planes(x, False), w, b), ref, mag, max_gate=False)


def test_conv1x1_rejects_without_cuda(pkg, monkeypatch):
    import torch.cuda
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: pytest.fail("touched CUDA"))
    x = torch.zeros((2, 64, 8, 8))
    w = torch.zeros((19, 64, 1, 1))
    b = torch.zeros(19)
    with pytest.raises(ValueError, match="CUDA"):
        pkg.conv1x1(x, w, b)                                          # CPU tensors
    with pytest.raises(ValueError, match="CUDA"):
        pkg.conv1x1(x, w)
    with pytest.raises(ValueError, match="float32"):
        pkg.conv1x1(x.double(), w.double(), b.double())
    with pytest.raises(ValueError, match="float32"):
        pkg.conv1x1(x, w, b.half())
    for xs, ws, bs in (((2, 64, 8, 8), (19, 64, 3, 3), (19,)),        # not 1x1
                       ((2, 64, 8, 8), (19, 32, 1, 1), (19,)),        # Cin mismatch
                       ((2, 64, 8, 8), (19, 64, 1, 1), (20,)),        # bias of the wrong length
                       ((2, 64, 8, 8), (19, 64, 1, 1), (19, 1)),      # bias not 1-D
                       ((2, 64, 12, 12), (19, 64, 1, 1), (19,)),      # H*W = 144: not a multiple of 64
                       ((2, 64, 4, 4), (19, 64, 1, 1), (19,)),        # H*W = 16
                       ((2, 4097, 8, 8), (19, 4097, 1, 1), (19,)),    # Cin > 4096
                       ((2, 64, 8, 8), (4097, 64, 1, 1), (4097,)),    # Cout > 4096
                       ((1025, 64, 64, 64), (19, 64, 1, 1), (19,)),   # N*H*W > 2^22
                       ((64, 8, 8), (19, 64, 1, 1), (19,))):          # not 4-D
        with pytest.raises(ValueError, match="expected|unsupported"):
            pkg.conv1x1(torch.zeros(xs), torch.zeros(ws), torch.zeros(bs))


def test_abi_validation_without_gpu(pkg):
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    assert L.cdr_conv1x1_train_workspace_bytes(64, 2048, 300, 8, 8, C.byref(s), C.byref(w)) == 0
    assert s.value >= 2 * 64 * 64 * 2048 * 2 and w.value > 0
    assert L.cdr_conv1x1_train_workspace_bytes(1, 1, 1, 8, 8, C.byref(s), C.byref(w)) == 0
    for n, cin, cout, h, wd in ((64, 2048, 300, 12, 12), (64, 2048, 300, 4, 4), (0, 64, 64, 8, 8), (1, 0, 64, 8, 8),
                                (1, 64, 0, 8, 8), (1, 4097, 64, 8, 8), (1, 64, 4097, 8, 8), (1025, 64, 64, 64, 64),
                                (1, 64, 64, 0, 64)):
        assert L.cdr_conv1x1_train_workspace_bytes(n, cin, cout, h, wd, C.byref(s), C.byref(w)) == 1
        assert b"cdr_conv1x1_train_workspace_bytes" in L.cdr_last_error()
    assert L.cdr_conv1x1_train_workspace_bytes(1, 64, 64, 8, 8, None, None) == 1
    assert L.cdr_conv1x1_train_forward(None, None, None, 1, 64, 64, 8, 8, None, None, 0, None, 0, None) == 1
    assert b"cdr_conv1x1_train_forward" in L.cdr_last_error()
    assert L.cdr_conv1x1_train_backward(None, None, None, 1, 64, 64, 8, 8, None, None, None, None, 0, None) == 1
    assert b"cdr_conv1x1_train_backward" in L.cdr_last_error()
    fake = C.c_void_p(1 << 20)                                        # never dereferenced: the shape check comes first
    assert L.cdr_conv1x1_train_forward(fake, fake, None, 1, 64, 64, 12, 12, fake, fake, 1 << 30, fake, 1 << 30,
                                       None) == 1
    assert b"cdr_conv1x1_train_forward" in L.cdr_last_error()
    assert L.cdr_conv1x1_train_backward(fake, fake, fake, 1, 64, 64, 12, 12, fake, None, None, fake, 1 << 30, None) == 1
    assert b"cdr_conv1x1_train_backward" in L.cdr_last_error()
    odd = C.c_void_p((1 << 20) + 4)                                   # misaligned: rejected before any CUDA call
    assert L.cdr_conv1x1_train_forward(odd, fake, None, 1, 64, 64, 8, 8, fake, fake, 1 << 30, fake, 1 << 30, None) == 1
