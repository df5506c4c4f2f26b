"""CPU: the argument checks of stem_conv and max_pool3x3 and of their cdr_* entry points, none of which may touch CUDA;
the shape table of test_gpu_stem_train.py against its slice mirror and the workspace the library reports; the
strictness of the per-element gate on the stem's weight gradient; and a CPU mirror of the max-pool's selection and
summation rule against torch's CPU max-pool."""
import ctypes as C
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

from train_conv_checks import GATE_C, f16_planes, gate


def _domain():
    """tests/test_gpu_stem_train.py (its shape table and slice mirror), imported without a GPU."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "test_gpu_stem_train.py")
    spec = importlib.util.spec_from_file_location("_stem_train_domain", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_shape_table_covers_the_plan():
    """The table reaches one chunk per slice, several with a ragged last slice, slices ending mid-image, H != W both
    ways and the B = 64 view; every shape is in the domain."""
    D = _domain()
    assert all(D.slices(n, h, w) == sl for n, h, w, sl in D.TABLE)
    assert all(h % 16 == 0 and w % 64 == 0 and n * (h // 2) * (w // 2) <= 1 << 22 for n, h, w, _ in D.TABLE)
    chunks = [(n * (h // 4) * (w // 64), (h // 4) * (w // 64), sl) for n, h, w, sl in D.TABLE]
    assert any(c == sl for c, _, sl in chunks) and any(c % sl and c > sl for c, _, sl in chunks)
    assert any((-(-c // sl)) % per_img and c > sl for c, per_img, sl in chunks)       # a slice ends mid-image
    assert any(h > w for _, h, w, _ in D.TABLE) and any(h < w for _, h, w, _ in D.TABLE)
    assert (64, 256, 256) in {t[:3] for t in D.TABLE}
    assert max(D.slices(n, 256, 256) for n in range(1, 257)) <= D.TARGET_SLICES


def test_slice_mirror_fits_the_reported_workspace(pkg):
    """The backward workspace holds the wgrad partials, [slices][64][147] fp32 after a 256-byte scale slot: a mirror
    that counted more slices than the library would not fit; saved holds x as fp16 hi / lo planes."""
    D = _domain()
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    for n, h, wd, sl in D.TABLE + [(256, 256, 256, D.slices(256, 256, 256))]:
        assert L.cdr_stem_train_workspace_bytes(n, 3, 64, h, wd, C.byref(s), C.byref(w)) == 0
        assert w.value >= 256 + sl * 64 * 147 * 4
        assert s.value >= 2 * n * 3 * h * wd * 2


def test_per_element_gate_catches_a_lost_lo_plane():
    """An fp64 emulation of the weight gradient through both planes of x and dy passes the per-element gate; dropping
    the lo plane of x, or of dy, fails it.  So the gate's constant is tight enough to see either lo plane."""
    assert GATE_C <= 2.0 ** -14
    g = torch.Generator().manual_seed(0)
    x = torch.randn((2, 3, 32, 64), generator=g).double()
    dy = torch.randn((2, 64, 16, 32), generator=g).double()

    def wgrad(xv, dyv):
        w = torch.zeros((64, 3, 7, 7), dtype=torch.float64, requires_grad=True)
        (dw,) = torch.autograd.grad(F.conv2d(xv, w, stride=2, padding=3), (w,), dyv)
        return dw
    ref, mag = wgrad(x, dy), wgrad(x.abs(), dy.abs())
    gate("dw", wgrad(f16_planes(x, True), f16_planes(dy, True)), ref, mag)
    for xv, dyv in ((f16_planes(x, False), f16_planes(dy, True)), (f16_planes(x, True), f16_planes(dy, False))):
        with pytest.raises(AssertionError, match="per-element gate"):
            gate("dw", wgrad(xv, dyv), ref, mag, max_gate=False)


def test_ops_reject_without_cuda(pkg, monkeypatch):
    import torch.cuda
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: pytest.fail("touched CUDA"))
    x, w = torch.zeros((2, 3, 32, 64)), torch.zeros((64, 3, 7, 7))
    with pytest.raises(ValueError, match="requires grad"):
        pkg.stem_conv(x.clone().requires_grad_(True), w)
    with pytest.raises(ValueError, match="CUDA"):
        pkg.stem_conv(x, w)
    with pytest.raises(ValueError, match="float32"):
        pkg.stem_conv(x.double(), w.double())
    for xs, ws in (((2, 3, 32, 64), (64, 3, 5, 5)),       # not 7x7
                   ((2, 3, 32, 64), (64, 4, 7, 7)),       # Cin mismatch
                   ((2, 4, 32, 64), (64, 4, 7, 7)),       # Cin = 4
                   ((2, 3, 32, 64), (128, 3, 7, 7)),      # Cout = 128
                   ((2, 3, 24, 64), (64, 3, 7, 7)),       # H % 16
                   ((2, 3, 32, 96), (64, 3, 7, 7)),       # W % 64
                   ((257, 3, 256, 256), (64, 3, 7, 7)),   # N*(H/2)*(W/2) > 2^22
                   ((3, 32, 64), (64, 3, 7, 7))):         # not 4-D
        with pytest.raises(ValueError, match="expected|unsupported"):
            pkg.stem_conv(torch.zeros(xs), torch.zeros(ws))
    with pytest.raises(ValueError, match="CUDA"):
        pkg.max_pool3x3(torch.zeros((1, 2, 5, 5)))
    with pytest.raises(ValueError, match="float32"):
        pkg.max_pool3x3(torch.zeros((1, 2, 5, 5), dtype=torch.float64))
    with pytest.raises(ValueError, match="expected"):
        pkg.max_pool3x3(torch.zeros((2, 5, 5)))
    with pytest.raises(ValueError, match="unsupported"):
        pkg.max_pool3x3(torch.zeros((1, 0, 5, 5)))


def test_abi_validation_without_gpu(pkg):
    L = pkg._lib.lib()
    s, w = C.c_size_t(), C.c_size_t()
    assert L.cdr_stem_train_workspace_bytes(64, 3, 64, 256, 256, C.byref(s), C.byref(w)) == 0
    assert L.cdr_stem_train_workspace_bytes(256, 3, 64, 256, 256, C.byref(s), C.byref(w)) == 0
    for args in ((0, 3, 64, 256, 256), (1, 4, 64, 256, 256), (1, 3, 32, 256, 256), (1, 3, 64, 24, 256),
                 (1, 3, 64, 256, 96), (1, 3, 64, 0, 64), (1, 3, 64, 16, 0), (257, 3, 64, 256, 256)):
        assert L.cdr_stem_train_workspace_bytes(*args, C.byref(s), C.byref(w)) == 1, args
        assert b"cdr_stem_train_workspace_bytes" in L.cdr_last_error()
    assert L.cdr_stem_train_workspace_bytes(1, 3, 64, 16, 64, None, None) == 1
    assert L.cdr_stem_train_forward(None, None, 1, 3, 64, 16, 64, None, None, 0, None, 0, None) == 1
    assert b"cdr_stem_train_forward" in L.cdr_last_error()
    assert L.cdr_stem_train_backward(None, None, None, 1, 3, 64, 16, 64, None, None, None, 0, None) == 1
    assert b"cdr_stem_train_backward" in L.cdr_last_error()
    fake = C.c_void_p(1 << 20)                                        # never dereferenced: the checks come first
    assert L.cdr_stem_train_backward(fake, fake, fake, 1, 3, 64, 16, 64, fake, fake, fake, 1 << 30, None) == 1
    assert b"dx must be NULL" in L.cdr_last_error()
    assert L.cdr_stem_train_forward(fake, fake, 1, 3, 64, 24, 64, fake, fake, 1 << 30, fake, 1 << 30, None) == 1
    odd = C.c_void_p((1 << 20) + 4)                                   # misaligned
    assert L.cdr_stem_train_forward(odd, fake, 1, 3, 64, 16, 64, fake, fake, 1 << 30, fake, 1 << 30, None) == 1
    assert L.cdr_stem_train_backward(fake, fake, fake, 1, 3, 64, 16, 64, None, odd, fake, 1 << 30, None) == 1
    assert L.cdr_stem_train_forward(fake, fake, 1, 3, 64, 16, 64, fake, fake, 16, fake, 1 << 30, None) == 3
    assert b"saved" in L.cdr_last_error()
    # max-pool: null pointers, sizes, alignment
    assert L.cdr_maxpool3x3_train_forward(None, 1, 1, 5, 5, fake, fake, None) == 1
    assert L.cdr_maxpool3x3_train_forward(fake, 1, 1, 5, 5, fake, None, None) == 1
    assert L.cdr_maxpool3x3_train_backward(None, fake, 1, 1, 5, 5, fake, None) == 1
    for n, c, h, wd in ((0, 1, 5, 5), (1, 0, 5, 5), (1, 1, 0, 5), (1, 1, 5, 0), (1024, 1024, 64, 32)):
        assert L.cdr_maxpool3x3_train_forward(fake, n, c, h, wd, fake, fake, None) == 1
        assert b"cdr_maxpool3x3_train_forward" in L.cdr_last_error()
        assert L.cdr_maxpool3x3_train_backward(fake, fake, n, c, h, wd, fake, None) == 1
    assert L.cdr_maxpool3x3_train_forward(C.c_void_p((1 << 20) + 2), 1, 1, 5, 5, fake, fake, None) == 1
    assert L.cdr_maxpool3x3_train_backward(fake, fake, 1, 1, 5, 5, C.c_void_p((1 << 20) + 1), None) == 1


def test_forward_train_binds_the_stem_ops_at_import(pkg):
    from fast_3d_human_pose_estimation_b200 import autograd as AG, encoder as E
    assert E._stem_conv is AG.stem_conv and E._max_pool3x3 is AG.max_pool3x3


# ---- the max-pool's selection and summation rule, mirrored on the CPU ----
def _pool_mirror(x, dy):
    """Scan each window row-major from its first in-image element, replace on > or NaN; dx[e] = sum from +0.0 in
    (oy, ox) order of dy over the windows whose argmax is e.  -> (y, window positions, dx)"""
    n, c, h, w = x.shape
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    y = torch.empty((n, c, ho, wo), dtype=x.dtype)
    pos = torch.empty((n, c, ho, wo), dtype=torch.int64)
    for oy in range(ho):
        for ox in range(wo):
            m = torch.full((n, c), float("-inf"), dtype=x.dtype)
            iy0, ix0 = max(2 * oy - 1, 0), max(2 * ox - 1, 0)
            p = torch.full((n, c), (iy0 - 2 * oy + 1) * 3 + (ix0 - 2 * ox + 1), dtype=torch.int64)
            for iy in range(iy0, min(2 * oy + 2, h)):
                for ix in range(ix0, min(2 * ox + 2, w)):
                    v = x[:, :, iy, ix]
                    take = (v > m) | torch.isnan(v)
                    m = torch.where(take, v, m)
                    p = torch.where(take, torch.full_like(p, (iy - 2 * oy + 1) * 3 + (ix - 2 * ox + 1)), p)
            y[:, :, oy, ox], pos[:, :, oy, ox] = m, p
    dx = torch.empty_like(x)
    for iy in range(h):
        for ix in range(w):
            s = torch.zeros((n, c), dtype=x.dtype)
            for oy in range(iy // 2, min((iy + 1) // 2, ho - 1) + 1):
                for ox in range(ix // 2, min((ix + 1) // 2, wo - 1) + 1):
                    hit = pos[:, :, oy, ox] == (iy - 2 * oy + 1) * 3 + (ix - 2 * ox + 1)
                    s = torch.where(hit, s + dy[:, :, oy, ox], s)
            dx[:, :, iy, ix] = s
    return y, pos, dx


@pytest.mark.parametrize("kind", ["ties", "nonfinite", "relu"])
@pytest.mark.parametrize("shape", [(2, 3, 9, 11), (1, 2, 1, 5), (1, 2, 2, 2), (2, 1, 6, 1)])
def test_pool_rule_matches_torch_cpu(kind, shape):
    g = torch.Generator().manual_seed(sum(shape))
    if kind == "ties":
        x = torch.randint(1, 4, shape, generator=g).float()
    elif kind == "relu":
        x = torch.randn(shape, generator=g).clamp_min(0)
    else:
        x = torch.randn(shape, generator=g)
        r = torch.rand(shape, generator=g)
        x[r < 0.15] = float("nan")
        x[(r >= 0.15) & (r < 0.25)] = float("inf")
        x[(r >= 0.25) & (r < 0.35)] = float("-inf")
    xr = x.clone().requires_grad_(True)
    yr, idx = F.max_pool2d_with_indices(xr, 3, 2, 1)
    dy = torch.randn(yr.shape, generator=g)
    yr.backward(dy)
    y, pos, dx = _pool_mirror(x, dy)
    w = shape[3]
    ho, wo = yr.shape[2:]
    oy = torch.arange(ho).view(-1, 1)
    ox = torch.arange(wo).view(1, -1)
    flat = (2 * oy - 1 + pos // 3) * w + (2 * ox - 1 + pos % 3)        # the window position as torch's flat index
    assert torch.equal(flat, idx)
    assert torch.equal(y.view(torch.int32), yr.detach().view(torch.int32))
    assert torch.equal(dx.view(torch.int32), xr.grad.view(torch.int32))
