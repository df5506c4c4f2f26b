"""Differentiable forms of the path's non-conv operators (SURVEY §8f rank 3, first slice).

``train_cdr.py:105-127`` back-propagates its losses through ``CDRNet.process_heatmap``
(models/cdrnet.py:120-149), ``CDRNet.dlt`` (:151-179) and ``CanonicalFusion.ftl`` (:45-56).  These
``torch.autograd.Function`` s run forward AND backward in libcdrhead.so, on the reference's own
tensor layouts (NCHW heat-maps / feature maps, (B,J,2) joints, (B,3,4) projections), so a training
script can swap them in one call at a time:

    kp  = soft_argmax_2d(heatmap, scale=4.0)          # == process_heatmap(heatmap) * 4.0
    xyz = dlt(P_l, P_r, kp_l, kp_r)                   # == stack([dlt(projs, kps[:, j]) for j ...], 1)
    z   = ftl(feat, mats)                             # == CanonicalFusion.ftl(feat, mats)

Projection matrices carry no gradient (they are data in the reference).  CUDA fp32 only; no fallback.

The decoder's transposed convolutions have one too, forward and backward on the f16x2 tensor-core GEMM at fp32
accuracy (independent of torch's TF32 flags):

    y = conv_transpose2d(x, weight)                   # == F.conv_transpose2d(x, weight, stride=2, padding=1)

and so do the head's 1x1 convolutions (the fusion block's and ``decoder.final_layer``), bias included:

    y = conv1x1(x, weight, bias)                      # == F.conv2d(x, weight, bias) for a (Cout, Cin, 1, 1) weight

and so do the encoder's 3x3 convolutions, at stride 1 and 2:

    y = conv3x3(x, weight, stride)                    # == F.conv2d(x, weight, stride=stride, padding=1), no bias
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


def _chk(t, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32):
        raise TypeError(f"{name}: CUDA float32 tensor expected (there is no CPU fallback)")
    return t.contiguous()


class _SoftArgmax2D(torch.autograd.Function):
    @staticmethod
    def forward(ctx, heat, scale):
        heat = _chk(heat, "soft_argmax_2d: heat")
        assert heat.dim() == 4, "heat-maps must be (B, J, H, W)"
        b, j, h, w = heat.shape
        kp = torch.empty((b, j, 2), dtype=torch.float32, device=heat.device)
        L = _lib.lib()
        with torch.cuda.device(heat.device):
            _lib.check(L.cdr_softargmax(_lib.ptr(heat), b * j, h, w, float(scale), _lib.ptr(kp),
                                        _lib.current_stream_ptr(heat.device)))
        ctx.save_for_backward(heat)
        ctx.scale = float(scale)
        return kp

    @staticmethod
    def backward(ctx, grad_kp):
        (heat,) = ctx.saved_tensors
        b, j, h, w = heat.shape
        g = _chk(grad_kp, "soft_argmax_2d: grad")
        out = torch.empty_like(heat)
        L = _lib.lib()
        with torch.cuda.device(heat.device):
            _lib.check(L.cdr_softargmax_backward(_lib.ptr(heat), _lib.ptr(g), b * j, h, w, ctx.scale, _lib.ptr(out),
                                                 _lib.current_stream_ptr(heat.device)))
        return out, None


class _DLT(torch.autograd.Function):
    @staticmethod
    def forward(ctx, P_l, P_r, kp_l, kp_r):
        P_l, P_r = _chk(P_l, "dlt: P_l"), _chk(P_r, "dlt: P_r")
        kp_l, kp_r = _chk(kp_l, "dlt: kp_l"), _chk(kp_r, "dlt: kp_r")
        b, j = kp_l.shape[:2]
        assert P_l.shape == (b, 3, 4) and P_r.shape == (b, 3, 4) and kp_r.shape == (b, j, 2) == kp_l.shape
        xyz = torch.empty((b, j, 3), dtype=torch.float32, device=kp_l.device)
        L = _lib.lib()
        with torch.cuda.device(kp_l.device):
            _lib.check(L.cdr_dlt(_lib.ptr(P_l), _lib.ptr(P_r), _lib.ptr(kp_l), _lib.ptr(kp_r), b, j, _lib.ptr(xyz),
                                 _lib.current_stream_ptr(kp_l.device)))
        ctx.save_for_backward(P_l, P_r, kp_l, kp_r)
        return xyz

    @staticmethod
    def backward(ctx, grad_xyz):
        P_l, P_r, kp_l, kp_r = ctx.saved_tensors
        b, j = kp_l.shape[:2]
        g = _chk(grad_xyz, "dlt: grad")
        gl, gr = torch.empty_like(kp_l), torch.empty_like(kp_r)
        L = _lib.lib()
        with torch.cuda.device(kp_l.device):
            _lib.check(L.cdr_dlt_backward(_lib.ptr(P_l), _lib.ptr(P_r), _lib.ptr(kp_l), _lib.ptr(kp_r), _lib.ptr(g), b, j,
                                          _lib.ptr(gl), _lib.ptr(gr), _lib.current_stream_ptr(kp_l.device)))
        return None, None, gl, gr


def _ftl_nchw(x, mats):
    """out[b, r*blk + c, p] = sum_k mats[b,r,k] * x[b, k*blk + c, p] on NCHW: for one sample the (c, p) plane of a
    coordinate block is contiguous, so it is cdr_ftl with one "pixel" per sample and blocks of blk*H*W elements."""
    b, c, h, w = x.shape
    rows, cols = mats.shape[1:]
    assert c % cols == 0, "channels must split into mats.shape[2] coordinate blocks"
    blk = (c // cols) * h * w
    out = torch.empty((b, rows * (c // cols), h, w), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    with torch.cuda.device(x.device):
        _lib.check(L.cdr_ftl(_lib.ptr(x), cols * blk, _lib.ptr(mats), rows, cols, blk, b, 1, _lib.ptr(out), rows * blk,
                             rows * blk, _lib.current_stream_ptr(x.device)))
    return out


class _FTL(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mats):
        x, mats = _chk(x, "ftl: x"), _chk(mats, "ftl: mats")
        assert x.dim() == 4 and mats.dim() == 3 and mats.shape[0] == x.shape[0]
        ctx.save_for_backward(mats)
        return _ftl_nchw(x, mats)

    @staticmethod
    def backward(ctx, grad_out):
        (mats,) = ctx.saved_tensors
        if ctx.needs_input_grad[1]:
            raise NotImplementedError("ftl: projection matrices carry no gradient (data in the reference)")
        return _ftl_nchw(_chk(grad_out, "ftl: grad"), mats.transpose(1, 2).contiguous()), None


def soft_argmax_2d(heat, scale=1.0):
    """(B,J,H,W) logits -> (B,J,2) = scale * spatial-softmax centre of mass, (x, y) order."""
    return _SoftArgmax2D.apply(heat, scale)


def dlt(P_l, P_r, kp_l, kp_r):
    """(B,3,4) x2, (B,J,2) x2 -> (B,J,3): per-joint two-view DLT triangulation."""
    return _DLT.apply(P_l, P_r, kp_l, kp_r)


def ftl(x, mats):
    """CanonicalFusion.ftl on NCHW: x (B, K*blk, H, W), mats (B, R, K) -> (B, R*blk, H, W)."""
    return _FTL.apply(x, mats)


def _deconv_args(x, weight):
    """Checks of conv_transpose2d's inputs, all before any CUDA call: ValueError, there is no fallback."""
    if not (isinstance(x, torch.Tensor) and isinstance(weight, torch.Tensor)):
        raise ValueError("conv_transpose2d: x and weight must be tensors")
    if x.dim() != 4 or weight.dim() != 4 or tuple(weight.shape[2:]) != (4, 4) or weight.shape[0] != x.shape[1]:
        raise ValueError(f"conv_transpose2d: x (N, Cin, H, W) and weight (Cin, Cout, 4, 4) expected, got "
                         f"{tuple(x.shape)} and {tuple(weight.shape)}")
    n, cin, h, w = x.shape
    cout = weight.shape[1]
    if n < 1 or cin % 64 or cout % 64 or h != w or h not in (8, 16, 32):
        raise ValueError(f"conv_transpose2d: unsupported shape x {tuple(x.shape)}, weight {tuple(weight.shape)} "
                         "(Cin and Cout multiples of 64, H == W in {8, 16, 32})")
    if x.dtype != torch.float32 or weight.dtype != torch.float32:
        raise ValueError(f"conv_transpose2d: float32 expected, got {x.dtype} and {weight.dtype}")
    if not (x.is_cuda and weight.is_cuda) or x.device != weight.device:
        raise ValueError("conv_transpose2d: x and weight must be CUDA tensors on one device (there is no CPU fallback)")
    return x.contiguous(), weight.contiguous()


class _ConvTranspose2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight):
        x, weight = _deconv_args(x, weight)
        n, cin, h, w = x.shape
        cout = weight.shape[1]
        L = _lib.lib()
        saved_b, ws_b = C.c_size_t(), C.c_size_t()
        _lib.check(L.cdr_deconv_train_workspace_bytes(n, cin, cout, h, w, C.byref(saved_b), C.byref(ws_b)))
        dev = x.device
        y = torch.empty((n, cout, 2 * h, 2 * w), dtype=torch.float32, device=dev)
        saved = torch.empty(saved_b.value, dtype=torch.uint8, device=dev)     # x as fp16 planes, for the weight gradient
        ws = torch.empty(ws_b.value, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.cdr_deconv_train_forward(_lib.ptr(x), _lib.ptr(weight), n, cin, cout, h, w, _lib.ptr(y),
                                                  _lib.ptr(saved), saved_b.value, _lib.ptr(ws), ws_b.value,
                                                  _lib.current_stream_ptr(dev)))
        ctx.save_for_backward(saved, weight)
        ctx.dims = (n, cin, cout, h, w)
        ctx.ws_bytes = ws_b.value
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y):
        saved, weight = ctx.saved_tensors
        n, cin, cout, h, w = ctx.dims
        need_x, need_w = ctx.needs_input_grad[:2]
        if not (need_x or need_w):
            return None, None
        dy = _chk(grad_y, "conv_transpose2d: grad")
        dev = dy.device
        dx = torch.empty((n, cin, h, w), dtype=torch.float32, device=dev) if need_x else None
        dw = torch.empty((cin, cout, 4, 4), dtype=torch.float32, device=dev) if need_w else None
        ws = torch.empty(ctx.ws_bytes, dtype=torch.uint8, device=dev)
        L = _lib.lib()
        with torch.cuda.device(dev):
            _lib.check(L.cdr_deconv_train_backward(_lib.ptr(saved), _lib.ptr(weight), _lib.ptr(dy), n, cin, cout, h, w,
                                                   _lib.ptr(dx), _lib.ptr(dw), _lib.ptr(ws), ctx.ws_bytes,
                                                   _lib.current_stream_ptr(dev)))
        return dx, dw


def conv_transpose2d(x, weight):
    """F.conv_transpose2d(x, weight, stride=2, padding=1) for 4x4 kernels without bias, forward and backward on
    libcdrhead at fp32 accuracy.  x (N, Cin, H, W), weight (Cin, Cout, 4, 4): CUDA float32, Cin and Cout multiples
    of 64, H == W in {8, 16, 32}; anything else raises ValueError."""
    return _ConvTranspose2d.apply(x, weight)


def _aligned(t):
    """t contiguous with a 16-byte-aligned address (a contiguous view may start mid-allocation)."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _conv1x1_args(x, weight, bias):
    """Checks of conv1x1's inputs, all before any CUDA call: ValueError, there is no fallback."""
    ts = (x, weight) if bias is None else (x, weight, bias)
    if not all(isinstance(t, torch.Tensor) for t in ts):
        raise ValueError("conv1x1: x, weight and bias must be tensors")
    if x.dim() != 4 or weight.dim() != 4 or tuple(weight.shape[2:]) != (1, 1) or weight.shape[1] != x.shape[1]:
        raise ValueError(f"conv1x1: x (N, Cin, H, W) and weight (Cout, Cin, 1, 1) expected, got {tuple(x.shape)} and "
                         f"{tuple(weight.shape)}")
    n, cin, h, w = x.shape
    cout = weight.shape[0]
    if bias is not None and tuple(bias.shape) != (cout,):
        raise ValueError(f"conv1x1: bias of shape ({cout},) expected, got {tuple(bias.shape)}")
    if not (n >= 1 and 1 <= cin <= 4096 and 1 <= cout <= 4096 and (h * w) % 64 == 0 and h * w > 0
            and n * h * w <= 1 << 22):
        raise ValueError(f"conv1x1: unsupported shape x {tuple(x.shape)}, weight {tuple(weight.shape)} "
                         "(1 <= Cin, Cout <= 4096, H*W a multiple of 64, N*H*W <= 2^22)")
    if any(t.dtype != torch.float32 for t in ts):
        raise ValueError(f"conv1x1: float32 expected, got {', '.join(str(t.dtype) for t in ts)}")
    if not all(t.is_cuda and t.device == x.device for t in ts):
        raise ValueError("conv1x1: x, weight and bias must be CUDA tensors on one device (there is no CPU fallback)")
    return _aligned(x), _aligned(weight), None if bias is None else _aligned(bias)


class _Conv1x1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        x, weight, bias = _conv1x1_args(x, weight, bias)
        n, cin, h, w = x.shape
        cout = weight.shape[0]
        L = _lib.lib()
        saved_b, ws_b = C.c_size_t(), C.c_size_t()
        _lib.check(L.cdr_conv1x1_train_workspace_bytes(n, cin, cout, h, w, C.byref(saved_b), C.byref(ws_b)))
        dev = x.device
        y = torch.empty((n, cout, h, w), dtype=torch.float32, device=dev)
        saved = torch.empty(saved_b.value, dtype=torch.uint8, device=dev)     # x as fp16 planes, for the weight gradient
        ws = torch.empty(ws_b.value, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.cdr_conv1x1_train_forward(_lib.ptr(x), _lib.ptr(weight), _lib.ptr(bias), n, cin, cout, h, w,
                                                   _lib.ptr(y), _lib.ptr(saved), saved_b.value, _lib.ptr(ws), ws_b.value,
                                                   _lib.current_stream_ptr(dev)))
        ctx.save_for_backward(saved, weight)
        ctx.dims = (n, cin, cout, h, w)
        ctx.ws_bytes = ws_b.value
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y):
        saved, weight = ctx.saved_tensors
        n, cin, cout, h, w = ctx.dims
        need_x, need_w, need_b = ctx.needs_input_grad[:3]
        if not (need_x or need_w or need_b):
            return None, None, None
        dy = _aligned(_chk(grad_y, "conv1x1: grad"))
        dev = dy.device
        dx = torch.empty((n, cin, h, w), dtype=torch.float32, device=dev) if need_x else None
        dw = torch.empty((cout, cin, 1, 1), dtype=torch.float32, device=dev) if need_w else None
        db = torch.empty((cout,), dtype=torch.float32, device=dev) if need_b else None
        ws = torch.empty(ctx.ws_bytes, dtype=torch.uint8, device=dev)
        L = _lib.lib()
        with torch.cuda.device(dev):
            _lib.check(L.cdr_conv1x1_train_backward(_lib.ptr(saved), _lib.ptr(weight), _lib.ptr(dy), n, cin, cout, h, w,
                                                    _lib.ptr(dx), _lib.ptr(dw), _lib.ptr(db), _lib.ptr(ws), ctx.ws_bytes,
                                                    _lib.current_stream_ptr(dev)))
        return dx, dw, db


def conv1x1(x, weight, bias=None):
    """F.conv2d(x, weight, bias) for a (Cout, Cin, 1, 1) weight, forward and backward on libcdrhead at fp32 accuracy.
    x (N, Cin, H, W), bias (Cout) or None: CUDA float32, 1 <= Cin, Cout <= 4096, H*W a multiple of 64,
    N*H*W <= 2^22; anything else raises ValueError."""
    return _Conv1x1.apply(x, weight, bias)


def _conv3x3_args(x, weight, stride):
    """Checks of conv3x3's inputs, all before any CUDA call: ValueError, there is no fallback."""
    if not (isinstance(x, torch.Tensor) and isinstance(weight, torch.Tensor)):
        raise ValueError("conv3x3: x and weight must be tensors")
    if x.dim() != 4 or weight.dim() != 4 or tuple(weight.shape[2:]) != (3, 3) or weight.shape[1] != x.shape[1]:
        raise ValueError(f"conv3x3: x (N, Cin, H, W) and weight (Cout, Cin, 3, 3) expected, got {tuple(x.shape)} and "
                         f"{tuple(weight.shape)}")
    n, cin, h, w = x.shape
    cout = weight.shape[0]
    ok = type(stride) is int and stride in (1, 2) and n >= 1 and all(64 <= c <= 2048 and c % 64 == 0 for c in (cin, cout))
    ok = ok and h % stride == 0 and w % stride == 0
    ho, wo = (h // stride, w // stride) if ok else (0, 0)
    if not (ok and wo in (8, 16, 32, 64) and (ho * wo == 64 or (ho * wo) % 128 == 0) and n * ho * wo <= 1 << 22):
        raise ValueError(f"conv3x3: unsupported shape x {tuple(x.shape)}, weight {tuple(weight.shape)}, stride {stride!r} "
                         "(stride 1 or 2, Cin and Cout multiples of 64 in [64, 2048], H and W divisible by the stride; "
                         "output W a power of two in [8, 64], output H*W = 64 or a multiple of 128, N*H*W <= 2^22)")
    if x.dtype != torch.float32 or weight.dtype != torch.float32:
        raise ValueError(f"conv3x3: float32 expected, got {x.dtype} and {weight.dtype}")
    if not (x.is_cuda and weight.is_cuda) or x.device != weight.device:
        raise ValueError("conv3x3: x and weight must be CUDA tensors on one device (there is no CPU fallback)")
    return _aligned(x), _aligned(weight)


class _Conv3x3(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, stride):
        x, weight = _conv3x3_args(x, weight, stride)
        n, cin, h, w = x.shape
        cout = weight.shape[0]
        L = _lib.lib()
        saved_b, ws_b = C.c_size_t(), C.c_size_t()
        _lib.check(L.cdr_conv3x3_train_workspace_bytes(n, cin, cout, h, w, stride, C.byref(saved_b), C.byref(ws_b)))
        dev = x.device
        y = torch.empty((n, cout, h // stride, w // stride), dtype=torch.float32, device=dev)
        saved = torch.empty(saved_b.value, dtype=torch.uint8, device=dev)     # x as fp16 planes, for the weight gradient
        ws = torch.empty(ws_b.value, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.cdr_conv3x3_train_forward(_lib.ptr(x), _lib.ptr(weight), n, cin, cout, h, w, stride,
                                                   _lib.ptr(y), _lib.ptr(saved), saved_b.value, _lib.ptr(ws), ws_b.value,
                                                   _lib.current_stream_ptr(dev)))
        ctx.save_for_backward(saved, weight)
        ctx.dims = (n, cin, cout, h, w, stride)
        ctx.ws_bytes = ws_b.value
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y):
        saved, weight = ctx.saved_tensors
        n, cin, cout, h, w, stride = ctx.dims
        need_x, need_w = ctx.needs_input_grad[:2]
        if not (need_x or need_w):
            return None, None, None
        dy = _aligned(_chk(grad_y, "conv3x3: grad"))
        dev = dy.device
        dx = torch.empty((n, cin, h, w), dtype=torch.float32, device=dev) if need_x else None
        dw = torch.empty((cout, cin, 3, 3), dtype=torch.float32, device=dev) if need_w else None
        ws = torch.empty(ctx.ws_bytes, dtype=torch.uint8, device=dev)
        L = _lib.lib()
        with torch.cuda.device(dev):
            _lib.check(L.cdr_conv3x3_train_backward(_lib.ptr(saved), _lib.ptr(weight), _lib.ptr(dy), n, cin, cout, h, w,
                                                    stride, _lib.ptr(dx), _lib.ptr(dw), _lib.ptr(ws), ctx.ws_bytes,
                                                    _lib.current_stream_ptr(dev)))
        return dx, dw, None


def conv3x3(x, weight, stride=1):
    """F.conv2d(x, weight, stride=stride, padding=1) for a (Cout, Cin, 3, 3) weight without bias, forward and backward
    on libcdrhead at fp32 accuracy.  x (N, Cin, H, W): CUDA float32, stride 1 or 2, Cin and Cout multiples of 64 in
    [64, 2048], H and W divisible by the stride, the output's width a power of two in [8, 64], its H*W 64 or a multiple
    of 128 and N*H*W <= 2^22; anything else raises ValueError."""
    return _Conv3x3.apply(x, weight, stride)
