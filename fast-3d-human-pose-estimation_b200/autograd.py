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

and the encoder's stem: its 7x7 convolution (forward and weight gradient; its input, the image batch, gets no gradient)
and its max-pool (bit for bit torch's):

    y = stem_conv(x, weight)                          # == F.conv2d(x, weight, stride=2, padding=3), no bias
    p = max_pool3x3(y)                                # == F.max_pool2d(y, 3, stride=2, padding=1)
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import Callable

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


def _aligned(t):
    """t contiguous with a 16-byte-aligned address (a contiguous view may start mid-allocation)."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


@dataclasses.dataclass(frozen=True)
class _TrainConvOp:
    """One training convolution of libcdrhead: what the shared Function needs to know about it."""
    name: str            # the public function, for messages
    lib: str             # its C entry points cdr_<lib>_train_{workspace_bytes,forward,backward}
    k: int               # kernel size
    cin_dim: int         # the weight's Cin dimension: 0 for a transposed conv's (Cin, Cout, k, k), 1 for a conv's
    has_bias: bool
    out_hw: Callable     # (h, w, *extra int args) -> the output's (H, W)
    data_grad: bool = True   # False: the op has no input gradient, and x must not require one


_DECONV = _TrainConvOp("conv_transpose2d", "deconv", 4, 0, False, lambda h, w: (2 * h, 2 * w))
_CONV1X1 = _TrainConvOp("conv1x1", "conv1x1", 1, 1, True, lambda h, w: (h, w))
_CONV3X3 = _TrainConvOp("conv3x3", "conv3x3", 3, 1, False, lambda h, w, s: (h // s, w // s))
_STEM = _TrainConvOp("stem_conv", "stem", 7, 1, False, lambda h, w: (h // 2, w // 2), data_grad=False)


def _train_conv_args(op, x, weight, bias, extra):
    """Checks of a training conv's inputs, all before any CUDA call: ValueError, there is no fallback.  The shape's
    domain is the library's: cdr_<lib>_train_workspace_bytes decides it without a device, and its byte counts are the
    ones the forward uses.  -> x, weight, bias, the C shape arguments, saved bytes, workspace bytes."""
    ts = (x, weight) if bias is None else (x, weight, bias)
    if not all(isinstance(t, torch.Tensor) for t in ts):
        raise ValueError(f"{op.name}: x, weight and bias must be tensors")
    if not op.data_grad and x.requires_grad:
        raise ValueError(f"{op.name}: x requires grad, but the op has no input gradient (its input is the image batch)")
    if x.dim() != 4 or weight.dim() != 4 or tuple(weight.shape[2:]) != (op.k, op.k) or \
            weight.shape[op.cin_dim] != x.shape[1]:
        layout = "Cin, Cout" if op.cin_dim == 0 else "Cout, Cin"
        raise ValueError(f"{op.name}: x (N, Cin, H, W) and weight ({layout}, {op.k}, {op.k}) expected, got "
                         f"{tuple(x.shape)} and {tuple(weight.shape)}")
    n, cin, h, w = x.shape
    cout = weight.shape[1 - op.cin_dim]
    if bias is not None and tuple(bias.shape) != (cout,):
        raise ValueError(f"{op.name}: bias of shape ({cout},) expected, got {tuple(bias.shape)}")
    if not all(type(e) is int for e in extra):
        raise ValueError(f"{op.name}: an int stride expected, got {extra[0]!r}")
    L = _lib.lib()
    dims = (n, cin, cout, h, w, *extra)
    saved_b, ws_b = C.c_size_t(), C.c_size_t()
    if getattr(L, f"cdr_{op.lib}_train_workspace_bytes")(*dims, C.byref(saved_b), C.byref(ws_b)):
        raise ValueError(f"{op.name}: unsupported shape x {tuple(x.shape)}, weight {tuple(weight.shape)}"
                         f"{''.join(f', stride {e!r}' for e in extra)} ({L.cdr_last_error().decode(errors='replace')})")
    if any(t.dtype != torch.float32 for t in ts):
        raise ValueError(f"{op.name}: float32 expected, got {', '.join(str(t.dtype) for t in ts)}")
    if not all(t.is_cuda and t.device == x.device for t in ts):
        raise ValueError(f"{op.name}: x, weight and bias must be CUDA tensors on one device (there is no CPU fallback)")
    return (_aligned(x), _aligned(weight), None if bias is None else _aligned(bias), dims, saved_b.value,
            ws_b.value)


class _TrainConv(torch.autograd.Function):
    """conv_transpose2d, conv1x1, conv3x3 and stem_conv: forward and backward through the op's cdr_<lib>_train_* entry
    points.
    extra: the int arguments that follow (n, cin, cout, h, w) in them (conv3x3's stride)."""

    @staticmethod
    def forward(ctx, op, x, weight, bias, *extra):
        x, weight, bias, dims, saved_b, ws_b = _train_conv_args(op, x, weight, bias, extra)
        n, _, cout, h, w = dims[:5]
        L = _lib.lib()
        dev = x.device
        y = torch.empty((n, cout, *op.out_hw(h, w, *extra)), dtype=torch.float32, device=dev)
        saved = torch.empty(saved_b, dtype=torch.uint8, device=dev)     # x as fp16 planes, for the weight gradient
        ws = torch.empty(ws_b, dtype=torch.uint8, device=dev)
        b = (_lib.ptr(bias),) if op.has_bias else ()
        with torch.cuda.device(dev):
            _lib.check(getattr(L, f"cdr_{op.lib}_train_forward")(_lib.ptr(x), _lib.ptr(weight), *b, *dims, _lib.ptr(y),
                                                                  _lib.ptr(saved), saved_b, _lib.ptr(ws), ws_b,
                                                                  _lib.current_stream_ptr(dev)))
        ctx.save_for_backward(saved, weight)
        ctx.op, ctx.dims, ctx.ws_bytes = op, dims, ws_b
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y):
        saved, weight = ctx.saved_tensors
        op, dims = ctx.op, ctx.dims
        n, cin, cout, h, w = dims[:5]
        need_x, need_w, need_b = ctx.needs_input_grad[1:4]
        no_extra = (None,) * (len(dims) - 5)
        if not (need_x or need_w or need_b):
            return (None, None, None, None, *no_extra)
        dy = _aligned(_chk(grad_y, f"{op.name}: grad"))
        dev = dy.device
        dx = torch.empty((n, cin, h, w), dtype=torch.float32, device=dev) if need_x else None
        dw = torch.empty(weight.shape, dtype=torch.float32, device=dev) if need_w else None
        db = torch.empty((cout,), dtype=torch.float32, device=dev) if need_b else None
        ws = torch.empty(ctx.ws_bytes, dtype=torch.uint8, device=dev)
        b = (_lib.ptr(db),) if op.has_bias else ()
        L = _lib.lib()
        with torch.cuda.device(dev):
            _lib.check(getattr(L, f"cdr_{op.lib}_train_backward")(_lib.ptr(saved), _lib.ptr(weight), _lib.ptr(dy), *dims,
                                                                   _lib.ptr(dx), _lib.ptr(dw), *b, _lib.ptr(ws),
                                                                   ctx.ws_bytes, _lib.current_stream_ptr(dev)))
        return (None, dx, dw, db, *no_extra)


def conv_transpose2d(x, weight):
    """F.conv_transpose2d(x, weight, stride=2, padding=1) for 4x4 kernels without bias, forward and backward on
    libcdrhead at fp32 accuracy.  x (N, Cin, H, W), weight (Cin, Cout, 4, 4): CUDA float32, Cin and Cout multiples
    of 64, H == W in {8, 16, 32}; anything else raises ValueError."""
    return _TrainConv.apply(_DECONV, x, weight, None)


def conv1x1(x, weight, bias=None):
    """F.conv2d(x, weight, bias) for a (Cout, Cin, 1, 1) weight, forward and backward on libcdrhead at fp32 accuracy.
    x (N, Cin, H, W), bias (Cout) or None: CUDA float32, 1 <= Cin, Cout <= 4096, H*W a multiple of 64,
    N*H*W <= 2^22; anything else raises ValueError."""
    return _TrainConv.apply(_CONV1X1, x, weight, bias)


def conv3x3(x, weight, stride=1):
    """F.conv2d(x, weight, stride=stride, padding=1) for a (Cout, Cin, 3, 3) weight without bias, forward and backward
    on libcdrhead at fp32 accuracy.  x (N, Cin, H, W): CUDA float32, stride 1 or 2, Cin and Cout multiples of 64 in
    [64, 2048], H and W divisible by the stride, the output's width a power of two in [8, 64], its H*W 64 or a multiple
    of 128 and N*H*W <= 2^22; anything else raises ValueError."""
    return _TrainConv.apply(_CONV3X3, x, weight, None, stride)


def stem_conv(x, weight):
    """F.conv2d(x, weight, stride=2, padding=3) for the ResNet stem's (64, 3, 7, 7) weight without bias, forward and
    weight gradient on libcdrhead at fp32 accuracy.  There is no input gradient: x is the image batch, and an x that
    requires grad raises ValueError.  x (N, 3, H, W): CUDA float32, H % 16 == 0, W % 64 == 0, N*(H/2)*(W/2) <= 2^22;
    anything else raises ValueError."""
    return _TrainConv.apply(_STEM, x, weight, None)


class _MaxPool3x3(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        if not isinstance(x, torch.Tensor) or x.dim() != 4:
            raise ValueError("max_pool3x3: x (N, C, H, W) expected")
        n, c, h, w = x.shape
        if min(n, c, h, w) < 1 or n * c * h * w >= 1 << 31:
            raise ValueError(f"max_pool3x3: unsupported shape {tuple(x.shape)} (every size >= 1, N*C*H*W < 2^31)")
        if x.dtype != torch.float32:
            raise ValueError(f"max_pool3x3: float32 expected, got {x.dtype}")
        if not x.is_cuda:
            raise ValueError("max_pool3x3: a CUDA tensor expected (there is no CPU fallback)")
        x = x.contiguous()
        ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
        y = torch.empty((n, c, ho, wo), dtype=torch.float32, device=x.device)
        argmax = torch.empty((n, c, ho, wo), dtype=torch.uint8, device=x.device)    # window position ky * 3 + kx
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().cdr_maxpool3x3_train_forward(_lib.ptr(x), n, c, h, w, _lib.ptr(y), _lib.ptr(argmax),
                                                               _lib.current_stream_ptr(x.device)))
        ctx.save_for_backward(argmax)
        ctx.in_shape = (n, c, h, w)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_y):
        (argmax,) = ctx.saved_tensors
        n, c, h, w = ctx.in_shape
        dy = _chk(grad_y, "max_pool3x3: grad")
        dx = torch.empty((n, c, h, w), dtype=torch.float32, device=dy.device)
        with torch.cuda.device(dy.device):
            _lib.check(_lib.lib().cdr_maxpool3x3_train_backward(_lib.ptr(argmax), _lib.ptr(dy), n, c, h, w, _lib.ptr(dx),
                                                                _lib.current_stream_ptr(dy.device)))
        return dx


def max_pool3x3(x):
    """F.max_pool2d(x, 3, stride=2, padding=1) on NCHW float32 CUDA tensors, forward and backward on libcdrhead, equal
    to torch's CUDA kernels bit for bit (ties go to the first maximum in row-major order, a NaN wins).  Keeps one byte
    per output for the backward instead of torch's int64 index.  Any N, C, H, W >= 1 with N*C*H*W < 2^31; anything else
    raises ValueError."""
    return _MaxPool3x3.apply(x)
