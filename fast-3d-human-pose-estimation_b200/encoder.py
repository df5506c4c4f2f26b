"""ResNet backbone — stays on torch/cuDNN (BASELINE.json north_star).

Not part of the hand-written hot path; it only produces the (B,2048,8,8)
latent the head consumes.  The module tree reproduces the reference's
``state_dict`` key names (``conv1``, ``bn1``, ``layer{1..4}.<i>.{conv1,bn1,
conv2,bn2,conv3,bn3,downsample.0,downsample.1}``; reference
models/encoder.py:79-131) so ``best.pth`` / ``latest.pth`` checkpoints load,
and creates parameters in the same order so a seeded random init matches.
"""
import ctypes as C

import torch
import torch.nn.functional as F
from torch import nn

# bound once, at import: the encoder's training forward does not follow a later rebinding of ``autograd.conv1x1`` (the
# head's training-step tests swap that name for cuDNN's to compare the head's 1x1 convs alone)
from .autograd import conv1x1 as _conv1x1, conv3x3 as _conv3x3, max_pool3x3 as _max_pool3x3, stem_conv as _stem_conv

_SPEC = {18: ("basic", (2, 2, 2, 2)), 34: ("basic", (3, 4, 6, 3)),
         50: ("bottleneck", (3, 4, 6, 3)), 101: ("bottleneck", (3, 4, 23, 3)),
         152: ("bottleneck", (3, 8, 36, 3))}


def _bn(c):
    return nn.BatchNorm2d(c, momentum=0.1)


class _Block(nn.Module):
    """Residual block.  ``kind='bottleneck'``: 1x1 -> 3x3(stride) -> 1x1(x4)
    (reference models/encoder.py:38-76).  ``kind='basic'``: two 3x3 convs that
    BOTH carry the stride, as the reference does (models/encoder.py:6-35)."""

    def __init__(self, kind, cin, planes, stride, downsample):
        super().__init__()
        if kind == "bottleneck":
            self.conv1 = nn.Conv2d(cin, planes, 1, bias=False)
            self.bn1 = _bn(planes)
            self.conv2 = nn.Conv2d(planes, planes, 3, stride, 1, bias=False)
            self.bn2 = _bn(planes)
            self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
            self.bn3 = _bn(planes * 4)
        else:
            self.conv1 = nn.Conv2d(cin, planes, 3, stride, 1, bias=False)
            self.bn1 = _bn(planes)
            self.conv2 = nn.Conv2d(planes, planes, 3, stride, 1, bias=False)
            self.bn2 = _bn(planes)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.kind = kind

    def forward(self, x):
        y = self.relu(self.bn1(self.conv1(x)))
        if self.kind == "bottleneck":
            y = self.relu(self.bn2(self.conv2(y)))
            y = self.bn3(self.conv3(y))
        else:
            y = self.bn2(self.conv2(y))
        r = x if self.downsample is None else self.downsample(x)
        return self.relu(y + r)


class ResNet(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        kind, counts = _SPEC[cfg.MODEL.NUM_LAYERS]
        exp = 4 if kind == "bottleneck" else 1
        self.conv1 = nn.Conv2d(3, 64, 7, 2, 3, bias=False)
        self.bn1 = _bn(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(3, 2, 1)
        cin = 64
        for li, (planes, n, stride) in enumerate(
                zip((64, 128, 256, 512), counts, (1, 2, 2, 2)), start=1):
            blocks = []
            for bi in range(n):
                s = stride if bi == 0 else 1
                ds = None
                if bi == 0 and (s != 1 or cin != planes * exp):
                    ds = nn.Sequential(nn.Conv2d(cin, planes * exp, 1, s, bias=False),
                                       _bn(planes * exp))
                blocks.append(_Block(kind, cin, planes, s, ds))
                cin = planes * exp
            setattr(self, f"layer{li}", nn.Sequential(*blocks))
        self.out_channels = cin
        self.kind = kind

    def forward(self, x):
        x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        return self.layer4(self.layer3(self.layer2(self.layer1(x))))

    def forward_train(self, x, stem_on_library=False):
        """``forward`` in training mode with every Bottleneck block on libcdrhead, forward and backward at fp32 accuracy
        whatever torch's TF32 flags say: conv1 / conv3 and the downsample conv (on the stride-2 slice, an exact identity
        for a 1x1 conv) through ``conv1x1``, conv2 through ``conv3x3``, every BatchNorm through ``batch_norm_train``
        (batch statistics and the running-stat update, as nn.BatchNorm2d in training mode).  The stem (7x7 conv over 3
        channels, BatchNorm, ReLU, max-pool) stays on torch unless ``stem_on_library=True``: then its conv runs through
        ``stem_conv`` (fp32 accuracy, forward and weight gradient; x, the image batch, gets no gradient), its BatchNorm
        + ReLU through ``batch_norm_train`` and its max-pool through ``max_pool3x3`` (torch's bits).  The library's shape
        limits apply: at N images per call, 256 x 256 inputs are inside them for every N up to 64.
        ``CDRNet(..., train_encoder_on_library=True)`` calls it for each view from ``forward_train``."""
        if self.kind != "bottleneck":
            raise ValueError("ResNet.forward_train: only Bottleneck encoders (ResNet-50/101/152) train on the library")
        from .losses import batch_norm_train
        if stem_on_library:
            x = _max_pool3x3(batch_norm_train(_stem_conv(x, self.conv1.weight), self.bn1, relu=True))
        else:
            x = self.maxpool(self.relu(self.bn1(self.conv1(x))))
        for layer in (self.layer1, self.layer2, self.layer3, self.layer4):
            for b in layer:
                x = _bottleneck_train(b, x)
        return x


def _bottleneck_train(b, x):
    """one Bottleneck block of ResNet.forward_train: relu(bn3(conv3(relu(bn2(conv2(relu(bn1(conv1(x)))))))) + r)"""
    from .losses import batch_norm_train
    y = batch_norm_train(_conv1x1(x, b.conv1.weight), b.bn1, relu=True)
    y = batch_norm_train(_conv3x3(y, b.conv2.weight, b.conv2.stride[0]), b.bn2, relu=True)
    y = batch_norm_train(_conv1x1(y, b.conv3.weight), b.bn3)
    r = x
    if b.downsample is not None:
        conv, bn = b.downsample[0], b.downsample[1]
        s = conv.stride[0]
        r = batch_norm_train(_conv1x1(x if s == 1 else x[:, :, ::s, ::s], conv.weight), bn)
    return F.relu(y + r)


IMAGENET_MEAN = (0.485, 0.456, 0.406)      # inference.py:42-43
IMAGENET_STD = (0.229, 0.224, 0.225)


class TcEncoder:
    """A Bottleneck ``ResNet`` on libcdrhead (SURVEY §8f rank 1; include/cdrhead.h ``cdr_encoder_*``):
    layer1..layer4 on the tcgen05 tap-GEMM kernel, the 7x7 stem + max-pool on a warp-MMA kernel
    (``cdr_encoder_forward_images``; in bf16 mode images with H % 16 or W % 64 != 0 fall back to a cuDNN bf16
    stem whose channels-last output is the same NHWC layout).  Eval-mode BN folded, fp32 accumulation.
    ``precision='bf16'``: bf16 activations; ``precision='fp32'``: the reference's precision — scaled fp16 hi/lo planes,
    3 MMAs per product, residual add on planes, three-term fp16 stem (1.5e-6 of max from the fp64 network).  Inference only;
    weights are re-packed when a parameter changes.  ``rows(x)`` returns the latents as bf16
    pixel-major rows (n*h*w, 2048) — what ``cdr_head_forward_rows`` consumes — or, in fp32 mode, the opaque
    "fp16 planes" uint8 buffer ``cdr_head_forward_planes`` consumes; ``__call__`` returns
    the reference's (n, 2048, h, w) fp32 tensor."""

    def __init__(self, resnet, precision="bf16"):
        blocks = [b for li in range(1, 5) for b in getattr(resnet, f"layer{li}")]
        if any(b.kind != "bottleneck" for b in blocks):
            # (the reference's BasicBlock puts the stride on BOTH 3x3 convs, models/encoder.py:9-14, so its ResNet-18/34
            # fail with a shape mismatch at layer2's residual add: there is nothing to accelerate)
            raise NotImplementedError("the tcgen05 encoder covers the Bottleneck ResNets (50/101/152)")
        if precision not in ("bf16", "fp32"):
            raise ValueError(f"TcEncoder precision must be 'bf16' or 'fp32', got {precision!r}")
        # 'fp32': the reference's precision on the tensor cores — scaled fp16 hi/lo planes, 3 MMAs per product, fp32
        # three-term fp16 stem (include/cdrhead.h: cdr_encoder_create_prec).  rows() then returns the opaque "fp16 planes" buffer
        self.precision = precision
        self.resnet, self.blocks = resnet, blocks
        self._box, self._key, self._stem = None, None, None
        self.torch_stem = False          # True: force the cuDNN stem (A/B timing)

    @property
    def _handle(self):
        return self._box.handle if self._box is not None else None

    def retain(self):
        """(box, key) of the packed encoder for a captured graph (workspace.HandleBox)."""
        if self._box is None:
            raise RuntimeError("nothing packed yet: run one forward before capturing")
        return self._box.retain(), self._key

    def key_now(self, device):
        return (str(device),) + tuple((t.data_ptr(), t._version) for t in self._tensors())

    def __deepcopy__(self, memo):
        import copy
        return TcEncoder(copy.deepcopy(self.resnet, memo), self.precision)     # device handles are never shared or copied

    def __getstate__(self):
        return {"resnet": self.resnet, "blocks": self.blocks, "_box": None, "_key": None, "_stem": None,
                "torch_stem": self.torch_stem, "precision": self.precision}

    def _tensors(self):
        r = self.resnet
        ts = [r.conv1.weight, r.bn1.weight, r.bn1.bias, r.bn1.running_mean, r.bn1.running_var]
        for b in self.blocks:
            mods = [(b.conv1, b.bn1), (b.conv2, b.bn2), (b.conv3, b.bn3)]
            if b.downsample is not None:
                mods.append((b.downsample[0], b.downsample[1]))
            for c, n in mods:
                ts += [c.weight, n.weight, n.bias, n.running_mean, n.running_var]
        return ts

    def _pack(self, device):
        from . import _lib, workspace as _wsmod
        key = self.key_now(device)
        if key == self._key:
            return self._box.handle
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("encoder parameters changed (or were never packed) during a CUDA-graph capture")
        r = self.resnet
        for bn in [r.bn1] + [m for b in self.blocks for m in b.modules() if isinstance(m, nn.BatchNorm2d)]:
            if abs(bn.eps - 1e-5) > 1e-12:
                raise ValueError(f"BatchNorm eps={bn.eps}: the packing kernels fold the default 1e-5")
        self.release()
        L = _lib.lib()
        keep = []

        def cb(conv, bn):
            v = _lib.CdrConvBn()
            for name, t in (("weight", conv.weight), ("bn_weight", bn.weight), ("bn_bias", bn.bias),
                            ("bn_mean", bn.running_mean), ("bn_var", bn.running_var)):
                t = t.detach().to(device=device, dtype=torch.float32).contiguous()
                keep.append(t)
                setattr(v, name, t.data_ptr())
            return v
        arr = (_lib.CdrEncoderBlock * len(self.blocks))()
        for i, b in enumerate(self.blocks):
            arr[i].conv1, arr[i].conv2, arr[i].conv3 = cb(b.conv1, b.bn1), cb(b.conv2, b.bn2), cb(b.conv3, b.bn3)
            if b.downsample is not None:
                arr[i].downsample = cb(b.downsample[0], b.downsample[1])
            arr[i].planes, arr[i].stride = b.conv2.out_channels, b.conv2.stride[0]
        spec = _lib.CdrEncoderSpec(len(self.blocks), arr, self.resnet.conv1.out_channels,
                                   cb(self.resnet.conv1, self.resnet.bn1))
        handle = C.c_void_p()
        with torch.cuda.device(device):
            prec = _lib.CDR_PREC_F16X2 if self.precision == "fp32" else _lib.CDR_PREC_BF16
            _lib.check(L.cdr_encoder_create_prec(C.byref(spec), prec, _lib.current_stream_ptr(device), C.byref(handle)))
        # stem: BN folded into the conv, bf16 channels-last
        r = self.resnet
        sc = (r.bn1.weight.double() / torch.sqrt(r.bn1.running_var.double() + r.bn1.eps))
        w = (r.conv1.weight.double() * sc.reshape(-1, 1, 1, 1)).to(device=device, dtype=torch.bfloat16)
        bias = (r.bn1.bias.double() - r.bn1.running_mean.double() * sc).to(device=device, dtype=torch.bfloat16)
        self._stem = (w.contiguous(memory_format=torch.channels_last), bias)
        self._box, self._key = _wsmod.HandleBox(handle, lambda h: _lib.lib().cdr_encoder_destroy(h)), key
        return handle

    def release(self):
        if self._box is not None:
            self._box.release()          # destroyed now unless a captured graph still holds it
        self._box, self._key = None, None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def stem(self, x):
        """(n,3,S,S) -> (n, S/4, S/4, 64) bf16 NHWC (conv 7x7 s2 + BN + ReLU + max-pool 3x3 s2)."""
        w, b = self._stem
        r = self.resnet
        y = F.conv2d(x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last), w, b,
                     stride=r.conv1.stride, padding=r.conv1.padding)
        y = F.max_pool2d(F.relu_(y), 3, 2, 1)
        return y.permute(0, 2, 3, 1)          # a view: channels-last storage is NHWC

    def rows(self, x, out=None, mean=IMAGENET_MEAN, std=IMAGENET_STD):
        """x: (n,3,S,S) float CUDA images as the reference feeds its model, or raw (n,S,S,3) uint8 CUDA
        frames, normalised on the fly with torchvision's ToTensor + Normalize(mean, std)
        (inference.py:40-44).  -> (rows (n*h*w, C) bf16, (h, w, C))."""
        from . import _lib, workspace as _wsmod
        if not x.is_cuda:
            raise RuntimeError("the tcgen05 encoder has no CPU path")
        if self.resnet.training:
            raise RuntimeError("the tcgen05 encoder is inference-only; call .eval() first")
        dev = x.device
        handle = self._pack(dev)
        L = _lib.lib()
        u8 = x.dtype == torch.uint8
        if u8:
            n, H, W, c = x.shape
            if c != 3:
                raise ValueError(f"uint8 frames must be (n,H,W,3), got {tuple(x.shape)}")
            if H % 16 or W % 64:
                raise ValueError("uint8 frames need H % 16 == 0 and W % 64 == 0")
        else:
            n, _, H, W = x.shape
        native_stem = H % 16 == 0 and W % 64 == 0 and (u8 or not self.torch_stem)
        planes = self.precision == "fp32"
        if planes and not native_stem:
            raise ValueError("the fp32 tcgen05 encoder needs images with H % 16 == 0 and W % 64 == 0")
        if native_stem:
            xin = x.detach().contiguous() if u8 else x.detach().to(torch.float32).contiguous()
            h, w = H // 4, W // 4
        else:
            with torch.no_grad():
                xin = self.stem(x)
            if not xin.is_contiguous():
                xin = xin.contiguous()
            _, h, w, _ = xin.shape
        oh, ow, oc = C.c_int(), C.c_int(), C.c_int()
        _lib.check(L.cdr_encoder_out_shape(handle, h, w, C.byref(oh), C.byref(ow), C.byref(oc)))
        nbytes = C.c_size_t()
        if native_stem:
            _lib.check(L.cdr_encoder_workspace_bytes_images(handle, n, H, W, C.byref(nbytes)))
        else:
            _lib.check(L.cdr_encoder_workspace_bytes(handle, n, h, w, C.byref(nbytes)))
        ws = _wsmod.current(dev).get("encoder", dev, nbytes.value)     # per stream, or the enclosing pipeline's own
        if planes:
            obytes = C.c_size_t()
            _lib.check(L.cdr_encoder_out_bytes(handle, n, h, w, C.byref(obytes)))
            if out is None:
                out = torch.empty(obytes.value, dtype=torch.uint8, device=dev)
            elif out.dtype != torch.uint8 or out.numel() < obytes.value:
                raise ValueError(f"out must be a uint8 CUDA buffer of {obytes.value} bytes")
        elif out is None:
            out = torch.empty((n * oh.value * ow.value, oc.value), dtype=torch.bfloat16, device=dev)
        st = _lib.current_stream_ptr(dev)
        with torch.cuda.device(dev):
            if u8:
                m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
                _lib.check(L.cdr_encoder_forward_frames_u8(handle, _lib.ptr(xin), m3, s3, n, H, W, _lib.ptr(out),
                                                           _lib.ptr(ws), nbytes.value, st))
            elif native_stem:
                _lib.check(L.cdr_encoder_forward_images(handle, _lib.ptr(xin), n, H, W, _lib.ptr(out), _lib.ptr(ws),
                                                        nbytes.value, st))
            else:
                _lib.check(L.cdr_encoder_forward(handle, _lib.ptr(xin), n, h, w, _lib.ptr(out), _lib.ptr(ws),
                                                 nbytes.value, st))
        return out, (oh.value, ow.value, oc.value)

    @staticmethod
    def planes_to_rows(buf, rows, channels):
        """Decode an "fp16 planes" buffer (include/cdrhead.h) into an fp32 (rows, channels) tensor — a format
        conversion for tests and ``__call__``; the head consumes the buffer as it is."""
        stride = -(-rows * channels * 2 // 1024) * 1024
        hi = buf[:rows * channels * 2].view(torch.float16).reshape(rows, channels)
        lo = buf[stride:stride + rows * channels * 2].view(torch.float16).reshape(rows, channels)
        scale = buf[2 * stride + 4:2 * stride + 8].view(torch.float32)
        return (hi.double() + lo.double() / 2048.0) / scale.double()

    def __call__(self, x):
        rows, (h, w, c) = self.rows(x)
        n = x.shape[0]
        if self.precision == "fp32":
            rows = self.planes_to_rows(rows, n * h * w, c)
        return rows.reshape(n, h, w, c).permute(0, 3, 1, 2).float()
