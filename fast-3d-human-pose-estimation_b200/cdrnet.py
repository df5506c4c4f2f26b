"""Drop-in ``CDRNet`` / ``PoseResNet`` / ``PoseDecoder`` whose head runs in libcdrhead.so.

Mirrors the reference's module interface (models/cdrnet.py:88-268,
models/poseresnet.py:10-21, models/decoder.py:7-46):

* same constructor arguments, same ``state_dict`` key names and parameter
  creation order (so ``load_state_dict(torch.load('best.pth'))`` and a seeded
  random init both match the reference);
* ``forward(xs, proj_list) -> (pred_2ds, pred_3ds)`` with the same shapes,
  dtypes and device.

What differs is *where the arithmetic runs*: the ResNet encoder stays an
``nn.Module`` on torch/cuDNN; everything after it (pinv, canonical fusion with
the feature-transform layer, deconvolution decoder, soft-argmax, DLT) is one call
into the C ABI (``cdr_head_forward``, include/cdrhead.h) on the current CUDA
stream.  The ``nn.Conv2d`` / ``nn.BatchNorm2d`` children of ``CF`` and
``decoder`` are parameter containers only: they are BN-folded and re-laid-out
into a device-side handle the first time ``forward`` runs and whenever a
parameter changes (``load_state_dict``, ``.to()``, in-place edits).

Inference only: the reference's training step (autograd through the head,
train-mode BN) is out of scope for this build — calling ``forward`` in
training mode raises.  There is no CPU / PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import functools
import os

import torch
from torch import nn

from . import _lib
from . import workspace as _wsmod
from .encoder import ResNet, TcEncoder

PINV_RTOL_FP32 = 4 * float(torch.finfo(torch.float32).eps)  # torch.linalg.pinv default, (3,4) fp32


def _conv_bn_relu(cin, cout):
    return nn.Sequential(nn.Conv2d(cin, cout, kernel_size=1, stride=1),
                         nn.BatchNorm2d(cout), nn.ReLU(inplace=True))


class CanonicalFusion(nn.Module):
    """Parameter container for reference models/cdrnet.py:10-43."""

    def __init__(self, in_dim=2048, hid_ch1=300, hid_ch2=300, n_views=2):
        super().__init__()
        self.conv_layer1 = _conv_bn_relu(in_dim, hid_ch1)
        self.conv_layer2 = nn.Sequential(
            nn.Conv2d(n_views * hid_ch2, hid_ch2, kernel_size=1, stride=1),
            nn.BatchNorm2d(hid_ch2), nn.ReLU(inplace=True),
            nn.Conv2d(hid_ch2, hid_ch2, kernel_size=1, stride=1),
            nn.BatchNorm2d(hid_ch2), nn.ReLU(inplace=True))
        self.out_layer = nn.ModuleList([_conv_bn_relu(hid_ch1, in_dim) for _ in range(n_views)])

    def forward(self, *a, **k):
        raise RuntimeError("CanonicalFusion is a parameter container; call CDRNet.forward")


class PoseDecoder(nn.Module):
    """models/decoder.py:7-46.  ``forward`` runs ``cdr_decoder_forward``."""

    def __init__(self, cfg, precision="fp32"):
        super().__init__()
        self.deconv1 = self._deconv(2048, 256)
        self.deconv2 = self._deconv(256, 256)
        self.deconv3 = self._deconv(256, 256)
        self.final_layer = nn.Conv2d(256, cfg.MODEL.NUM_JOINTS, kernel_size=1, stride=1, padding=0)
        self.num_joints = cfg.MODEL.NUM_JOINTS
        self._packed = _PackedWeights(self, precision, has_fusion=False)

    @staticmethod
    def _deconv(cin, cout):
        return nn.Sequential(
            nn.ConvTranspose2d(cin, cout, kernel_size=4, stride=2, padding=1, output_padding=0,
                               bias=False),
            nn.BatchNorm2d(cout, momentum=0.1), nn.ReLU(inplace=True))

    def init_weights(self):
        """models/decoder.py:48-73."""
        for seq in (self.deconv1, self.deconv2, self.deconv3):
            nn.init.normal_(seq[0].weight, std=0.001)
            nn.init.constant_(seq[1].weight, 1)
            nn.init.constant_(seq[1].bias, 0)
        nn.init.normal_(self.final_layer.weight, std=0.001)
        nn.init.constant_(self.final_layer.bias, 0)

    def forward(self, x):
        _require_eval(self)
        x = _as_f32_cuda(x, "PoseDecoder input")
        n = x.shape[0]
        if tuple(x.shape[1:]) != (2048, 8, 8):
            raise ValueError(f"PoseDecoder expects (N,2048,8,8) features, got {tuple(x.shape)}")
        handle = self._packed.get(_decoder_tensors(self, ""), x.device)
        L = _lib.lib()
        nbytes = C.c_size_t()
        _lib.check(L.cdr_decoder_workspace_bytes(handle, n, C.byref(nbytes)))
        ws = _workspace(x.device, nbytes.value)
        out = torch.empty((n, self.num_joints, 64, 64), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):        # launches go to the CURRENT device: make it the tensors' device
            _lib.check(L.cdr_decoder_forward(handle, _lib.ptr(x), n, _lib.ptr(out), _lib.ptr(ws),
                                             nbytes.value, _lib.current_stream_ptr(x.device)))
        return out

    def forward_rows(self, rows, n_images=None):
        """The same on latents given as bf16 pixel-major rows (n*64, 2048) — the tcgen05 encoder's output — or
        (uint8 buffer + n_images) as the fp32 tcgen05 encoder's "fp16 planes" buffer (include/cdrhead.h)."""
        _require_eval(self)
        planes = rows.dtype == torch.uint8
        if planes:
            if not (rows.is_cuda and rows.is_contiguous() and n_images):
                raise ValueError("forward_rows on an fp16-planes buffer needs a contiguous CUDA uint8 tensor and n_images")
        elif not (rows.is_cuda and rows.dtype == torch.bfloat16 and rows.is_contiguous() and rows.dim() == 2
                  and rows.shape[1] == 2048 and rows.shape[0] % 64 == 0):
            raise ValueError("forward_rows expects a contiguous CUDA bf16 tensor of shape (n*64, 2048)")
        n = int(n_images) if planes else rows.shape[0] // 64
        handle = self._packed.get(_decoder_tensors(self, ""), rows.device)
        L = _lib.lib()
        nbytes = C.c_size_t()
        _lib.check(L.cdr_decoder_workspace_bytes(handle, n, C.byref(nbytes)))
        ws = _workspace(rows.device, nbytes.value)
        out = torch.empty((n, self.num_joints, 64, 64), dtype=torch.float32, device=rows.device)
        with torch.cuda.device(rows.device):
            fn = L.cdr_decoder_forward_planes if planes else L.cdr_decoder_forward_rows
            _lib.check(fn(handle, _lib.ptr(rows), n, _lib.ptr(out), _lib.ptr(ws), nbytes.value,
                          _lib.current_stream_ptr(rows.device)))
        return out


def _default_encoder_precision(value):
    """``encoder_precision=None`` (the default of CDRNet / PoseResNet): the environment variable
    ``CDR_ENCODER_PRECISION`` ('fp32' | 'bf16' | 'torch') or 'torch'.  It lets the reference's unmodified drivers, which
    construct ``CDRNet(config)`` with no extra arguments (inference.py:28, baseline.py:27), run the ENCODER on this
    library too — ``CDR_ENCODER_PRECISION=fp32 python inference.py`` — without touching their source."""
    if value is not None:
        return value
    return os.environ.get("CDR_ENCODER_PRECISION", "torch")


def _require_eval(m):
    if m.training:
        raise RuntimeError(
            f"{type(m).__name__}: the B200 head is inference-only (eval-mode BN folded into the "
            "convs, no autograd); call .eval() first")


def _as_f32_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what} must be a CUDA tensor: the CDRNet head has no CPU path")
    return t.detach().to(torch.float32).contiguous()


def _workspace(device, nbytes, slot="head"):
    """Scratch for one forward (torch-owned; the library never allocates caller-visible memory): the buffer of
    the current (device, stream), or of the enclosing graph/pipeline (workspace.py)."""
    return _wsmod.current(device).get(slot, device, nbytes)


def _convbn(conv, bn):
    s = _lib.CdrConvBn()
    s.weight = conv.weight.data_ptr()
    s.bias = conv.bias.data_ptr() if conv.bias is not None else None
    if bn is not None:
        s.bn_weight = bn.weight.data_ptr()
        s.bn_bias = bn.bias.data_ptr()
        s.bn_mean = bn.running_mean.data_ptr()
        s.bn_var = bn.running_var.data_ptr()
    return s


def _decoder_tensors(dec, _prefix):
    return [dec.deconv1, dec.deconv2, dec.deconv3, dec.final_layer]


class _PackedWeights:
    """Owns the CdrWeights handle of one module and re-packs it when parameters change.

    The handle lives in a reference-counted ``HandleBox``: captured CUDA graphs ``retain()`` it, so a re-pack
    (load_state_dict, optimizer step, ``.to()``) after a capture cannot free the pool the graph's kernels read —
    the graph holder notices the changed signature at its next replay and refuses to run on stale weights."""

    BN_EPS = 1e-5            # folded by the packing kernels (csrc/pack.cu, gemm_tc.cu)

    def __init__(self, owner, precision, has_fusion):
        if precision not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}, got {precision!r}")
        self.precision = precision
        self.has_fusion = has_fusion
        self._box = None
        self._sig = None
        self._last = None          # (modules, device, cf) of the last get(): lets signature_now() recompute

    @property
    def _handle(self):
        return self._box.handle if self._box is not None else None

    def _collect(self, dec, device, cf):
        params = []
        mods = ([cf.conv_layer1, cf.conv_layer2, cf.out_layer[0], cf.out_layer[1]] if cf is not None
                else []) + list(dec)
        for m in mods:
            params += list(m.parameters()) + list(m.buffers())
        return mods, params

    def _signature(self, tensors, device):
        return (str(device), self.precision) + tuple((t.data_ptr(), t._version) for t in tensors)

    def signature_now(self):
        """Signature of the parameters as they are now (None before the first get())."""
        if self._last is None:
            return None
        dec, device, cf = self._last
        return self._signature(self._collect(dec, device, cf)[1], device)

    def retain(self):
        """(box, signature) of the current handle for a graph holder; the box must be release()d."""
        if self._box is None:
            raise RuntimeError("nothing packed yet: run one forward before capturing")
        return self._box.retain(), self._sig

    def get(self, modules, device, cf=None):
        dec = modules
        mods, params = self._collect(dec, device, cf)
        for t in params:
            if t.is_floating_point() and (t.dtype != torch.float32 or t.device != device):
                raise RuntimeError("head parameters must be float32 on the input's device "
                                   f"(found {t.dtype} on {t.device}, input on {device})")
        sig = self._signature(params, device)
        self._last = (dec, device, cf)
        if self._box is not None and sig == self._sig:
            return self._box.handle
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("head parameters changed (or were never packed) while a CUDA graph is being captured: "
                               "packing allocates and synchronises; run one eager forward first")
        for m in mods:
            for sub in m.modules():
                if isinstance(sub, nn.BatchNorm2d) and abs(sub.eps - self.BN_EPS) > 1e-12:
                    raise ValueError(f"BatchNorm eps={sub.eps}: the packing kernels fold the default eps "
                                     f"{self.BN_EPS} (models/cdrnet.py:19, models/decoder.py:34)")
        self.release()
        src = _lib.CdrWeightPtrs()
        src.num_joints = dec[3].out_channels
        src.has_fusion = 1 if cf is not None else 0
        if cf is not None:
            src.cf_conv1 = _convbn(cf.conv_layer1[0], cf.conv_layer1[1])
            src.cf_conv2a = _convbn(cf.conv_layer2[0], cf.conv_layer2[1])
            src.cf_conv2b = _convbn(cf.conv_layer2[3], cf.conv_layer2[4])
            for v in range(2):
                src.cf_out[v] = _convbn(cf.out_layer[v][0], cf.out_layer[v][1])
            src.fusion_hid_ch1 = cf.conv_layer1[0].out_channels          # 0 / 0 would mean the defaults 300 / 400
            src.fusion_hid_ch2 = cf.conv_layer2[3].out_channels
        for i in range(3):
            src.deconv[i] = _convbn(dec[i][0], dec[i][1])
        src.final_layer = _convbn(dec[3], None)
        handle = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(_lib.lib().cdr_weights_create(
                C.byref(src), _lib.PRECISIONS[self.precision], _lib.current_stream_ptr(device),
                C.byref(handle)))
        self._box = _wsmod.HandleBox(handle, lambda h: _lib.lib().cdr_weights_destroy(h))
        self._sig = sig
        return handle

    def release(self):
        if self._box is not None:
            self._box.release()          # destroyed now unless a captured graph still holds it
            self._box = None
            self._sig = None

    def __deepcopy__(self, memo):
        return _PackedWeights(None, self.precision, self.has_fusion)  # handles are not shared

    def __getstate__(self):
        return {"precision": self.precision, "has_fusion": self.has_fusion,
                "_box": None, "_sig": None, "_last": None}

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class CDRNet(nn.Module):
    """Reference models/cdrnet.py:88-268 with the post-encoder path on libcdrhead.so.

    Extra keyword ``precision``: 'fp32' (default) = fp32-accurate results on the tcgen05 tensor cores — decoder and
    conv_layer1 on scaled fp16 two-term operands (f16x2), the rest of the fusion block on 3xTF32; 'tf32x3' = 3xTF32
    everywhere; 'fp32_ffma' = the same arithmetic on CUDA cores (cross-check); 'bf16' = bf16 operands on tcgen05."""

    def __init__(self, cfg, n_views=2, nj=19, fusion_in_dim=2048, fusion_hid_ch1=300,
                 fusion_hid_ch2=400, precision="fp32", encoder_precision=None, trainable=False, train_encoder_on_library=False,
                 train_stem_on_library=False):
        """encoder_precision: 'fp32' — this library's tcgen05 encoder at the reference's precision (scaled fp16 hi/lo
        planes, 3 MMAs per product; needs precision='fp32'); 'torch' (default — the reference's nn.Module on torch/cuDNN, fp32) or
        'bf16' (Bottleneck stages on libcdrhead's tcgen05 kernels, stem on cuDNN bf16; SURVEY §8f).
        trainable: opt in to ``forward`` in training mode (``forward_train``, SURVEY §8f rank 3 slice).
        train_encoder_on_library: ``forward_train`` runs a Bottleneck encoder through ``ResNet.forward_train`` (its 1x1 /
        3x3 convs and BatchNorms on libcdrhead at fp32 accuracy) instead of the torch modules (DESIGN.md §7).
        train_stem_on_library: with ``train_encoder_on_library``, the encoder's stem (7x7 conv, BatchNorm + ReLU,
        max-pool) trains on libcdrhead as well (``ResNet.forward_train(x, stem_on_library=True)``)."""
        super().__init__()
        if train_stem_on_library and not train_encoder_on_library:
            raise ValueError("train_stem_on_library=True needs train_encoder_on_library=True")
        self.trainable = bool(trainable)
        self.train_encoder_on_library = bool(train_encoder_on_library)
        self.train_stem_on_library = bool(train_stem_on_library)
        encoder_precision = _default_encoder_precision(encoder_precision)
        if encoder_precision not in ("torch", "bf16", "fp32"):
            raise ValueError(f"encoder_precision must be 'torch', 'bf16' or 'fp32', got {encoder_precision!r}")
        if encoder_precision == "fp32" and precision not in ("fp32", "f16x2"):
            raise ValueError("encoder_precision='fp32' (fp16-plane latents) needs the fp32 head (precision='fp32')")
        self.encoder_precision = encoder_precision
        if n_views != 2 or fusion_in_dim != 2048:
            # the reference itself only runs in this configuration: CanonicalFusion has exactly two out_layer heads and
            # forward returns views 0 and 1 (models/cdrnet.py:32-43,255), the decoder takes 2048 channels
            # (models/decoder.py:8-9) — shown on the unmodified reference in tests/test_oracle_golden.py
            raise NotImplementedError(
                "n_views must be 2 and fusion_in_dim 2048: the reference's own forward fails otherwise "
                "(models/cdrnet.py:32-43,255, models/decoder.py:8-9)")
        if fusion_hid_ch2 * 3 != fusion_hid_ch1 * 4:
            raise ValueError(
                f"fusion_hid_ch2 must be 4/3 of fusion_hid_ch1 (got {fusion_hid_ch1} / {fusion_hid_ch2}): the 4x3 / 3x4 "
                "feature transforms map 3 channel blocks to 4 and back (models/cdrnet.py:45-56,65,79)")
        if fusion_hid_ch1 % 12 != 0 or not 12 <= fusion_hid_ch1 <= 3072:
            raise NotImplementedError("fusion_hid_ch1 must be a multiple of 12 in 12..3072 (FTL blocks of whole 128-bit vectors)")
        self.encoder = ResNet(cfg)
        self.CF = CanonicalFusion(in_dim=fusion_in_dim, hid_ch1=fusion_hid_ch1,
                                  hid_ch2=fusion_hid_ch2, n_views=n_views)
        self.decoder = PoseDecoder(cfg, precision)
        self.n_views = n_views
        self.nj = nj
        self._packed = _PackedWeights(self, precision, has_fusion=True)
        self._tc_encoder = TcEncoder(self.encoder, encoder_precision) if encoder_precision != "torch" else None

    @property
    def precision(self):
        return self._packed.precision

    def init_weights(self, pretrained=""):
        """models/cdrnet.py:103-118: decoder N(0, 1e-3) init + encoder.* keys of a checkpoint."""
        import os
        if not os.path.isfile(pretrained):
            raise ValueError("Pretrained model '{}' does not exist.".format(pretrained))
        self.decoder.init_weights()
        ckpt = torch.load(pretrained)
        self.load_state_dict({k: v for k, v in ckpt.items() if k.startswith("encoder")},
                             strict=False)

    def head(self, feats, proj_list, proj_inv_list=None, taps=False, img_size=256, feat_rows=None, out_xyz=None):
        """The hot path: encoder latents -> (pred_2ds, pred_3ds).  models/cdrnet.py:236-268.

        feats: list[2] of (B,2048,8,8); proj_list: list[2] of (B,3,4).  ``proj_inv_list``
        overrides the on-device pseudo-inverse.  ``taps=True`` also returns the stage
        tensors the parity tests compare.  ``feat_rows`` (instead of ``feats``): the latents as
        bf16 pixel-major rows (2*B*64, 2048), left view first — the tcgen05 encoder's output.
        ``out_xyz``: a contiguous (B,J,3) fp32 CUDA tensor the 3D joints are written into (e.g. this rank's slot
        of a multi-GPU gather buffer, dist.GatherBuffer) instead of a fresh tensor."""
        _require_eval(self)
        pl = _as_f32_cuda(proj_list[0], "proj_list")
        pr = _as_f32_cuda(proj_list[1], "proj_list")
        b = pl.shape[0]
        fl = fr = None
        planes = feat_rows is not None and feat_rows.dtype == torch.uint8     # the fp32 encoder's fp16-planes buffer
        if planes:
            if not (feat_rows.is_cuda and feat_rows.is_contiguous() and feat_rows.numel() >= 2 * (2 * b * 64 * 2048 * 2) + 8):
                raise ValueError("feat_rows (fp16 planes) must be the contiguous CUDA uint8 buffer TcEncoder.rows returned")
        elif feat_rows is not None:
            if not (feat_rows.is_cuda and feat_rows.dtype == torch.bfloat16 and feat_rows.is_contiguous()
                    and tuple(feat_rows.shape) == (2 * b * 64, 2048)):
                raise ValueError("feat_rows must be a contiguous CUDA bf16 tensor of shape (2*B*64, 2048)")
        else:
            fl = _as_f32_cuda(feats[0], "features")
            fr = _as_f32_cuda(feats[1], "features")
            if tuple(fl.shape) != (b, 2048, 8, 8) or fr.shape != fl.shape:
                raise ValueError(f"expected two (B,2048,8,8) latents, got {tuple(fl.shape)} / {tuple(fr.shape)}")
        if tuple(pl.shape) != (b, 3, 4) or tuple(pr.shape) != (b, 3, 4):
            raise ValueError(f"proj_list entries must be (B,3,4), got {tuple(pl.shape)} / {tuple(pr.shape)}")
        dev = pl.device
        j = self.decoder.num_joints
        if j != self.nj:
            raise ValueError(f"nj={self.nj} but cfg.MODEL.NUM_JOINTS={j} (the reference would fail in dlt)")
        pil = pir = None
        if proj_inv_list is not None:
            pil = _as_f32_cuda(proj_inv_list[0], "proj_inv_list")
            pir = _as_f32_cuda(proj_inv_list[1], "proj_inv_list")
        handle = self._packed.get(_decoder_tensors(self.decoder, "decoder."), dev, cf=self.CF)
        L = _lib.lib()
        nbytes = C.c_size_t()
        _lib.check(L.cdr_head_workspace_bytes(handle, b, C.byref(nbytes)))
        ws = _workspace(dev, nbytes.value)
        kp_l = torch.empty((b, j, 2), dtype=torch.float32, device=dev)
        kp_r = torch.empty((b, j, 2), dtype=torch.float32, device=dev)
        if out_xyz is not None:
            if not (out_xyz.is_cuda and out_xyz.dtype == torch.float32 and out_xyz.is_contiguous()
                    and tuple(out_xyz.shape) == (b, j, 3) and out_xyz.device == dev):
                raise ValueError(f"out_xyz must be a contiguous ({b},{j},3) float32 tensor on {dev}")
            xyz = out_xyz
        else:
            xyz = torch.empty((b, j, 3), dtype=torch.float32, device=dev)
        tap_struct, tap_out = None, None
        if taps:
            tap_out = {
                "pinv": torch.empty((2, b, 4, 3), dtype=torch.float32, device=dev),
                "cf_cat": torch.empty((b, 64, 2 * self.CF.conv_layer2[3].out_channels), dtype=torch.float32, device=dev),
                "cf_f": torch.empty((b, 64, self.CF.conv_layer2[3].out_channels), dtype=torch.float32, device=dev),
                "f_out": torch.empty((2, b, 64, 2048), dtype=torch.float32, device=dev),
                "heatmaps": torch.empty((2, b, j, 64, 64), dtype=torch.float32, device=dev),
            }
            tap_struct = _lib.CdrHeadTaps()
            for k, t in tap_out.items():
                setattr(tap_struct, k, t.data_ptr())
        with torch.cuda.device(dev):
            if feat_rows is not None:
                _lib.check((L.cdr_head_forward_planes if planes else L.cdr_head_forward_rows)(
                    handle, _lib.ptr(feat_rows), _lib.ptr(pl), _lib.ptr(pr), _lib.ptr(pil),
                    _lib.ptr(pir), PINV_RTOL_FP32, b, int(img_size), _lib.ptr(kp_l), _lib.ptr(kp_r),
                    _lib.ptr(xyz), C.byref(tap_struct) if taps else None, _lib.ptr(ws), nbytes.value,
                    _lib.current_stream_ptr(dev)))
            else:
                _lib.check(L.cdr_head_forward(
                    handle, _lib.ptr(fl), _lib.ptr(fr), _lib.ptr(pl), _lib.ptr(pr), _lib.ptr(pil),
                    _lib.ptr(pir), PINV_RTOL_FP32, b, int(img_size), _lib.ptr(kp_l), _lib.ptr(kp_r),
                    _lib.ptr(xyz), C.byref(tap_struct) if taps else None, _lib.ptr(ws), nbytes.value,
                    _lib.current_stream_ptr(dev)))
        if taps:
            return [kp_l, kp_r], xyz, tap_out
        return [kp_l, kp_r], xyz

    def forward(self, xs, proj_list):
        """xs: list[2] of (B,3,S,S) images; proj_list: list[2] of (B,3,4).
        Returns ([kp_left, kp_right] each (B,J,2) in image pixels, xyz (B,J,3))."""
        if self.training and self.trainable:
            return self.forward_train(xs, proj_list)
        _require_eval(self)
        img_size = int(xs[0].size(2))                             # models/cdrnet.py:229
        if self._tc_encoder is not None and xs[0].shape[-1] == 256 and xs[0].shape[-2] == 256:
            # both views through the tcgen05 encoder as one batch; its bf16 rows feed the head directly
            rows, _ = self._tc_encoder.rows(torch.cat([xs[0], xs[1]], 0))
            return self.head(None, proj_list, img_size=img_size, feat_rows=rows)
        with torch.no_grad():
            zs = [self.encoder(xs[i]) for i in range(self.n_views)]  # :231-234 (torch/cuDNN)
        return self.head(zs, proj_list, img_size=img_size)


    def forward_train(self, xs, proj_list):
        """The training-mode forward of train_cdr.py:105 (models/cdrnet.py:224-268 with autograd), SURVEY §8f rank 3
        — an explicit HYBRID, not a fallback of the inference path.  Every convolution of the head runs forward and
        backward in libcdrhead.so at fp32 accuracy, independent of torch's TF32 flags (autograd.py): the decoder's three
        transposed convolutions (``conv_transpose2d`` on the weights of ``decoder.deconv{1,2,3}.0``) and the 1x1 convs
        of the fusion block and ``decoder.final_layer`` (``conv1x1``, bias included).  The head's train-mode BatchNorm +
        ReLU (losses.py: batch statistics, running-stat update), the three operators the reference hand-rolls —
        ``ftl`` (:45-56), ``process_heatmap`` (:120-149) and ``dlt`` (:151-179) — and the pseudo-inverse run forward
        AND backward in libcdrhead.so too (autograd.py, losses.py).  With ``train_encoder_on_library=True`` a Bottleneck
        encoder (ResNet-50/101/152) trains on the library as well (``ResNet.forward_train``): its 1x1 convs through
        ``conv1x1``, its 3x3 convs through ``conv3x3`` and its BatchNorms through ``batch_norm_train``, one call per view
        so that BatchNorm sees per-view batch statistics, as in the reference; otherwise the encoder runs on torch (cuDNN
        + torch autograd).  The encoder's stem (7x7 conv, BatchNorm, ReLU, max-pool) stays with torch unless
        ``train_stem_on_library=True``, which puts it on the library too (``stem_conv``, ``batch_norm_train``,
        ``max_pool3x3``).  The optimizer always stays with torch.  Needs ``CDRNet(..., trainable=True)``; projection
        matrices get no gradient (data in the reference)."""
        from .autograd import conv1x1, conv_transpose2d, dlt, ftl, soft_argmax_2d
        if not self.trainable:
            raise RuntimeError("forward_train needs CDRNet(..., trainable=True)")
        pl = _as_f32_cuda(proj_list[0], "proj_list")
        pr = _as_f32_cuda(proj_list[1], "proj_list")
        b = pl.shape[0]
        img_size = int(xs[0].size(2))                                         # :229
        pinv = torch.empty((2, b, 4, 3), dtype=torch.float32, device=pl.device)
        with torch.cuda.device(pl.device):
            st = _lib.current_stream_ptr(pl.device)
            for v, p in enumerate((pl, pr)):                                  # :236-237
                _lib.check(_lib.lib().cdr_pinv(_lib.ptr(p), b, PINV_RTOL_FP32, _lib.ptr(pinv[v]), st))
        from .losses import batch_norm_train

        def cbr(seq, x, i=0):
            """1x1 conv -> train-mode BatchNorm + ReLU, both on libcdrhead"""
            return batch_norm_train(conv1x1(x, seq[i].weight, seq[i].bias), seq[i + 1], relu=True)

        def dcbr(seq, x):
            """transposed conv on libcdrhead -> train-mode BatchNorm + ReLU"""
            return batch_norm_train(conv_transpose2d(x, seq[0].weight), seq[1], relu=True)
        enc = self.encoder.forward_train if self.train_encoder_on_library else self.encoder
        if self.train_stem_on_library:
            enc = functools.partial(enc, stem_on_library=True)
        feats = [enc(xs[v]) for v in range(2)]                                # :231-234, one call per view
        cf = self.CF
        z = torch.cat([ftl(cbr(cf.conv_layer1, feats[v]), pinv[v]) for v in range(2)], dim=1)      # :62-70
        f = cbr(cf.conv_layer2, cbr(cf.conv_layer2, z), 3)                    # :74
        projs = (pl, pr)
        kps = []
        for v in range(2):
            o = cbr(cf.out_layer[v], ftl(f, projs[v]))                        # :79-81
            d = self.decoder
            h = conv1x1(dcbr(d.deconv3, dcbr(d.deconv2, dcbr(d.deconv1, o))), d.final_layer.weight,
                        d.final_layer.bias)                                   # models/decoder.py:39-46
            kps.append(soft_argmax_2d(h, img_size / h.shape[2]))              # :243-250
        return kps, dlt(pl, pr, kps[0], kps[1])                               # :252-268

    def forward_frames(self, frames, proj_list, mean=None, std=None, img_size=None):
        """Device-side input pipeline (SURVEY §8f rank 2): frames = [left, right] raw uint8 CUDA tensors
        (B,H,W,3) — or one (2B,H,W,3) tensor, left half first — instead of inference.py:40-52's
        PIL -> ToTensor -> Normalize -> .to(device).  Needs ``encoder_precision='fp32'`` or ``'bf16'``."""
        from .encoder import IMAGENET_MEAN, IMAGENET_STD
        _require_eval(self)
        if self._tc_encoder is None:
            raise RuntimeError("forward_frames needs CDRNet(..., encoder_precision='fp32' or 'bf16')")
        x = frames if isinstance(frames, torch.Tensor) else torch.cat([frames[0], frames[1]], 0)
        rows, _ = self._tc_encoder.rows(x, mean=IMAGENET_MEAN if mean is None else tuple(float(v) for v in mean),
                                        std=IMAGENET_STD if std is None else tuple(float(v) for v in std))
        return self.head(None, proj_list, img_size=int(img_size or x.shape[1]), feat_rows=rows)


class PoseResNet(nn.Module):
    """models/poseresnet.py:10-38: ResNet encoder (torch/cuDNN) + PoseDecoder (libcdrhead)."""

    def __init__(self, cfg, precision="fp32", encoder_precision=None):
        super().__init__()
        encoder_precision = _default_encoder_precision(encoder_precision)
        if encoder_precision not in ("torch", "bf16", "fp32"):
            raise ValueError(f"encoder_precision must be 'torch', 'bf16' or 'fp32', got {encoder_precision!r}")
        if encoder_precision == "fp32" and precision not in ("fp32", "f16x2"):
            raise ValueError("encoder_precision='fp32' (fp16-plane latents) needs the fp32 decoder (precision='fp32')")
        self.encoder = ResNet(cfg)
        self.decoder = PoseDecoder(cfg, precision)
        self.encoder_precision = encoder_precision
        self._tc_encoder = TcEncoder(self.encoder, encoder_precision) if encoder_precision != "torch" else None

    def forward(self, x):
        """x: (N,3,256,256) float images — or, with encoder_precision='fp32' / 'bf16', raw (N,256,256,3) uint8 frames."""
        if self._tc_encoder is not None and self.decoder._packed.precision != "fp32_ffma" and \
                tuple(x.shape[-3:] if x.dtype == torch.uint8 else x.shape[-2:])[:2] == (256, 256):
            rows, _ = self._tc_encoder.rows(x)
            return self.decoder.forward_rows(rows, n_images=x.shape[0])
        with torch.no_grad():
            feats = self.encoder(x)
        return self.decoder(feats)

    def init_weights(self, pretrained=""):
        import os
        if not os.path.isfile(pretrained):
            raise ValueError("Pretrained model '{}' does not exist.".format(pretrained))
        self.decoder.init_weights()
        ckpt = torch.load(pretrained)
        self.load_state_dict({k: v for k, v in ckpt.items() if k.startswith("encoder")},
                             strict=False)
