"""ctypes binding of libcdrhead.so (include/cdrhead.h).

There is no fallback: if the shared library is missing or a call fails, this
module raises.  ``build()`` compiles it in-tree with nvcc for sm_100a.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CDR_LIB_PATH") or os.path.join(_HERE, "libcdrhead.so")   # override: A/B builds of the same ABI
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "cdrhead.h")

CDR_PREC_FP32 = 0
CDR_PREC_BF16 = 1
CDR_PREC_TF32X3 = 2
CDR_PREC_F16X2 = 3
# "fp32" / "f16x2": fp32-accurate results on the tcgen05 tensor cores — the default.  Fusion block and decoder on
#              scaled fp16 two-term operands (3 kind::f16 MMAs per product; gemm_tc.cu: kModeF16X2)
# "tf32x3"   : 3xTF32 split (kind::tf32) everywhere
# "fp32_ffma": the same arithmetic on CUDA cores (FFMA), kept as the in-library cross-check
# "bf16"     : bf16 operands on the tensor cores
PRECISIONS = {"fp32": CDR_PREC_F16X2, "f16x2": CDR_PREC_F16X2, "tf32x3": CDR_PREC_TF32X3, "fp32_ffma": CDR_PREC_FP32,
              "bf16": CDR_PREC_BF16}

_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_vp = C.c_void_p


class CdrConvBn(C.Structure):
    _fields_ = [(n, _vp) for n in ("weight", "bias", "bn_weight", "bn_bias", "bn_mean", "bn_var")]


class CdrWeightPtrs(C.Structure):
    _fields_ = [("num_joints", C.c_int), ("has_fusion", C.c_int),
                ("cf_conv1", CdrConvBn), ("cf_conv2a", CdrConvBn), ("cf_conv2b", CdrConvBn),
                ("cf_out", CdrConvBn * 2), ("deconv", CdrConvBn * 3), ("final_layer", CdrConvBn),
                ("fusion_hid_ch1", C.c_int), ("fusion_hid_ch2", C.c_int)]


class CdrHeadTaps(C.Structure):
    _fields_ = [(n, _vp) for n in ("pinv", "cf_cat", "cf_f", "f_out", "heatmaps")]


class CdrEncoderBlock(C.Structure):
    _fields_ = [("conv1", CdrConvBn), ("conv2", CdrConvBn), ("conv3", CdrConvBn), ("downsample", CdrConvBn),
                ("planes", C.c_int), ("stride", C.c_int)]


class CdrEncoderSpec(C.Structure):
    _fields_ = [("num_blocks", C.c_int), ("blocks", C.POINTER(CdrEncoderBlock)), ("in_channels", C.c_int),
                ("stem", CdrConvBn)]


class CdrError(RuntimeError):
    pass


# name -> (restype, argtypes); kept in step with include/cdrhead.h (tests/test_abi.py checks)
_SIGNATURES = {
    "cdr_abi_version": (C.c_int, []),
    "cdr_last_error": (C.c_char_p, []),
    "cdr_debug_words": (C.POINTER(C.c_uint), []),
    "cdr_launch_count": (C.c_ulonglong, []),
    "cdr_launch_count_reset": (None, []),
    "cdr_stage_timing_begin": (C.c_int, [_vp]),
    "cdr_stage_timing_end": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "cdr_weights_create": (C.c_int, [C.POINTER(CdrWeightPtrs), C.c_int, _vp, C.POINTER(_vp)]),
    "cdr_weights_destroy": (C.c_int, [_vp]),
    "cdr_head_workspace_bytes": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_size_t)]),
    "cdr_decoder_workspace_bytes": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_size_t)]),
    "cdr_head_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_double, C.c_int, C.c_int,
                                   _vp, _vp, _vp, C.POINTER(CdrHeadTaps), _vp, C.c_size_t, _vp]),
    "cdr_decoder_forward": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "cdr_decoder_forward_rows": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "cdr_head_forward_rows": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_double, C.c_int, C.c_int,
                                        _vp, _vp, _vp, C.POINTER(CdrHeadTaps), _vp, C.c_size_t, _vp]),
    "cdr_head_forward_planes": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_double, C.c_int, C.c_int,
                                          _vp, _vp, _vp, C.POINTER(CdrHeadTaps), _vp, C.c_size_t, _vp]),
    "cdr_decoder_forward_planes": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "cdr_encoder_create": (C.c_int, [C.POINTER(CdrEncoderSpec), _vp, C.POINTER(_vp)]),
    "cdr_encoder_create_prec": (C.c_int, [C.POINTER(CdrEncoderSpec), C.c_int, _vp, C.POINTER(_vp)]),
    "cdr_encoder_out_bytes": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "cdr_encoder_destroy": (C.c_int, [_vp]),
    "cdr_encoder_workspace_bytes": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "cdr_encoder_out_shape": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                        C.POINTER(C.c_int)]),
    "cdr_encoder_forward": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "cdr_encoder_workspace_bytes_images": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "cdr_encoder_forward_images": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "cdr_encoder_forward_frames_u8": (C.c_int, [_vp, _vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_int,
                                                C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "cdr_bn_train_forward": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_double, C.c_double, _vp, _vp, C.c_int,
                                       _vp, _vp, _vp, _vp]),
    "cdr_bn_train_backward": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    "cdr_joint_loss_scratch_bytes": (C.c_size_t, []),
    "cdr_joint_loss_forward": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_double, _vp, _vp, _vp]),
    "cdr_joint_loss_backward": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_double, _vp, _vp, _vp]),
    "cdr_pinv": (C.c_int, [_vp, C.c_int, C.c_double, _vp, _vp]),
    "cdr_projection_matrices": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, _vp]),
    "cdr_ftl": (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp,
                          C.c_int, C.c_int, _vp]),
    "cdr_softargmax": (C.c_int, [_vp, C.c_longlong, C.c_int, C.c_int, C.c_float, _vp, _vp]),
    "cdr_dlt": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp]),
    "cdr_softargmax_dlt": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_longlong, C.c_int, C.c_int,
                                     C.c_int, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp]),
    "cdr_argmax": (C.c_int, [_vp, C.c_longlong, C.c_int, C.c_int, C.c_float, _vp, _vp, _vp, _vp]),
    "cdr_triangulate_u8": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_longlong, C.c_int,
                                     _vp, _vp]),
    "cdr_mpjpe_scratch_bytes": (C.c_size_t, [C.c_longlong]),
    "cdr_mpjpe_partial": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int,
                                    C.c_longlong, C.c_int, _vp, _vp, _vp]),
    "cdr_mpjpe_reduce": (C.c_int, [_vp, C.c_longlong, C.c_int, _vp, _vp, _vp]),
    "cdr_softargmax_backward": (C.c_int, [_vp, _vp, C.c_longlong, C.c_int, C.c_int, C.c_float, _vp, _vp]),
    "cdr_dlt_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp]),
    "cdr_deconv_train_workspace_bytes": (C.c_int, [C.c_int] * 5 + [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "cdr_deconv_train_forward": (C.c_int, [_vp, _vp] + [C.c_int] * 5 + [_vp, _vp, C.c_size_t, _vp, C.c_size_t, _vp]),
    "cdr_deconv_train_backward": (C.c_int, [_vp, _vp, _vp] + [C.c_int] * 5 + [_vp, _vp, _vp, C.c_size_t, _vp]),
    "cdr_conv1x1_train_workspace_bytes": (C.c_int, [C.c_int] * 5 + [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "cdr_conv1x1_train_forward": (C.c_int, [_vp, _vp, _vp] + [C.c_int] * 5 + [_vp, _vp, C.c_size_t, _vp, C.c_size_t,
                                                                             _vp]),
    "cdr_conv1x1_train_backward": (C.c_int, [_vp, _vp, _vp] + [C.c_int] * 5 + [_vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "cdr_conv3x3_train_workspace_bytes": (C.c_int, [C.c_int] * 6 + [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "cdr_conv3x3_train_forward": (C.c_int, [_vp, _vp] + [C.c_int] * 6 + [_vp, _vp, C.c_size_t, _vp, C.c_size_t, _vp]),
    "cdr_conv3x3_train_backward": (C.c_int, [_vp, _vp, _vp] + [C.c_int] * 6 + [_vp, _vp, _vp, C.c_size_t, _vp]),
    "cdr_stem_train_workspace_bytes": (C.c_int, [C.c_int] * 5 + [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "cdr_stem_train_forward": (C.c_int, [_vp, _vp] + [C.c_int] * 5 + [_vp, _vp, C.c_size_t, _vp, C.c_size_t, _vp]),
    "cdr_stem_train_backward": (C.c_int, [_vp, _vp, _vp] + [C.c_int] * 5 + [_vp, _vp, _vp, C.c_size_t, _vp]),
    "cdr_maxpool3x3_train_forward": (C.c_int, [_vp] + [C.c_int] * 4 + [_vp, _vp, _vp]),
    "cdr_maxpool3x3_train_backward": (C.c_int, [_vp, _vp] + [C.c_int] * 4 + [_vp, _vp]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def build(verbose: bool = False) -> str:
    """Compile libcdrhead.so in-tree (nvcc, sm_100a, -lineinfo)."""
    script = os.path.join(_HERE, "csrc", "build.sh")
    res = subprocess.run(["bash", script], capture_output=True, text=True)
    if res.returncode != 0:
        raise CdrError("building libcdrhead.so failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout)
    return LIB_PATH


def lib() -> C.CDLL:
    """Load the library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CdrError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the CDRNet head)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        got = handle.cdr_abi_version()
        if got != 1:
            raise CdrError(f"libcdrhead.so ABI version {got} != 1")
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().cdr_last_error()
        raise CdrError(f"libcdrhead error {rc}: {msg.decode(errors='replace') if msg else '?'}")


def stage_timing_begin(device=None):
    check(lib().cdr_stage_timing_begin(current_stream_ptr(device)))


def stage_timing_end(capacity=512):
    """-> list of (stage label, milliseconds) for every launch since stage_timing_begin."""
    names = C.create_string_buffer(48 * capacity)
    ms = (C.c_float * capacity)()
    n = C.c_int()
    check(lib().cdr_stage_timing_end(capacity, names, ms, C.byref(n)))
    raw = names.raw
    return [(raw[i * 48:(i + 1) * 48].split(b"\0", 1)[0].decode(), float(ms[i])) for i in range(n.value)]


def ptr(t):
    """Device (or host) address of a torch tensor / None -> c_void_p."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def current_stream_ptr(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
