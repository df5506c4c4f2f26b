// Shared helpers for libcdrhead.so (sm_100a only).
#pragma once
#include <stdlib.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/cdrhead.h"

namespace cdr {

// thread-local error string + launch counter (the only mutable global state)
void set_error(const char* fmt, ...);
void count_launch(const char* kernel);
// label attached to subsequent launches in the stage-timing record (api.cu)
void set_stage(const char* label);
void timing_restart();

#define CDR_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      cdr::set_error(__VA_ARGS__);               \
      return CDR_ERR_INVALID;                    \
    }                                            \
  } while (0)

#define CDR_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      cdr::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),        \
                     __FILE__, __LINE__);                                           \
      (void)cudaGetLastError(); /* reported here: do not leave it for the next call's launch check */ \
      return CDR_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

// check the launch that just happened
#define CDR_LAUNCH_OK(name)                                                         \
  do {                                                                              \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess) {                                                        \
      cdr::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));      \
      return CDR_ERR_CUDA;                                                          \
    }                                                                               \
    cdr::count_launch(name);                                                        \
  } while (0)

// Per-device caches: a process may drive several GPUs (the Python shim wraps every call in
// torch.cuda.device(dev)), and both the SM count and a kernel's opt-in to > 48 KB of dynamic shared
// memory (cudaFuncSetAttribute) belong to the CURRENT device, not to the process.
constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 0;
  return dev;
}
inline int num_sms() {
  static int n[kMaxDevices] = {};
  const int dev = current_device();
  if (n[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n[dev] = v;
  }
  return n[dev];
}
// one flag word per kernel instantiation (a function-local static at the call site), one bit per device
// Device scalars written by a predecessor kernel (scale / amax slots) are read with __ldcg (L2), never through the
// non-coherent L1 path.  MEASURED (round 2): with the FTL / layout kernels launched by programmatic dependent launch too,
// a kernel that starts early shares an SM with its still-running predecessors, whose own __ldg of the same 128-byte
// line (all slots live in one) left a stale copy in that SM's L1 — conv outputs scaled by 1/0 in ~1 of 10 runs.  With
// every predecessor-written word read through L2 the race is gone, but the L2-only loads cost the FTL kernels more
// (12 -> 20 us) than the overlapped prologues returned (+2 % -> -1 % on the step), so the layout kernels are plain
// launches again; only the tap-GEMM / tail kernels (which never co-reside: one 220 KB CTA per SM) and the merge kernel
// (it shares SMs with the tail's last CTAs but reads only their records, which no co-resident CTA ever loads) chain by PDL.

struct DeviceOnce {
  unsigned long long mask = 0;
  bool need() const { return !((mask >> current_device()) & 1ull); }
  void done() { mask |= 1ull << current_device(); }
};

template <typename T>
__host__ __device__ constexpr T ceil_div(T a, T b) { return (a + b - 1) / b; }
template <typename T>
__host__ __device__ constexpr T round_up(T a, T b) { return ceil_div(a, b) * b; }

// ---- 3xTF32 operand split.  hi = x rounded to nearest-even at tf32 precision (11 significant
// bits, exactly a tf32 value), lo = x - hi (exact, |lo| <= 2^-11 |x|, random sign), so hi + lo
// reproduces x bit for bit for the consumers that add the planes.  The tensor core sees lo
// through its own 11-bit window; because lo's sign is random that residue (<= 2^-21 |x|) is
// unbiased.  (A truncating split hi = x & ~0x1fff leaves a same-signed residue in every
// product, which does not average out over K: ~1e-5 relative error in the heat-maps.)
__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t u = __float_as_uint(x);
  u += 0xFFFu + ((u >> 13) & 1u);
  return __uint_as_float(u & 0xFFFFE000u);
}
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = tf32_rn(x);
  lo = x - hi;
}

// ---- power-of-two scale of the scaled fp16 hi/lo planes (gemm_tc.cu: kFmtF16P): s = 2^(13 - ilogb(amax)) puts the
// largest |x| in [2^13, 2^14), 4x below fp16 max.  The exponent is capped at 127 so that s stays a finite float for
// amax < 2^-114 (uncapped, s = +Inf and the encode x * s turns every element into +-Inf or NaN); 1/s = 2^-127 is then an
// exact subnormal, as the library never flushes denormals.  A zero, infinite or NaN amax gives s = 1.  For amax in
// [2^-114, FLT_MAX] this is exactly 2^(13 - ilogb(amax)).
constexpr int kF16TargetExp = 13;
__device__ __forceinline__ int f16_pow2_exp(float amax) {
  if (!(amax > 0.f && amax <= 3.40282347e38f)) return 0;
  const int e = kF16TargetExp - ilogbf(amax);
  return e < 127 ? e : 127;
}
__device__ __forceinline__ float f16_pow2_scale(float amax) { return ldexpf(1.f, f16_pow2_exp(amax)); }

// ---- fixed geometry of the head (models/cdrnet.py:89-91, models/decoder.py:8-13) ----
constexpr int kFeatC = 2048;   // encoder channels = fusion_in_dim
constexpr int kFeatHW = 64;    // 8x8 latent
constexpr int kHid1 = 300;     // fusion_hid_ch1
constexpr int kHid1Pad = 304;  // channel pitch of 300-channel buffers (16-B rows for bf16, K%16 for fp32)
constexpr int kHid2 = 400;     // fusion_hid_ch2
constexpr int kFtlBlk = 100;   // channels per FTL "coordinate" block: 300/3 = 400/4
// Runtime fusion widths (models/cdrnet.py:89-91: fusion_hid_ch1 / fusion_hid_ch2; the defaults above).  The reference's
// forward only type-checks when hid_ch2 = 4/3 hid_ch1 (the 4x3 / 3x4 feature transforms map 3 blocks to 4 and back);
// this library additionally wants the block size to be a multiple of 4 (128-bit FTL, 16-byte rows): hid_ch1 % 12 == 0.
struct FusionDims {
  int h1 = kHid1, h1p = kHid1Pad, h2 = kHid2, blk = kFtlBlk;
  int n1_pad() const { return (h1 + 127) / 128 * 128; }     // packed output channels of conv_layer1 (N tiles of 128)
  int n2_pad() const { return (h2 + 127) / 128 * 128; }
};
inline bool fusion_dims_ok(int h1, int h2) { return h1 >= 12 && h1 % 12 == 0 && h1 <= 3072 && h2 * 3 == h1 * 4; }
inline FusionDims make_fusion_dims(int h1, int h2) {
  FusionDims d;
  if (h1 > 0) { d.h1 = h1; d.h2 = h2; d.h1p = (h1 + 15) / 16 * 16; d.blk = h1 / 3; }
  return d;
}
constexpr int kDecC = 256;     // deconv output channels
constexpr int kHeat = 64;      // heat-map side
constexpr int kMaxJoints = 64;

}  // namespace cdr
