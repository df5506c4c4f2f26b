// ResNet stem on B200: conv 7x7 stride 2 pad 3 (3 -> 64) + eval BN + ReLU, then max-pool 3x3 stride 2
// pad 1 (reference models/encoder.py:93-97,122-125), fp32 NCHW images in, bf16 NHWC rows out — the
// layout the tcgen05 bottleneck kernels read.
//
// Cin = 3 rules out the TMA/UMMA operand path (a pixel is 6 bytes), and K = 147 is tiny, so the conv
// is an implicit GEMM on warp-level mma.sync (m16n8k16 bf16, fp32 accumulate) fed from a shared-memory
// image patch: A[m][k] = patch[base(m) + off(k)], with the K axis laid out as 7 rows of 22 (21 taps*
// channels + 1 zero pad) so that a fragment's (k, k+1) pair is one aligned 32-bit LDS.  HBM-bound by
// design (100 MB in, 268 MB out per 128 images); the pool is a second, purely streaming kernel.
#include <stdlib.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "kernels.h"

namespace cdr {

constexpr int kStemCo = 64;
constexpr int kStemKy = 7, kStemRow = 22;          // K' = ky * 22 + (kx * 3 + ci), slot 21 of a row is a zero weight
constexpr int kStemK = 160;                        // 7 * 22 = 154, padded to a multiple of 16
constexpr int kStemWPitch = 168;                   // weight row pitch (elements): conflict-free B-fragment loads
constexpr int kTileH = 8, kTileW = 32;             // conv-output tile of one CTA pass: one row per warp
constexpr int kPatchH = 2 * kTileH + 5;            // 21 input rows
constexpr int kPatchW = 2 * kTileW + 5;            // 69 input columns
constexpr int kPatchPitch = 208;                   // 69 * 3 = 207 elements per patch row, padded to even

// conv1 (64,3,7,7) + bn1 -> bf16 [64][kStemWPitch] in the K' order above, fp32 folded bias [64]
__global__ void pack_stem_kernel(CdrConvBn s, __nv_bfloat16* __restrict__ w, float* __restrict__ bias) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kStemCo * kStemWPitch) return;
  const int n = idx / kStemWPitch, k = idx - n * kStemWPitch;
  const double sc = (double)s.bn_weight[n] / sqrt((double)s.bn_var[n] + 1e-5);
  if (k == 0) bias[n] = (float)((double)s.bn_bias[n] - (double)s.bn_mean[n] * sc);
  float v = 0.f;
  const int ky = k / kStemRow, r = k - ky * kStemRow;
  if (ky < kStemKy && r < 21) {
    const int kx = r / 3, ci = r - kx * 3;
    v = (float)((double)s.weight[((n * 3 + ci) * 7 + ky) * 7 + kx] * sc);
  }
  w[idx] = __float2bfloat16_rn(v);
}

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Input pixel fetch.  kU8 = false: fp32 NCHW tensors as the reference feeds its model (already normalised).
// kU8 = true: raw uint8 HWC frames with torchvision's ToTensor + Normalize (inference.py:40-44) applied on
// the fly in the same fp32 operation order — x / 255, - mean, / std — so the bf16 patch is bit-identical
// to converting the reference's preprocessed tensor (SURVEY §8f rank 2: 4x fewer bytes over PCIe, no
// host-side torchvision pass).
struct StemNorm {
  float mean[3], std[3];
};

// grid (conv rows / 8, images); each CTA walks the W/64 column tiles of its row band.
template <bool kU8>
__global__ void __launch_bounds__(256)
stem_conv_kernel(const void* __restrict__ xin, int H, int W, const StemNorm nrm, const __nv_bfloat16* __restrict__ wpk,
                 const float* __restrict__ bias, __nv_bfloat16* __restrict__ out) {
  __shared__ __align__(16) __nv_bfloat16 s_w[kStemCo * kStemWPitch];     // 21.5 KB
  __shared__ __align__(16) __nv_bfloat16 s_p[kPatchH * kPatchPitch];     // 8.7 KB
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int img = blockIdx.y, oy0 = blockIdx.x * kTileH;
  const int Ho = H >> 1, Wo = W >> 1;
  for (int i = threadIdx.x; i < kStemCo * kStemWPitch / 8; i += 256)
    reinterpret_cast<uint4*>(s_w)[i] = __ldg(reinterpret_cast<const uint4*>(wpk) + i);
  float bv[8][2];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    bv[nt][0] = __ldg(bias + nt * 8 + 2 * t);
    bv[nt][1] = __ldg(bias + nt * 8 + 2 * t + 1);
  }
  // per-lane patch offsets of the two k-pairs of every k-step: off(k') = ky * pitch + r
  int koff[kStemK / 16][2];
#pragma unroll
  for (int s = 0; s < kStemK / 16; ++s) {
#pragma unroll
    for (int hk = 0; hk < 2; ++hk) {
      const int k = 16 * s + 8 * hk + 2 * t;
      const int ky = k / kStemRow, r = k - ky * kStemRow;
      koff[s][hk] = ky < kStemKy ? ky * kPatchPitch + r : 0;       // padded k: weight is zero, any address does
    }
  }
  const float* xi = reinterpret_cast<const float*>(xin) + (size_t)img * 3 * H * W;
  const uint8_t* xu = reinterpret_cast<const uint8_t*>(xin) + (size_t)img * 3 * H * W;
  for (int ox0 = 0; ox0 < Wo; ox0 += kTileW) {
    __syncthreads();                                   // previous pass done with the patch (and s_w visible)
    const int iy0 = 2 * oy0 - 3, ix0 = 2 * ox0 - 3;
    if constexpr (!kU8) {
      for (int i = threadIdx.x; i < kPatchH * 3 * kPatchW; i += 256) {
        const int col = i % kPatchW, rc = i / kPatchW;
        const int ci = rc % 3, row = rc / 3;
        const int iy = iy0 + row, ix = ix0 + col;
        float v = 0.f;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(xi + ((size_t)ci * H + iy) * W + ix);
        s_p[row * kPatchPitch + col * 3 + ci] = __float2bfloat16_rn(v);
      }
    } else {
      for (int i = threadIdx.x; i < kPatchH * 3 * kPatchW; i += 256) {
        const int e = i % (3 * kPatchW), row = i / (3 * kPatchW);     // e = col * 3 + ci: contiguous in HWC
        const int col = e / 3, ci = e - col * 3;
        const int iy = iy0 + row, ix = ix0 + col;
        float v = 0.f;                                                 // zero padding applies AFTER normalisation
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
          const float u = (float)__ldg(xu + ((size_t)iy * W + ix) * 3 + ci);
          v = __fdiv_rn(__fsub_rn(__fdiv_rn(u, 255.f), nrm.mean[ci]), nrm.std[ci]);
        }
        s_p[row * kPatchPitch + e] = __float2bfloat16_rn(v);
      }
    }
    if (threadIdx.x < kPatchH) s_p[threadIdx.x * kPatchPitch + 207] = __float2bfloat16_rn(0.f);
    __syncthreads();
    float acc[2][8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
    // this warp: conv row `warp` of the tile, columns mt*16 + {g, g+8}
    const int base0 = (2 * warp) * kPatchPitch + 6 * g;          // pixel (warp, g): patch origin, in elements
#pragma unroll
    for (int s = 0; s < kStemK / 16; ++s) {
      uint32_t a[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const int b = base0 + 6 * 16 * mt;
        a[mt][0] = *reinterpret_cast<const uint32_t*>(s_p + b + koff[s][0]);
        a[mt][1] = *reinterpret_cast<const uint32_t*>(s_p + b + 48 + koff[s][0]);       // column g + 8
        a[mt][2] = *reinterpret_cast<const uint32_t*>(s_p + b + koff[s][1]);
        a[mt][3] = *reinterpret_cast<const uint32_t*>(s_p + b + 48 + koff[s][1]);
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const __nv_bfloat16* wr = s_w + (nt * 8 + g) * kStemWPitch + 16 * s + 2 * t;
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(wr);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(wr + 8);
        mma_bf16_16816(acc[0][nt], a[0], b0, b1);
        mma_bf16_16816(acc[1][nt], a[1], b0, b1);
      }
    }
    // + bias, ReLU, bf16, NHWC: pixel (oy0 + warp, ox0 + mt*16 + g [+8]), channels nt*8 + 2t, +1
    const int oy = oy0 + warp;
    if (oy < Ho) {
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
        for (int hr = 0; hr < 2; ++hr) {
          const int ox = ox0 + mt * 16 + g + 8 * hr;
          if (ox < Wo) {
            __nv_bfloat16* o = out + (((size_t)img * Ho + oy) * Wo + ox) * kStemCo + 2 * t;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
              const float v0 = fmaxf(acc[mt][nt][2 * hr] + bv[nt][0], 0.f);
              const float v1 = fmaxf(acc[mt][nt][2 * hr + 1] + bv[nt][1], 0.f);
              *reinterpret_cast<__nv_bfloat162*>(o + nt * 8) = __floats2bfloat162_rn(v0, v1);
            }
          }
        }
      }
    }
  }
}

// max-pool 3x3 stride 2 pad 1 on NHWC bf16 (values are post-ReLU, so 0 is the identity of the max)
__global__ void __launch_bounds__(256)
maxpool3s2_nhwc_kernel(const __nv_bfloat16* __restrict__ in, int Hi, int Wi, int C8, long long total,
                       __nv_bfloat16* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c8 = (int)(idx % C8);
  long long r = idx / C8;
  const int Wo = Wi >> 1, Ho = Hi >> 1;
  const int ox = (int)(r % Wo);
  r /= Wo;
  const int oy = (int)(r % Ho);
  const long long img = r / Ho;
  __nv_bfloat162 m[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) m[e] = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int iy = 2 * oy + dy;
    if (iy < 0 || iy >= Hi) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int ix = 2 * ox + dx;
      if (ix < 0 || ix >= Wi) continue;
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(in + ((img * Hi + iy) * Wi + ix) * (long long)(C8 * 8)) + c8);
      const __nv_bfloat162* v = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
      for (int e = 0; e < 4; ++e) m[e] = __hmax2(m[e], v[e]);
    }
  }
  reinterpret_cast<uint4*>(out + ((img * Ho + oy) * Wo + ox) * (long long)(C8 * 8))[c8] = *reinterpret_cast<const uint4*>(m);
}

int launch_pack_stem(const CdrConvBn& s, void* w, float* bias, cudaStream_t st) {
  CDR_CHECK_ARG(s.weight && s.bn_weight && s.bn_bias && s.bn_mean && s.bn_var && w && bias, "pack_stem: bad args");
  pack_stem_kernel<<<ceil_div(kStemCo * kStemWPitch, 256), 256, 0, st>>>(s, (__nv_bfloat16*)w, bias);
  CDR_LAUNCH_OK("pack_stem_kernel");
  return CDR_OK;
}
size_t stem_weight_bytes() { return (size_t)kStemCo * kStemWPitch * sizeof(__nv_bfloat16); }

// x (n,3,H,W) fp32 -> conv_out (n,H/2,W/2,64) bf16 scratch -> pooled (n,H/4,W/4,64) bf16
int launch_stem(const void* x, int is_u8, const float* mean, const float* std, int n, int H, int W, const void* w,
                const float* bias, void* conv_out, void* pooled, cudaStream_t st) {
  CDR_CHECK_ARG(x && w && bias && conv_out && pooled && n > 0, "stem: bad args");
  CDR_CHECK_ARG(!is_u8 || (mean && std), "stem: uint8 frames need mean / std");
  StemNorm nrm{};
  for (int c = 0; c < 3; ++c) {
    nrm.mean[c] = is_u8 ? mean[c] : 0.f;
    nrm.std[c] = is_u8 ? std[c] : 1.f;
  }
  CDR_CHECK_ARG(H % 16 == 0 && W % 64 == 0, "stem: image %dx%d must have H %% 16 == 0 and W %% 64 == 0", H, W);
  CDR_CHECK_ARG(((uintptr_t)conv_out & 15) == 0 && ((uintptr_t)pooled & 15) == 0 && ((uintptr_t)w & 15) == 0, "stem: alignment");
  const int Ho = H / 2, Wo = W / 2;
  if (is_u8)
    stem_conv_kernel<true><<<dim3(Ho / kTileH, n), 256, 0, st>>>(x, H, W, nrm, (const __nv_bfloat16*)w, bias,
                                                               (__nv_bfloat16*)conv_out);
  else
    stem_conv_kernel<false><<<dim3(Ho / kTileH, n), 256, 0, st>>>(x, H, W, nrm, (const __nv_bfloat16*)w, bias,
                                                                (__nv_bfloat16*)conv_out);
  CDR_LAUNCH_OK("stem_conv_kernel");
  const long long total = (long long)n * (Ho / 2) * (Wo / 2) * (kStemCo / 8);
  maxpool3s2_nhwc_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(
      (const __nv_bfloat16*)conv_out, Ho, Wo, kStemCo / 8, total, (__nv_bfloat16*)pooled);
  CDR_LAUNCH_OK("maxpool3s2_nhwc_kernel");
  return CDR_OK;
}


// max-pool 3x3 stride 2 pad 1 on NHWC fp32 (post-ReLU) -> scaled fp16 hi/lo planes; slot = {amax (complete), scale}.
// The pooled tensor's scale comes from the EXACT maximum (max-pool commutes with max): the fp32-accurate stem conv
// atomicMax-es its post-ReLU outputs into slot[0], this kernel turns that into slot[1] = 2^(13 - ilogb(amax)).
__global__ void __launch_bounds__(256)
maxpool3s2_f16p_kernel(const float* __restrict__ in, int Hi, int Wi, int C8, long long total, __half* __restrict__ hi,
                       __half* __restrict__ lo, float* __restrict__ slot) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const float a = __ldg(slot);
  const float s = f16_pow2_scale(a);
  if (idx == 0) slot[1] = s;
  if (idx >= total) return;
  const int c8 = (int)(idx % C8);
  long long r = idx / C8;
  const int Wo = Wi >> 1, Ho = Hi >> 1;
  const int ox = (int)(r % Wo);
  r /= Wo;
  const int oy = (int)(r % Ho);
  const long long img = r / Ho;
  float m[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) m[e] = 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int iy = 2 * oy + dy;
    if (iy < 0 || iy >= Hi) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int ix = 2 * ox + dx;
      if (ix < 0 || ix >= Wi) continue;
      const float4* q = reinterpret_cast<const float4*>(in + ((img * Hi + iy) * Wi + ix) * (long long)(C8 * 8)) + 2 * c8;
      const float4 q0 = __ldg(q), q1 = __ldg(q + 1);
      m[0] = fmaxf(m[0], q0.x); m[1] = fmaxf(m[1], q0.y); m[2] = fmaxf(m[2], q0.z); m[3] = fmaxf(m[3], q0.w);
      m[4] = fmaxf(m[4], q1.x); m[5] = fmaxf(m[5], q1.y); m[6] = fmaxf(m[6], q1.z); m[7] = fmaxf(m[7], q1.w);
    }
  }
  __align__(16) __half h8[8];
  __align__(16) __half l8[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float X = m[e] * s;
    h8[e] = __float2half_rn(X);
    l8[e] = __float2half_rn((X - __half2float(h8[e])) * 2048.f);
  }
  const long long o = ((img * Ho + oy) * Wo + ox) * (long long)(C8 * 8) + 8 * c8;
  *reinterpret_cast<uint4*>(hi + o) = *reinterpret_cast<const uint4*>(h8);
  *reinterpret_cast<uint4*>(lo + o) = *reinterpret_cast<const uint4*>(l8);
}


// ------------------------------------------------------------------------------------------
// The stem at fp32 accuracy for the f16x2 ("fp32") encoder, on the tensor cores (DESIGN.md §7): the bf16 kernel's implicit GEMM on warp-level mma.sync.m16n8k16, with BOTH operands as fp16 hi/lo
// pairs and three MMAs per product — x w = xh wh + 2^-11 (xh wl + xl wh) (+ 2^-22 xl wl, dropped) — exactly the f16x2
// scheme of gemm_tc.cu.  fp16 products are exact in the fp32 accumulators; main and correction terms accumulate
// separately (K = 147: no long same-signed chain).  Pixels need no scale (|x| < 65504; the lo plane keeps values down
// to 2^-36 absolute), weights carry one power-of-two scale per output channel (2^-t undone in the epilogue).
constexpr int kT16W = 16;                          // conv-output tile of one CTA pass: 8 rows x 16 columns, one row per warp
constexpr int kP16W = 2 * kT16W + 5;               // 37 input columns
constexpr int kP16Pitch = 112;                     // 37 * 3 = 111 elements per patch row, padded to even
constexpr int kStem16SmemBytes = (2 * kStemCo * kStemWPitch + 2 * kPatchH * kP16Pitch) * (int)sizeof(__half);

// conv1 (64,3,7,7) + bn1 -> fp16 hi / lo [64][kStemWPitch] in the K' order of the bf16 kernel, wsi[64] = 2^-t, bias[64].
// A null bn_weight (the training forward) packs the conv alone: BN scale 1, bias 0 (pack.cu's convention).
__global__ void pack_stem_f16x2_kernel(CdrConvBn s, __half* __restrict__ w_hi, __half* __restrict__ w_lo,
                                       float* __restrict__ wsi, float* __restrict__ bias) {
  const int n = blockIdx.x;                        // one block per output channel
  __shared__ float red[8];
  const double sc = s.bn_weight ? (double)s.bn_weight[n] / sqrt((double)s.bn_var[n] + 1e-5) : 1.0;
  auto val = [&](int k) -> float {
    const int ky = k / kStemRow, r = k - ky * kStemRow;
    if (ky >= kStemKy || r >= 21) return 0.f;
    const int kx = r / 3, ci = r - kx * 3;
    return (float)((double)s.weight[((n * 3 + ci) * 7 + ky) * 7 + kx] * sc);
  };
  float mx = 0.f;
  for (int k = threadIdx.x; k < kStemWPitch; k += blockDim.x) mx = fmaxf(mx, fabsf(val(k)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) mx = fmaxf(mx, red[i]);
  const int t = f16_pow2_exp(mx);
  if (threadIdx.x == 0) {
    wsi[n] = ldexpf(1.f, -t);
    bias[n] = s.bn_weight ? (float)((double)s.bn_bias[n] - (double)s.bn_mean[n] * sc) : 0.f;
  }
  const float up = ldexpf(1.f, t);
  for (int k = threadIdx.x; k < kStemWPitch; k += blockDim.x) {
    const float X = val(k) * up;
    const __half h = __float2half_rn(X);
    w_hi[n * kStemWPitch + k] = h;
    w_lo[n * kStemWPitch + k] = __float2half_rn((X - __half2float(h)) * 2048.f);
  }
}

__device__ __forceinline__ void mma_f16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// grid (conv rows / 8, images); each CTA walks the W/32 column tiles of its row band.
// kTrain = false (inference): + bias, ReLU, fp32 NHWC output + amax.  kTrain = true (stem_conv training forward): x is
// encoded times the power-of-two tensor scale of its exact amax (x_slot[0]), exactly as stem_x_planes_kernel writes the
// saved planes, and the raw conv (no bias, no ReLU, the scale undone) is written as fp32 NCHW, the layout
// batch_norm_train reads; bias and amax_out are unused.
template <bool kU8, bool kTrain = false>
__global__ void __launch_bounds__(256, 2)
stem_conv_f16x2_kernel(const void* __restrict__ xin, int H, int W, const StemNorm nrm, const __half* __restrict__ wpk_hi,
                       const __half* __restrict__ wpk_lo, const float* __restrict__ wsi, const float* __restrict__ bias,
                       float* __restrict__ out, float* __restrict__ amax_out, const float* __restrict__ x_slot) {
  static_assert(!(kU8 && kTrain), "the training stem reads fp32 images");
  extern __shared__ __align__(16) unsigned char smem_h[];
  __half* s_wh = reinterpret_cast<__half*>(smem_h);                 // [64][168]
  __half* s_wl = s_wh + kStemCo * kStemWPitch;
  __half* s_ph = s_wl + kStemCo * kStemWPitch;                      // [21][112]
  __half* s_pl = s_ph + kPatchH * kP16Pitch;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int img = blockIdx.y, oy0 = blockIdx.x * kTileH;
  const int Ho = H >> 1, Wo = W >> 1;
  for (int i = threadIdx.x; i < kStemCo * kStemWPitch / 8; i += 256) {
    reinterpret_cast<uint4*>(s_wh)[i] = __ldg(reinterpret_cast<const uint4*>(wpk_hi) + i);
    reinterpret_cast<uint4*>(s_wl)[i] = __ldg(reinterpret_cast<const uint4*>(wpk_lo) + i);
  }
  float bv[8][2], sv[8][2];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if constexpr (!kTrain) {
      bv[nt][0] = __ldg(bias + nt * 8 + 2 * t);
      bv[nt][1] = __ldg(bias + nt * 8 + 2 * t + 1);
    }
    sv[nt][0] = __ldg(wsi + nt * 8 + 2 * t);
    sv[nt][1] = __ldg(wsi + nt * 8 + 2 * t + 1);
  }
  float xs = 1.f, xs_inv = 1.f;                      // training: x's tensor scale and its inverse (powers of two)
  if constexpr (kTrain) {
    xs = f16_pow2_scale(__ldcg(x_slot));
    xs_inv = 1.f / xs;
  }
  int koff[kStemK / 16][2];
#pragma unroll
  for (int s = 0; s < kStemK / 16; ++s) {
#pragma unroll
    for (int hk = 0; hk < 2; ++hk) {
      const int k = 16 * s + 8 * hk + 2 * t;
      const int ky = k / kStemRow, r = k - ky * kStemRow;
      koff[s][hk] = ky < kStemKy ? ky * kP16Pitch + r : 0;         // padded k: weight is zero, any address does
    }
  }
  const float* xi = reinterpret_cast<const float*>(xin) + (size_t)img * 3 * H * W;
  const uint8_t* xu = reinterpret_cast<const uint8_t*>(xin) + (size_t)img * 3 * H * W;
  float mx = 0.f;
  for (int ox0 = 0; ox0 < Wo; ox0 += kT16W) {
    __syncthreads();                                   // previous pass done with the patch (and the weights visible)
    const int iy0 = 2 * oy0 - 3, ix0 = 2 * ox0 - 3;
    for (int i = threadIdx.x; i < kPatchH * 3 * kP16W; i += 256) {
      int row, e;
      float v = 0.f;
      if constexpr (!kU8) {
        const int col = i % kP16W, rc = i / kP16W;
        const int ci = rc % 3;
        row = rc / 3;
        e = col * 3 + ci;
        const int iy = iy0 + row, ix = ix0 + col;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(xi + ((size_t)ci * H + iy) * W + ix);
        if constexpr (kTrain) v *= xs;
      } else {
        e = i % (3 * kP16W);
        row = i / (3 * kP16W);
        const int col = e / 3, ci = e - col * 3;
        const int iy = iy0 + row, ix = ix0 + col;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {                // zero padding applies AFTER normalisation
          const float u = (float)__ldg(xu + ((size_t)iy * W + ix) * 3 + ci);
          v = __fdiv_rn(__fsub_rn(__fdiv_rn(u, 255.f), nrm.mean[ci]), nrm.std[ci]);
        }
      }
      const __half h = __float2half_rn(v);
      s_ph[row * kP16Pitch + e] = h;
      s_pl[row * kP16Pitch + e] = __float2half_rn((v - __half2float(h)) * 2048.f);
    }
    if (threadIdx.x < kPatchH) {
      s_ph[threadIdx.x * kP16Pitch + 111] = __float2half_rn(0.f);
      s_pl[threadIdx.x * kP16Pitch + 111] = __float2half_rn(0.f);
    }
    __syncthreads();
    float am[8][4], ac[8][4];                          // main (hi hi) and correction (hi lo + lo hi) accumulators
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) am[nt][e] = ac[nt][e] = 0.f;
    // this warp: conv row `warp` of the tile, columns {g, g + 8}
    const int base0 = (2 * warp) * kP16Pitch + 6 * g;
#pragma unroll
    for (int s = 0; s < kStemK / 16; ++s) {
      uint32_t ah[4], al[4];
      ah[0] = *reinterpret_cast<const uint32_t*>(s_ph + base0 + koff[s][0]);
      ah[1] = *reinterpret_cast<const uint32_t*>(s_ph + base0 + 48 + koff[s][0]);       // column g + 8
      ah[2] = *reinterpret_cast<const uint32_t*>(s_ph + base0 + koff[s][1]);
      ah[3] = *reinterpret_cast<const uint32_t*>(s_ph + base0 + 48 + koff[s][1]);
      al[0] = *reinterpret_cast<const uint32_t*>(s_pl + base0 + koff[s][0]);
      al[1] = *reinterpret_cast<const uint32_t*>(s_pl + base0 + 48 + koff[s][0]);
      al[2] = *reinterpret_cast<const uint32_t*>(s_pl + base0 + koff[s][1]);
      al[3] = *reinterpret_cast<const uint32_t*>(s_pl + base0 + 48 + koff[s][1]);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int wo = (nt * 8 + g) * kStemWPitch + 16 * s + 2 * t;
        const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(s_wh + wo), bh1 = *reinterpret_cast<const uint32_t*>(s_wh + wo + 8);
        const uint32_t bl0 = *reinterpret_cast<const uint32_t*>(s_wl + wo), bl1 = *reinterpret_cast<const uint32_t*>(s_wl + wo + 8);
        mma_f16_16816(am[nt], ah, bh0, bh1);
        mma_f16_16816(ac[nt], ah, bl0, bl1);
        mma_f16_16816(ac[nt], al, bh0, bh1);
      }
    }
    // (main + 2^-11 corr) * 2^-t + bias, ReLU, fp32 NHWC: pixel (oy0 + warp, ox0 + g [+8]), channels nt*8 + 2t, +1
    const int oy = oy0 + warp;
    if constexpr (kTrain) {
      // ((main + 2^-11 corr) * 2^-t) / s_x, fp32 NCHW: for one channel, lanes g = 0..7 store 8 consecutive pixels, so
      // every store fills whole 32-byte sectors.  The domain (n * Ho * Wo <= 2^22) keeps y below 2^28 elements.
      const int hw = Ho * Wo;
      int o = ((img * kStemCo + 2 * t) * Ho + oy) * Wo + ox0 + g;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt, o += 8 * hw) {
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
          for (int hr = 0; hr < 2; ++hr)
            out[o + e * hw + 8 * hr] = fmaf(ac[nt][2 * hr + e], 1.f / 2048.f, am[nt][2 * hr + e]) * sv[nt][e] * xs_inv;
      }
    } else if (oy < Ho) {
#pragma unroll
      for (int hr = 0; hr < 2; ++hr) {
        const int ox = ox0 + g + 8 * hr;
        if (ox < Wo) {
          float* o = out + (((size_t)img * Ho + oy) * Wo + ox) * kStemCo + 2 * t;
#pragma unroll
          for (int nt = 0; nt < 8; ++nt) {
            const float v0 = fmaxf(fmaf(fmaf(ac[nt][2 * hr], 1.f / 2048.f, am[nt][2 * hr]), sv[nt][0], bv[nt][0]), 0.f);
            const float v1 = fmaxf(fmaf(fmaf(ac[nt][2 * hr + 1], 1.f / 2048.f, am[nt][2 * hr + 1]), sv[nt][1], bv[nt][1]), 0.f);
            mx = fmaxf(mx, fmaxf(v0, v1));
            *reinterpret_cast<float2*>(o + nt * 8) = make_float2(v0, v1);
          }
        }
      }
    }
  }
  if constexpr (!kTrain) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) atomicMax(reinterpret_cast<unsigned int*>(amax_out), __float_as_uint(mx));   // mx >= 0
  }
}

// packed buffer of the fp32-accurate stem: [fp16 hi [64][168] | fp16 lo | wsi [64]]
constexpr size_t kStem16PlaneBytes = (size_t)kStemCo * kStemWPitch * sizeof(__half);             // 21504
int launch_pack_stem_f16x2(const CdrConvBn& s, void* w, float* bias, cudaStream_t st) {
  CDR_CHECK_ARG(s.weight && s.bn_weight && s.bn_bias && s.bn_mean && s.bn_var && w && bias, "pack_stem: bad args");
  uint8_t* b = reinterpret_cast<uint8_t*>(w);
  pack_stem_f16x2_kernel<<<kStemCo, 64, 0, st>>>(s, reinterpret_cast<__half*>(b), reinterpret_cast<__half*>(b + kStem16PlaneBytes),
                                                 reinterpret_cast<float*>(b + 2 * kStem16PlaneBytes), bias);
  CDR_LAUNCH_OK("pack_stem_f16x2_kernel");
  return CDR_OK;
}
size_t stem_weight_bytes_f16x2() { return 2 * kStem16PlaneBytes + kStemCo * sizeof(float); }

int launch_stem_f32(const void* x, int is_u8, const float* mean, const float* std, int n, int H, int W, const void* w,
                    const float* bias, float* conv_out, void* pooled_hi, void* pooled_lo, float* slot, cudaStream_t st) {
  CDR_CHECK_ARG(x && w && bias && conv_out && pooled_hi && pooled_lo && slot && n > 0, "stem: bad args");
  CDR_CHECK_ARG(!is_u8 || (mean && std), "stem: uint8 frames need mean / std");
  StemNorm nrm{};
  for (int c = 0; c < 3; ++c) {
    nrm.mean[c] = is_u8 ? mean[c] : 0.f;
    nrm.std[c] = is_u8 ? std[c] : 1.f;
  }
  CDR_CHECK_ARG(H % 16 == 0 && W % 64 == 0, "stem: image %dx%d must have H %% 16 == 0 and W %% 64 == 0", H, W);
  CDR_CHECK_ARG(((uintptr_t)conv_out & 15) == 0 && ((uintptr_t)pooled_hi & 15) == 0 && ((uintptr_t)pooled_lo & 15) == 0 &&
                    ((uintptr_t)w & 15) == 0, "stem: alignment");
  static DeviceOnce attr_set[2];
  const int Ho = H / 2, Wo = W / 2;
  const uint8_t* b = reinterpret_cast<const uint8_t*>(w);
  const __half* wh = reinterpret_cast<const __half*>(b);
  const __half* wl = reinterpret_cast<const __half*>(b + kStem16PlaneBytes);
  const float* wsi = reinterpret_cast<const float*>(b + 2 * kStem16PlaneBytes);
  if (is_u8) {
    if (attr_set[1].need()) {
      CDR_CUDA(cudaFuncSetAttribute(stem_conv_f16x2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kStem16SmemBytes));
      attr_set[1].done();
    }
    stem_conv_f16x2_kernel<true><<<dim3(Ho / kTileH, n), 256, kStem16SmemBytes, st>>>(x, H, W, nrm, wh, wl, wsi, bias, conv_out, slot,
                                                                                      nullptr);
  } else {
    if (attr_set[0].need()) {
      CDR_CUDA(cudaFuncSetAttribute(stem_conv_f16x2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kStem16SmemBytes));
      attr_set[0].done();
    }
    stem_conv_f16x2_kernel<false><<<dim3(Ho / kTileH, n), 256, kStem16SmemBytes, st>>>(x, H, W, nrm, wh, wl, wsi, bias, conv_out, slot,
                                                                                       nullptr);
  }
  CDR_LAUNCH_OK("stem_conv_f16x2_kernel");
  const long long total = (long long)n * (Ho / 2) * (Wo / 2) * (kStemCo / 8);
  maxpool3s2_f16p_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(
      conv_out, Ho, Wo, kStemCo / 8, total, (__half*)pooled_hi, (__half*)pooled_lo, slot);
  CDR_LAUNCH_OK("maxpool3s2_f16p_kernel");
  return CDR_OK;
}


// ------------------------------------------------------------------------------------------
// Training the stem (DESIGN.md §7): stem_conv = Conv2d(3, 64, 7, stride 2, padding 3, bias=False) forward and weight
// gradient at fp32 accuracy, and the 3x3 stride-2 pad-1 max-pool forward and backward on NCHW fp32.  No data gradient of
// the conv: its input is the image batch.
//   forward  x -> one power-of-two tensor scale from its exact amax -> the x planes (saved for the weight gradient) and
//            stem_conv_f16x2_kernel<false, true> on the weight packed per call (pack_stem_f16x2_kernel, no BN)
//   wgrad    dW[co][ci][ky][kx] = sum over pixels of dy[co][p] x[ci][tap(p, ky, kx)]: M = 64, N = 3 x 7 x 8 (kx padded
//            to 8), K = the n*Ho*Wo pixels in chunks of 2 output rows x 32 columns, split into K slices
//            (stem_train_slices) -> fp32 partials -> wgrad_reduce (fixed slice order: bitwise deterministic, no atomics)
// saved: [x hi planes | x lo planes | {amax, scale} of x], each 256-byte aligned, the planes in x's NCHW order.
// workspace: forward [packed weight | bias]; backward [{amax, scale} of dy | partials [slices][64][147]].
constexpr int kStemWgRows = 2, kStemWgCols = 32;      // a K chunk: 2 output rows x 32 output columns = 64 pixels
constexpr int kStemWgPatchRows = 2 * kStemWgRows + 5; // 9 input rows
constexpr int kStemWgPatchCols = 2 * kStemWgCols + 6; // 70 input columns: column 2j + kx of the patch, j < 32, kx < 8
constexpr int kStemWgKxPitch = 40;                    // one kx copy of a patch row: 32 halves + 8 (conflict-free B loads)
constexpr int kStemWgRowHalves = 8 * kStemWgKxPitch;  // a patch row as 8 kx copies: entry j of copy kx = column 2j + kx
constexpr int kStemWgDyPitch = 64 + 8;                // one output channel of a dy chunk: 64 pixels + 8 (ldmatrix rows)
constexpr int kStemWgThreads = 7 * 32;                // warp = ky: its 3 n-tiles are (ci, ky, kx = 0..7), ci = 0..2
constexpr int kStemWgDrain = 8;                       // chunks (512 pixels) between drains of the accumulators
constexpr int kStemWgXHalves = 2 * 3 * kStemWgPatchRows * kStemWgRowHalves;
constexpr int kStemWgDyHalves = 2 * kStemCo * kStemWgDyPitch;
constexpr int kStemWgSmemBytes = (kStemWgXHalves + kStemWgDyHalves) * (int)sizeof(__half) +
                                 kStemWgThreads * 48 * (int)sizeof(float);     // + every lane's 48 drained sums
constexpr int kStemWgTaps = 3 * 49;                   // dW row: (ci, ky, kx)
constexpr int kStemWgTargetSlices = 2 * 148;          // two CTAs per SM, one wave of a 148-SM B200

struct StemTrainPlan {
  long long x_elems;
  size_t plane_bytes, saved_bytes, ws_fwd, ws_bwd;
  int chunks, cps, slices;                            // wgrad: K chunks, chunks per slice, slices
};
// A function of the shape only, so the summation order of dW (and dW, bit for bit) does not depend on the device.
static StemTrainPlan stem_train_plan(int n, int H, int W) {
  StemTrainPlan p;
  p.x_elems = (long long)n * 3 * H * W;
  p.plane_bytes = round_up<size_t>((size_t)p.x_elems * sizeof(__half), 256);
  p.saved_bytes = 2 * p.plane_bytes + 256;
  p.ws_fwd = 2 * kStem16PlaneBytes + round_up<size_t>(kStemCo * sizeof(float), 256) + round_up<size_t>(kStemCo * sizeof(float), 256);
  p.chunks = n * (H / 2 / kStemWgRows) * (W / 2 / kStemWgCols);
  p.cps = ceil_div(p.chunks, kStemWgTargetSlices);
  p.slices = ceil_div(p.chunks, p.cps);
  p.ws_bwd = 256 + (size_t)p.slices * kStemCo * kStemWgTaps * sizeof(float);
  return p;
}
size_t stem_train_saved_bytes(int n, int H, int W) { return stem_train_plan(n, H, W).saved_bytes; }
size_t stem_train_workspace_bytes(int n, int H, int W) {
  const StemTrainPlan p = stem_train_plan(n, H, W);
  return p.ws_fwd > p.ws_bwd ? p.ws_fwd : p.ws_bwd;
}

__device__ __forceinline__ void f16_split(float X, __half& h, __half& l) {
  h = __float2half_rn(X);
  l = __float2half_rn((X - __half2float(h)) * 2048.f);
}

// x (NCHW fp32, x_elems a multiple of 4) -> scaled fp16 hi / lo planes in the same order; slot = {amax (complete), scale}
__global__ void __launch_bounds__(256)
stem_x_planes_kernel(const float4* __restrict__ x, long long n4, uint2* __restrict__ hi, uint2* __restrict__ lo,
                     float* __restrict__ slot) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const float s = f16_pow2_scale(__ldcg(slot));
  if (i == 0) slot[1] = s;
  if (i >= n4) return;
  const float4 v = __ldg(x + i);
  __align__(8) __half h[4], l[4];
  f16_split(v.x * s, h[0], l[0]);
  f16_split(v.y * s, h[1], l[1]);
  f16_split(v.z * s, h[2], l[2]);
  f16_split(v.w * s, h[3], l[3]);
  hi[i] = *reinterpret_cast<const uint2*>(h);
  lo[i] = *reinterpret_cast<const uint2*>(l);
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const __half* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
}

// grid = slices; CTA b sums chunks [b * cps, min((b + 1) * cps, chunks)) into part[b] (64 x 147, times s_x * s_dy).
// A = dy (64 channels x 16 pixels per k-step: ldmatrix from the [co][pixel] chunk), B = x (16 pixels x 8 kx of one
// (ci, ky): the pixel pair (k, k+1) of a fragment is columns 2ox + kx and 2ox + 2 + kx, adjacent in the patch row's kx
// copy).  fp16 products are exact; main and correction terms accumulate apart and are drained into fp32 sums in shared
// memory every kStemWgDrain chunks, so no accumulation chain grows with K.
__global__ void __launch_bounds__(kStemWgThreads, 2)
stem_wgrad_kernel(const __half* __restrict__ x_hi, const __half* __restrict__ x_lo, const float* __restrict__ dy, int H,
                  int W, int chunks, int cps, float* __restrict__ dy_slot, float* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char smem_wg[];
  __half* s_xh = reinterpret_cast<__half*>(smem_wg);                 // [ci][patch row][kx][kStemWgKxPitch]
  __half* s_xl = s_xh + kStemWgXHalves / 2;
  __half* s_dh = s_xh + kStemWgXHalves;                               // [co][kStemWgDyPitch]
  __half* s_dl = s_dh + kStemCo * kStemWgDyPitch;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int ky = warp;
  float* tot = reinterpret_cast<float*>(s_dh + kStemWgDyHalves) + warp * 48 * 32 + lane;   // this lane's sums, 32 apart
  const int Ho = H >> 1, Wo = W >> 1;
  const int cols_t = Wo / kStemWgCols, rows_t = Ho / kStemWgRows;
  const float sdy = f16_pow2_scale(__ldcg(dy_slot));
  if (blockIdx.x == 0 && threadIdx.x == 0) dy_slot[1] = sdy;
#pragma unroll
  for (int i = 0; i < 48; ++i) tot[i * 32] = 0.f;
  float am[4][3][4], ac[4][3][4];                    // [m-tile: 16 channels][ci][fragment]
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
      for (int e = 0; e < 4; ++e) am[mt][ci][e] = ac[mt][ci][e] = 0.f;
  const int c_end = min(chunks, (blockIdx.x + 1) * cps);
  int since = 0;
  for (int c = blockIdx.x * cps; c < c_end; ++c) {
    const int tx = c % cols_t, r = c / cols_t;
    const int oy0 = (r % rows_t) * kStemWgRows, ox0 = tx * kStemWgCols, img = r / rows_t;
    __syncthreads();                                 // the previous chunk's fragments are read
    // dy: 64 channels x 2 rows x 32 columns, scaled and split -> [co][row * 32 + column]
    for (int i = threadIdx.x; i < kStemCo * kStemWgRows * kStemWgCols / 4; i += kStemWgThreads) {
      const int q = i & 7, rr = (i >> 3) & 1, co = i >> 4;
      const float4 v = __ldg(reinterpret_cast<const float4*>(dy + (((size_t)img * kStemCo + co) * Ho + oy0 + rr) * Wo + ox0) + q);
      __align__(8) __half h[4], l[4];
      f16_split(v.x * sdy, h[0], l[0]);
      f16_split(v.y * sdy, h[1], l[1]);
      f16_split(v.z * sdy, h[2], l[2]);
      f16_split(v.w * sdy, h[3], l[3]);
      const int o = co * kStemWgDyPitch + rr * kStemWgCols + 4 * q;
      *reinterpret_cast<uint2*>(s_dh + o) = *reinterpret_cast<const uint2*>(h);
      *reinterpret_cast<uint2*>(s_dl + o) = *reinterpret_cast<const uint2*>(l);
    }
    // x: 3 channels x 9 input rows x 70 columns of both planes (zero outside the image), each value into the kx copies
    // that read it
    const int iy0 = 2 * oy0 - 3, ix0 = 2 * ox0 - 3;
    for (int i = threadIdx.x; i < 3 * kStemWgPatchRows * kStemWgPatchCols; i += kStemWgThreads) {
      const int col = i % kStemWgPatchCols, rc = i / kStemWgPatchCols;     // rc = ci * 9 + patch row
      const int iy = iy0 + rc % kStemWgPatchRows, ix = ix0 + col;
      __half h = __float2half_rn(0.f), l = h;
      if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
        const size_t o = (((size_t)img * 3 + rc / kStemWgPatchRows) * H + iy) * W + ix;
        h = __ldg(x_hi + o);
        l = __ldg(x_lo + o);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int kx = (col & 1) + 2 * k, j = (col - kx) >> 1;
        if (j >= 0 && j < kStemWgCols) {
          s_xh[rc * kStemWgRowHalves + kx * kStemWgKxPitch + j] = h;
          s_xl[rc * kStemWgRowHalves + kx * kStemWgKxPitch + j] = l;
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < kStemWgRows * kStemWgCols / 16; ++s) {      // k-step: output row s / 2, columns 16 (s % 2) + 0..15
      const int rr = s >> 1, j0 = 16 * (s & 1);
      uint32_t bh[3][2], bl[3][2];
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        const int o = (ci * kStemWgPatchRows + 2 * rr + ky) * kStemWgRowHalves + g * kStemWgKxPitch + j0 + 2 * t;
        bh[ci][0] = *reinterpret_cast<const uint32_t*>(s_xh + o);
        bh[ci][1] = *reinterpret_cast<const uint32_t*>(s_xh + o + 8);
        bl[ci][0] = *reinterpret_cast<const uint32_t*>(s_xl + o);
        bl[ci][1] = *reinterpret_cast<const uint32_t*>(s_xl + o + 8);
      }
      const int arow = (lane & 7) + ((lane >> 3) & 1) * 8, acol = rr * kStemWgCols + j0 + (lane >> 4) * 8;
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        uint32_t ah[4], al[4];
        ldsm_x4(ah, s_dh + (16 * mt + arow) * kStemWgDyPitch + acol);
        ldsm_x4(al, s_dl + (16 * mt + arow) * kStemWgDyPitch + acol);
#pragma unroll
        for (int ci = 0; ci < 3; ++ci) {
          mma_f16_16816(am[mt][ci], ah, bh[ci][0], bh[ci][1]);
          mma_f16_16816(ac[mt][ci], ah, bl[ci][0], bl[ci][1]);
          mma_f16_16816(ac[mt][ci], al, bh[ci][0], bh[ci][1]);
        }
      }
    }
    if (++since == kStemWgDrain || c + 1 == c_end) {
      since = 0;
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int ci = 0; ci < 3; ++ci)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            tot[((mt * 3 + ci) * 4 + e) * 32] += fmaf(ac[mt][ci][e], 1.f / 2048.f, am[mt][ci][e]);
            am[mt][ci][e] = ac[mt][ci][e] = 0.f;
          }
    }
  }
  // fragment e of (mt, ci): channel 16 mt + g (+8 for e >= 2), kx = 2t + (e & 1); kx = 7 is padding
  float* pp = part + (size_t)blockIdx.x * kStemCo * kStemWgTaps;
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int co = 16 * mt + g + 8 * (e >> 1), kx = 2 * t + (e & 1);
        if (kx < 7) pp[co * kStemWgTaps + ci * 49 + ky * 7 + kx] = tot[((mt * 3 + ci) * 4 + e) * 32];
      }
}

int stem_train_slices(int n, int H, int W) { return stem_train_plan(n, H, W).slices; }

int launch_stem_train_forward(const float* x, const float* weight, int n, int H, int W, float* y, void* saved,
                              void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const StemTrainPlan p = stem_train_plan(n, H, W);
  if (workspace_bytes < p.ws_fwd) {
    set_error("cdr_stem_train_forward: workspace %zu < required %zu bytes", workspace_bytes, p.ws_fwd);
    return CDR_ERR_WORKSPACE;
  }
  set_stage("stem_train_fwd");
  uint8_t* sv = reinterpret_cast<uint8_t*>(saved);
  __half* xh = reinterpret_cast<__half*>(sv);
  __half* xl = reinterpret_cast<__half*>(sv + p.plane_bytes);
  float* slot = reinterpret_cast<float*>(sv + 2 * p.plane_bytes);
  CDR_CUDA(cudaMemsetAsync(slot, 0, 2 * sizeof(float), st));
  if (int rc = launch_amax_f32(x, nullptr, p.x_elems, slot, st)) return rc;
  const long long n4 = p.x_elems / 4;
  stem_x_planes_kernel<<<(unsigned)ceil_div<long long>(n4, 256), 256, 0, st>>>(
      reinterpret_cast<const float4*>(x), n4, reinterpret_cast<uint2*>(xh), reinterpret_cast<uint2*>(xl), slot);
  CDR_LAUNCH_OK("stem_x_planes_kernel");
  uint8_t* b = reinterpret_cast<uint8_t*>(workspace);
  float* bias = reinterpret_cast<float*>(b + p.ws_fwd - round_up<size_t>(kStemCo * sizeof(float), 256));
  CdrConvBn cb{};
  cb.weight = weight;
  pack_stem_f16x2_kernel<<<kStemCo, 64, 0, st>>>(cb, reinterpret_cast<__half*>(b), reinterpret_cast<__half*>(b + kStem16PlaneBytes),
                                                  reinterpret_cast<float*>(b + 2 * kStem16PlaneBytes), bias);
  CDR_LAUNCH_OK("pack_stem_f16x2_kernel");
  static DeviceOnce attr_set;
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(stem_conv_f16x2_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kStem16SmemBytes));
    attr_set.done();
  }
  stem_conv_f16x2_kernel<false, true><<<dim3(H / 2 / kTileH, n), 256, kStem16SmemBytes, st>>>(
      x, H, W, StemNorm{}, reinterpret_cast<const __half*>(b), reinterpret_cast<const __half*>(b + kStem16PlaneBytes),
      reinterpret_cast<const float*>(b + 2 * kStem16PlaneBytes), nullptr, y, nullptr, slot);
  CDR_LAUNCH_OK("stem_conv_f16x2_kernel");
  set_stage(nullptr);
  return CDR_OK;
}

int launch_stem_train_backward(const void* saved, const float* dy, int n, int H, int W, float* dweight, void* workspace,
                               size_t workspace_bytes, cudaStream_t st) {
  const StemTrainPlan p = stem_train_plan(n, H, W);
  if (workspace_bytes < p.ws_bwd) {
    set_error("cdr_stem_train_backward: workspace %zu < required %zu bytes", workspace_bytes, p.ws_bwd);
    return CDR_ERR_WORKSPACE;
  }
  if (!dweight) return CDR_OK;
  set_stage("stem_train_bwd");
  const uint8_t* sv = reinterpret_cast<const uint8_t*>(saved);
  const float* x_slot = reinterpret_cast<const float*>(sv + 2 * p.plane_bytes);
  float* dy_slot = reinterpret_cast<float*>(workspace);
  float* part = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + 256);
  CDR_CUDA(cudaMemsetAsync(dy_slot, 0, 2 * sizeof(float), st));
  if (int rc = launch_amax_f32(dy, nullptr, (long long)n * kStemCo * (H / 2) * (W / 2), dy_slot, st)) return rc;
  static DeviceOnce attr_set;
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(stem_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStemWgSmemBytes));
    attr_set.done();
  }
  stem_wgrad_kernel<<<p.slices, kStemWgThreads, kStemWgSmemBytes, st>>>(
      reinterpret_cast<const __half*>(sv), reinterpret_cast<const __half*>(sv + p.plane_bytes), dy, H, W, p.chunks, p.cps,
      dy_slot, part);
  CDR_LAUNCH_OK("stem_wgrad_kernel");
  if (int rc = launch_wgrad_reduce(part, p.slices, 1, kStemCo, kStemWgTaps, kStemWgTaps, x_slot + 1, dy_slot + 1, dweight, st))
    return rc;
  set_stage(nullptr);
  return CDR_OK;
}


// ---- max-pool 3x3 stride 2 pad 1 on NCHW fp32 with the selection rule of torch's CUDA NCHW kernel: the window is
// scanned in row-major order from its first in-image element, and an element replaces the maximum when it is larger or
// NaN (ties: the first maximum; a NaN window: its last NaN).  argmax keeps one byte per output, the window position
// ky * 3 + kx.  Each thread handles 4 consecutive outputs (forward) or inputs (backward) of one row; stores are 16-byte
// (4-byte for argmax) when the 4 elements are whole and aligned.
__global__ void __launch_bounds__(256)
maxpool3x3_train_fwd_kernel(const float* __restrict__ x, int H, int W, int Ho, int Wo, long long total,
                            float* __restrict__ y, uint8_t* __restrict__ argmax) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int wq = (Wo + 3) >> 2;
  const int q = (int)(idx % wq);
  const long long r = idx / wq;
  const int oy = (int)(r % Ho);
  const long long plane = r / Ho;
  const float* xp = x + plane * H * W;
  const int y0 = 2 * oy - 1, ya = max(y0, 0), yb = min(y0 + 2, H - 1);
  float m[4];
  uint8_t pos[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int ox = 4 * q + k, x0 = 2 * ox - 1, xa = max(x0, 0), xb = min(x0 + 2, W - 1);
    float mv = -INFINITY;
    int mp = (ya - y0) * 3 + (xa - x0);
    if (ox < Wo) {
      for (int iy = ya; iy <= yb; ++iy)
        for (int ix = xa; ix <= xb; ++ix) {
          const float v = __ldg(xp + (long long)iy * W + ix);
          if (v > mv || isnan(v)) {
            mv = v;
            mp = (iy - y0) * 3 + (ix - x0);
          }
        }
    }
    m[k] = mv;
    pos[k] = (uint8_t)mp;
  }
  const long long o = r * Wo + 4 * q;
  float* yo = y + o;
  uint8_t* ao = argmax + o;
  if (4 * q + 4 <= Wo && ((uintptr_t)yo & 15) == 0 && ((uintptr_t)ao & 3) == 0) {
    *reinterpret_cast<float4*>(yo) = make_float4(m[0], m[1], m[2], m[3]);
    *reinterpret_cast<uchar4*>(ao) = make_uchar4(pos[0], pos[1], pos[2], pos[3]);
  } else {
    for (int k = 0; k < 4 && 4 * q + k < Wo; ++k) {
      yo[k] = m[k];
      ao[k] = pos[k];
    }
  }
}

// dx[iy][ix] = the sum, from +0.0 and in (oy, ox) order, of dy over the (at most 4) windows whose argmax is (iy, ix):
// the order of torch's CUDA NCHW backward, so dx matches it bit for bit.  No atomics.
__global__ void __launch_bounds__(256)
maxpool3x3_train_bwd_kernel(const uint8_t* __restrict__ argmax, const float* __restrict__ dy, int H, int W, int Ho, int Wo,
                            long long total, float* __restrict__ dx) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int wq = (W + 3) >> 2;
  const int q = (int)(idx % wq);
  const long long r = idx / wq;
  const int iy = (int)(r % H);
  const long long plane = r / H;
  const uint8_t* ap = argmax + plane * Ho * Wo;
  const float* dp = dy + plane * Ho * Wo;
  const int oya = iy >> 1, oyb = min((iy + 1) >> 1, Ho - 1);
  float s[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int ix = 4 * q + k, oxa = ix >> 1, oxb = min((ix + 1) >> 1, Wo - 1);
    float acc = 0.f;
    if (ix < W) {
      for (int oy = oya; oy <= oyb; ++oy)
        for (int ox = oxa; ox <= oxb; ++ox) {
          const long long o = (long long)oy * Wo + ox;
          if (__ldg(ap + o) == (iy - 2 * oy + 1) * 3 + (ix - 2 * ox + 1)) acc += __ldg(dp + o);
        }
    }
    s[k] = acc;
  }
  float* xo = dx + r * W + 4 * q;
  if (4 * q + 4 <= W && ((uintptr_t)xo & 15) == 0) {
    *reinterpret_cast<float4*>(xo) = make_float4(s[0], s[1], s[2], s[3]);
  } else {
    for (int k = 0; k < 4 && 4 * q + k < W; ++k) xo[k] = s[k];
  }
}

int launch_maxpool3x3_train_forward(const float* x, int n, int c, int H, int W, float* y, uint8_t* argmax, cudaStream_t st) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long total = (long long)n * c * Ho * ((Wo + 3) / 4);
  maxpool3x3_train_fwd_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(x, H, W, Ho, Wo, total, y, argmax);
  CDR_LAUNCH_OK("maxpool3x3_train_fwd_kernel");
  return CDR_OK;
}
int launch_maxpool3x3_train_backward(const uint8_t* argmax, const float* dy, int n, int c, int H, int W, float* dx,
                                     cudaStream_t st) {
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const long long total = (long long)n * c * H * ((W + 3) / 4);
  maxpool3x3_train_bwd_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(argmax, dy, H, W, Ho, Wo, total, dx);
  CDR_LAUNCH_OK("maxpool3x3_train_bwd_kernel");
  return CDR_OK;
}

}  // namespace cdr
