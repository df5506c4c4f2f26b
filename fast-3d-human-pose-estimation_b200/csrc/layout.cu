// Layout kernels: NCHW -> pixel-major rows, and the feature transform layer (FTL).
// Both are pure data movement / AXPY work: HBM-bound, coalesced 128-byte accesses.
#include <cuda_fp16.h>
#include <initializer_list>

#include "kernels.h"

namespace cdr {

// (n_img, C, HW) fp32  ->  (n_img*HW, out_pitch) rows of C channels.  One 32-channel x
// 64-pixel tile per block through padded shared memory so that both the reads (along
// pixels) and the writes (along channels) are full 128-byte lines.
template <typename TOut>
__global__ void __launch_bounds__(256)
nchw_to_rows_kernel(const float* __restrict__ in, const float* __restrict__ in2, int n_first, int C, int HW,
                    TOut* __restrict__ out, int out_pitch) {
  __shared__ float tile[32][65];
  const int c0 = blockIdx.x * 32, p0 = blockIdx.y * 64, img = blockIdx.z;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const float* base = img < n_first ? in + (size_t)img * C * HW : in2 + (size_t)(img - n_first) * C * HW;
  for (int c = ty; c < 32; c += 8) {
    const float* src = base + (size_t)(c0 + c) * HW + p0;
    if (c0 + c < C) {
      if (p0 + tx < HW) tile[c][tx] = src[tx];
      if (p0 + tx + 32 < HW) tile[c][tx + 32] = src[tx + 32];
    }
  }
  __syncthreads();
  if (c0 + tx < C) {
    for (int pp = ty; pp < 64; pp += 8) {
      if (p0 + pp < HW)
        out[((size_t)img * HW + p0 + pp) * out_pitch + c0 + tx] = (TOut)tile[tx][pp];
    }
  }
}

// 16-bit outputs, fast path (C % 64 == 0, HW % 64 == 0): 64-channel x 64-pixel tiles, float2 loads along
// pixels, one packed pair of channels (4 bytes) per lane on the way out, so a warp writes a full 128-byte
// line per instruction.  kF16P: scaled fp16 hi/lo planes (scale from *amax, gemm_tc.cu: kFmtF16P).
template <bool kF16P>
__global__ void __launch_bounds__(256)
nchw_to_rows16_kernel(const float* __restrict__ in, const float* __restrict__ in2, int n_first, int C, int HW,
                      void* __restrict__ out_hi, void* __restrict__ out_lo, int out_pitch,
                      const float* __restrict__ amax, float* __restrict__ scale_out) {
  __shared__ float tile[64][65];
  float s = 1.f;
  if constexpr (kF16P) {
    const float a = __ldg(amax);
    s = f16_pow2_scale(a);
    if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) *scale_out = s;
  }
  const int c0 = blockIdx.x * 64, p0 = blockIdx.y * 64, img = blockIdx.z;
  const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* base = img < n_first ? in + (size_t)img * C * HW : in2 + (size_t)(img - n_first) * C * HW;
  {   // all 8 loads of a thread are issued before the first dependent store (one load in flight per thread caps
      // the kernel at ~2.5 TB/s: 2048 threads x 8 B per SM against ~1 us of DRAM latency)
    float2 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      v[i] = __ldg(reinterpret_cast<const float2*>(base + (size_t)(c0 + ty + 8 * i) * HW + p0) + lane);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      tile[ty + 8 * i][2 * lane] = v[i].x;
      tile[ty + 8 * i][2 * lane + 1] = v[i].y;
    }
  }
  __syncthreads();
  for (int pp = ty; pp < 64; pp += 8) {
    const float x0 = tile[2 * lane][pp] * s, x1 = tile[2 * lane + 1][pp] * s;
    const size_t o = ((size_t)img * HW + p0 + pp) * out_pitch + c0 + 2 * lane;
    if constexpr (kF16P) {
      const __half2 h = __floats2half2_rn(x0, x1);
      const float2 hf = __half22float2(h);
      *reinterpret_cast<__half2*>(reinterpret_cast<__half*>(out_hi) + o) = h;
      *reinterpret_cast<__half2*>(reinterpret_cast<__half*>(out_lo) + o) =
          __floats2half2_rn((x0 - hf.x) * 2048.f, (x1 - hf.y) * 2048.f);
    } else {
      *reinterpret_cast<__nv_bfloat162*>(reinterpret_cast<__nv_bfloat16*>(out_hi) + o) = __floats2bfloat162_rn(x0, x1);
    }
  }
}

// in2 (optional): a second (n_img, C, HW) tensor whose rows follow the first one's in `out`
template <typename TOut>
static int launch_nchw_to_rows(const float* in, const float* in2, int n_img, int C, int HW, TOut* out, int out_pitch,
                               cudaStream_t st) {
  CDR_CHECK_ARG(in && out && n_img > 0 && C > 0 && HW > 0 && out_pitch >= C, "nchw_to_rows: bad args");
  dim3 grid(ceil_div(C, 32), ceil_div(HW, 64), in2 ? 2 * n_img : n_img);
  nchw_to_rows_kernel<TOut><<<grid, 256, 0, st>>>(in, in2, n_img, C, HW, out, out_pitch);
  CDR_LAUNCH_OK("nchw_to_rows_kernel");
  return CDR_OK;
}
int launch_nchw_to_rows_f32(const float* in, const float* in2, int n_img, int C, int HW, float* out, int out_pitch,
                            cudaStream_t st) {
  return launch_nchw_to_rows<float>(in, in2, n_img, C, HW, out, out_pitch, st);
}
int launch_nchw_to_rows_bf16(const float* in, const float* in2, int n_img, int C, int HW, __nv_bfloat16* out,
                             int out_pitch, cudaStream_t st) {
  if (C % 64 == 0 && HW % 64 == 0 && out_pitch == C && ((uintptr_t)in & 7) == 0 && (!in2 || ((uintptr_t)in2 & 7) == 0)) {
    CDR_CHECK_ARG(in && out && n_img > 0 && out_pitch >= C, "nchw_to_rows: bad args");
    dim3 grid(C / 64, HW / 64, in2 ? 2 * n_img : n_img);
    nchw_to_rows16_kernel<false><<<grid, 256, 0, st>>>(in, in2, n_img, C, HW, out, nullptr, out_pitch, nullptr, nullptr);
    CDR_LAUNCH_OK("nchw_to_rows16_kernel");
    return CDR_OK;
  }
  return launch_nchw_to_rows<__nv_bfloat16>(in, in2, n_img, C, HW, out, out_pitch, st);
}

// split-plane variant for the 3xTF32 path (common.cuh: split_tf32)
__global__ void __launch_bounds__(256)
nchw_to_rows_split_kernel(const float* __restrict__ in, const float* __restrict__ in2, int n_first, int C, int HW,
                          float* __restrict__ out_hi, float* __restrict__ out_lo, int out_pitch) {
  __shared__ float tile[32][65];
  const int c0 = blockIdx.x * 32, p0 = blockIdx.y * 64, img = blockIdx.z;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* base = img < n_first ? in + (size_t)img * C * HW : in2 + (size_t)(img - n_first) * C * HW;
  for (int c = ty; c < 32; c += 8) {
    const float* src = base + (size_t)(c0 + c) * HW + p0;
    if (c0 + c < C) {
      if (p0 + tx < HW) tile[c][tx] = src[tx];
      if (p0 + tx + 32 < HW) tile[c][tx + 32] = src[tx + 32];
    }
  }
  __syncthreads();
  if (c0 + tx < C) {
    for (int pp = ty; pp < 64; pp += 8) {
      if (p0 + pp < HW) {
        const float v = tile[tx][pp];
        float hi, lo;
        split_tf32(v, hi, lo);
        const size_t o = ((size_t)img * HW + p0 + pp) * out_pitch + c0 + tx;
        out_hi[o] = hi;
        out_lo[o] = lo;
      }
    }
  }
}
int launch_nchw_to_rows_split(const float* in, const float* in2, int n_img, int C, int HW, float* out_hi, float* out_lo,
                              int out_pitch, cudaStream_t st) {
  CDR_CHECK_ARG(in && out_hi && out_lo && n_img > 0 && C > 0 && HW > 0 && out_pitch >= C, "nchw_to_rows_split: bad args");
  dim3 grid(ceil_div(C, 32), ceil_div(HW, 64), in2 ? 2 * n_img : n_img);
  nchw_to_rows_split_kernel<<<grid, 256, 0, st>>>(in, in2, n_img, C, HW, out_hi, out_lo, out_pitch);
  CDR_LAUNCH_OK("nchw_to_rows_split_kernel");
  return CDR_OK;
}

// max |x| over a flat fp32 array -> atomicMax into *amax (pre-zeroed; non-negative floats order
// like their bit patterns)
__global__ void __launch_bounds__(256)
amax_f32_kernel(const float* __restrict__ in_a, const float* __restrict__ in_b, long long n, float* __restrict__ amax) {
  const float* __restrict__ in = blockIdx.y == 0 ? in_a : in_b;     // grid.y = number of tensors (1 or 2)
  float m = 0.f;
  const long long n4 = n >> 2;
  const float4* in4 = reinterpret_cast<const float4*>(in);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(in4 + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(in[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(amax), __float_as_uint(m));
}
int launch_amax_f32(const float* in, const float* in2, long long n, float* amax, cudaStream_t st) {
  CDR_CHECK_ARG(in && amax && n > 0 && ((uintptr_t)in & 15) == 0 && ((uintptr_t)in2 & 15) == 0, "amax_f32: bad args");
  const long long want = ceil_div<long long>(n >> 2, 256 * 4);
  const unsigned gx = (unsigned)(want < 1 ? 1 : want > 4 * num_sms() ? 4 * num_sms() : want);
  amax_f32_kernel<<<dim3(gx, in2 ? 2 : 1), 256, 0, st>>>(in, in2, n, amax);
  CDR_LAUNCH_OK("amax_f32_kernel");
  return CDR_OK;
}

// scaled fp16 hi/lo planes (gemm_tc.cu: kFmtF16P): X = x * s with s = 2^(13 - ilogb(amax)) (common.cuh: f16_pow2_scale),
// hi = rn_f16(X), lo = rn_f16((X - hi) * 2^11); block (0,0,0) publishes s.  Columns [C, out_pitch) of every row are
// written as zeros: a padded K pitch reaches the GEMM, and stale bytes there could be NaN (NaN * 0 poisons the sum).
__global__ void __launch_bounds__(256)
nchw_to_rows_f16p_kernel(const float* __restrict__ in, const float* __restrict__ in2, int n_first, int C, int HW,
                         __half* __restrict__ out_hi, __half* __restrict__ out_lo, int out_pitch,
                         const float* __restrict__ amax, float* __restrict__ scale_out) {
  __shared__ float tile[32][65];
  const float a = __ldg(amax);
  const float s = f16_pow2_scale(a);
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) *scale_out = s;
  const int c0 = blockIdx.x * 32, p0 = blockIdx.y * 64, img = blockIdx.z;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* base = img < n_first ? in + (size_t)img * C * HW : in2 + (size_t)(img - n_first) * C * HW;
  for (int c = ty; c < 32; c += 8) {
    const float* src = base + (size_t)(c0 + c) * HW + p0;
    if (c0 + c < C) {
      if (p0 + tx < HW) tile[c][tx] = src[tx];
      if (p0 + tx + 32 < HW) tile[c][tx + 32] = src[tx + 32];
    }
  }
  __syncthreads();
  if (c0 + tx < out_pitch) {
    const bool pad = c0 + tx >= C;
    for (int pp = ty; pp < 64; pp += 8) {
      if (p0 + pp < HW) {
        const float X = pad ? 0.f : tile[tx][pp] * s;
        const __half h = __float2half_rn(X);
        const size_t o = ((size_t)img * HW + p0 + pp) * out_pitch + c0 + tx;
        out_hi[o] = h;
        out_lo[o] = __float2half_rn((X - __half2float(h)) * 2048.f);
      }
    }
  }
}
int launch_nchw_to_rows_f16p(const float* in, const float* in2, int n_img, int C, int HW, void* out_hi, void* out_lo,
                             int out_pitch, const float* amax, float* scale_out, cudaStream_t st) {
  CDR_CHECK_ARG(in && out_hi && out_lo && amax && scale_out && n_img > 0 && C > 0 && HW > 0 && out_pitch >= C,
                "nchw_to_rows_f16p: bad args");
  if (C % 64 == 0 && HW % 64 == 0 && out_pitch == C && ((uintptr_t)in & 7) == 0 && (!in2 || ((uintptr_t)in2 & 7) == 0)) {
    dim3 grid16(C / 64, HW / 64, in2 ? 2 * n_img : n_img);
    nchw_to_rows16_kernel<true><<<grid16, 256, 0, st>>>(in, in2, n_img, C, HW, out_hi, out_lo, out_pitch, amax, scale_out);
    CDR_LAUNCH_OK("nchw_to_rows16_kernel");
    return CDR_OK;
  }
  dim3 grid(ceil_div(out_pitch, 32), ceil_div(HW, 64), in2 ? 2 * n_img : n_img);
  nchw_to_rows_f16p_kernel<<<grid, 256, 0, st>>>(in, in2, n_img, C, HW, (__half*)out_hi, (__half*)out_lo, out_pitch, amax,
                                                 scale_out);
  CDR_LAUNCH_OK("nchw_to_rows_f16p_kernel");
  return CDR_OK;
}

// One launch instead of {amax pass, transposition}: per-ROW scales.  A scale that multiplies a whole A row factors
// out of the GEMM, so every pixel may carry its own s = 2^(13 - ilogb(max_c |x[c, px]|)) (tighter than one tensor
// scale, and no global reduction before the first store).  A cluster of 8 CTAs owns one image (HW = 64 pixels): each
// CTA reduces |x| over its share of the channels, the partial maxima meet through distributed shared memory,
// then each CTA transposes its share again (the re-read hits L2) and stores the scaled fp16 hi/lo planes.
// row_scale[img*64 + px] = s; *amax_out (optional, pre-zeroed) = max |x| of the whole tensor.
constexpr int kRsCluster = 8;     // CTAs per image
__device__ __forceinline__ unsigned int ld_cluster_u32(const unsigned int* local, unsigned int rank) {
  unsigned int a = (unsigned int)__cvta_generic_to_shared(local), r, v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(r) : "memory");
  return v;
}
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__global__ void __cluster_dims__(kRsCluster, 1, 1) __launch_bounds__(256)
nchw_to_rows_f16p_rowscale_kernel(const float* __restrict__ in, const float* __restrict__ in2, int n_first, int C,
                                  __half* __restrict__ out_hi, __half* __restrict__ out_lo, int out_pitch,
                                  float* __restrict__ row_scale, float* __restrict__ amax_out) {
  constexpr int HW = 64;
  __shared__ unsigned int smax[HW];
  __shared__ float sscale[HW];
  __shared__ float tile[64][65];
  const int quarter = blockIdx.x, img = blockIdx.y;
  const int cq = C / kRsCluster, c_begin = quarter * cq;
  const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* base = (img < n_first ? in + (size_t)img * C * HW : in2 + (size_t)(img - n_first) * C * HW) +
                      (size_t)c_begin * HW;
  if (threadIdx.x < HW) smax[threadIdx.x] = 0u;
  __syncthreads();
  {   // pass 1: this thread always sees pixels 4*px4 .. 4*px4+3 (256 threads = 16 channels x 16 float4 per sweep)
    const int px4 = threadIdx.x & 15, cl = threadIdx.x >> 4;
    float m[4] = {0.f, 0.f, 0.f, 0.f};
    for (int cb = cl; cb < cq; cb += 128) {          // cq % 64 == 0 and 128 = 8 sweeps: batches of 8 (or 4) loads in flight
      float4 v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
        v[i] = cb + 16 * i < cq ? __ldg(reinterpret_cast<const float4*>(base + (size_t)(cb + 16 * i) * HW) + px4)
                                : float4{0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        m[0] = fmaxf(m[0], fabsf(v[i].x)); m[1] = fmaxf(m[1], fabsf(v[i].y));
        m[2] = fmaxf(m[2], fabsf(v[i].z)); m[3] = fmaxf(m[3], fabsf(v[i].w));
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      m[j] = fmaxf(m[j], __shfl_xor_sync(0xffffffffu, m[j], 16));
      if (lane < 16) atomicMax(&smax[4 * px4 + j], __float_as_uint(m[j]));     // non-negative floats order like uints
    }
  }
  cluster_barrier();
  if (threadIdx.x < HW) {
    unsigned int mx = 0u;
#pragma unroll
    for (unsigned int r = 0; r < kRsCluster; ++r) {
      const unsigned int v = ld_cluster_u32(&smax[threadIdx.x], r);
      mx = v > mx ? v : mx;
    }
    const float a = __uint_as_float(mx);
    const float s = f16_pow2_scale(a);
    sscale[threadIdx.x] = s;
    if (quarter == 0) {
      row_scale[(size_t)img * HW + threadIdx.x] = s;
      if (amax_out) {
        float w = a;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) w = fmaxf(w, __shfl_xor_sync(0xffffffffu, w, o));
        if (lane == 0) atomicMax(reinterpret_cast<unsigned int*>(amax_out), __float_as_uint(w));
      }
    }
  }
  cluster_barrier();     // the peers have read smax (it may die with this CTA), sscale is visible to the block
  // pass 2: 64-channel x 64-pixel tiles as nchw_to_rows16_kernel; the next tile's loads are in flight while this one
  // is transposed and stored
  float2 v[8];
  auto load_tile = [&](int c0) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      v[i] = __ldg(reinterpret_cast<const float2*>(base + (size_t)(c0 + ty + 8 * i) * HW) + lane);
  };
  load_tile(0);
  for (int c0 = 0; c0 < cq; c0 += 64) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      tile[ty + 8 * i][2 * lane] = v[i].x;
      tile[ty + 8 * i][2 * lane + 1] = v[i].y;
    }
    __syncthreads();
    if (c0 + 64 < cq) load_tile(c0 + 64);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int pp = ty + 8 * i;
      const float s = sscale[pp];
      const float x0 = tile[2 * lane][pp] * s, x1 = tile[2 * lane + 1][pp] * s;
      const size_t o = ((size_t)img * HW + pp) * out_pitch + c_begin + c0 + 2 * lane;
      const __half2 h = __floats2half2_rn(x0, x1);
      const float2 hf = __half22float2(h);
      *reinterpret_cast<__half2*>(out_hi + o) = h;
      *reinterpret_cast<__half2*>(out_lo + o) = __floats2half2_rn((x0 - hf.x) * 2048.f, (x1 - hf.y) * 2048.f);
    }
    __syncthreads();
  }
}
// true: the one-launch per-row-scale form covers this shape (the caller falls back to amax + tensor scale otherwise)
bool nchw_rowscale_ok(const float* in, const float* in2, int n_img, int C, int HW, int out_pitch) {
  return (in2 ? 2 * n_img : n_img) <= 65535 && HW == 64 && C % (64 * kRsCluster) == 0 && out_pitch % 2 == 0 && ((uintptr_t)in & 15) == 0 && (!in2 || ((uintptr_t)in2 & 15) == 0);
}
int launch_nchw_to_rows_f16p_rowscale(const float* in, const float* in2, int n_img, int C, int HW, void* out_hi,
                                      void* out_lo, int out_pitch, float* row_scale, float* amax_out, cudaStream_t st) {
  CDR_CHECK_ARG(in && out_hi && out_lo && row_scale && n_img > 0 && out_pitch >= C && nchw_rowscale_ok(in, in2, n_img, C, HW, out_pitch),
                "nchw_to_rows_f16p_rowscale: bad args");
  dim3 grid(kRsCluster, in2 ? 2 * n_img : n_img);
  nchw_to_rows_f16p_rowscale_kernel<<<grid, 256, 0, st>>>(in, in2, n_img, C, (__half*)out_hi, (__half*)out_lo, out_pitch,
                                                          row_scale, amax_out);
  CDR_LAUNCH_OK("nchw_to_rows_f16p_rowscale_kernel");
  return CDR_OK;
}

// FTL (models/cdrnet.py:45-56) on pixel-major rows.  With z.reshape(b, N, -1) the k-th
// "coordinate" of channel c is channel k*blk + c of the same pixel (SURVEY.md A.2), so
//   out[row, r*blk + c] = sum_k mats[img(row)][r][k] * in[row, k*blk + c].
// One thread per (row, c); consecutive threads walk consecutive channels.
// Both views in one launch: blockIdx.y = view picks (in, mats, out) from FtlViews.
template <typename T>
struct FtlViews {
  const T* in[2];
  const T* in_lo[2];
  const float* mats[2];
  T* out[2];
  T* out_lo[2];
};
template <typename T, int ROWS, int COLS>
__global__ void __launch_bounds__(256)
ftl_kernel(const FtlViews<T> fv, int in_pitch, int blk, long long total, int hw, int out_pitch, int out_fill) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int view = blockIdx.y;
  const T* __restrict__ in = fv.in[view];
  const float* __restrict__ mats = fv.mats[view];
  T* __restrict__ out = fv.out[view];
  const long long row = idx / blk;
  const int c = (int)(idx - row * blk);
  const float* m = mats + (row / hw) * (ROWS * COLS);
  float x[COLS];
#pragma unroll
  for (int k = 0; k < COLS; ++k) x[k] = (float)in[row * in_pitch + k * blk + c];
  T* o = out + row * out_pitch;
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < COLS; ++k) acc = fmaf(__ldg(m + r * COLS + k), x[k], acc);
    o[r * blk + c] = (T)acc;
  }
  if (c < out_fill - ROWS * blk) o[ROWS * blk + c] = (T)0.f;  // zero the pad columns
}

// 128-bit form of the two FTL kernels (blk, pitches and pad all multiples of 4 channels, 16-byte aligned
// planes — the head's 100-channel blocks at pitch 304 / 400 / 800): one thread per (row, 4 channels), so a
// warp reads and writes whole 128-byte lines (fp32) and issues a quarter of the memory instructions.
struct Vec4 { float v[4]; };
__device__ __forceinline__ Vec4 ld4(const float* p) {
  const float4 q = __ldg(reinterpret_cast<const float4*>(p));
  return Vec4{{q.x, q.y, q.z, q.w}};
}
__device__ __forceinline__ Vec4 ld4(const __nv_bfloat16* p) {
  const uint2 q = __ldg(reinterpret_cast<const uint2*>(p));
  return Vec4{{__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xffff0000u), __uint_as_float(q.y << 16),
               __uint_as_float(q.y & 0xffff0000u)}};
}
__device__ __forceinline__ void st4(float* p, const Vec4& a) {
  *reinterpret_cast<float4*>(p) = make_float4(a.v[0], a.v[1], a.v[2], a.v[3]);
}
__device__ __forceinline__ void st4(__nv_bfloat16* p, const Vec4& a) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(a.v[0], a.v[1]), hi = __floats2bfloat162_rn(a.v[2], a.v[3]);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}

template <typename T, int ROWS, int COLS>
__global__ void __launch_bounds__(256)
ftl_vec_kernel(const FtlViews<T> fv, int in_pitch, int blk, long long total4, int hw, int out_pitch, int out_fill) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total4) return;
  const bool v1 = blockIdx.y != 0;   // select, not index: a dynamically indexed __grid_constant__ struct is copied to local memory
  const int blk4 = blk >> 2;
  const long long row = idx / blk4;
  const int c = (int)(idx - row * blk4) << 2;
  const float* m = (v1 ? fv.mats[1] : fv.mats[0]) + (row / hw) * (ROWS * COLS);
  const T* __restrict__ in = (v1 ? fv.in[1] : fv.in[0]) + row * in_pitch + c;
  Vec4 x[COLS];
#pragma unroll
  for (int k = 0; k < COLS; ++k) x[k] = ld4(in + k * blk);
  T* __restrict__ o = (v1 ? fv.out[1] : fv.out[0]) + row * out_pitch + c;
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    Vec4 acc{{0.f, 0.f, 0.f, 0.f}};
#pragma unroll
    for (int k = 0; k < COLS; ++k) {
      const float mk = __ldg(m + r * COLS + k);
#pragma unroll
      for (int e = 0; e < 4; ++e) acc.v[e] = fmaf(mk, x[k].v[e], acc.v[e]);
    }
    st4(o + r * blk, acc);
  }
  if (c < out_fill - ROWS * blk) st4(o + ROWS * blk, Vec4{{0.f, 0.f, 0.f, 0.f}});   // zero the pad columns
}

template <int ROWS, int COLS>
__global__ void __launch_bounds__(256)
ftl_split_vec_kernel(const FtlViews<float> fv, int in_pitch, int blk, long long total4, int hw, int out_pitch,
                     int out_fill) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool v1 = blockIdx.y != 0;   // select, not index: a dynamically indexed __grid_constant__ struct is copied to local memory
  if (idx < total4) {
    const int blk4 = blk >> 2;
    const long long row = idx / blk4;
    const int c = (int)(idx - row * blk4) << 2;
    const float* m = (v1 ? fv.mats[1] : fv.mats[0]) + (row / hw) * (ROWS * COLS);
    const long long i0 = row * in_pitch + c;
    Vec4 x[COLS];
#pragma unroll
    for (int k = 0; k < COLS; ++k) {
      const Vec4 h = ld4((v1 ? fv.in[1] : fv.in[0]) + i0 + k * blk), l = ld4((v1 ? fv.in_lo[1] : fv.in_lo[0]) + i0 + k * blk);
#pragma unroll
      for (int e = 0; e < 4; ++e) x[k].v[e] = h.v[e] + l.v[e];     // exact: hi + lo reconstructs the fp32 value
    }
    const long long o = row * out_pitch + c;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      Vec4 hi, lo;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < COLS; ++k) acc = fmaf(__ldg(m + r * COLS + k), x[k].v[e], acc);
        split_tf32(acc, hi.v[e], lo.v[e]);
      }
      st4((v1 ? fv.out[1] : fv.out[0]) + o + r * blk, hi);
      st4((v1 ? fv.out_lo[1] : fv.out_lo[0]) + o + r * blk, lo);
    }
    if (c < out_fill - ROWS * blk) {
      st4((v1 ? fv.out[1] : fv.out[0]) + o + ROWS * blk, Vec4{{0.f, 0.f, 0.f, 0.f}});
      st4((v1 ? fv.out_lo[1] : fv.out_lo[0]) + o + ROWS * blk, Vec4{{0.f, 0.f, 0.f, 0.f}});
    }
  }
}

// can the 128-bit kernels run?  every plane pointer 4-element aligned, every stride a multiple of 4 channels
static bool ftl_vec_ok(int elem_bytes, int in_pitch, int blk, int out_pitch, int out_fill, int rows,
                       std::initializer_list<const void*> ptrs) {
  if ((blk | in_pitch | out_pitch | (out_fill - rows * blk)) & 3) return false;
  for (const void* p : ptrs)
    if (p && ((uintptr_t)p & (uintptr_t)(4 * elem_bytes - 1))) return false;
  return true;
}

template <int ROWS, int COLS>
__global__ void __launch_bounds__(256)
ftl_split_kernel(const FtlViews<float> fv, int in_pitch, int blk, long long total, int hw, int out_pitch, int out_fill) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int view = blockIdx.y;
  const float* __restrict__ in_hi = fv.in[view];
  const float* __restrict__ in_lo = fv.in_lo[view];
  const float* __restrict__ mats = fv.mats[view];
  float* __restrict__ out_hi = fv.out[view];
  float* __restrict__ out_lo = fv.out_lo[view];
  if (idx >= total) return;
  const long long row = idx / blk;
  const int c = (int)(idx - row * blk);
  const float* m = mats + (row / hw) * (ROWS * COLS);
  float x[COLS];
#pragma unroll
  for (int k = 0; k < COLS; ++k) {
    const long long i = row * in_pitch + k * blk + c;
    x[k] = in_hi[i] + in_lo[i];          // exact: hi + lo reconstructs the fp32 value
  }
  const long long o = row * out_pitch;
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < COLS; ++k) acc = fmaf(__ldg(m + r * COLS + k), x[k], acc);
    float hi, lo;
    split_tf32(acc, hi, lo);
    out_hi[o + r * blk + c] = hi;
    out_lo[o + r * blk + c] = lo;
  }
  if (c < out_fill - ROWS * blk) {
    out_hi[o + ROWS * blk + c] = 0.f;
    out_lo[o + ROWS * blk + c] = 0.f;
  }
}

int launch_ftl_split2(const float* const in_hi[2], const float* const in_lo[2], int in_pitch, const float* const mats[2],
                      int rows, int cols, int blk, int n, int hw, float* const out_hi[2], float* const out_lo[2],
                      int out_pitch, int out_fill, int views, cudaStream_t st) {
  CDR_CHECK_ARG(views == 1 || views == 2, "ftl_split: 1 or 2 views");
  FtlViews<float> fv{};
  for (int v = 0; v < views; ++v) {
    CDR_CHECK_ARG(in_hi[v] && in_lo[v] && mats[v] && out_hi[v] && out_lo[v], "ftl_split: bad args");
    fv.in[v] = in_hi[v]; fv.in_lo[v] = in_lo[v]; fv.mats[v] = mats[v]; fv.out[v] = out_hi[v]; fv.out_lo[v] = out_lo[v];
  }
  CDR_CHECK_ARG(n > 0 && hw > 0 && blk > 0, "ftl_split: bad args");
  const long long total = (long long)n * hw * blk;
  if ((rows == 4 && cols == 3 || rows == 3 && cols == 4) &&
      ftl_vec_ok(4, in_pitch, blk, out_pitch, out_fill, rows,
                 {in_hi[0], in_lo[0], out_hi[0], out_lo[0], views > 1 ? in_hi[1] : nullptr, views > 1 ? in_lo[1] : nullptr,
                  views > 1 ? out_hi[1] : nullptr, views > 1 ? out_lo[1] : nullptr})) {
    const dim3 grid4((unsigned)ceil_div<long long>(total / 4, 256), views);
    if (rows == 4)
      ftl_split_vec_kernel<4, 3><<<grid4, 256, 0, st>>>(fv, in_pitch, blk, total / 4, hw, out_pitch, out_fill);
    else
      ftl_split_vec_kernel<3, 4><<<grid4, 256, 0, st>>>(fv, in_pitch, blk, total / 4, hw, out_pitch, out_fill);
    CDR_LAUNCH_OK("ftl_split_vec_kernel");
    return CDR_OK;
  }
  const dim3 grid((unsigned)ceil_div<long long>(total, 256), views);
  if (rows == 4 && cols == 3)
    ftl_split_kernel<4, 3><<<grid, 256, 0, st>>>(fv, in_pitch, blk, total, hw, out_pitch, out_fill);
  else if (rows == 3 && cols == 4)
    ftl_split_kernel<3, 4><<<grid, 256, 0, st>>>(fv, in_pitch, blk, total, hw, out_pitch, out_fill);
  else {
    set_error("ftl_split: only (4x3) and (3x4) matrices are supported");
    return CDR_ERR_UNSUPPORTED;
  }
  CDR_LAUNCH_OK("ftl_split_kernel");
  return CDR_OK;
}

// FTL on scaled fp16 hi/lo planes (gemm_tc.cu: kFmtF16P), both directions of the fp32-grade fusion block: the value is
// (hi + lo * 2^-11) / s_in (exact in fp32: 22 significant bits), the product is formed in fp32 and stored with
// s_out = 2^(13 - ilogb(bound)), bound = max|in| * max_row ||M||_1 >= max|out| (so nothing overflows fp16 without a
// reduction over the output first).  One thread per (row, 4 channels): 8-byte accesses.
struct Half4 { __half2 a, b; };
__device__ __forceinline__ Half4 ldh4(const __half* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  Half4 h;
  h.a = *reinterpret_cast<const __half2*>(&u.x);
  h.b = *reinterpret_cast<const __half2*>(&u.y);
  return h;
}
__device__ __forceinline__ void sth4(__half* p, __half2 a, __half2 b) {
  uint2 u;
  u.x = *reinterpret_cast<const uint32_t*>(&a);
  u.y = *reinterpret_cast<const uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}
template <int ROWS, int COLS>
__global__ void __launch_bounds__(256)
ftl_f16p_vec_kernel(const FtlViews<__half> fv, int in_pitch, int blk, long long total4, int hw, int out_pitch,
                    int out_fill, const float* __restrict__ scale_in, const float* __restrict__ amax_in,
                    const float* __restrict__ l1max, float* __restrict__ scale_out, float* __restrict__ amax_out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool v1 = blockIdx.y != 0;
  const float inv_s = 1.f / __ldg(scale_in);          // powers of two: exact
  const float bound = __ldg(amax_in) * __ldg(l1max);
  const float s_out = f16_pow2_scale(bound);
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *scale_out = s_out;
  float amax = 0.f;
  if (idx < total4) {
    const int blk4 = blk >> 2;
    const long long row = idx / blk4;
    const int c = (int)(idx - row * blk4) << 2;
    const float* m = (v1 ? fv.mats[1] : fv.mats[0]) + (row / hw) * (ROWS * COLS);
    const long long i0 = row * in_pitch + c;
    Vec4 x[COLS];
#pragma unroll
    for (int k = 0; k < COLS; ++k) {
      const Half4 h = ldh4((v1 ? fv.in[1] : fv.in[0]) + i0 + k * blk), l = ldh4((v1 ? fv.in_lo[1] : fv.in_lo[0]) + i0 + k * blk);
      const float2 h0 = __half22float2(h.a), h1 = __half22float2(h.b), l0 = __half22float2(l.a), l1 = __half22float2(l.b);
      x[k].v[0] = fmaf(l0.x, 1.f / 2048.f, h0.x) * inv_s; x[k].v[1] = fmaf(l0.y, 1.f / 2048.f, h0.y) * inv_s;
      x[k].v[2] = fmaf(l1.x, 1.f / 2048.f, h1.x) * inv_s; x[k].v[3] = fmaf(l1.y, 1.f / 2048.f, h1.y) * inv_s;
    }
    const long long o = row * out_pitch + c;
    __half* oh = v1 ? fv.out[1] : fv.out[0];
    __half* ol = v1 ? fv.out_lo[1] : fv.out_lo[0];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      float X[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < COLS; ++k) acc = fmaf(__ldg(m + r * COLS + k), x[k].v[e], acc);
        amax = fmaxf(amax, fabsf(acc));
        X[e] = acc * s_out;
      }
      const __half2 ha = __floats2half2_rn(X[0], X[1]), hb = __floats2half2_rn(X[2], X[3]);
      const float2 fa = __half22float2(ha), fb = __half22float2(hb);
      sth4(oh + o + r * blk, ha, hb);
      sth4(ol + o + r * blk, __floats2half2_rn((X[0] - fa.x) * 2048.f, (X[1] - fa.y) * 2048.f),
           __floats2half2_rn((X[2] - fb.x) * 2048.f, (X[3] - fb.y) * 2048.f));
    }
    if (c < out_fill - ROWS * blk) {
      const __half2 z = __floats2half2_rn(0.f, 0.f);
      sth4(oh + o + ROWS * blk, z, z);
      sth4(ol + o + ROWS * blk, z, z);
    }
  }
  if (amax_out) {   // max |out|: the next conv's output-scale bound
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(amax_out), __float_as_uint(amax));
  }
}
int launch_ftl_f16p2(const void* const in_hi[2], const void* const in_lo[2], int in_pitch, const float* const mats[2],
                     int rows, int cols, int blk, int n, int hw, void* const out_hi[2], void* const out_lo[2],
                     int out_pitch, int out_fill, const float* scale_in, const float* amax_in, const float* l1max,
                     float* scale_out, float* amax_out, cudaStream_t st) {
  FtlViews<__half> fv{};
  for (int v = 0; v < 2; ++v) {
    CDR_CHECK_ARG(in_hi[v] && in_lo[v] && mats[v] && out_hi[v] && out_lo[v], "ftl_f16p: bad args");
    fv.in[v] = (const __half*)in_hi[v]; fv.in_lo[v] = (const __half*)in_lo[v]; fv.mats[v] = mats[v];
    fv.out[v] = (__half*)out_hi[v]; fv.out_lo[v] = (__half*)out_lo[v];
  }
  CDR_CHECK_ARG(n > 0 && hw > 0 && blk > 0 && scale_in && amax_in && l1max && scale_out, "ftl_f16p: bad args");
  CDR_CHECK_ARG((rows == 4 && cols == 3 || rows == 3 && cols == 4) &&
                    ftl_vec_ok(2, in_pitch, blk, out_pitch, out_fill, rows,
                               {in_hi[0], in_lo[0], out_hi[0], out_lo[0], in_hi[1], in_lo[1], out_hi[1], out_lo[1]}),
                "ftl_f16p: (4x3) / (3x4) matrices on 4-channel-aligned planes only");
  const long long total = (long long)n * hw * blk;
  const dim3 grid4((unsigned)ceil_div<long long>(total / 4, 256), 2);
  if (rows == 4)
    ftl_f16p_vec_kernel<4, 3><<<grid4, 256, 0, st>>>(fv, in_pitch, blk, total / 4, hw, out_pitch, out_fill, scale_in,
                                                     amax_in, l1max, scale_out, amax_out);
  else
    ftl_f16p_vec_kernel<3, 4><<<grid4, 256, 0, st>>>(fv, in_pitch, blk, total / 4, hw, out_pitch, out_fill, scale_in,
                                                     amax_in, l1max, scale_out, amax_out);
  CDR_LAUNCH_OK("ftl_f16p_vec_kernel");
  return CDR_OK;
}

// max over samples and rows of the L1 row norm of two sets of small matrices (both views each):
// out[0] <- set A (a0, a1: n matrices of ra x ca each), out[1] <- set B.  One block; inflated by 2^-20 so that the
// rounded sum stays an upper bound.
__global__ void __launch_bounds__(256)
mats_l1max_kernel(const float* __restrict__ a0, const float* __restrict__ a1, int ra, int ca,
                  const float* __restrict__ b0, const float* __restrict__ b1, int rb, int cb, int n,
                  float* __restrict__ out) {
  __shared__ float red[2][8];
  float mx[2] = {0.f, 0.f};
  for (int set = 0; set < 2; ++set) {
    const int R = set ? rb : ra, Cc = set ? cb : ca;
    const long long total = 2LL * n * R;
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
      const long long mat = i / R;
      const int r = (int)(i - mat * R);
      const float* base = set ? (mat < n ? b0 + mat * R * Cc : b1 + (mat - n) * R * Cc)
                              : (mat < n ? a0 + mat * R * Cc : a1 + (mat - n) * R * Cc);
      float sum = 0.f;
      for (int k = 0; k < Cc; ++k) sum += fabsf(__ldg(base + r * Cc + k));
      mx[set] = fmaxf(mx[set], sum);
    }
  }
#pragma unroll
  for (int set = 0; set < 2; ++set) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx[set] = fmaxf(mx[set], __shfl_xor_sync(0xffffffffu, mx[set], o));
    if ((threadIdx.x & 31) == 0) red[set][threadIdx.x >> 5] = mx[set];
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    float m = 0.f;
    for (int w = 0; w < 8; ++w) m = fmaxf(m, red[threadIdx.x][w]);
    out[threadIdx.x] = m * (1.f + 9.5367431640625e-07f);
  }
}
int launch_mats_l1max(const float* a0, const float* a1, int ra, int ca, const float* b0, const float* b1, int rb, int cb,
                      int n, float* out, cudaStream_t st) {
  CDR_CHECK_ARG(a0 && a1 && b0 && b1 && out && n > 0, "mats_l1max: bad args");
  mats_l1max_kernel<<<1, 256, 0, st>>>(a0, a1, ra, ca, b0, b1, rb, cb, n, out);
  CDR_LAUNCH_OK("mats_l1max_kernel");
  return CDR_OK;
}

template <typename T>
int launch_ftl2(const T* const in[2], int in_pitch, const float* const mats[2], int rows, int cols, int blk, int n,
                int hw, T* const out[2], int out_pitch, int out_fill, int views, cudaStream_t st) {
  CDR_CHECK_ARG(views == 1 || views == 2, "cdr_ftl: 1 or 2 views");
  FtlViews<T> fv{};
  for (int v = 0; v < views; ++v) {
    CDR_CHECK_ARG(in[v] && mats[v] && out[v], "cdr_ftl: bad args");
    fv.in[v] = in[v]; fv.mats[v] = mats[v]; fv.out[v] = out[v];
  }
  CDR_CHECK_ARG(n > 0 && hw > 0 && blk > 0, "cdr_ftl: bad args");
  CDR_CHECK_ARG(in_pitch >= cols * blk && out_pitch >= rows * blk && out_fill >= rows * blk &&
                    out_fill <= out_pitch && out_fill - rows * blk <= blk,
                "cdr_ftl: pitches too small for %dx%d blocks of %d", rows, cols, blk);
  const long long total = (long long)n * hw * blk;
  if ((rows == 4 && cols == 3 || rows == 3 && cols == 4) &&
      ftl_vec_ok((int)sizeof(T), in_pitch, blk, out_pitch, out_fill, rows,
                 {in[0], out[0], views > 1 ? in[1] : nullptr, views > 1 ? out[1] : nullptr})) {
    const dim3 grid4((unsigned)ceil_div<long long>(total / 4, 256), views);
    if (rows == 4)
      ftl_vec_kernel<T, 4, 3><<<grid4, 256, 0, st>>>(fv, in_pitch, blk, total / 4, hw, out_pitch, out_fill);
    else
      ftl_vec_kernel<T, 3, 4><<<grid4, 256, 0, st>>>(fv, in_pitch, blk, total / 4, hw, out_pitch, out_fill);
    CDR_LAUNCH_OK("ftl_vec_kernel");
    return CDR_OK;
  }
  const dim3 grid((unsigned)ceil_div<long long>(total, 256), views);
  if (rows == 4 && cols == 3)
    ftl_kernel<T, 4, 3><<<grid, 256, 0, st>>>(fv, in_pitch, blk, total, hw, out_pitch, out_fill);
  else if (rows == 3 && cols == 4)
    ftl_kernel<T, 3, 4><<<grid, 256, 0, st>>>(fv, in_pitch, blk, total, hw, out_pitch, out_fill);
  else {
    set_error("cdr_ftl: only (4x3) and (3x4) matrices are supported, got %dx%d", rows, cols);
    return CDR_ERR_UNSUPPORTED;
  }
  CDR_LAUNCH_OK("ftl_kernel");
  return CDR_OK;
}
template int launch_ftl2<float>(const float* const[2], int, const float* const[2], int, int, int, int, int, float* const[2], int, int, int, cudaStream_t);
template int launch_ftl2<__nv_bfloat16>(const __nv_bfloat16* const[2], int, const float* const[2], int, int, int, int, int, __nv_bfloat16* const[2], int, int, int, cudaStream_t);

template <typename T>
int launch_ftl(const T* in, int in_pitch, const float* mats, int rows, int cols, int blk, int n,
               int hw, T* out, int out_pitch, int out_fill, cudaStream_t st) {
  const T* ins[2] = {in, nullptr};
  const float* ms[2] = {mats, nullptr};
  T* outs[2] = {out, nullptr};
  return launch_ftl2<T>(ins, in_pitch, ms, rows, cols, blk, n, hw, outs, out_pitch, out_fill, 1, st);
}
template int launch_ftl<float>(const float*, int, const float*, int, int, int, int, int, float*, int, int, cudaStream_t);
template int launch_ftl<__nv_bfloat16>(const __nv_bfloat16*, int, const float*, int, int, int, int, int, __nv_bfloat16*, int, int, cudaStream_t);

}  // namespace cdr

extern "C" int cdr_ftl(const float* in, int in_pitch, const float* mats, int rows, int cols, int blk,
                       int n, int hw, float* out, int out_pitch, int out_fill, void* stream) {
  return cdr::launch_ftl<float>(in, in_pitch, mats, rows, cols, blk, n, hw, out, out_pitch, out_fill,
                                (cudaStream_t)stream);
}
