// bf16 implicit-GEMM on the 5th-gen tensor cores (tcgen05 + TMEM + TMA), sm_100a.
//
// Same "tap-GEMM" arithmetic as gemm_ffma.cu — C[m,n] = sum_tap sum_k A[shift_tap(m),k] W[n][tap,k]
// over pixel-major bf16 activations — mapped to the Blackwell execution model:
//
//   * persistent CTAs (one per SM), 192 threads = 6 warps with fixed roles:
//       warp 0  TMA producer   one elected lane issues cp.async.bulk.tensor loads:
//                              A tile = 128 pixels x 64 channels.  For 1x1 convs a 2-D box of the
//                              (pixels, channels) matrix; for the transposed convs a 4-D box
//                              (64ch, W, rows, images) of the NHWC tensor whose start coordinate is
//                              shifted by the tap (dy,dx) — the TMA unit zero-fills out-of-range
//                              pixels, so the im2col never exists and borders cost nothing.
//                              B tile = BN output channels x 64 of the K-major packed weights.
//       warp 1  MMA issuer     one lane issues tcgen05.mma (M=128, N=BN, K=16, kind::f16, bf16 in,
//                              fp32 accumulate in TMEM); tcgen05.commit releases smem stages and
//                              publishes finished accumulators.  Also owns TMEM alloc/dealloc.
//       warps 2-5 epilogue     tcgen05.ld the 128 x BN fp32 accumulator (one TMEM lane = one pixel
//                              per thread), + folded-BN bias, ReLU, convert, store: pixel-major bf16
//                              rows, the transposed-conv phase scatter, or planar fp32 heat-maps.
//   * 128B-swizzled smem tiles shared by TMA and the UMMA descriptors, 4-6 stage mbarrier ring;
//   * two TMEM accumulator buffers (2 x BN columns) so the epilogue of tile i overlaps the
//     main loop of tile i+1.
//
// Tile order: consecutive CTAs take the 4 phases / N-tiles of the SAME 128-pixel block, so the
// shifted A tiles they share hit in L2; the packed weights (<= 16 MB) stay L2-resident.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <type_traits>
#include <utility>

#include "jacobi.cuh"
#include "ptx.cuh"
#include "tc_api.h"

namespace cdr {

// ------------------------------------------------------------------------------------------
// Storage formats of an activation / weight tensor.
//   kFmtBF16 : one bf16 plane.
//   kFmtTF32P: two fp32 planes hi = rn_tf32(x), lo = x - hi (common.cuh: split_tf32).
//   kFmtF16P : two fp16 planes of X = x * s (s a power of two, per tensor for activations, per
//              output channel for weights): hi = rn_f16(X), lo = rn_f16((X - hi) * 2^11).
//              X = hi + lo * 2^-11 to 2^-24 relative (fp16 subnormals: 2^-36 absolute), i.e. fp32
//              precision for every value within 2^-27 of the scaled maximum.
enum ActFmt { kFmtBF16 = 0, kFmtTF32P = 1, kFmtF16P = 2 };
__host__ __device__ constexpr int fmt_elem(int fmt) { return fmt == kFmtTF32P ? 4 : 2; }
__host__ __device__ constexpr int fmt_planes(int fmt) { return fmt == kFmtBF16 ? 1 : 2; }
constexpr float kLoScale = 2048.f;            // 2^11: the lo plane of kFmtF16P is stored times this

// ------------------------------------------------------------------------------------------
// tensor maps
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  }
  return fn;
}

// dims[0] innermost (contiguous); strides in elements for dims 1..rank-1; fmt = ActFmt of the tensor
static int make_tmap(CUtensorMap* map, const void* base, int fmt, int rank, const uint64_t* dims,
                     const uint64_t* strides_elems, const uint32_t* box, const uint32_t* elem_strides = nullptr) {
  const int elem_bytes = fmt_elem(fmt);
  const CUtensorMapDataType dtype = fmt == kFmtBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                    : fmt == kFmtTF32P ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                                       : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  auto enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return CDR_ERR_CUDA;
  }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bdim[5], estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = elem_strides ? elem_strides[i] : 1;
    if (i > 0) gstr[i - 1] = strides_elems[i - 1] * (uint64_t)elem_bytes;
  }
  CUresult r = enc(map, dtype, (cuuint32_t)rank, const_cast<void*>(base),
                   gdim, gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu %llu, box %u %u)",
              (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return CDR_ERR_CUDA;
  }
  return CDR_OK;
}

// ------------------------------------------------------------------------------------------
constexpr int kTcBM = 128;
constexpr int kABytes = kTcBM * 128;             // 128 rows x one 128-byte swizzle row = 16 KB
constexpr int kSmemBudget = 224 * 1024;          // of the 227 KB a CTA may own
constexpr int kStageBufBytes = 32 * 128;         // TMA-store staging per epilogue warp: 32 rows x 128 B

// Operand kinds.
//   kKindBF16  : bf16 operands, kind::f16, one MMA per K=16 step.
//   kKindTF32X3: fp32 accuracy on the tensor cores.  Every fp32 operand is stored as two fp32
//                planes hi = rn_tf32(x), lo = x - hi (common.cuh: split_tf32); x*y ~= hi*hi' + hi*lo' + lo*hi' with kind::tf32 MMAs accumulating in
//                fp32 (dropped lo*lo' term ~2^-22 relative, random sign).
//   kKindF16X2 : fp32 accuracy at the full 16-bit tensor rate.  Operands in kFmtF16P; with
//                x = (xh + xl 2^-11)/s and w = (wh + wl 2^-11)/t:  x*w*s*t = xh*wh + 2^-11 (xh*wl + xl*wh)
//                + 2^-22 xl*wl.  The main term and the (2^11-scaled) correction terms accumulate in
//                separate TMEM accumulators (the same two the 3xTF32 kernel uses); the epilogue
//                adds main + 2^-11 corr and undoes s*t.  Dropped term: 2^-24 relative.  fp16
//                products are exact in fp32, so this is strictly more accurate than 3xTF32 (2^-22)
//                while each product costs 3 kind::f16 MMAs instead of 3 half-rate kind::tf32 MMAs,
//                and the activations move half the bytes (2 x fp16 instead of 2 x fp32).
//                The tensor scale s is data-dependent: the producing kernel derives it from a
//                rigorous bound |out| <= amax(in) * max_row ||W||_1 + max|bias| (amax(in) measured by
//                ITS producer with atomicMax), so nothing can overflow fp16 and one layer of bound
//                looseness (~2^7) is far inside the format's 2^27 full-precision window.
enum TcKind { kKindBF16 = 0, kKindTF32X3 = 1, kKindF16X2 = 2 };
// kTapConv4s2: 4x4 stride-2 pad-1 conv (16 taps), the data gradient of a k4 s2 p1 transposed conv (deconv_train_backward)
enum TapMode { kTapNone = 0, kTapDeconv = 1, kTapConv3 = 2, kTapConv4s2 = 3 };
template <int KIND> struct KindTraits;
template <> struct KindTraits<kKindBF16>   { static constexpr int kElem = 2, kBK = 64, kPlanes = 1, kFmt = kFmtBF16; };
template <> struct KindTraits<kKindTF32X3> { static constexpr int kElem = 4, kBK = 32, kPlanes = 2, kFmt = kFmtTF32P; };
template <> struct KindTraits<kKindF16X2>  { static constexpr int kElem = 2, kBK = 64, kPlanes = 2, kFmt = kFmtF16P; };

template <int BN, int KIND, int OFMT, int CL = 0>
struct TcCfg {
  static constexpr int kBK = KindTraits<KIND>::kBK;
  static constexpr int kPlanes = KindTraits<KIND>::kPlanes;
  static constexpr int kBRows = CL == 2 ? BN / 2 : BN;           // CL = 2 (cta_group::2): each CTA of the pair stages half of B
  static constexpr int kBBytes = kBRows * 128;
  static constexpr int kStageBytes = kPlanes * (kABytes + kBBytes);
  // Epilogue: 8 warps for wide tiles — two per TMEM lane quarter, each owning half of the columns —
  // because with short K loops (the 256-channel transposed convs: 16 K-blocks per tile) the epilogue,
  // not the MMA, paces the kernel (measured: the MMA issuer spinning on tmem_empty).
  static constexpr int kEpiWarps = BN >= 128 ? 8 : 4;
  static constexpr int kThreads = 64 + 32 * kEpiWarps;
  static constexpr int kColsPerWarp = BN / (kEpiWarps / 4);
  // 16-bit row-major outputs leave through swizzled smem staging + TMA tensor stores (full 128-byte
  // lines, issued by one lane, asynchronous) instead of 32 scattered 16-byte stores per warp instruction.
  static constexpr bool kTmaStore = BN >= 64 && OFMT != kFmtTF32P;
  // two staging buffers per warp where smem allows (bf16, BN <= 128): a warp never waits for its previous
  // store to drain — the memory-bound encoder layers are paced by epilogue bytes in flight
  static constexpr int kStageBufs = (KIND == kKindBF16 && BN <= 128) ? 2 : 1;
  static constexpr int kStagingBytes = kTmaStore ? kEpiWarps * kStageBufs * kStageBufBytes : 0;
  static constexpr int kStagesFit = (kSmemBudget - kStagingBytes) / kStageBytes;
  static constexpr int kStages = kStagesFit > 8 ? 8 : kStagesFit;
  static constexpr int kAccBufs = KIND != kKindBF16 ? 4 : 2;     // see the TMEM column map in the kernel
  static constexpr int kTmemCols = (kAccBufs * BN <= 32) ? 32 : (kAccBufs * BN <= 64) ? 64
                                   : (kAccBufs * BN <= 128) ? 128 : (kAccBufs * BN <= 256) ? 256 : 512;
  static_assert(kAccBufs * BN <= 512, "TMEM has 512 columns");
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + kStagingBytes + 1024 /*align*/ + 512 /*barriers*/;
  static_assert(BN % 32 == 0 && BN >= 32 && BN <= 256, "UMMA N for M=128; 32-column epilogue slabs");
  static_assert(kStages >= 2, "pipeline too shallow");
  static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
};

struct TcGemmParams {
  int M;                  // output rows (pixels) per group
  int n_img, H, W;        // pixel grid of the A operand
  int cin;                // K per tap
  int ntaps;              // 1 or 4
  int a4d;                // 1: A through the 4-D NHWC map (shifted / strided taps), 0: 2-D (rows, channels)
  int tap_mode;           // kTapNone: 1 tap; kTapDeconv: 4 taps of output phase g; kTapConv3: 9 taps (3x3, pad 1);
                          // kTapConv4s2: 16 taps (4x4, stride 2, pad 1)
  int stride;             // 4-D A: input pixel = stride * output pixel + tap shift (map carries the element stride)
  int has_res;            // residual tensor (rows like C, same format) added before the ReLU: its 128 x 128 tile travels
                          // through the operand ring as one extra stage per tile (BN = 128; bf16, or f16x2 hi/lo planes)
  const float* res_scale; // kFmtF16P residual: its tensor scale s and max |x| (unscaled; enters the output-scale bound)
  const float* res_amax;
  int box_rows, box_imgs; // 4-D box: W x box_rows x box_imgs pixels = 128
  int half_dim, half_step;// CTA pairs: coordinate (2 = row, 3 = image) and step that separate the two 64-pixel half boxes
  int groups;             // phases (deconv) or independent problems stacked along rows
  int a_group_rows;       // 2-D A: row offset per group
  int b_group_rows;       // weight-row offset per group
  int n_tiles;            // N tiles of BN per group
  int n;                  // valid output channels
  const float* bias;      // (groups?, n_pad)
  int bias_group_stride;
  void* C;                // bf16 rows, or the hi plane (kFmtTF32P / kFmtF16P), or planar fp32 heat-maps
  void* C_lo;             // the lo plane
  // kKindF16X2 operands / kFmtF16P outputs (device scalars live in the workspace "slots")
  const float* wsi;       // per packed weight row: 2^-t (undoes the weight scale)
  int wsi_group_stride;
  const float* scale_in;  // s of the A tensor
  const float* scale_in_rows;   // (optional) one s per A row instead (2-D A only): layout.cu's per-pixel scales
  const float* amax_in;   // max |x| of the A tensor (unscaled)   } bound for the output scale
  const float* norms;     // layer {max_row ||W||_1, max |bias|}   }
  float* amax_out;        // atomicMax target: max |out| (unscaled), pre-zeroed
  float* scale_out;       // s chosen for the output tensor
  long long c_group_stride;
  int c_pitch, c_fill;
  int relu;
  int out_mode;           // kOutRows / kOutDeconv or kOutPlanar (fp32)
  int planar_deconv;      // kOutPlanar of a kTapDeconv launch: output phase g scattered to (2y + g/2, 2x + g%2) of a 2H x 2W map
  int num_tiles;
};

struct EpiScale {          // per-thread epilogue constants of the scaled formats
  float a_inv = 1.f;       // 1 / s(A tensor)
  float r_inv = 1.f;       // 1 / s(residual tensor)
  float s_out = 1.f;       // s(output tensor)
  float amax = 0.f;        // running max |out| of this thread
};

// + scale (f16x2), bias, ReLU for one 32-column slab of a finished row.  `floor` = 0 (ReLU) or -inf
// (none): one FMNMX per element instead of a branch; the column mask only runs on the slab that
// straddles the layer's last channel.  (The first version spent ~35 instructions per element here —
// per-element predicates and masks — and made every short-K layer epilogue-issue-bound.)
template <int KIND>
__device__ __forceinline__ void finish_slab(const TcGemmParams& p, const float (&acc)[32], float (&v)[32], int n0c,
                                            const float* __restrict__ bias, const float* __restrict__ wsi,
                                            const EpiScale& es, float floor) {
#pragma unroll
  for (int j4 = 0; j4 < 8; ++j4) {
    float4 x = make_float4(acc[4 * j4], acc[4 * j4 + 1], acc[4 * j4 + 2], acc[4 * j4 + 3]);
    if constexpr (KIND == kKindF16X2) {
      const float4 w4 = __ldg(reinterpret_cast<const float4*>(wsi + n0c) + j4);
      x.x *= es.a_inv * w4.x; x.y *= es.a_inv * w4.y; x.z *= es.a_inv * w4.z; x.w *= es.a_inv * w4.w;
    }
    const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + n0c) + j4);
    v[4 * j4] = fmaxf(x.x + b4.x, floor);
    v[4 * j4 + 1] = fmaxf(x.y + b4.y, floor);
    v[4 * j4 + 2] = fmaxf(x.z + b4.z, floor);
    v[4 * j4 + 3] = fmaxf(x.w + b4.w, floor);
  }
  if (n0c + 32 > p.n) {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (n0c + j >= p.n) v[j] = 0.f;
  }
}

// 16-bit encodings of a finished slab: 16 packed words per plane
template <int OFMT>
__device__ __forceinline__ void encode_slab(const float (&v)[32], uint32_t (&hi)[16], uint32_t (&lo)[16],
                                            bool row_ok, EpiScale& es) {
  if constexpr (OFMT == kFmtF16P) {
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const float x0 = v[2 * e], x1 = v[2 * e + 1];
      if (row_ok) es.amax = fmaxf(es.amax, fmaxf(fabsf(x0), fabsf(x1)));
      const float X0 = x0 * es.s_out, X1 = x1 * es.s_out;
      const __half2 hh = __floats2half2_rn(X0, X1);
      const float2 hf = __half22float2(hh);
      const __half2 ll = __floats2half2_rn((X0 - hf.x) * kLoScale, (X1 - hf.y) * kLoScale);
      hi[e] = *reinterpret_cast<const uint32_t*>(&hh);
      lo[e] = *reinterpret_cast<const uint32_t*>(&ll);
    }
  } else {
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const __nv_bfloat162 b = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
      hi[e] = *reinterpret_cast<const uint32_t*>(&b);
    }
  }
}

// Direct global stores of one finished slab (planar heat-maps, fp32 planes, and the narrow tiles).
template <int KIND, int OFMT>
__device__ __forceinline__ void store_slab(const TcGemmParams& p, const float (&acc)[32], int n0c, int g, bool row_ok,
                                           size_t orow, int img, int pix, int HW, const float* __restrict__ bias,
                                           const float* __restrict__ wsi, EpiScale& es) {
  float v[32];
  finish_slab<KIND>(p, acc, v, n0c, bias, wsi, es, p.relu ? 0.f : -INFINITY);
  if (!row_ok) return;
  if (p.out_mode == kOutPlanar) {
    float* __restrict__ C = reinterpret_cast<float*>(p.C);
    if (p.planar_deconv) {
      const int y = pix / p.W, x = pix - y * p.W;
      const size_t o = (size_t)(2 * y + (g >> 1)) * (2 * p.W) + 2 * x + (g & 1);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (n0c + j < p.n) C[((size_t)img * p.n + n0c + j) * (4 * HW) + o] = v[j];
      return;
    }
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (n0c + j < p.n) C[((size_t)img * p.n + n0c + j) * HW + pix] = v[j];
    return;
  }
  const size_t off = (p.out_mode == kOutDeconv ? 0 : (size_t)g * p.c_group_stride) + orow * p.c_pitch + n0c;
  if constexpr (OFMT == kFmtTF32P) {
    float* __restrict__ Ch = reinterpret_cast<float*>(p.C) + off;
    float* __restrict__ Cl = reinterpret_cast<float*>(p.C_lo) + off;
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
      if (n0c + j4 * 4 < p.c_fill) {
        float hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) split_tf32(v[j4 * 4 + e], hi[e], lo[e]);
        *reinterpret_cast<float4*>(Ch + j4 * 4) = make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(Cl + j4 * 4) = make_float4(lo[0], lo[1], lo[2], lo[3]);
      }
    }
  } else {
    uint32_t hi[16], lo[16];
    encode_slab<OFMT>(v, hi, lo, true, es);
    uint16_t* __restrict__ Ch = reinterpret_cast<uint16_t*>(p.C) + off;
#pragma unroll
    for (int j8 = 0; j8 < 4; ++j8)
      if (n0c + j8 * 8 < p.c_fill)
        *reinterpret_cast<uint4*>(Ch + j8 * 8) = make_uint4(hi[4 * j8], hi[4 * j8 + 1], hi[4 * j8 + 2], hi[4 * j8 + 3]);
    if constexpr (OFMT == kFmtF16P) {
      uint16_t* __restrict__ Cl = reinterpret_cast<uint16_t*>(p.C_lo) + off;
#pragma unroll
      for (int j8 = 0; j8 < 4; ++j8)
        if (n0c + j8 * 8 < p.c_fill)
          *reinterpret_cast<uint4*>(Cl + j8 * 8) = make_uint4(lo[4 * j8], lo[4 * j8 + 1], lo[4 * j8 + 2], lo[4 * j8 + 3]);
    }
  }
}

// One warp's 32 rows x 64 columns of 16-bit output: registers -> 128B-swizzled staging -> one TMA
// tensor store.  `words` = this lane's row, 32 packed words (64 values).  The staging buffer is
// private to the warp; the previous store's read of it is awaited first.
struct StoreCoord {
  int rows;      // kOutRows: (c, m, g)
  int m, g;
  int px, x0, py, r0;   // kOutDeconv: (c, px, x, py, img*H + y)
};
template <int kPending>
__device__ __forceinline__ void tma_store_block(const TcGemmParams& p, const void* tmap, uint8_t* stage, int lane,
                                                const uint32_t (&words)[32], int c0, const StoreCoord& sc) {
  if (lane == 0) ptx::bulk_wait_read<kPending>();   // the store that last used THIS buffer has read it
  __syncwarp();
  const uint32_t base = ptx::smem_u32(stage) + (uint32_t)lane * 128u;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    ptx::st_shared_v4(base + (uint32_t)((j ^ (lane & 7)) << 4), words[4 * j], words[4 * j + 1], words[4 * j + 2],
                      words[4 * j + 3]);
  ptx::fence_proxy_async();
  __syncwarp();
  if (lane == 0) {
    if (p.out_mode == kOutDeconv) ptx::tma_store_5d(tmap, stage, c0, sc.px, sc.x0, sc.py, sc.r0);
    else ptx::tma_store_3d(tmap, stage, c0, sc.m, sc.g);
    ptx::bulk_commit();
  }
}

// K-blocks accumulated inside TMEM before the split kinds' main term is drained into fp32 registers.
// The tensor core adds into its fp32 accumulator with round-toward-zero; over a long K chain
// of same-signed partial sums that bias grows linearly (measured: 1e-5 relative at K=2048, 40x
// worse than FFMA).  The cross-chunk sum is done by the epilogue warps in registers with round-to-nearest.
// Chains of 8 K-blocks (32 MMAs): heat-maps 3.1e-6 of max vs the fp64 oracle, 2D joints 2.9e-4 px (gates 2e-5 / 1e-3;
// the reference's own fp32 sits at 5.8e-4 px); chains of 4 gave 1.7e-6 / 1.8e-4 px.  8 halves the number of chunk
// hand-backs between the MMA issuer and the epilogue warps — what made cta_group::2 pairs lose on the 16-K-block layers
// (every hand-back crosses the cluster): f16x2 deconv2 / deconv3 on pairs 154 / 600 us with chunks of 4, 132 / 527 with 8.
constexpr int kSplitChunk = 8;

// CL = 1: CTA pairs (thread-block clusters of 2).  The two CTAs of a pair work on the two N tiles of the SAME
// 128-pixel block and output phase, so they need the same A tile: each loads half of it (64 pixels) and
// multicasts it into both CTAs' stage (tmap_a / tmap_a_lo then carry the half box) — one L2 read feeds two
// SMs.  ncu on the f16x2 transposed convs (BN = 128: 64 KB of operands per 12 MMAs) showed 12.3 TB/s of
// L2->SM traffic and the tensor pipe at 84 % of what the bf16 kernel reaches; with the shared A tile the
// traffic drops by a quarter.  Protocol: a stage may be refilled only when BOTH CTAs' MMAs have released
// it, so empty[s] counts two arrivals and every release is a multicast commit to both CTAs; everything
// else (TMEM, epilogue) stays per CTA.  Both CTAs run the same number of tiles (even n_tiles and grid).
//
// CL = 2: CTA pairs driving ONE tensor-core op (tcgen05.mma.cta_group::2, M = 256).  The pair takes two consecutive
// 128-pixel blocks of the same output phase and N tile; each CTA stages its own A rows and HALF of the B tile (BN/2
// weight rows), the leader (rank 0) issues every MMA for both, each CTA's accumulator rows live in its own TMEM and its
// own epilogue warps drain them.  Per SM and MMA the tensor core then reads A + B/2 from shared memory instead of
// A + B, and a stage shrinks from 64 to 48 KB (f16x2, BN = 128): 4 stages instead of 3.  The idea: with BN = 128 an MMA
// reads 8 KB of operands in the 64 cycles it computes — the 128 B/clk the shared memory delivers.  MEASURED on B200
// (B = 64, parity green): f16x2 deconv1 / 2 / 3 344 / 176 / 674 us with the multicast pairs (CL = 1) -> 353 / 189 / 716 us
// with cta_group::2 — 3-8 % SLOWER, while the kernel was still ISSUE-bound (one thread fed the tensor cores of two SMs
// through the ELECT loops described at the issuer).  With the converged issuer the picture is the expected one: ncu
// shows the f16x2 tail's tensor pipe active 65 % with the issuer stalled ON the UTCHMMA instructions and the TMA
// producer on a full ring — operand reads (8 KB per 64-cycle MMA) plus TMA fills (64 KB per K block) ask 213 B/clk of
// a 128 B/clk shared memory.  Re-measured: f16x2 deconv1 (128 K blocks per tile) 310 -> 274 us; deconv2 / deconv3 (16 K
// blocks per tile) 153 -> 154 / 604 -> 600 with main-term chunks of 4 K blocks (every chunk hand-back crosses the
// cluster) and 153 -> 132 / 604 -> 527 with chunks of 8 (now the default); bf16 deconv1 / 2 / 3 103 -> 95, 57 -> 53,
// 208 -> 180 us.  Enabled for the decoder's transposed convs (tc_decoder sets TcLaunch::pair2).  Protocol: one "full" barrier per stage, the leader's — both CTAs'
// TMA loads count their bytes on it (cp.async.bulk.tensor.cta_group::2); stage release, chunk / tile completion are
// multicast commits to both CTAs' barriers; "accumulator drained" arrivals of the peer's epilogue warps go to the
// leader's barriers through the cluster window (mapa + mbarrier.arrive.shared::cluster).
//
// kMN (f16x2, BN = 128, CL = 0): weight gradients, K = pixels.  One tile = 128 channels of A (M) x 128 channels of B (N)
// of one group g = slice * taps + tap and one K slice.  Both operands are read straight from the pixel-major fp16 planes,
// so they are MN-major (channels contiguous): A = two 64-channel x 64-pixel boxes; B = the same 64 pixels in the same
// (img, y, x) order.  tap_mode kTapConv4s2: a k4 s2 p1 transposed conv (deconv_train_backward; A = x, B = dy through the
// stride-2 box shifted by (kx - 1, ky - 1), 16 taps).  kTapConv3: a 3x3 pad-1 conv at stride p.stride
// (conv3x3_train_backward; A = dy, B = x through the stride-1 or stride-2 box shifted by (kx - 1, ky - 1), 9 taps).
// kTapNone: a 1x1 conv (conv1x1_train_backward; A = dy, B = x, both 2-D maps, 1 tap).  The UMMA descriptors carry the MN-major SWIZZLE_128B layout (LBO = the 8 KB between
// the two 64-channel halves, SBO = 1024 B between 8-pixel groups) and the instruction descriptor the transpose bits.
// The epilogue stores the raw fp32 tile (still times s_x * s_dy) into the slice's partial; wgrad_reduce_kernel sums
// the slices in a fixed order.
template <int BN, int KIND, int OFMT, int CL, bool kMN = false>
__global__ void __launch_bounds__(TcCfg<BN, KIND, OFMT, CL>::kThreads, 1)
tap_gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a_lo,
                   const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_b_lo,
                   const __grid_constant__ CUtensorMap tmap_c, const __grid_constant__ CUtensorMap tmap_c_lo,
                   const __grid_constant__ CUtensorMap tmap_r, const __grid_constant__ CUtensorMap tmap_r_lo,
                   const TcGemmParams p) {
  using Cfg = TcCfg<BN, KIND, OFMT, CL>;
  // layers that may carry a residual: the bf16 and the f16x2 -> fp16-plane kernels with BN = 128, one CTA per tile
  constexpr bool kResOK = CL == 0 && BN == 128 && ((KIND == kKindBF16 && OFMT == kFmtBF16) || (KIND == kKindF16X2 && OFMT == kFmtF16P));
  constexpr int S = Cfg::kStages;
  constexpr int kTcBK = Cfg::kBK;
  constexpr bool kSplit = KIND != kKindBF16;
  constexpr bool kPair2 = CL == 2;
  static_assert(!kPair2 || KIND != kKindTF32X3, "cta_group::2 is wired for the kind::f16 operand kinds");
  static_assert(!kMN || (KIND == kKindF16X2 && BN == 128 && CL == 0), "MN-major operands: f16x2, BN = 128, one CTA per tile");
  constexpr int kEpiWarps = Cfg::kEpiWarps;
  constexpr int kCols = Cfg::kColsPerWarp;       // columns of the tile owned by one epilogue warp
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // stage s: [A (16 KB) | A_lo (split kinds) | B (BN*128 B) | B_lo (split kinds)], every piece 1024-aligned
  auto stage_a = [&](int s, int plane) { return smem + (size_t)s * Cfg::kStageBytes + (size_t)plane * kABytes; };
  auto stage_b = [&](int s, int plane) {
    return smem + (size_t)s * Cfg::kStageBytes + (size_t)Cfg::kPlanes * kABytes + (size_t)plane * Cfg::kBBytes;
  };
  uint8_t* staging = smem + (size_t)S * Cfg::kStageBytes;               // [kEpiWarps][4 KB], 1024-aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + Cfg::kStagingBytes);
  uint64_t* full = bars;                      // [S]  TMA -> MMA
  uint64_t* empty = bars + S;                 // [S]  MMA -> TMA
  uint64_t* tmem_full = bars + 2 * S;         // [2]  finished tile accumulator (bf16) / correction accumulator (split)
  uint64_t* tmem_empty = bars + 2 * S + 2;    // [2]
  uint64_t* chunk_full = bars + 2 * S + 4;    // [2]  split kinds: main-term chunk accumulator
  uint64_t* chunk_empty = bars + 2 * S + 6;   // [2]
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 8);
  uint32_t* res_cnt = reinterpret_cast<uint32_t*>(bars + 2 * S + 9);   // [S] epilogue warps done with a residual stage

  // warp index through a shuffle: ptxas then KNOWS it is warp-uniform, so the role branches below are uniform control
  // flow and whatever the MMA-issuer warp computes inside them can live in uniform registers (see the issuer)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  // Programmatic dependent launch: let the next tap-GEMM's CTAs take over SMs as ours retire (its barrier
  // init / TMEM alloc / descriptor prefetch then overlap our tail and the wave-quantisation gap) ...
  ptx::grid_dep_launch();
  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
    if (kSplit) {
      ptx::prefetch_tmap(&tmap_a_lo);
      ptx::prefetch_tmap(&tmap_b_lo);
    }
    if (Cfg::kTmaStore && p.out_mode != kOutPlanar) {
      ptx::prefetch_tmap(&tmap_c);
      if (OFMT == kFmtF16P) ptx::prefetch_tmap(&tmap_c_lo);
    }
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], CL == 1 ? 2 : 1);    // CL = 1: released by the MMA issuers of both CTAs of the pair
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], kPair2 ? 2 * kEpiWarps : kEpiWarps);     // one arrive per epilogue warp (of both CTAs)
      ptx::mbar_init(&chunk_full[a], 1);
      ptx::mbar_init(&chunk_empty[a], kPair2 ? 2 * kEpiWarps : kEpiWarps);
    }
    for (int s = 0; s < S; ++s) res_cnt[s] = 0;
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (kPair2) ptx::tmem_alloc_2sm<Cfg::kTmemCols>(tmem_base_slot);
    else ptx::tmem_alloc<Cfg::kTmemCols>(tmem_base_slot);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CL != 0) ptx::cluster_sync();       // the peer's barriers exist before anything is multicast
  ptx::tc_fence_after();
  const uint32_t cta_rank = CL ? ptx::cluster_ctarank() : 0u;
  // tile walk: CL = 2 pairs walk PAIR tiles (two consecutive pixel blocks), everything else walks tiles
  const int tile0 = kPair2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = kPair2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  auto tile_m0 = [&](int tile) {
    const int mt = tile / (p.n_tiles * p.groups);
    return (kPair2 ? mt * 2 + (int)cta_rank : mt) * kTcBM;
  };
  // "this accumulator / chunk buffer is drained": to the leader's barrier when a pair shares one MMA issuer
  auto arrive_issuer = [&](uint64_t* bar) {
    if (kPair2 && cta_rank != 0) ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(bar), 0));
    else ptx::mbar_arrive(bar);
  };
  // ... and do not touch anything the previous kernel wrote (activations, scale slots) before it is complete
  ptx::grid_dep_wait();
  const uint32_t tmem_base = *tmem_base_slot;
  // TMEM columns: bf16 : [0,BN) [BN,2BN)               two tile accumulators
  //               split: [0,BN) [BN,2BN)               two main-term chunk accumulators
  //                      [2BN,3BN) [3BN,4BN)           two correction-term tile accumulators

  const int kb_per_tap = (p.cin + kTcBK - 1) / kTcBK;
  const int num_kb = p.ntaps * kb_per_tap;
  const int HW = p.H * p.W;

  if (warp == 0) {
    // ===================================================================== TMA producer
    // converged like the MMA issuer (UTMALDG takes its tensor-map pointer / barrier from uniform registers too): the
    // whole warp walks the tiles and waits, one elected lane arms the barrier and issues the loads of a K block
    {
      uint32_t it = 0;
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step) {
        const int n_tile = tile % p.n_tiles;
        const int g = (tile / p.n_tiles) % p.groups;
        const int m0 = tile_m0(tile);
        const int py = g >> 1, px = g & 1;
        const int img0 = m0 / HW, y0 = (m0 - img0 * HW) / p.W;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t par = (it / S) & 1;
          ptx::mbar_wait(&empty[s], par ^ 1u);
          // every coordinate is computed here, in warp-uniform code; the elected lane only issues
          const int tap = kb / kb_per_tap;
          const int k0 = (kb - tap * kb_per_tap) * kTcBK;
          int dy = 0, dx = 0;
          if (p.tap_mode == kTapDeconv) {
            dy = py - (tap >> 1); dx = px - (tap & 1);
          } else if (p.tap_mode == kTapConv3) {
            dy = tap / 3 - 1; dx = tap - (tap / 3) * 3 - 1;
          } else if (p.tap_mode == kTapConv4s2) {
            dy = (tap >> 2) - 1; dx = (tap & 3) - 1;
          }
          const int ys = p.stride * y0 + dy;
          const int arow = g * p.a_group_rows + m0;
          const int bk = tap * p.cin + k0;
          const int brow = g * p.b_group_rows + n_tile * BN + (kPair2 ? (int)cta_rank * (BN / 2) : 0);   // CL = 2: my half of B
          if constexpr (kMN) {
            // wgrad: g = slice * kw^2 + (ky * kw + kx), kw = 4 (kTapConv4s2), 3 (kTapConv3) or 1 (kTapNone); 64 pixels
            // of A from k0 of the slice (p.cin pixels per slice; for the 4-D box a block is whole rows of one image since
            // W | 64 | H*W) and the B pixels they pair with: the same ones, or (stride * y - 1 + ky, stride * x - 1 + kx)
            const int kw = p.tap_mode == kTapConv4s2 ? 4 : p.tap_mode == kTapConv3 ? 3 : 1;
            const int sl = g / (kw * kw), wt = g - sl * kw * kw, wky = wt / kw, wkx = wt - wky * kw;
            const int pix0 = sl * p.cin + k0;
            const int wimg = pix0 / HW, wy = (pix0 - wimg * HW) / p.W;
            const int co0 = n_tile * BN;
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&full[s], Cfg::kStageBytes);
#pragma unroll
              for (int pl = 0; pl < 2; ++pl) {
                const CUtensorMap* ma = pl ? &tmap_a_lo : &tmap_a;
                const CUtensorMap* mb = pl ? &tmap_b_lo : &tmap_b;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  ptx::tma_load_2d(stage_a(s, pl) + h * (kABytes / 2), ma, &full[s], m0 + 64 * h, pix0);
                  if (kw > 1)
                    ptx::tma_load_4d(stage_b(s, pl) + h * (Cfg::kBBytes / 2), mb, &full[s], co0 + 64 * h, wkx - 1,
                                     p.stride * wy + wky - 1, wimg);
                  else
                    ptx::tma_load_2d(stage_b(s, pl) + h * (Cfg::kBBytes / 2), mb, &full[s], co0 + 64 * h, pix0);
                }
              }
            }
          } else if constexpr (kPair2) {
            // both CTAs count their bytes on the LEADER's barrier of this stage; the leader expects the sum
            const uint32_t full_leader = ptx::mapa_u32(ptx::smem_u32(&full[s]), 0);
            if (ptx::elect_one()) {
              if (cta_rank == 0) ptx::mbar_arrive_expect_tx(&full[s], 2 * Cfg::kStageBytes);
              if (p.a4d) {
                ptx::tma_load_4d_2sm(stage_a(s, 0), &tmap_a, full_leader, k0, dx, ys, img0);
                if (kSplit) ptx::tma_load_4d_2sm(stage_a(s, 1), &tmap_a_lo, full_leader, k0, dx, ys, img0);
              } else {
                ptx::tma_load_2d_2sm(stage_a(s, 0), &tmap_a, full_leader, k0, arow);
                if (kSplit) ptx::tma_load_2d_2sm(stage_a(s, 1), &tmap_a_lo, full_leader, k0, arow);
              }
              ptx::tma_load_2d_2sm(stage_b(s, 0), &tmap_b, full_leader, bk, brow);
              if (kSplit) ptx::tma_load_2d_2sm(stage_b(s, 1), &tmap_b_lo, full_leader, bk, brow);
            }
          } else {
            // CL = 1: my half of the A tile (64 pixels = 8 KB per plane), delivered to both CTAs of the pair
            const int yh = ys + (CL == 1 && p.half_dim == 2 ? (int)cta_rank * p.half_step : 0);
            const int ih = img0 + (CL == 1 && p.half_dim == 3 ? (int)cta_rank * p.half_step : 0);
            const uint32_t off = CL == 1 ? cta_rank * (uint32_t)(kABytes / 2) : 0u;
            const int arow_h = arow + (CL == 1 ? (int)cta_rank * (kTcBM / 2) : 0);
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&full[s], Cfg::kStageBytes);
              if (p.a4d) {
                if constexpr (CL == 1) {
                  ptx::tma_load_4d_mc(stage_a(s, 0) + off, &tmap_a, &full[s], k0, dx, yh, ih, 3);
                  if (kSplit) ptx::tma_load_4d_mc(stage_a(s, 1) + off, &tmap_a_lo, &full[s], k0, dx, yh, ih, 3);
                } else {
                  ptx::tma_load_4d(stage_a(s, 0), &tmap_a, &full[s], k0, dx, ys, img0);
                  if (kSplit) ptx::tma_load_4d(stage_a(s, 1), &tmap_a_lo, &full[s], k0, dx, ys, img0);
                }
              } else if constexpr (CL == 1) {
                ptx::tma_load_2d_mc(stage_a(s, 0) + off, &tmap_a, &full[s], k0, arow_h, 3);
                if (kSplit) ptx::tma_load_2d_mc(stage_a(s, 1) + off, &tmap_a_lo, &full[s], k0, arow_h, 3);
              } else {
                ptx::tma_load_2d(stage_a(s, 0), &tmap_a, &full[s], k0, arow);
                if (kSplit) ptx::tma_load_2d(stage_a(s, 1), &tmap_a_lo, &full[s], k0, arow);
              }
              ptx::tma_load_2d(stage_b(s, 0), &tmap_b, &full[s], bk, brow);
              if (kSplit) ptx::tma_load_2d(stage_b(s, 1), &tmap_b_lo, &full[s], bk, brow);
            }
          }
          __syncwarp();
        }
        if constexpr (kResOK) {
          if (p.has_res) {
            // the tile's residual (128 rows x 128 channels: bf16 = one 32 KB stage, fp16 hi/lo planes = one 64 KB
            // stage) rides the ring: prefetched up to S stages ahead of the epilogue that consumes it, released by
            // the epilogue warps.  Boxes of 64 channels: [hi c0 | hi c0+64 | lo c0 | lo c0+64], 16 KB each
            const int s = it % S;
            ptx::mbar_wait(&empty[s], ((it / S) & 1) ^ 1u);
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&full[s], Cfg::kStageBytes);
              ptx::tma_load_3d(stage_a(s, 0), &tmap_r, &full[s], n_tile * BN, m0, 0);
              ptx::tma_load_3d(stage_a(s, 0) + kABytes, &tmap_r, &full[s], n_tile * BN + 64, m0, 0);
              if constexpr (KIND == kKindF16X2) {
                ptx::tma_load_3d(stage_a(s, 0) + 2 * kABytes, &tmap_r_lo, &full[s], n_tile * BN, m0, 0);
                ptx::tma_load_3d(stage_a(s, 0) + 3 * kABytes, &tmap_r_lo, &full[s], n_tile * BN + 64, m0, 0);
              }
            }
            __syncwarp();
            ++it;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (CL = 2: the leader's, for the pair)
    // The WHOLE warp runs this loop, converged; one elected lane issues the tcgen05 instructions.  Round 1 ran it as
    // `if (lane == 0)`: inside that divergent region ptxas cannot prove any value uniform, and UTCHMMA takes its
    // descriptors / TMEM address from UNIFORM registers — so every MMA was wrapped in an ELECT / R2UR.BROADCAST /
    // BRA.U.ANY loop: 244 SASS instructions per K block of the f16x2 kernel, one thread, ~1650 cycles for 12 MMAs whose
    // tensor-core floor is 768 (ncu source page, profiles/r02_*: the issuing warp never waited on a barrier, the TMA
    // producer sat on a full ring, the epilogue warps on chunk_full — the kernel was ISSUE-bound).  Converged, the
    // operands are warp-uniform by construction (kernel parameters, block index, loop counters, the TMEM base through
    // a shuffle) and the loop shrinks to the MMAs plus a handful of uniform adds.
    if (!kPair2 || cta_rank == 0) {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      // instruction descriptor: D=f32, A/B format (kind::f16: 0 = f16, 1 = bf16; kind::tf32: 2), both K-major,
      // N=BN, M=128
      constexpr uint32_t fmt = KIND == kKindTF32X3 ? 2u : KIND == kKindBF16 ? 1u : 0u;
      // (kMN: bits 15 / 16 = A / B MN-major)
      constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) |
                                 ((uint32_t)((kPair2 ? 2 * kTcBM : kTcBM) >> 4) << 24) | (kMN ? (3u << 15) : 0u);
      auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t acc_flag) {
        if constexpr (KIND == kKindTF32X3) ptx::umma_tf32(d, a, b, idesc, acc_flag);
        else if constexpr (kPair2) ptx::umma_f16_2sm(d, a, b, idesc, acc_flag);
        else ptx::umma_f16(d, a, b, idesc, acc_flag);
      };
      // completion of everything issued so far -> `bar` (CL = 2: the barrier at that offset in BOTH CTAs)
      auto commit = [&](uint64_t* bar) {
        if constexpr (kPair2) ptx::umma_commit_2sm_mc(bar, 3);
        else ptx::umma_commit(bar);
      };
      // smem matrix descriptor (K-major, SWIZZLE_128B): LBO=1, SBO=1024 B, version=1, layout=2.  kMN (MN-major,
      // SWIZZLE_128B): LBO = 8 KB from the first 64 channels to the next 64, SBO = 1024 B from one 8-pixel group to the next
      constexpr uint64_t desc_hi = ((uint64_t)(kMN ? (kABytes / 2) >> 4 : 1) << 16) | ((uint64_t)(1024 >> 4) << 32) |
                                   ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
      static_assert(!kMN || Cfg::kBBytes == kABytes, "kMN: A and B halves are both 8 KB apart");
      // K step of 16: 32 bytes inside the swizzle row (K-major), 16 pixel rows of 128 bytes (MN-major); descriptor units of 16 B
      constexpr uint64_t kStep = kMN ? 128 : 2;
      auto desc = [&](const uint8_t* ptr) { return desc_hi | (uint64_t)((ptx::smem_u32(ptr) >> 4) & 0x3FFF); };
      auto release_stage = [&](int s) {
        if constexpr (CL == 1) ptx::umma_commit_mc(&empty[s], 3);   // the peer multicasts into this stage too
        else commit(&empty[s]);
      };
      uint32_t it = 0, tl = 0, ch = 0;
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++tl) {
        const int acc = tl & 1;
        ptx::mbar_wait(&tmem_empty[acc], ((tl >> 1) & 1) ^ 1u);
        ptx::tc_fence_after();
        if constexpr (!kSplit) {
          const uint32_t d_tmem = tb + (uint32_t)(acc * BN);
          for (int kb = 0; kb < num_kb; ++kb, ++it) {
            const int s = it % S;
            ptx::mbar_wait(&full[s], (it / S) & 1);
            ptx::tc_fence_after();
            const uint64_t da = desc(stage_a(s, 0)), db = desc(stage_b(s, 0));
            if (ptx::elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)    // +32 bytes (= 2 x 16 B) per K step (16 bf16) inside the swizzle row
                mma(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), (kb | k) != 0);
              release_stage(s);                    // smem stage reusable once these MMAs retire
            }
            __syncwarp();
          }
        } else {
          const uint32_t d_corr = tb + (uint32_t)((2 + acc) * BN);
          for (int kb0 = 0; kb0 < num_kb; kb0 += kSplitChunk, ++ch) {
            const int buf = ch & 1;
            ptx::mbar_wait(&chunk_empty[buf], ((ch >> 1) & 1) ^ 1u);
            ptx::tc_fence_after();
            const uint32_t d_main = tb + (uint32_t)(buf * BN);
            const int kb1 = kb0 + kSplitChunk < num_kb ? kb0 + kSplitChunk : num_kb;
            for (int kb = kb0; kb < kb1; ++kb, ++it) {
              const int s = it % S;
              ptx::mbar_wait(&full[s], (it / S) & 1);
              ptx::tc_fence_after();
              const uint64_t da = desc(stage_a(s, 0)), dal = desc(stage_a(s, 1));
              const uint64_t db = desc(stage_b(s, 0)), dbl = desc(stage_b(s, 1));
              const uint32_t first = kb != 0, first_main = kb > kb0;
              if (ptx::elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {        // K step = 8 tf32 / 16 f16 = 32 bytes (kMN: 2 KB)
                  const uint64_t o = kStep * (uint64_t)k;
                  mma(d_corr, dal + o, db + o, k ? 1u : first);            // lo*hi  } whole-tile chain: these
                  mma(d_corr, da + o, dbl + o, 1u);                        // hi*lo  } terms are 2^-11 of the main one
                  mma(d_main, da + o, db + o, k ? 1u : first_main);        // hi*hi, short chain
                }
                release_stage(s);
              }
              __syncwarp();
            }
            if (ptx::elect_one()) commit(&chunk_full[buf]);   // main-term chunk ready to be drained
            __syncwarp();
          }
        }
        if (ptx::elect_one()) commit(&tmem_full[acc]);         // tile (bf16) / correction accumulator (split) complete
        __syncwarp();
        if constexpr (kResOK) {
          if (p.has_res) {
            // The residual stage belongs to the epilogue, but this warp must still OBSERVE its phase: an
            // mbarrier wait can only tell the current phase from the one before it.  Skipping the phase let a
            // later wait on the same stage (S uses on) mistake "residual still loading" for "next K-block
            // landed" whenever the residual's HBM load outlasted S-1 K-blocks of MMAs — the tensor core then
            // consumed the residual as operands and empty[s] got two arrivals: a launch failure once in
            // ~10^7 tiles (found by stressing the encoder; the tests never hit it).
            ptx::mbar_wait(&full[it % S], (it / S) & 1);
            ++it;
          }
        }
      }
    }
  } else {
    // ===================================================================== epilogue (warps 2..)
    const int q = warp & 3;                        // TMEM lane quarter this warp may access
    const int ew = warp - 2;                       // epilogue warp index
    const int cb0 = (ew >> 2) * kCols;             // first tile column owned by this warp
    uint8_t* stage = staging + (size_t)ew * Cfg::kStageBufs * kStageBufBytes;
    int sbuf = 0;                                  // staging buffer of this warp's next store
    uint32_t tl = 0, ch = 0, it_e = 0;             // it_e: ring position of the current tile's residual stage
    EpiScale es;
    if constexpr (KIND == kKindF16X2)
      if (!p.scale_in_rows) es.a_inv = 1.f / __ldcg(p.scale_in);   // powers of two: exact
    if constexpr (OFMT == kFmtF16P) {
      if (p.out_mode != kOutPlanar) {
        float bound = __ldcg(p.amax_in) * __ldg(p.norms) + __ldg(p.norms + 1);
        if constexpr (kResOK)
          if (p.has_res && p.res_amax) bound += __ldcg(p.res_amax);       // |conv + residual| <= bound(conv) + max |residual|
        es.s_out = f16_pow2_scale(bound);
        if (blockIdx.x == 0 && threadIdx.x == 64) *p.scale_out = es.s_out;
      }
    }
    if constexpr (kResOK && KIND == kKindF16X2)
      if (p.has_res) es.r_inv = 1.f / __ldcg(p.res_scale);
    const bool use_tma = Cfg::kTmaStore && p.out_mode != kOutPlanar;
    const float relu_floor = p.relu ? 0.f : -INFINITY;
    for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++tl) {
      const int n_tile = tile % p.n_tiles;
      const int g = (tile / p.n_tiles) % p.groups;
      const int m0 = tile_m0(tile);
      const int acc = tl & 1;
      const int mw = m0 + q * 32;                  // first pixel of this warp
      const int m = mw + lane;                     // this thread's pixel
      const bool row_ok = m < p.M;
      if constexpr (KIND == kKindF16X2)
        if (p.scale_in_rows) es.a_inv = row_ok ? 1.f / __ldcg(p.scale_in_rows + (size_t)g * p.a_group_rows + m) : 1.f;
      const int n0 = n_tile * BN + cb0;            // first output channel of this warp
      const float* __restrict__ bias = p.bias + (size_t)g * p.bias_group_stride;
      const float* __restrict__ wsi = KIND == kKindF16X2 ? p.wsi + (size_t)g * p.wsi_group_stride : nullptr;
      size_t orow = (size_t)(row_ok ? m : 0);
      int img = 0, pix = 0;
      StoreCoord sc{};
      if (p.out_mode == kOutDeconv) {
        img = (int)(orow / HW);
        pix = (int)(orow - (size_t)img * HW);
        const int y = pix / p.W, x = pix - y * p.W;
        orow = ((size_t)img * 2 * p.H + 2 * y + (g >> 1)) * (size_t)(2 * p.W) + 2 * x + (g & 1);
        sc.px = g & 1; sc.py = g >> 1;
        sc.x0 = mw % p.W; sc.r0 = mw / p.W;        // merged (img, y) row index of the warp's first pixel
      } else if (p.out_mode == kOutPlanar) {
        img = (int)(orow / HW);
        pix = (int)(orow - (size_t)img * HW);
      } else {
        sc.m = mw; sc.g = g;
      }
      const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);

      // one finished 32-column slab (fp32, scale/bias/ReLU still to apply) -> its destination
      uint32_t resw[32];               // this thread's 64 residual values (bf16 pairs) of the current tile
      bool has_res_vals = false;
      uint32_t res_row = 0;            // f16x2: smem address of this thread's residual row in the hi box (lo: + 2 boxes)
      bool res_in_smem = false;
      auto emit = [&](const float (&a32)[32], int c, auto half_c, uint32_t (&wh)[32], uint32_t (&wl)[32]) {
        constexpr int half = decltype(half_c)::value;     // which 32-column half of a 64-column store block
        // c = column inside the warp's range; TMA path gathers two slabs (64 columns) per store
        if (!use_tma) {
          store_slab<KIND, OFMT>(p, a32, n0 + c, g, row_ok, orow, img, pix, HW, bias, wsi, es);
          return;
        }
        if constexpr (Cfg::kTmaStore) {
          float v[32];
          finish_slab<KIND>(p, a32, v, n0 + c, bias, wsi, es, (has_res_vals || res_in_smem) ? -INFINITY : relu_floor);
          if (has_res_vals) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              v[2 * j] = fmaxf(v[2 * j] + __uint_as_float(resw[half * 16 + j] << 16), relu_floor);
              v[2 * j + 1] = fmaxf(v[2 * j + 1] + __uint_as_float(resw[half * 16 + j] & 0xffff0000u), relu_floor);
            }
          }
          if constexpr (kResOK && KIND == kKindF16X2) {
            if (res_in_smem) {
              // 32 columns of this row = four 16-byte chunks per plane, at swizzled positions (chunk ^ (row & 7))
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t o = (uint32_t)(((half * 4 + j) ^ (lane & 7)) << 4);
                uint32_t h4[4], l4[4];
                ptx::ld_shared_v4(res_row + o, h4[0], h4[1], h4[2], h4[3]);
                ptx::ld_shared_v4(res_row + 2 * kABytes + o, l4[0], l4[1], l4[2], l4[3]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&h4[e]));
                  const float2 lf = __half22float2(*reinterpret_cast<const __half2*>(&l4[e]));
                  const int c8 = 8 * j + 2 * e;
                  v[c8] = fmaxf(v[c8] + fmaf(lf.x, 1.f / kLoScale, hf.x) * es.r_inv, relu_floor);
                  v[c8 + 1] = fmaxf(v[c8 + 1] + fmaf(lf.y, 1.f / kLoScale, hf.y) * es.r_inv, relu_floor);
                }
              }
            }
          }
          uint32_t h16[16], l16[16];
          encode_slab<OFMT>(v, h16, l16, row_ok, es);
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            wh[half * 16 + e] = h16[e];
            if constexpr (OFMT == kFmtF16P) wl[half * 16 + e] = l16[e];
          }
          if (half == 1) {
            const int c0 = n0 + c - 32;            // first channel of the 64-column block
            if (c0 < p.c_fill) {
              tma_store_block<Cfg::kStageBufs - 1>(p, &tmap_c, stage + sbuf * kStageBufBytes, lane, wh, c0, sc);
              if constexpr (Cfg::kStageBufs > 1) sbuf ^= 1;
              if constexpr (OFMT == kFmtF16P) tma_store_block<0>(p, &tmap_c_lo, stage, lane, wl, c0, sc);
            }
          }
        }
      };

      if constexpr (!kSplit) {
        ptx::mbar_wait(&tmem_full[acc], (tl >> 1) & 1);
        ptx::tc_fence_after();
        uint32_t wh[32], wl[32];
#pragma unroll 1
        for (int c = 0; c < kCols; c += 64) {
          // 64 columns per TMEM round trip (one wait for two loads) when the warp owns that many
          uint32_t r0[32], r1[32];
          ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)(acc * BN + cb0 + c), r0);
          if (kCols >= 64) ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)(acc * BN + cb0 + c + 32), r1);
          ptx::tmem_ld_wait();
          if (c + 64 >= kCols) {
            // all TMEM reads of this accumulator are complete -> hand it back before the stores
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) arrive_issuer(&tmem_empty[acc]);
          }
          if constexpr (kResOK && KIND == kKindBF16) {
            if (p.has_res) {
              // residual stage of this tile: after the tile's K-blocks in ring order
              it_e += (uint32_t)num_kb;
              const int s = it_e % S;
              ptx::mbar_wait(&full[s], (it_e / S) & 1);
              const uint32_t rb = ptx::smem_u32(stage_a(s, 0)) + (uint32_t)((ew >> 2) * kABytes) +
                                  (uint32_t)(q * 32 + lane) * 128u;
#pragma unroll
              for (int j = 0; j < 8; ++j)
                ptx::ld_shared_v4(rb + (uint32_t)((j ^ (lane & 7)) << 4), resw[4 * j], resw[4 * j + 1], resw[4 * j + 2],
                                  resw[4 * j + 3]);
              has_res_vals = true;
              __threadfence_block();
              __syncwarp();
              if (lane == 0 && atomicAdd(&res_cnt[s], 1u) == (uint32_t)(kEpiWarps - 1)) {
                res_cnt[s] = 0;
                ptx::mbar_arrive(&empty[s]);       // last of the 8 warps hands the stage back to the producer
              }
              ++it_e;
            }
          }
          float a32[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) a32[j] = __uint_as_float(r0[j]);
          emit(a32, c, std::integral_constant<int, 0>{}, wh, wl);
          if (kCols >= 64) {
#pragma unroll
            for (int j = 0; j < 32; ++j) a32[j] = __uint_as_float(r1[j]);
            emit(a32, c + 32, std::integral_constant<int, 1>{}, wh, wl);
          }
        }
      } else {
        // running fp32 sum of this thread's output row, round-to-nearest
        float sum[kCols];
#pragma unroll
        for (int j = 0; j < kCols; ++j) sum[j] = 0.f;
        for (int kb0 = 0; kb0 < num_kb; kb0 += kSplitChunk, ++ch) {
          const int buf = ch & 1;
          ptx::mbar_wait(&chunk_full[buf], (ch >> 1) & 1);
          ptx::tc_fence_after();
#pragma unroll
          for (int c = 0; c < kCols; c += 32) {
            uint32_t r[32];
            ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)(buf * BN + cb0 + c), r);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) sum[c + j] += __uint_as_float(r[j]);
          }
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) arrive_issuer(&chunk_empty[buf]);
        }
        ptx::mbar_wait(&tmem_full[acc], (tl >> 1) & 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int c = 0; c < kCols; c += 32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)((2 + acc) * BN + cb0 + c), r);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if constexpr (KIND == kKindF16X2) sum[c + j] = fmaf(__uint_as_float(r[j]), 1.f / kLoScale, sum[c + j]);
            else sum[c + j] += __uint_as_float(r[j]);
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) arrive_issuer(&tmem_empty[acc]);
        if constexpr (kMN) {
          // the slice's raw partial: row ci of (slice, tap) = g, columns co (pitch c_pitch, first c_fill written)
          if (row_ok) {
            float* __restrict__ dst = reinterpret_cast<float*>(p.C) + ((size_t)g * p.M + m) * p.c_pitch + n0;
#pragma unroll
            for (int c = 0; c < kCols; c += 4)
              if (n0 + c < p.c_fill)
                *reinterpret_cast<float4*>(dst + c) = make_float4(sum[c], sum[c + 1], sum[c + 2], sum[c + 3]);
          }
          continue;
        }
        int res_stage = -1;
        if constexpr (kResOK && KIND == kKindF16X2) {
          if (p.has_res) {
            // residual stage of this tile: after the tile's K-blocks in ring order; this warp's 64 columns are box
            // (ew >> 2) of each plane, this thread's row is q * 32 + lane
            it_e += (uint32_t)num_kb;
            res_stage = (int)(it_e % S);
            ptx::mbar_wait(&full[res_stage], (it_e / S) & 1);
            res_row = ptx::smem_u32(stage_a(res_stage, 0)) + (uint32_t)((ew >> 2) * kABytes) + (uint32_t)(q * 32 + lane) * 128u;
            res_in_smem = true;
            ++it_e;
          }
        }
        uint32_t wh[32], wl[32];
#pragma unroll
        for (int c = 0; c < kCols; c += 64) {
          float a32[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) a32[j] = sum[c + j];
          emit(a32, c, std::integral_constant<int, 0>{}, wh, wl);
          if (kCols >= 64) {
#pragma unroll
            for (int j = 0; j < 32; ++j) a32[j] = sum[(c + 32) % kCols + j];
            emit(a32, c + 32, std::integral_constant<int, 1>{}, wh, wl);
          }
        }
        if constexpr (kResOK && KIND == kKindF16X2) {
          if (res_stage >= 0) {
            __threadfence_block();
            __syncwarp();
            if (lane == 0 && atomicAdd(&res_cnt[res_stage], 1u) == (uint32_t)(kEpiWarps - 1)) {
              res_cnt[res_stage] = 0;
              ptx::mbar_arrive(&empty[res_stage]);     // last of the 8 warps hands the stage back to the producer
            }
          }
        }
      }
    }
    if constexpr (Cfg::kTmaStore) {
      if (use_tma && lane == 0) ptx::bulk_wait_all0();
      (void)it_e;     // our stores have landed before the CTA retires
    }
    if constexpr (OFMT == kFmtF16P) {
      if (p.out_mode != kOutPlanar && p.amax_out) {
        float mx = es.amax;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) atomicMax(reinterpret_cast<unsigned int*>(p.amax_out), __float_as_uint(mx));   // mx >= 0
      }
    }
  }

  // ------------------------------------------------------------------ teardown
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CL != 0) ptx::cluster_sync();       // the peer's last stage releases arrive on OUR barriers
  if (warp == 1) {
    ptx::tc_fence_after();
    if constexpr (kPair2) ptx::tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base);
    else ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------
// host side: packed layers, launches, orchestration
struct TcLayer {            // one packed conv: K-major B operand (1 plane bf16 / 2 planes fp32 or fp16) + bias
  int kind = kKindBF16;
  void* w[2] = {nullptr, nullptr};
  float* bias = nullptr;
  float* wsi = nullptr;     // kKindF16X2: per packed row 2^-t
  float* norms = nullptr;   // {max_row ||W'||_1, max |bias'|} (layers whose output is stored in kFmtF16P)
  CUtensorMap map[2];
  int rows = 0, k = 0, k_pitch = 0, bn = 0, n_pad = 0;
};
// Pack modes (TcWeights.kind): 0 = every layer bf16, 1 = every layer 3xTF32,
// 2 = every layer f16x2 (the library's "fp32" precision): the fusion block and the decoder run on scaled fp16 hi/lo
//     planes (half the MMA time of 3xTF32).
enum TcMode { kModeBF16 = 0, kModeTF32X3 = 1, kModeF16X2 = 2 };
static inline int mode_kind(int mode) {
  return mode == kModeBF16 ? kKindBF16 : mode == kModeTF32X3 ? kKindTF32X3 : kKindF16X2;
}
static inline int kind_fmt(int kind) {
  return kind == kKindBF16 ? kFmtBF16 : kind == kKindTF32X3 ? kFmtTF32P : kFmtF16P;
}
struct TcPack {
  int mode = kModeBF16;
  TcLayer cf1, cf2a, cf2b, out, dc[3], fin;
};
struct Act {                // an activation buffer: 1 plane (bf16) or hi/lo planes
  void* p[2] = {nullptr, nullptr};
  int fmt = kFmtBF16;
};
static inline Act act_offset(const Act& a, size_t elems) {
  Act r;
  r.fmt = a.fmt;
  const int elem_bytes = fmt_elem(a.fmt);
  r.p[0] = a.p[0] ? (uint8_t*)a.p[0] + elems * elem_bytes : nullptr;
  r.p[1] = a.p[1] ? (uint8_t*)a.p[1] + elems * elem_bytes : nullptr;
  return r;
}

// Device scalars of the scaled fp16 tensors, one pair per tensor, in the workspace.
struct ScaleSlot {
  float* amax = nullptr;    // max |x| (atomicMax by the producer; zeroed at the start of a forward)
  float* scale = nullptr;   // s
};
// an "fp16 planes" buffer (include/cdrhead.h): [hi plane | lo plane | {amax, scale}] — defined with the encoder
static Act planes_act(const void* buf, size_t rows, int channels, ScaleSlot* sl);

struct TcLaunch {
  Act A;                    // activations
  int a_pitch;
  int n_img, H, W, cin, deconv, groups;
  long long a_rows_total;   // 2-D map: total rows addressable (groups stacked)
  const TcLayer* layer;
  int b_group_rows, n;
  int bias_group_stride;
  Act C;                    // output planes (or planar fp32 heat-maps in C.p[0])
  long long c_group_stride;
  int c_pitch, c_fill, relu, out_mode;
  ScaleSlot in_slot, out_slot;   // kFmtF16P tensors
  const float* in_row_scale;     // overrides in_slot.scale: one scale per A row (2-D A)
  // encoder convs: H, W above are the OUTPUT pixel grid; the input grid is (stride*H, stride*W)
  int conv3;                     // 3x3, pad 1 (9 taps)
  int conv4s2;                   // 4x4, stride 2 (set stride = 2), pad 1 (16 taps)
  int planar_deconv;             // kOutPlanar + deconv: fp32 NCHW output of the 2H x 2W map (phase scatter)
  int stride;                    // 0/1 or 2
  const void* res;               // residual rows (n channels, pitch res_pitch; bf16, or the hi plane of kFmtF16P) added
  const void* res_lo;            // before the ReLU; kFmtF16P: the lo plane and the residual tensor's scale slot
  ScaleSlot res_slot;
  int res_pitch;
  int pair2;                     // run as cta_group::2 CTA pairs (kernel parameter CL = 2) if the geometry allows
};

// The tap-GEMM, decoder-tail and merge kernels are launched with programmatic dependent launch (PDL): the next kernel's
// CTAs take over SMs as ours retire.  Measured on B200: encoder 4.58 -> 4.39 ms, bf16 head 94.9 k -> 97.7 k pairs/s.  `pair`: thread-block clusters
// of 2 CTAs (multicast pairs, cta_group::2 pairs).
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, bool pair, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchAttribute attr[2];
  int n_attr = 0;
  if (pair) {
    attr[n_attr].id = cudaLaunchAttributeClusterDimension;
    attr[n_attr].val.clusterDim.x = 2;
    attr[n_attr].val.clusterDim.y = 1;
    attr[n_attr].val.clusterDim.z = 1;
    ++n_attr;
  }
  attr[n_attr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n_attr].val.programmaticStreamSerializationAllowed = 1;
  ++n_attr;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = n_attr;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// cta_group::2 pairs (kernel template parameter CL = 2).  The pair takes two consecutive 128-pixel blocks: an even number
// of pixel blocks, no residual, unit stride.  Where they pay (measured, see the kernel comment) the caller asks for them
// with TcLaunch::pair2.
static bool tc_pair2_ok(const TcLaunch& l) {
  if (!l.pair2 || l.res || l.stride > 1) return false;
  const long long m = (long long)l.n_img * l.H * l.W;
  return m % (2 * kTcBM) == 0;
}
// can this launch run as multicast CTA pairs (CL = 1)?  the pair shares one A tile: an even number of N tiles per pixel
// block.  Not for residual layers (DESIGN.md §7: measured slower, the pair runs in lock step and a residual stage is only
// free once BOTH epilogues have read theirs).
static bool tc_cluster_ok(const TcLaunch& l, int bn) {
  if (l.res || l.stride > 1 || (l.layer->n_pad / bn) % 2 != 0) return false;
  if (l.deconv || l.conv3) {
    if (l.W > kTcBM || kTcBM % l.W != 0) return false;
    int rows = kTcBM / l.W;
    if (rows > l.H) rows = l.H;
    const int imgs = kTcBM / (l.W * rows);
    return imgs >= 2 ? imgs % 2 == 0 : rows % 2 == 0;
  }
  return true;
}

template <int BN, int KIND, int OFMT, int CL = 0>
static int launch_tc_t(const TcLaunch& l, cudaStream_t st) {
  using Cfg = TcCfg<BN, KIND, OFMT, CL>;
  constexpr int kElem = KindTraits<KIND>::kElem;
  constexpr int kBK = Cfg::kBK;
  constexpr int kAFmt = KindTraits<KIND>::kFmt;
  static DeviceOnce attr_set;   // per instantiation AND per device
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(tap_gemm_tc_kernel<BN, KIND, OFMT, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)Cfg::kSmemBytes));
    attr_set.done();
  }
  TcGemmParams p{};
  const int HW = l.H * l.W;
  p.M = l.n_img * HW;
  p.n_img = l.n_img; p.H = l.H; p.W = l.W; p.cin = l.cin;
  const int stride = l.stride > 1 ? l.stride : 1;
  const bool a4d = l.deconv || l.conv3 || l.conv4s2 || stride > 1;
  p.tap_mode = l.deconv ? kTapDeconv : l.conv3 ? kTapConv3 : l.conv4s2 ? kTapConv4s2 : kTapNone;
  p.ntaps = l.deconv ? 4 : l.conv3 ? 9 : l.conv4s2 ? 16 : 1;
  CDR_CHECK_ARG(!l.conv4s2 || stride == 2, "tap_gemm_tc: the 4x4 tap mode is the stride-2 conv");
  p.planar_deconv = l.planar_deconv;
  CDR_CHECK_ARG(!l.planar_deconv || (l.deconv && l.out_mode == kOutPlanar), "tap_gemm_tc: phase scatter needs a planar deconv");
  p.a4d = a4d;
  p.stride = stride;
  p.has_res = l.res != nullptr;
  p.groups = l.groups;
  p.a_group_rows = a4d ? 0 : p.M;
  p.b_group_rows = l.b_group_rows;
  p.n_tiles = l.layer->n_pad / BN;
  p.n = l.n;
  p.bias = l.layer->bias; p.bias_group_stride = l.bias_group_stride;
  p.C = l.C.p[0]; p.C_lo = l.C.p[1];
  p.c_group_stride = l.c_group_stride; p.c_pitch = l.c_pitch; p.c_fill = l.c_fill;
  p.relu = l.relu; p.out_mode = l.out_mode;
  p.wsi = l.layer->wsi; p.wsi_group_stride = l.b_group_rows;
  p.scale_in = l.in_slot.scale;
  p.scale_in_rows = l.in_row_scale;
  p.amax_in = l.in_slot.amax;
  p.norms = l.layer->norms;
  p.amax_out = l.out_slot.amax; p.scale_out = l.out_slot.scale;
  const int m_tiles = ceil_div(p.M, kTcBM);
  p.num_tiles = m_tiles * p.groups * p.n_tiles;
  if (CL == 2) {                      // the kernel walks PAIR tiles: two consecutive pixel blocks each
    CDR_CHECK_ARG(p.M % (2 * kTcBM) == 0 && !l.res && stride == 1, "tap_gemm_tc: cta_group::2 needs an even number of "
                  "full 128-pixel blocks, unit stride and no residual");
    p.num_tiles = (m_tiles / 2) * p.groups * p.n_tiles;
  }
  CDR_CHECK_ARG(l.layer->bn == BN && l.layer->n_pad % BN == 0, "tap_gemm_tc: layer packed for BN=%d, launched with %d",
                l.layer->bn, BN);
  CDR_CHECK_ARG(p.bias != nullptr, "tap_gemm_tc: every packed layer carries a (possibly zero) bias vector");
  CDR_CHECK_ARG(l.A.fmt == kAFmt, "tap_gemm_tc: A stored as format %d, kernel kind %d wants %d", l.A.fmt, KIND, kAFmt);
  CDR_CHECK_ARG((l.a_pitch * kElem) % 16 == 0 && ((uintptr_t)l.A.p[0] & 15) == 0, "tap_gemm_tc: A pitch/alignment");
  if (l.out_mode != kOutPlanar) {
    CDR_CHECK_ARG(l.C.fmt == OFMT, "tap_gemm_tc: output format %d, kernel writes %d", l.C.fmt, OFMT);
    CDR_CHECK_ARG((l.c_pitch * fmt_elem(OFMT)) % 16 == 0 && (l.c_fill * fmt_elem(OFMT)) % 16 == 0,
                  "tap_gemm_tc: output pitch / fill must be 16-byte multiples");
    if (OFMT == kFmtF16P)
      CDR_CHECK_ARG(p.amax_in && p.norms && p.scale_out, "tap_gemm_tc: fp16-plane output needs its scale slots");
  }
  if (KIND == kKindF16X2) {
    CDR_CHECK_ARG(p.wsi && (p.scale_in || p.scale_in_rows), "tap_gemm_tc: f16x2 operands need their scales");
    CDR_CHECK_ARG(!p.scale_in_rows || !p.a4d, "tap_gemm_tc: per-row scales need a 2-D A operand");
  }

  CUtensorMap tmap_a[2];
  for (int pl = 0; pl < KindTraits<KIND>::kPlanes; ++pl) {
    if (a4d) {
      CDR_CHECK_ARG(l.W <= kTcBM && kTcBM % l.W == 0, "tap_gemm_tc: W=%d must divide 128", l.W);
      int rows = kTcBM / l.W;
      if (rows > l.H) rows = l.H;
      const int imgs = kTcBM / (l.W * rows);
      CDR_CHECK_ARG(l.H % rows == 0 && l.cin % kBK == 0 && stride * l.W <= 256 && stride * rows <= 256,
                    "tap_gemm_tc: unsupported tap-conv geometry");
      p.box_rows = rows; p.box_imgs = imgs;
      int brows = rows, bimgs = imgs;
      if (CL == 1) {                          // each CTA of a pair loads (and multicasts) half of the box
        CDR_CHECK_ARG(stride == 1 && (imgs >= 2 ? imgs % 2 == 0 : rows % 2 == 0), "tap_gemm_tc: box cannot be halved");
        if (imgs >= 2) { bimgs = imgs / 2; p.half_dim = 3; p.half_step = bimgs; }
        else { brows = rows / 2; p.half_dim = 2; p.half_step = brows; }
      }
      const uint64_t iw = (uint64_t)stride * l.W, ih = (uint64_t)stride * l.H;      // input pixel grid
      const uint64_t dims[4] = {(uint64_t)l.cin, iw, ih, (uint64_t)l.n_img};
      const uint64_t strides[3] = {(uint64_t)l.a_pitch, (uint64_t)l.a_pitch * iw, (uint64_t)l.a_pitch * iw * ih};
      // a strided box spans stride*count input pixels and the TMA unit keeps every stride-th of them
      const uint32_t box[4] = {(uint32_t)kBK, (uint32_t)(stride * l.W), (uint32_t)(stride * brows), (uint32_t)bimgs};
      const uint32_t estr[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
      if (int rc = make_tmap(&tmap_a[pl], l.A.p[pl], kAFmt, 4, dims, strides, box, estr)) return rc;
    } else {
      const uint64_t dims[2] = {(uint64_t)l.cin, (uint64_t)l.a_rows_total};
      const uint64_t strides[1] = {(uint64_t)l.a_pitch};
      const uint32_t box[2] = {(uint32_t)kBK, (uint32_t)(CL == 1 ? kTcBM / 2 : kTcBM)};
      if (int rc = make_tmap(&tmap_a[pl], l.A.p[pl], kAFmt, 2, dims, strides, box)) return rc;
    }
  }
  if (KindTraits<KIND>::kPlanes == 1) tmap_a[1] = tmap_a[0];
  // output maps for the TMA-store epilogue: one warp stores 32 pixels x 64 channels per instruction
  CUtensorMap tmap_c[2] = {tmap_a[0], tmap_a[0]};
  if (Cfg::kTmaStore && l.out_mode != kOutPlanar) {
    for (int pl = 0; pl < fmt_planes(OFMT); ++pl) {
      CDR_CHECK_ARG(((uintptr_t)l.C.p[pl] & 15) == 0, "tap_gemm_tc: output alignment");
      if (l.out_mode == kOutDeconv) {
        // (n_img, 2H, 2W, C) seen from one output phase: offset = c + px*C + x*2C + py*2W*C + (img*H + y)*4W*C
        CDR_CHECK_ARG(l.W == 8 || l.W == 16 || l.W == 32, "tap_gemm_tc: deconv store box needs W in {8,16,32}");
        const uint64_t cp = (uint64_t)l.c_pitch;
        const uint64_t dims[5] = {(uint64_t)l.c_fill, 2, (uint64_t)l.W, 2, (uint64_t)l.n_img * l.H};
        const uint64_t strides[4] = {cp, 2 * cp, 2 * (uint64_t)l.W * cp, 4 * (uint64_t)l.W * cp};
        const uint32_t box[5] = {64, 1, (uint32_t)l.W, 1, (uint32_t)(32 / l.W)};
        if (int rc = make_tmap(&tmap_c[pl], l.C.p[pl], OFMT, 5, dims, strides, box)) return rc;
      } else {
        const uint64_t gs = l.groups > 1 ? (uint64_t)l.c_group_stride : (uint64_t)p.M * l.c_pitch;
        CDR_CHECK_ARG(gs % 8 == 0, "tap_gemm_tc: output group stride must be a 16-byte multiple");
        const uint64_t dims[3] = {(uint64_t)l.c_fill, (uint64_t)p.M, (uint64_t)l.groups};
        const uint64_t strides[2] = {(uint64_t)l.c_pitch, gs};
        const uint32_t box[3] = {64, 32, 1};
        if (int rc = make_tmap(&tmap_c[pl], l.C.p[pl], OFMT, 3, dims, strides, box)) return rc;
      }
    }
    if (fmt_planes(OFMT) == 1) tmap_c[1] = tmap_c[0];
  }
  CUtensorMap tmap_r = tmap_a[0], tmap_r_lo = tmap_a[0];
  if (l.res) {
    constexpr bool kResKernel = BN == 128 && CL != 2 && ((KIND == kKindBF16 && OFMT == kFmtBF16) ||
                                                         (KIND == kKindF16X2 && OFMT == kFmtF16P));
    CDR_CHECK_ARG(kResKernel && l.out_mode == kOutRows && l.groups == 1 && l.n % BN == 0 && l.c_fill == l.n,
                  "tap_gemm_tc: the residual add needs the bf16 / f16x2 BN=128 kernel and a multiple of 128 channels");
    CDR_CHECK_ARG(((uintptr_t)l.res & 15) == 0 && (l.res_pitch * 2) % 16 == 0, "tap_gemm_tc: residual alignment");
    const uint64_t dims[3] = {(uint64_t)l.c_fill, (uint64_t)p.M, 1};
    const uint64_t strides[2] = {(uint64_t)l.res_pitch, (uint64_t)p.M * l.res_pitch};
    const uint32_t box[3] = {64, 128, 1};     // half a residual tile: 128 rows x 64 channels
    if (int rc = make_tmap(&tmap_r, l.res, OFMT, 3, dims, strides, box)) return rc;
    if (OFMT == kFmtF16P) {
      CDR_CHECK_ARG(l.res_lo && ((uintptr_t)l.res_lo & 15) == 0 && l.res_slot.scale && l.res_slot.amax,
                    "tap_gemm_tc: an fp16-plane residual needs its lo plane and scale slot");
      if (int rc = make_tmap(&tmap_r_lo, l.res_lo, OFMT, 3, dims, strides, box)) return rc;
      p.res_scale = l.res_slot.scale; p.res_amax = l.res_slot.amax;
    }
  }
  // weight maps: the layer's own (box = BN rows), or for cta_group::2 a box of BN/2 rows — each CTA stages its half
  CUtensorMap tmap_b[2] = {l.layer->map[0], l.layer->map[KindTraits<KIND>::kPlanes - 1]};
  if (CL == 2) {
    for (int pl = 0; pl < KindTraits<KIND>::kPlanes; ++pl) {
      const uint64_t dims[2] = {(uint64_t)l.layer->k, (uint64_t)l.layer->rows};
      const uint64_t strides[1] = {(uint64_t)l.layer->k_pitch};
      const uint32_t box[2] = {(uint32_t)kBK, (uint32_t)(BN / 2)};
      if (int rc = make_tmap(&tmap_b[pl], l.layer->w[pl], kAFmt, 2, dims, strides, box)) return rc;
    }
    if (KindTraits<KIND>::kPlanes == 1) tmap_b[1] = tmap_b[0];
  }
  int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  if (CL == 2) grid = 2 * p.num_tiles < num_sms() ? 2 * p.num_tiles : num_sms();     // two CTAs per pair tile
  if (CL) {
    // CL = 1: CTA 2i / 2i+1 take tiles t / t+1 = the two N tiles of one pixel block, for the same number of rounds
    if (CL == 1)
      CDR_CHECK_ARG(p.n_tiles % 2 == 0, "tap_gemm_tc: CTA pairs need an even number of N tiles");
    grid &= ~1;
  }
  CDR_CUDA(launch_pdl(tap_gemm_tc_kernel<BN, KIND, OFMT, CL>, grid, Cfg::kThreads, Cfg::kSmemBytes, CL != 0, st, tmap_a[0],
                      tmap_a[1], tmap_b[0], tmap_b[1], tmap_c[0], tmap_c[1], tmap_r, tmap_r_lo, p));
  CDR_LAUNCH_OK("tap_gemm_tc_kernel");
  return CDR_OK;
}

static int launch_tc(const TcLaunch& l, cudaStream_t st) {
  const int bn = l.layer->bn, kind = l.layer->kind;
  const int ofmt = l.out_mode == kOutPlanar ? kind_fmt(kind) : l.C.fmt;
  if (kind == kKindBF16 && ofmt == kFmtBF16) {
    if (bn == 256 && tc_pair2_ok(l)) return launch_tc_t<256, kKindBF16, kFmtBF16, 2>(l, st);
    if (bn == 256) return launch_tc_t<256, kKindBF16, kFmtBF16>(l, st);
    if (bn == 128) return launch_tc_t<128, kKindBF16, kFmtBF16>(l, st);
    if (bn == 64) return launch_tc_t<64, kKindBF16, kFmtBF16>(l, st);
    if (bn == 32) return launch_tc_t<32, kKindBF16, kFmtBF16>(l, st);
  } else if (kind == kKindTF32X3 && ofmt == kFmtTF32P) {
    if (bn == 128) return launch_tc_t<128, kKindTF32X3, kFmtTF32P>(l, st);
    if (bn == 32) return launch_tc_t<32, kKindTF32X3, kFmtTF32P>(l, st);
  } else if (kind == kKindF16X2 && ofmt == kFmtF16P) {
    if (bn == 128 && tc_pair2_ok(l)) return launch_tc_t<128, kKindF16X2, kFmtF16P, 2>(l, st);
    if (bn == 128 && tc_cluster_ok(l, bn)) return launch_tc_t<128, kKindF16X2, kFmtF16P, 1>(l, st);
    if (bn == 128) return launch_tc_t<128, kKindF16X2, kFmtF16P>(l, st);
    if (bn == 32) return launch_tc_t<32, kKindF16X2, kFmtF16P>(l, st);
  }
  set_error("tap_gemm_tc: no kernel for kind %d BN %d output format %d", kind, bn, ofmt);
  return CDR_ERR_UNSUPPORTED;
}

// ------------------------------------------------------------------------------------------
// fused decoder tail: deconv3 + final 1x1 + soft-argmax partials (tail_tc.cuh)
}  // namespace cdr
#include "tail_tc.cuh"
#include "tail_pair_tc.cuh"
namespace cdr {

// CDR_FUSED_TAIL=0 keeps deconv3 / final 1x1 / soft-argmax as three launches (the tests' reference for the fused tail).  Read at
// every forward (one getenv) so a test can compare both paths inside one process.
static bool tc_use_fused_tail() {
  const char* e = getenv("CDR_FUSED_TAIL");
  return !(e && e[0] == '0');
}

struct TailLaunch {
  Act A;                    // d2: (n_img, 32, 32, 256) pixel-major
  int n_img, joints;
  const TcLayer* dc3;       // packed deconv3
  const TcLayer* fin;       // packed final layer (32 padded rows)
  ScaleSlot in_slot;        // f16x2: scale / amax of d2
  float* heat;              // optional planar heat-maps
  float4* part;             // optional soft-argmax partial records
};

// bf16: the single-CTA kernel of tail_tc.cuh
static int launch_tail(const TailLaunch& l, cudaStream_t st) {
  using Cfg = TailCfg;
  static DeviceOnce attr_set;
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(deconv_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes));
    attr_set.done();
  }
  CDR_CHECK_ARG(l.A.fmt == kFmtBF16 && l.dc3->kind == kKindBF16 && l.fin->kind == kKindBF16 && l.dc3->bn == Cfg::kBN &&
                    l.fin->n_pad == 32 && l.joints <= 32 && (l.heat || l.part),
                "deconv_tail: operand formats / packing do not match the kernel");
  CUtensorMap tmap_a;
  {
    const uint64_t dims[4] = {(uint64_t)kDecC, 32, 32, (uint64_t)l.n_img};
    const uint64_t strides[3] = {(uint64_t)kDecC, (uint64_t)kDecC * 32, (uint64_t)kDecC * 1024};
    const uint32_t box[4] = {64, 32, 4, 1};
    if (int rc = make_tmap(&tmap_a, l.A.p[0], kFmtBF16, 4, dims, strides, box)) return rc;
  }
  TailParams p{};
  p.n_img = l.n_img;
  p.num_units = (l.n_img * 1024 / kTcBM) * 4;
  p.joints = l.joints;
  p.bias = l.dc3->bias;
  p.bias_fin = l.fin->bias;
  p.heat = l.heat;
  p.part = l.part;
  const int grid = p.num_units < num_sms() ? p.num_units : num_sms();
  CDR_CUDA(launch_pdl(deconv_tail_kernel, grid, kTailThreads, Cfg::kSmemBytes, false, st, tmap_a, l.dc3->map[0],
                      l.fin->map[0], p));
  CDR_LAUNCH_OK("deconv_tail_kernel");
  return CDR_OK;
}

// f16x2: the same on cta_group::2 CTA pairs (tail_pair_tc.cuh).  Measured on B200 at B = 64: f16x2 653 -> 556 us; the bf16
// tail on pairs went 200 -> 203 us (its tile is 256 channels wide — operand reads were never its limit).
static int launch_tail_pair(const TailLaunch& l, cudaStream_t st) {
  using Cfg = TailPairCfg;
  static DeviceOnce attr_set;
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(deconv_tail_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes));
    attr_set.done();
  }
  CDR_CHECK_ARG(l.A.fmt == kFmtF16P && l.dc3->kind == kKindF16X2 && l.fin->kind == kKindF16X2 && l.dc3->bn == Cfg::kBN &&
                    l.fin->n_pad == 32 && l.joints <= 32 && (l.heat || l.part),
                "deconv_tail_pair: operand formats / packing do not match the kernel");
  CUtensorMap tmap_a[2], tmap_b[2], tmap_w16;
  for (int pl = 0; pl < 2; ++pl) {
    const uint64_t dims[4] = {(uint64_t)kDecC, 32, 32, (uint64_t)l.n_img};
    const uint64_t strides[3] = {(uint64_t)kDecC, (uint64_t)kDecC * 32, (uint64_t)kDecC * 1024};
    const uint32_t box[4] = {64, 32, 4, 1};
    if (int rc = make_tmap(&tmap_a[pl], l.A.p[pl], kFmtF16P, 4, dims, strides, box)) return rc;
    // each CTA of the pair stages half of the weight tile: a box of BN/2 rows
    const uint64_t bdims[2] = {(uint64_t)l.dc3->k, (uint64_t)l.dc3->rows};
    const uint64_t bstr[1] = {(uint64_t)l.dc3->k_pitch};
    const uint32_t bbox[2] = {64, (uint32_t)(Cfg::kBN / 2)};
    if (int rc = make_tmap(&tmap_b[pl], l.dc3->w[pl], kFmtF16P, 2, bdims, bstr, bbox)) return rc;
  }
  {   // 16-row boxes of the final layer's (hi) plane: each CTA's half of an N = 32 operand
    const uint64_t dims[2] = {(uint64_t)l.fin->k, (uint64_t)l.fin->rows};
    const uint64_t strides[1] = {(uint64_t)l.fin->k_pitch};
    const uint32_t box[2] = {64, 16};
    if (int rc = make_tmap(&tmap_w16, l.fin->w[0], kFmtF16P, 2, dims, strides, box)) return rc;
  }
  TailParams p{};
  p.n_img = l.n_img;
  p.num_units = (l.n_img * 1024 / kTcBM) * 4;
  p.joints = l.joints;
  p.bias = l.dc3->bias;
  p.wsi = l.dc3->wsi;
  p.scale_in = l.in_slot.scale;
  p.amax_in = l.in_slot.amax;
  p.norms = l.dc3->norms;
  p.bias_fin = l.fin->bias;
  p.wsi_fin = l.fin->wsi;
  p.heat = l.heat;
  p.part = l.part;
  CDR_CHECK_ARG(p.wsi && p.scale_in && p.amax_in && p.norms && p.wsi_fin, "deconv_tail_pair: f16x2 operands need their scales");
  int grid = p.num_units < num_sms() ? p.num_units : num_sms();
  grid &= ~1;
  CDR_CUDA(launch_pdl(deconv_tail_pair_kernel, grid, kTailThreads, Cfg::kSmemBytes, true, st, tmap_a[0], tmap_a[1], tmap_b[0],
                      tmap_b[1], l.fin->map[0], l.fin->map[1], tmap_w16, p));
  CDR_LAUNCH_OK("deconv_tail_pair_kernel");
  return CDR_OK;
}

static int launch_tail_merge(const float4* part, const float* P_l, const float* P_r, int batch, int joints, float scale,
                             float* kp_l, float* kp_r, float* xyz, cudaStream_t st) {
  TailMergeParams p{};
  p.part = part;
  p.P[0] = P_l; p.P[1] = P_r;
  p.kp[0] = kp_l; p.kp[1] = kp_r;
  p.xyz = xyz;
  p.batch = batch; p.joints = joints; p.scale = scale;
  // PDL: its launch latency hides behind the tail kernel (which lets dependents launch early); a half-warp per heat-map
  CDR_CUDA(launch_pdl(tail_merge_dlt_kernel, batch, 32 * (joints < 1 ? 1 : joints > 32 ? 32 : joints), 0, false, st, p));
  CDR_LAUNCH_OK("tail_merge_dlt_kernel");
  return CDR_OK;
}

// ------------------------------------------------------------------------------------------
// weight packing (K-major B operands) — BN folded in fp64 as in pack.cu
constexpr double kBnEpsTc = 1e-5;
__device__ __forceinline__ double tc_bn_scale(const CdrConvBn& s, int co) {
  return s.bn_weight ? (double)s.bn_weight[co] / sqrt((double)s.bn_var[co] + kBnEpsTc) : 1.0;
}
__device__ __forceinline__ float tc_folded_bias(const CdrConvBn& s, int co) {
  const double b = s.bias ? (double)s.bias[co] : 0.0;
  if (!s.bn_weight) return (float)b;
  return (float)((b - (double)s.bn_mean[co]) * tc_bn_scale(s, co) + (double)s.bn_bias[co]);
}
// folded weight of a 1x1 conv (Cout,Cin) at packed position (n, k)
__device__ __forceinline__ float conv1x1_weight(const CdrConvBn& s, int cout, int cin, int n, int k) {
  if (n >= cout || k >= cin) return 0.f;
  return (float)((double)s.weight[(size_t)n * cin + k] * tc_bn_scale(s, n));
}
// folded weight of a transposed conv (Cin,Cout,4,4) at packed position (phase, n, tap*Cin + ci).  kK = 3: the weight
// is (Cin,Cout,3,3), read as its 4x4 zero-padding at index 3 (a 3x3 stride-2 pad-1 conv's data gradient)
template <int kK = 4>
__device__ __forceinline__ float deconv_weight(const CdrConvBn& s, int cin, int cout, int phase, int n, int kk) {
  if (n >= cout) return 0.f;
  const int tap = kk / cin, ci = kk - tap * cin;
  const int py = phase >> 1, px = phase & 1, ty = tap >> 1, tx = tap & 1;
  const int ky = 1 - py + 2 * ty, kx = 1 - px + 2 * tx;
  if constexpr (kK == 3) {
    if (ky == 3 || kx == 3) return 0.f;
  }
  return (float)((double)s.weight[(((size_t)ci * cout + n) * kK + ky) * kK + kx] * tc_bn_scale(s, n));
}
template <bool kSplit>
__device__ __forceinline__ void store_weight(void* w0, void* w1, long long idx, float v) {
  if constexpr (kSplit) {
    float hi, lo;
    split_tf32(v, hi, lo);
    reinterpret_cast<float*>(w0)[idx] = hi;
    reinterpret_cast<float*>(w1)[idx] = lo;
  } else {
    reinterpret_cast<__nv_bfloat16*>(w0)[idx] = __float2bfloat16_rn(v);
  }
}
// (Cout,Cin) -> [n_pad][k_pitch]
template <bool kSplit>
__global__ void pack_conv1x1_tc_kernel(CdrConvBn s, int cout, int cin, int k_pitch, int n_pad, void* w0,
                                       void* w1, float* __restrict__ bias_out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n_pad) bias_out[idx] = idx < cout ? tc_folded_bias(s, (int)idx) : 0.f;
  if (idx >= (long long)n_pad * k_pitch) return;
  const int n = (int)(idx / k_pitch), k = (int)(idx % k_pitch);
  store_weight<kSplit>(w0, w1, idx, conv1x1_weight(s, cout, cin, n, k));
}
// (Cin,Cout,4,4) -> [phase][n_pad][tap*Cin + ci]
template <bool kSplit>
__global__ void pack_deconv_tc_kernel(CdrConvBn s, int cin, int cout, int n_pad, void* w0, void* w1,
                                      float* __restrict__ bias_out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n_pad) bias_out[idx] = idx < cout ? tc_folded_bias(s, (int)idx) : 0.f;
  const long long K = 4LL * cin, total = 4LL * n_pad * K;
  if (idx >= total) return;
  const int kk = (int)(idx % K);
  long long r = idx / K;
  const int n = (int)(r % n_pad), phase = (int)(r / n_pad);
  store_weight<kSplit>(w0, w1, idx, deconv_weight(s, cin, cout, phase, n, kk));
}

// One block per packed weight row: max |w| and ||w||_1 of the row (block reduction), then the row scaled by 2^t (max lands
// in [2^13, 2^14)) as fp16 hi/lo planes, wsi[row] = 2^-t, and (norms != NULL) atomicMax of the row's L1 norm and |bias|
// into norms[0..1] (the output-scale bound).
// folded weight of a conv (Cout,Cin,kh,kw) with `taps` = kh*kw at packed position (n, tap*Cin + ci), tap = ky*kw + kx
__device__ __forceinline__ float conv_taps_weight(const CdrConvBn& s, int cout, int cin, int taps, int n, int kk) {
  if (n >= cout || kk >= taps * cin) return 0.f;
  const int tap = kk / cin, ci = kk - tap * cin;
  return (float)((double)s.weight[((size_t)n * cin + ci) * taps + tap] * tc_bn_scale(s, n));
}
// the data-gradient operand W^T at packed position (ci, tap*Cout + co): kTaps = 16, a transposed conv's weight
// (Cin,Cout,4,4) with tap = ky*4 + kx; kTaps = 9, a 3x3 conv's weight (Cout,Cin,3,3) with the taps flipped,
// W[co][ci][2 - ky][2 - kx] for tap = ky*3 + kx; kTaps = 1, a 1x1 conv's weight (Cout,Cin).  Zero in the padded rows
// and K pitch.
template <int kTaps>
__device__ __forceinline__ float dgrad_weight(const CdrConvBn& s, int cin, int cout, int ci, int kk) {
  if (ci >= cin || kk >= kTaps * cout) return 0.f;
  const int tap = kk / cout, co = kk - tap * cout;
  if constexpr (kTaps == 1) return s.weight[(size_t)co * cin + ci];
  if constexpr (kTaps == 9) return s.weight[((size_t)co * cin + ci) * 9 + (8 - tap)];
  return s.weight[((size_t)ci * cout + co) * kTaps + tap];
}
// kDeconv: 0 = 1x1 conv, 1 = transposed conv (4 phases; kDeconvK = 3 reads a 3x3 weight, see deconv_weight), >= 2: conv
// with kDeconv taps in encoder order (use 9; the 1x1 convs of the encoder go through mode 0), < 0:
// dgrad_weight<-kDeconv> (`cout` = Cin rows, `cin` = Cout per tap)
template <int kDeconv, int kDeconvK = 4>
__global__ void __launch_bounds__(256)
pack_rows_f16_kernel(CdrConvBn s, int cout, int cin, int k_pitch, int n_pad, __half* __restrict__ w_hi,
                     __half* __restrict__ w_lo, float* __restrict__ wsi, float* __restrict__ bias_out,
                     float* __restrict__ norms) {
  __shared__ float red_max[8], red_sum[8];
  const int row = blockIdx.x;
  const int n = row % n_pad, phase = row / n_pad;
  auto val = [&](int kk) -> float {
    if constexpr (kDeconv >= 2) return conv_taps_weight(s, cout, cin, kDeconv, n, kk);
    if constexpr (kDeconv < 0) return dgrad_weight<-kDeconv>(s, cout, cin, n, kk);
    return kDeconv ? deconv_weight<kDeconvK>(s, cin, cout, phase, n, kk) : conv1x1_weight(s, cout, cin, n, kk);
  };
  float mx = 0.f, l1 = 0.f;
  for (int kk = threadIdx.x; kk < k_pitch; kk += blockDim.x) {
    const float a = fabsf(val(kk));
    mx = fmaxf(mx, a);
    l1 += a;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    l1 += __shfl_xor_sync(0xffffffffu, l1, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red_max[threadIdx.x >> 5] = mx;
    red_sum[threadIdx.x >> 5] = l1;
  }
  __syncthreads();
  mx = 0.f;
  l1 = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) {
    mx = fmaxf(mx, red_max[i]);
    l1 += red_sum[i];
  }
  const int t = f16_pow2_exp(mx);
  if (threadIdx.x == 0) {
    const float b = n < cout ? tc_folded_bias(s, n) : 0.f;
    wsi[row] = ldexpf(1.f, -t);
    if (phase == 0) bias_out[n] = b;
    if (norms) {
      atomicMax(reinterpret_cast<unsigned int*>(norms), __float_as_uint(l1 * 1.001f));   // non-negative floats
      atomicMax(reinterpret_cast<unsigned int*>(norms + 1), __float_as_uint(fabsf(b)));
    }
  }
  const float up = ldexpf(1.f, t);
  for (int kk = threadIdx.x; kk < k_pitch; kk += blockDim.x) {
    const float X = val(kk) * up;
    const __half h = __float2half_rn(X);
    w_hi[(size_t)row * k_pitch + kk] = h;
    w_lo[(size_t)row * k_pitch + kk] = __float2half_rn((X - __half2float(h)) * kLoScale);
  }
}

// plane(s) -> fp32 (parity taps)
__global__ void act_to_f32_kernel(const void* __restrict__ p0, const void* __restrict__ p1, int fmt,
                                  const float* __restrict__ scale, float* __restrict__ out, long long rows,
                                  int in_pitch, int cols) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  const long long r = idx / cols;
  const int c = (int)(idx - r * cols);
  const long long i = r * in_pitch + c;
  if (fmt == kFmtTF32P)
    out[idx] = reinterpret_cast<const float*>(p0)[i] + reinterpret_cast<const float*>(p1)[i];
  else if (fmt == kFmtF16P)
    out[idx] = (__half2float(reinterpret_cast<const __half*>(p0)[i]) +
                __half2float(reinterpret_cast<const __half*>(p1)[i]) * (1.f / kLoScale)) / *scale;
  else
    out[idx] = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p0)[i]);
}

// ------------------------------------------------------------------------------------------
static const int kTcDcCin[3] = {kFeatC, kDecC, kDecC};

struct Bump1K {
  uint8_t* base;
  size_t off = 0;
  explicit Bump1K(void* b) : base((uint8_t*)b) {}
  void* take(size_t bytes) {
    void* r = base ? base + off : nullptr;
    off += round_up<size_t>(bytes, 1024);
    return r;
  }
};

static void plan_layer(TcLayer& L, Bump1K& b, int kind, int rows, int k, int k_pitch, int bn, int n_pad, int bias_n,
                       bool want_norms) {
  const int elem = (kind == kKindTF32X3 ? 4 : 2);
  L.kind = kind;
  L.rows = rows; L.k = k; L.k_pitch = k_pitch; L.bn = bn; L.n_pad = n_pad;
  L.w[0] = b.take((size_t)rows * k_pitch * elem);
  L.w[1] = kind != kKindBF16 ? b.take((size_t)rows * k_pitch * elem) : nullptr;
  L.bias = (float*)b.take((size_t)bias_n * sizeof(float));
  L.wsi = kind == kKindF16X2 ? (float*)b.take((size_t)rows * sizeof(float)) : nullptr;
  L.norms = want_norms ? (float*)b.take(2 * sizeof(float)) : nullptr;
}

static size_t plan_tc_weights(TcPack& pk, const TcWeights& w, void* base) {
  Bump1K b(base);
  const int k = mode_kind(pk.mode);
  const int bn = k == kKindBF16 ? 256 : 128;
  const bool f16 = k == kKindF16X2;        // every output but the heat-maps is stored in kFmtF16P: each layer needs its norms
  if (w.has_fusion) {
    const FusionDims& fd = w.fd;
    const int n1 = fd.n1_pad(), n2 = fd.n2_pad();
    plan_layer(pk.cf1, b, k, n1, kFeatC, kFeatC, 128, n1, n1, f16);
    plan_layer(pk.cf2a, b, k, n2, 2 * fd.h2, 2 * fd.h2, 128, n2, n2, f16);
    plan_layer(pk.cf2b, b, k, n2, fd.h2, fd.h2, 128, n2, n2, f16);
    plan_layer(pk.out, b, k, 2 * kFeatC, fd.h1, fd.h1p, bn, kFeatC, 2 * kFeatC, f16);
  }
  for (int i = 0; i < 3; ++i)
    plan_layer(pk.dc[i], b, k, 4 * kDecC, 4 * kTcDcCin[i], 4 * kTcDcCin[i], bn, kDecC, kDecC, f16);
  plan_layer(pk.fin, b, k, w.fin_npad, kDecC, kDecC, 32, w.fin_npad, w.fin_npad, false);
  return b.off;
}

static int layer_maps(TcLayer& L) {
  const int fmt = kind_fmt(L.kind);
  const int bk = L.kind == kKindTF32X3 ? 32 : 64;
  for (int pl = 0; pl < fmt_planes(fmt); ++pl) {
    const uint64_t dims[2] = {(uint64_t)L.k, (uint64_t)L.rows};
    const uint64_t strides[1] = {(uint64_t)L.k_pitch};
    const uint32_t box[2] = {(uint32_t)bk, (uint32_t)L.bn};
    if (int rc = make_tmap(&L.map[pl], L.w[pl], fmt, 2, dims, strides, box)) return rc;
  }
  return CDR_OK;
}

int tc_weights_create(const CdrWeightPtrs& src, int mode, TcWeights& w, cudaStream_t st) {
  w.joints = src.num_joints;
  w.has_fusion = src.has_fusion;
  w.fin_npad = round_up(src.num_joints, 32);
  w.kind = mode;
  w.fd = make_fusion_dims(src.fusion_hid_ch1, src.fusion_hid_ch2);     // validated by cdr_weights_create
  TcPack* pk = new TcPack();
  pk->mode = mode;
  w.impl = pk;
  const size_t bytes = plan_tc_weights(*pk, w, nullptr);
  CDR_CUDA(cudaMalloc(&w.pool, bytes));
  CDR_CUDA(cudaMemsetAsync(w.pool, 0, bytes, st));      // norms start at 0 for the atomicMax
  plan_tc_weights(*pk, w, w.pool);
  // 1x1 conv (cout, cin) into rows [row_off, row_off + rows) of layer L
  auto pack1 = [&](const CdrConvBn& s, int cout, int cin, TcLayer& L, size_t row_off, size_t bias_off) -> int {
    const int rows = cout <= L.n_pad ? L.n_pad : cout;   // rows packed by this call
    const long long total = (long long)rows * L.k_pitch;
    const int elem = (L.kind == kKindTF32X3 ? 4 : 2);
    void* w0 = (uint8_t*)L.w[0] + row_off * L.k_pitch * elem;
    void* w1 = L.w[1] ? (uint8_t*)L.w[1] + row_off * L.k_pitch * elem : nullptr;
    const unsigned grid = (unsigned)ceil_div<long long>(total, 256);
    if (L.kind == kKindF16X2) {
      pack_rows_f16_kernel<0><<<rows, 256, 0, st>>>(s, cout, cin, L.k_pitch, rows, (__half*)w0, (__half*)w1, L.wsi + row_off,
                                                    L.bias + bias_off, L.norms);
      CDR_LAUNCH_OK("pack_rows_f16_kernel");
      return CDR_OK;
    }
    if (L.kind == kKindTF32X3)
      pack_conv1x1_tc_kernel<true><<<grid, 256, 0, st>>>(s, cout, cin, L.k_pitch, rows, w0, w1, L.bias + bias_off);
    else
      pack_conv1x1_tc_kernel<false><<<grid, 256, 0, st>>>(s, cout, cin, L.k_pitch, rows, w0, w1, L.bias + bias_off);
    CDR_LAUNCH_OK("pack_conv1x1_tc_kernel");
    return CDR_OK;
  };
  int rc;
  if (w.has_fusion) {
    const FusionDims& fd = w.fd;
    if ((rc = pack1(src.cf_conv1, fd.h1, kFeatC, pk->cf1, 0, 0))) return rc;
    if ((rc = pack1(src.cf_conv2a, fd.h2, 2 * fd.h2, pk->cf2a, 0, 0))) return rc;
    if ((rc = pack1(src.cf_conv2b, fd.h2, fd.h2, pk->cf2b, 0, 0))) return rc;
    for (int v = 0; v < 2; ++v)
      if ((rc = pack1(src.cf_out[v], kFeatC, fd.h1, pk->out, (size_t)v * kFeatC, (size_t)v * kFeatC))) return rc;
    if ((rc = layer_maps(pk->cf1)) || (rc = layer_maps(pk->cf2a)) || (rc = layer_maps(pk->cf2b)) ||
        (rc = layer_maps(pk->out)))
      return rc;
  }
  for (int i = 0; i < 3; ++i) {
    TcLayer& L = pk->dc[i];
    const int K = 4 * kTcDcCin[i];
    if (L.kind == kKindF16X2) {
      pack_rows_f16_kernel<1><<<4 * kDecC, 256, 0, st>>>(src.deconv[i], kDecC, kTcDcCin[i], K, kDecC,
                                                                  (__half*)L.w[0], (__half*)L.w[1], L.wsi, L.bias, L.norms);
      CDR_LAUNCH_OK("pack_rows_f16_kernel");
    } else {
      const long long total = 4LL * kDecC * K;
      const unsigned grid = (unsigned)ceil_div<long long>(total, 256);
      if (L.kind == kKindTF32X3)
        pack_deconv_tc_kernel<true><<<grid, 256, 0, st>>>(src.deconv[i], kTcDcCin[i], kDecC, kDecC, L.w[0], L.w[1], L.bias);
      else
        pack_deconv_tc_kernel<false><<<grid, 256, 0, st>>>(src.deconv[i], kTcDcCin[i], kDecC, kDecC, L.w[0], L.w[1], L.bias);
      CDR_LAUNCH_OK("pack_deconv_tc_kernel");
    }
    if ((rc = layer_maps(L))) return rc;
  }
  if ((rc = pack1(src.final_layer, w.joints, kDecC, pk->fin, 0, 0))) return rc;
  return layer_maps(pk->fin);
}

void tc_weights_destroy(TcWeights& w) {
  if (w.pool) cudaFree(w.pool);
  w.pool = nullptr;
  delete (TcPack*)w.impl;
  w.impl = nullptr;
}

// ------------------------------------------------------------------------------------------
constexpr int kNumSlots = 12;      // ScaleSlot pairs: 0 unused, 1 x1, 2 d1, 3 d2, 4 d3, 5 x0 (f16x2 mode);
                                   // fp16 fusion block: 6 y1, 7 z, 8 f1, 9 f2, 10 g, 11 {max row L1 of P+, of P}
struct TcHeadWs {
  float* pinv;
  float* slots;
  float* x0_rs;             // f16x2 mode: one scale per x0 row (layout.cu: nchw_to_rows_f16p_rowscale_kernel)
  Act x0, y1, z, f1, f2, g, x1, d1, d2, d3;
  float* hm;
  float4* part;             // fused decoder tail: soft-argmax partial records (2B, J, kTailSlots)
  size_t bytes;
};
static ScaleSlot slot(float* slots, int i) {
  ScaleSlot s;
  s.amax = slots + 2 * i;
  s.scale = slots + 2 * i + 1;
  return s;
}
static Act take_act(Bump1K& b, size_t elems, int fmt) {
  Act a;
  a.fmt = fmt;
  a.p[0] = b.take(elems * fmt_elem(fmt));
  a.p[1] = fmt_planes(fmt) == 2 ? b.take(elems * fmt_elem(fmt)) : nullptr;
  return a;
}
static TcHeadWs plan_tc_head(void* base, int B, int J, int mode, const FusionDims& fd) {
  Bump1K b(base);
  const size_t N = 2 * (size_t)B;
  const int ff = kind_fmt(mode_kind(mode)), df = ff;
  TcHeadWs w;
  w.pinv = (float*)b.take(N * 12 * sizeof(float));
  w.slots = (float*)b.take(2 * kNumSlots * sizeof(float));
  w.x0_rs = (float*)b.take(N * kFeatHW * sizeof(float));
  w.x0 = take_act(b, N * kFeatHW * kFeatC, ff);
  w.y1 = take_act(b, N * kFeatHW * fd.h1p, ff);
  w.z = take_act(b, (size_t)B * kFeatHW * 2 * fd.h2, ff);
  w.f1 = take_act(b, (size_t)B * kFeatHW * fd.h2, ff);
  w.f2 = take_act(b, (size_t)B * kFeatHW * fd.h2, ff);
  w.g = take_act(b, N * kFeatHW * fd.h1p, ff);
  w.x1 = take_act(b, N * kFeatHW * kFeatC, df);
  w.d1 = take_act(b, N * 256 * kDecC, df);
  w.d2 = take_act(b, N * 1024 * kDecC, df);
  w.d3 = take_act(b, N * 4096 * kDecC, df);
  w.hm = (float*)b.take(N * J * 4096 * sizeof(float));
  w.part = (float4*)b.take(N * J * kTailSlots * sizeof(float4));
  w.bytes = b.off;
  return w;
}
struct TcDecWs {
  float* slots;
  Act x1, d1, d2, d3;
  size_t bytes;
};
static TcDecWs plan_tc_dec(void* base, int N, int mode) {
  Bump1K b(base);
  const int df = kind_fmt(mode_kind(mode));
  TcDecWs w;
  w.slots = (float*)b.take(2 * kNumSlots * sizeof(float));
  w.x1 = take_act(b, (size_t)N * kFeatHW * kFeatC, df);
  w.d1 = take_act(b, (size_t)N * 256 * kDecC, df);
  w.d2 = take_act(b, (size_t)N * 1024 * kDecC, df);
  w.d3 = take_act(b, (size_t)N * 4096 * kDecC, df);
  w.bytes = b.off;
  return w;
}

int tc_head_workspace_bytes(const TcWeights& w, int batch, size_t* bytes) {
  *bytes = plan_tc_head(nullptr, batch, w.joints, w.kind, w.fd).bytes;
  return CDR_OK;
}
int tc_decoder_workspace_bytes(const TcWeights& w, int n_images, size_t* bytes) {
  *bytes = plan_tc_dec(nullptr, n_images, w.kind).bytes;
  return CDR_OK;
}

// NCHW fp32 latents (one tensor, or two whose rows are stacked: the stereo views) -> pixel-major rows
// in the format of `out`.  kFmtF16P (single tensor only): the tensor scale comes from the exact amax
// of the input (one extra pass over 0.5 MB / image).
// *row_scale (in: buffer of n rows or NULL; out: NULL when the tensor-scale form ran)
static int to_rows(const float* feat, const float* feat2, int n_img, const Act& out, ScaleSlot sl, float** row_scale,
                   cudaStream_t st) {
  float* rs = row_scale ? *row_scale : nullptr;
  if (row_scale) *row_scale = nullptr;
  if (out.fmt == kFmtBF16)
    return launch_nchw_to_rows_bf16(feat, feat2, n_img, kFeatC, kFeatHW, (__nv_bfloat16*)out.p[0], kFeatC, st);
  if (out.fmt == kFmtTF32P)
    return launch_nchw_to_rows_split(feat, feat2, n_img, kFeatC, kFeatHW, (float*)out.p[0], (float*)out.p[1], kFeatC, st);
  if (rs && nchw_rowscale_ok(feat, feat2, n_img, kFeatC, kFeatHW, kFeatC)) {
    *row_scale = rs;
    return launch_nchw_to_rows_f16p_rowscale(feat, feat2, n_img, kFeatC, kFeatHW, out.p[0], out.p[1], kFeatC, rs, sl.amax, st);
  }
  if (int rc = launch_amax_f32(feat, feat2, (long long)n_img * kFeatC * kFeatHW, sl.amax, st)) return rc;
  return launch_nchw_to_rows_f16p(feat, feat2, n_img, kFeatC, kFeatHW, out.p[0], out.p[1], kFeatC, sl.amax, sl.scale, st);
}
// FTL of both views in one launch
// kFmtF16P: in_slot = scale / amax of the input, out_slot = where the output's go, l1max = max row L1 norm of `mats`
static int ftl_act2(const Act& in0, const Act& in1, int in_pitch, const float* const mats[2], int rows, int cols, int blk, int n,
                    const Act& out0, const Act& out1, int out_pitch, int out_fill, ScaleSlot in_slot, ScaleSlot out_slot,
                    const float* l1max, cudaStream_t st) {
  if (in0.fmt == kFmtF16P) {
    const void* ih[2] = {in0.p[0], in1.p[0]};
    const void* il[2] = {in0.p[1], in1.p[1]};
    void* oh[2] = {out0.p[0], out1.p[0]};
    void* ol[2] = {out0.p[1], out1.p[1]};
    return launch_ftl_f16p2(ih, il, in_pitch, mats, rows, cols, blk, n, kFeatHW, oh, ol, out_pitch, out_fill,
                            in_slot.scale, in_slot.amax, l1max, out_slot.scale, out_slot.amax, st);
  }
  if (in0.fmt == kFmtBF16) {
    const __nv_bfloat16* ins[2] = {(const __nv_bfloat16*)in0.p[0], (const __nv_bfloat16*)in1.p[0]};
    __nv_bfloat16* outs[2] = {(__nv_bfloat16*)out0.p[0], (__nv_bfloat16*)out1.p[0]};
    return launch_ftl2<__nv_bfloat16>(ins, in_pitch, mats, rows, cols, blk, n, kFeatHW, outs, out_pitch, out_fill, 2, st);
  }
  const float* ih[2] = {(const float*)in0.p[0], (const float*)in1.p[0]};
  const float* il[2] = {(const float*)in0.p[1], (const float*)in1.p[1]};
  float* oh[2] = {(float*)out0.p[0], (float*)out1.p[0]};
  float* ol[2] = {(float*)out0.p[1], (float*)out1.p[1]};
  return launch_ftl_split2(ih, il, in_pitch, mats, rows, cols, blk, n, kFeatHW, oh, ol, out_pitch, out_fill, 2, st);
}

// Can this pack run deconv3 + final 1x1 (+ soft-argmax partials) as the one kernel of tail_tc.cuh?
static bool tail_fusable(const TcWeights& w) {
  const int dk = mode_kind(w.kind);
  const TcPack* pk = (const TcPack*)w.impl;
  return tc_use_fused_tail() && (dk == kKindBF16 || dk == kKindF16X2) && w.fin_npad == 32 &&
         pk->dc[2].bn == (dk == kKindBF16 ? 256 : 128);
}

// slots: x1 -> 1, d1 -> 2, d2 -> 3, d3 -> 4.  heat (planar fp32 heat-maps) and part (soft-argmax partial records) are
// the two possible products; part != NULL requires tail_fusable().
static int tc_decoder(const TcWeights& w, const Act& x1, int N, const Act& d1, const Act& d2, const Act& d3,
                      float* slots, float* heat, float4* part, cudaStream_t st) {
  const TcPack* pk = (const TcPack*)w.impl;
  static const char* const kDcName[3] = {"deconv1", "deconv2", "deconv3"};
  const bool fused = tail_fusable(w);
  CDR_CHECK_ARG(fused || !part, "tc_decoder: soft-argmax partials need the fused tail");
  Act in = x1;
  const Act outs[3] = {d1, d2, d3};
  int side = 8;
  for (int i = 0; i < (fused ? 2 : 3); ++i) {
    set_stage(kDcName[i]);
    TcLaunch l{};
    l.A = in; l.a_pitch = kTcDcCin[i]; l.n_img = N; l.H = l.W = side; l.cin = kTcDcCin[i];
    l.deconv = 1; l.groups = 4; l.layer = &pk->dc[i]; l.b_group_rows = kDecC; l.n = kDecC;
    l.bias_group_stride = 0;
    l.C = outs[i]; l.c_pitch = kDecC; l.c_fill = kDecC; l.relu = 1; l.out_mode = kOutDeconv;
    l.in_slot = slot(slots, 1 + i); l.out_slot = slot(slots, 2 + i);
    // cta_group::2 pairs: measured to pay on every bf16 (BN = 256) and f16x2 transposed conv (see the kernel comment)
    l.pair2 = mode_kind(w.kind) == kKindBF16 || mode_kind(w.kind) == kKindF16X2;
    if (int rc = launch_tc(l, st)) return rc;
    in = outs[i];
    side *= 2;
  }
  if (fused) {
    set_stage("deconv3_tail");
    TailLaunch t{};
    t.A = d2; t.n_img = N; t.joints = w.joints;
    t.dc3 = &pk->dc[2]; t.fin = &pk->fin;
    t.in_slot = slot(slots, 3);
    t.heat = heat; t.part = part;
    const bool bf = mode_kind(w.kind) == kKindBF16;
    // (n_img * 8 pixel blocks: always an even number, so the pair form applies to every batch)
    const int rc = bf ? launch_tail(t, st) : launch_tail_pair(t, st);
    set_stage(nullptr);
    return rc;
  }
  set_stage("final_1x1");
  TcLaunch l{};
  l.A = d3; l.a_pitch = kDecC; l.n_img = N; l.H = l.W = kHeat; l.cin = kDecC; l.groups = 1;
  l.a_rows_total = (long long)N * 4096;
  l.layer = &pk->fin; l.n = w.joints;
  l.C.p[0] = heat; l.relu = 0; l.out_mode = kOutPlanar;
  l.in_slot = slot(slots, 4);
  const int rc = launch_tc(l, st);
  set_stage(nullptr);
  return rc;
}

static int tap_to_f32(float* dst, const Act& src, const float* scale, long long rows, int pitch, int cols,
                      cudaStream_t st) {
  if (!dst) return CDR_OK;
  act_to_f32_kernel<<<(unsigned)ceil_div<long long>(rows * cols, 256), 256, 0, st>>>(
      src.p[0], src.p[1], src.fmt, scale, dst, rows, pitch, cols);
  CDR_LAUNCH_OK("act_to_f32_kernel");
  return CDR_OK;
}

// scaled fp16 planes from bf16 rows (a bf16 value times a power of two is an fp16 value unless it underflows)
__global__ void bf16_rows_to_f16p_kernel(const __nv_bfloat16* __restrict__ in, __half* __restrict__ hi,
                                         __half* __restrict__ lo, long long n, const float* __restrict__ amax,
                                         float* __restrict__ scale_out) {
  const float a = __ldg(amax);
  const float s = f16_pow2_scale(a);
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *scale_out = s;
  if (i >= n) return;
  const float X = __bfloat162float(in[i]) * s;
  const __half h = __float2half_rn(X);
  hi[i] = h;
  lo[i] = __float2half_rn((X - __half2float(h)) * kLoScale);
}
__global__ void amax_bf16_kernel(const __nv_bfloat16* __restrict__ in, long long n, float* __restrict__ amax) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(__bfloat162float(in[i])));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(amax), __float_as_uint(m));
}

// encoder output (bf16 rows) -> the fusion block's fp32 hi/lo planes: a bf16 value is a tf32 value, lo = 0
__global__ void bf16_rows_to_tf32p_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ hi,
                                          float* __restrict__ lo, long long n8) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const uint4 q = reinterpret_cast<const uint4*>(in)[i];
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
  float4 a, b;
  a.x = __uint_as_float(w[0] << 16); a.y = __uint_as_float(w[0] & 0xffff0000u);
  a.z = __uint_as_float(w[1] << 16); a.w = __uint_as_float(w[1] & 0xffff0000u);
  b.x = __uint_as_float(w[2] << 16); b.y = __uint_as_float(w[2] & 0xffff0000u);
  b.z = __uint_as_float(w[3] << 16); b.w = __uint_as_float(w[3] & 0xffff0000u);
  reinterpret_cast<float4*>(hi)[2 * i] = a;
  reinterpret_cast<float4*>(hi)[2 * i + 1] = b;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  reinterpret_cast<float4*>(lo)[2 * i] = z;
  reinterpret_cast<float4*>(lo)[2 * i + 1] = z;
}

// A side stream per (host thread, device) for work that can overlap the main chain of a forward (the pseudo-inverses).
// NULL when it cannot be created: everything then stays on the caller's stream.
struct SideLane {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
static SideLane* side_lane() {
  static thread_local SideLane lanes[kMaxDevices];
  SideLane& l = lanes[current_device()];
  if (!l.stream) {
    if (cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&l.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&l.join, cudaEventDisableTiming) != cudaSuccess) {
      (void)cudaGetLastError();
      l.stream = nullptr;
      return nullptr;
    }
  }
  return &l;
}

int tc_head_forward(const TcWeights& w, const void* feat_rows, int feat_planes, const float* feat_l, const float* feat_r,
                    const float* P_l, const float* P_r, const float* pinv_l, const float* pinv_r, double pinv_rtol,
                    int batch, float scale, float* kp2d_l, float* kp2d_r, float* xyz,
                    const CdrHeadTaps* taps, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const TcPack* pk = (const TcPack*)w.impl;
  const int mode = w.kind;
  const bool scaled = mode_kind(mode) == kKindF16X2;
  const bool fus16 = w.has_fusion && scaled;   // fusion activations in kFmtF16P (slots 6..11)
  const int B = batch, N = 2 * batch, J = w.joints;
  TcHeadWs ws = plan_tc_head(workspace, B, J, mode, w.fd);
  const FusionDims& fd = w.fd;
  if (ws.bytes > workspace_bytes) {
    set_error("cdr_head_forward: workspace %zu < required %zu bytes", workspace_bytes, ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  int rc;
  if (scaled) CDR_CUDA(cudaMemsetAsync(ws.slots, 0, 2 * kNumSlots * sizeof(float), st));
  set_stage("pinv");
  const float* pinv[2] = {pinv_l, pinv_r};
  SideLane* lane = nullptr;
  if (!pinv_l) {
    // The pseudo-inverses (2B threads of fp64 Jacobi: ~14 us of pure latency) are not needed before the inverse
    // FTL: they run on a side stream forked here and joined there, under the layout pass and conv_layer1.  The fork /
    // join are plain event record / wait pairs, which a CUDA-graph capture of `st` turns into graph edges.
    lane = side_lane();
    cudaStream_t ps = st;
    if (lane) {
      CDR_CUDA(cudaEventRecord(lane->fork, st));
      CDR_CUDA(cudaStreamWaitEvent(lane->stream, lane->fork, 0));
      ps = lane->stream;
    }
    if ((rc = launch_pinv2(P_l, P_r, B, pinv_rtol, ws.pinv, fus16 ? ws.slots + 2 * 11 : nullptr, ps))) return rc;
    pinv[0] = ws.pinv;
    pinv[1] = ws.pinv + (size_t)B * 12;
    if (lane) CDR_CUDA(cudaEventRecord(lane->join, lane->stream));
  } else if (fus16) {
    if ((rc = launch_mats_l1max(pinv[0], pinv[1], 4, 3, P_l, P_r, 3, 4, B, ws.slots + 2 * 11, st))) return rc;
  }
  Act x0 = ws.x0;
  float* x0_rs = nullptr;          // per-row scales of x0, when the layout pass produced them
  ScaleSlot x0_slot = slot(ws.slots, 5);
  if (feat_rows && feat_planes) {
    // latents as scaled fp16 hi/lo planes + {amax, scale} (the f16x2 encoder's output): conv_layer1's operand as is
    CDR_CHECK_ARG(x0.fmt == kFmtF16P, "cdr_head_forward_planes: fp16-plane latents need the fp32 (f16x2) head");
    x0 = planes_act(feat_rows, (size_t)N * kFeatHW, kFeatC, &x0_slot);
  } else if (feat_rows) {
    // latents already pixel-major bf16 rows, views stacked (the tcgen05 encoder's output layout)
    if (x0.fmt == kFmtBF16) {
      x0.p[0] = const_cast<void*>(feat_rows);
    } else if (x0.fmt == kFmtTF32P) {
      set_stage("rows_to_planes");
      const long long n8 = (long long)N * kFeatHW * kFeatC / 8;
      bf16_rows_to_tf32p_kernel<<<(unsigned)ceil_div<long long>(n8, 256), 256, 0, st>>>(
          (const __nv_bfloat16*)feat_rows, (float*)x0.p[0], (float*)x0.p[1], n8);
      CDR_LAUNCH_OK("bf16_rows_to_tf32p_kernel");
    } else {
      set_stage("rows_to_planes");
      const long long n = (long long)N * kFeatHW * kFeatC;
      const ScaleSlot sl = slot(ws.slots, 5);
      amax_bf16_kernel<<<4 * num_sms(), 256, 0, st>>>((const __nv_bfloat16*)feat_rows, n, sl.amax);
      CDR_LAUNCH_OK("amax_bf16_kernel");
      bf16_rows_to_f16p_kernel<<<(unsigned)ceil_div<long long>(n, 256), 256, 0, st>>>(
          (const __nv_bfloat16*)feat_rows, (__half*)x0.p[0], (__half*)x0.p[1], n, sl.amax, sl.scale);
      CDR_LAUNCH_OK("bf16_rows_to_f16p_kernel");
    }
  } else {
    set_stage("nchw_to_rows");
    x0_rs = ws.x0_rs;
    if ((rc = to_rows(feat_l, feat_r, B, ws.x0, slot(ws.slots, 5), &x0_rs, st))) return rc;
  }
  set_stage("cf_conv1");
  {
    TcLaunch l{};
    l.A = x0; l.a_pitch = kFeatC; l.n_img = N; l.H = l.W = 8; l.cin = kFeatC; l.groups = 1;
    l.a_rows_total = (long long)N * kFeatHW;
    l.layer = &pk->cf1; l.n = fd.h1;
    l.C = ws.y1; l.c_pitch = fd.h1p; l.c_fill = fd.h1p; l.relu = 1; l.out_mode = kOutRows;
    l.in_slot = x0_slot;
    l.in_row_scale = x0_rs;
    if (fus16) l.out_slot = slot(ws.slots, 6);
    l.pair2 = fus16;                 // cta_group::2 pairs: cf_conv1 49.5 -> 46.3 us, conv_layer2 38.0 -> 36.4 us (out_layer: slower)
    if ((rc = launch_tc(l, st))) return rc;
  }
  set_stage("ftl_inv");
  if (lane) CDR_CUDA(cudaStreamWaitEvent(st, lane->join, 0));      // join: the pseudo-inverses are complete
  if ((rc = ftl_act2(ws.y1, act_offset(ws.y1, (size_t)B * kFeatHW * fd.h1p), fd.h1p, pinv, 4, 3, fd.blk, B, ws.z,
                     act_offset(ws.z, (size_t)fd.h2), 2 * fd.h2, fd.h2, slot(ws.slots, 6), slot(ws.slots, 7),
                     ws.slots + 2 * 11, st)))
    return rc;
  set_stage("cf_conv2");
  {
    TcLaunch l{};
    l.A = ws.z; l.a_pitch = 2 * fd.h2; l.n_img = B; l.H = l.W = 8; l.cin = 2 * fd.h2; l.groups = 1;
    l.a_rows_total = (long long)B * kFeatHW;
    l.layer = &pk->cf2a; l.n = fd.h2;
    l.C = ws.f1; l.c_pitch = fd.h2; l.c_fill = fd.h2; l.relu = 1; l.out_mode = kOutRows;
    if (fus16) { l.in_slot = slot(ws.slots, 7); l.out_slot = slot(ws.slots, 8); l.pair2 = 1; }
    if ((rc = launch_tc(l, st))) return rc;
    l.A = ws.f1; l.a_pitch = fd.h2; l.cin = fd.h2; l.layer = &pk->cf2b; l.C = ws.f2;
    if (fus16) { l.in_slot = slot(ws.slots, 8); l.out_slot = slot(ws.slots, 9); }
    if ((rc = launch_tc(l, st))) return rc;
  }
  set_stage("ftl_fwd");
  const float* Pv[2] = {P_l, P_r};
  if ((rc = ftl_act2(ws.f2, ws.f2, fd.h2, Pv, 3, 4, fd.blk, B, ws.g, act_offset(ws.g, (size_t)B * kFeatHW * fd.h1p),
                     fd.h1p, fd.h1p, slot(ws.slots, 9), slot(ws.slots, 10),
                     ws.slots + 2 * 11 + 1, st)))
    return rc;
  set_stage("cf_out");
  {
    TcLaunch l{};
    l.A = ws.g; l.a_pitch = fd.h1p; l.n_img = B; l.H = l.W = 8; l.cin = fd.h1; l.groups = 2;
    l.a_rows_total = (long long)N * kFeatHW;
    l.layer = &pk->out; l.b_group_rows = kFeatC; l.n = kFeatC; l.bias_group_stride = kFeatC;
    l.C = ws.x1; l.c_group_stride = (long long)B * kFeatHW * kFeatC; l.c_pitch = kFeatC; l.c_fill = kFeatC;
    l.relu = 1; l.out_mode = kOutRows;
    l.out_slot = slot(ws.slots, 1);
    if (fus16) l.in_slot = slot(ws.slots, 10);
    if ((rc = launch_tc(l, st))) return rc;
  }
  if (tail_fusable(w)) {
    // deconv3 + final 1x1 + soft-argmax partials in one kernel: neither deconv3's activation nor (unless a tap asks
    // for them) the heat-maps touch HBM; a 64-CTA merge kernel finishes soft-argmax, scale and DLT
    float* heat = (taps && taps->heatmaps) ? ws.hm : nullptr;
    if ((rc = tc_decoder(w, ws.x1, N, ws.d1, ws.d2, ws.d3, ws.slots, heat, ws.part, st))) return rc;
    set_stage("merge_dlt");
    if ((rc = launch_tail_merge(ws.part, P_l, P_r, B, J, scale, kp2d_l, kp2d_r, xyz, st))) return rc;
  } else {
    if ((rc = tc_decoder(w, ws.x1, N, ws.d1, ws.d2, ws.d3, ws.slots, ws.hm, nullptr, st))) return rc;
    set_stage("softargmax_dlt");
    if ((rc = cdr_softargmax_dlt(ws.hm, ws.hm + (size_t)B * J * 4096, 0, P_l, P_r, B, J, kHeat, kHeat, scale,
                                 kp2d_l, kp2d_r, xyz, nullptr, nullptr, nullptr, nullptr, nullptr, st)))
      return rc;
  }
  set_stage(nullptr);
  if (taps) {
    if (taps->pinv) {
      CDR_CUDA(cudaMemcpyAsync(taps->pinv, pinv[0], (size_t)B * 48, cudaMemcpyDeviceToDevice, st));
      CDR_CUDA(cudaMemcpyAsync(taps->pinv + (size_t)B * 12, pinv[1], (size_t)B * 48, cudaMemcpyDeviceToDevice, st));
    }
    if ((rc = tap_to_f32(taps->cf_cat, ws.z, slot(ws.slots, 7).scale, (long long)B * kFeatHW, 2 * fd.h2, 2 * fd.h2, st))) return rc;
    if ((rc = tap_to_f32(taps->cf_f, ws.f2, slot(ws.slots, 9).scale, (long long)B * kFeatHW, fd.h2, fd.h2, st))) return rc;
    if ((rc = tap_to_f32(taps->f_out, ws.x1, slot(ws.slots, 1).scale, (long long)N * kFeatHW, kFeatC, kFeatC, st)))
      return rc;
    if (taps->heatmaps)
      CDR_CUDA(cudaMemcpyAsync(taps->heatmaps, ws.hm, (size_t)N * J * 4096 * 4, cudaMemcpyDeviceToDevice, st));
  }
  return CDR_OK;
}

// feat_rows != NULL: latents as bf16 pixel-major rows (n_images*64, 2048) instead of NCHW fp32
int tc_decoder_forward(const TcWeights& w, const void* feat_rows, int feat_planes, const float* feat, int n_images,
                       float* heatmaps, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  TcDecWs ws = plan_tc_dec(workspace, n_images, w.kind);
  if (ws.bytes > workspace_bytes) {
    set_error("cdr_decoder_forward: workspace %zu < required %zu bytes", workspace_bytes, ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  if (feat_rows && feat_planes) {
    // fp16 hi/lo planes + {amax, scale} from the f16x2 encoder: deconv1's operand as is; its slot (1) gets a copy
    CDR_CHECK_ARG(ws.x1.fmt == kFmtF16P, "cdr_decoder_forward_planes: fp16-plane latents need the fp32 (f16x2) decoder");
    ScaleSlot sl;
    const Act x1 = planes_act(feat_rows, (size_t)n_images * kFeatHW, kFeatC, &sl);
    CDR_CUDA(cudaMemsetAsync(ws.slots, 0, 2 * kNumSlots * sizeof(float), st));
    CDR_CUDA(cudaMemcpyAsync(slot(ws.slots, 1).amax, sl.amax, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return tc_decoder(w, x1, n_images, ws.d1, ws.d2, ws.d3, ws.slots, heatmaps, nullptr, st);
  }
  if (feat_rows) {
    Act x1 = ws.x1;
    const long long n = (long long)n_images * kFeatHW * kFeatC;
    set_stage("rows_to_planes");
    if (x1.fmt == kFmtBF16) {
      x1.p[0] = const_cast<void*>(feat_rows);
    } else if (x1.fmt == kFmtTF32P) {
      bf16_rows_to_tf32p_kernel<<<(unsigned)ceil_div<long long>(n / 8, 256), 256, 0, st>>>(
          (const __nv_bfloat16*)feat_rows, (float*)x1.p[0], (float*)x1.p[1], n / 8);
      CDR_LAUNCH_OK("bf16_rows_to_tf32p_kernel");
    } else {
      CDR_CUDA(cudaMemsetAsync(ws.slots, 0, 2 * kNumSlots * sizeof(float), st));
      const ScaleSlot sl = slot(ws.slots, 1);
      amax_bf16_kernel<<<4 * num_sms(), 256, 0, st>>>((const __nv_bfloat16*)feat_rows, n, sl.amax);
      CDR_LAUNCH_OK("amax_bf16_kernel");
      bf16_rows_to_f16p_kernel<<<(unsigned)ceil_div<long long>(n, 256), 256, 0, st>>>(
          (const __nv_bfloat16*)feat_rows, (__half*)x1.p[0], (__half*)x1.p[1], n, sl.amax, sl.scale);
      CDR_LAUNCH_OK("bf16_rows_to_f16p_kernel");
    }
    return tc_decoder(w, x1, n_images, ws.d1, ws.d2, ws.d3, ws.slots, heatmaps, nullptr, st);
  }
  if (ws.x1.fmt == kFmtF16P) CDR_CUDA(cudaMemsetAsync(ws.slots, 0, 2 * kNumSlots * sizeof(float), st));
  set_stage("nchw_to_rows");
  if (int rc = to_rows(feat, nullptr, n_images, ws.x1, slot(ws.slots, 1), nullptr, st)) return rc;
  return tc_decoder(w, ws.x1, n_images, ws.d1, ws.d2, ws.d3, ws.slots, heatmaps, nullptr, st);
}


// ==========================================================================================
// ResNet bottleneck encoder on the same tap-GEMM kernel (SURVEY §8f rank 1; reference
// models/encoder.py:38-131).  bf16 activations as pixel-major rows, BN folded into bf16 weights,
// fp32 accumulation; per Bottleneck: 1x1 (+ReLU) -> 3x3 stride s as 9 shifted TMA taps (+ReLU) ->
// 1x1 with the residual (identity, or the 1x1 stride-s downsample conv) added in the epilogue
// (+ReLU).  The stride-2 convs read their input through tensor maps with element stride 2.
// (Cout,Cin,kh,kw) -> [n_pad][tap*Cin + ci], tap = ky*kw + kx
__global__ void pack_conv_tc_kernel(CdrConvBn s, int cout, int cin, int taps, int n_pad, __nv_bfloat16* __restrict__ w,
                                    float* __restrict__ bias_out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n_pad) bias_out[idx] = idx < cout ? tc_folded_bias(s, (int)idx) : 0.f;
  const long long K = (long long)taps * cin;
  if (idx >= (long long)n_pad * K) return;
  const int n = (int)(idx / K), kk = (int)(idx % K);
  const int tap = kk / cin, ci = kk - tap * cin;
  float v = 0.f;
  if (n < cout) v = (float)((double)s.weight[((size_t)n * cin + ci) * taps + tap] * tc_bn_scale(s, n));
  w[idx] = __float2bfloat16_rn(v);
}

struct EncBlock {
  TcLayer c1, c2, c3, ds;
  int cin = 0, planes = 0, stride = 1, has_ds = 0;
};
struct EncPack {
  void* pool = nullptr;
  void* stem_w = nullptr;        // stem.cu: packed conv1 + bn1 (NULL: no stem in this handle)
  float* stem_b = nullptr;
  int kind = kKindBF16;          // kKindBF16: bf16 rows; kKindF16X2: scaled fp16 hi/lo planes (fp32-accurate)
  int n_blocks = 0, in_channels = 0, out_channels = 0, total_stride = 1;
  EncBlock* blocks = nullptr;
};

// N tile: 128 for the layers that carry a residual (it rides the ring as one stage) and for the
// memory-bound 1x1 projections (two staging buffers per warp); 256 for the MMA-bound 3x3 / reduce convs.
// f16x2: 128 everywhere (4 accumulators of BN columns fill the 512 TMEM columns).
static int enc_bn(int n, bool wide) { return n >= 256 && wide ? 256 : n >= 128 ? 128 : 64; }

static size_t plan_encoder(EncPack& e, const CdrEncoderSpec& spec, void* base) {
  Bump1K b(base);
  int cin = spec.in_channels;
  const bool f16 = e.kind == kKindF16X2;
  auto plan = [&](TcLayer& L, int n, int k, bool wide) {
    const int bn = f16 ? 128 : enc_bn(n, wide);
    const int n_pad = round_up(n, bn);
    plan_layer(L, b, e.kind, n_pad, k, k, bn, n_pad, n_pad, f16);
  };
  for (int i = 0; i < spec.num_blocks; ++i) {
    const CdrEncoderBlock& sb = spec.blocks[i];
    EncBlock& blk = e.blocks[i];
    blk.cin = cin; blk.planes = sb.planes; blk.stride = sb.stride; blk.has_ds = sb.downsample.weight != nullptr;
    const int p = sb.planes, o = 4 * sb.planes;
    plan(blk.c1, p, cin, true);
    plan(blk.c2, p, 9 * p, true);
    plan(blk.c3, o, p, false);
    if (blk.has_ds) plan(blk.ds, o, cin, false);
    cin = o;
  }
  if (spec.stem.weight) {
    e.stem_w = b.take(f16 ? stem_weight_bytes_f16x2() : stem_weight_bytes());
    e.stem_b = (float*)b.take(64 * sizeof(float));
  }
  return b.off;
}

int tc_encoder_create(const CdrEncoderSpec& spec, int kind, void** out, cudaStream_t st) {
  CDR_CHECK_ARG(spec.num_blocks > 0 && spec.blocks && spec.in_channels > 0 && spec.in_channels % 64 == 0,
                "cdr_encoder_create: bad spec");
  CDR_CHECK_ARG(kind == kKindBF16 || kind == kKindF16X2, "cdr_encoder_create: precision must be bf16 or f16x2");
  int cin = spec.in_channels, total_stride = 1;
  for (int i = 0; i < spec.num_blocks; ++i) {
    const CdrEncoderBlock& sb = spec.blocks[i];
    CDR_CHECK_ARG(sb.planes >= 64 && sb.planes % 64 == 0 && (sb.stride == 1 || sb.stride == 2),
                  "cdr_encoder_create: block %d: planes must be a multiple of 64, stride 1 or 2", i);
    const CdrConvBn* cs[3] = {&sb.conv1, &sb.conv2, &sb.conv3};
    for (const CdrConvBn* c : cs)
      CDR_CHECK_ARG(c->weight && c->bn_weight && c->bn_bias && c->bn_mean && c->bn_var,
                    "cdr_encoder_create: block %d: missing conv / BN tensor", i);
    const bool need_ds = sb.stride != 1 || cin != 4 * sb.planes;
    CDR_CHECK_ARG(need_ds == (sb.downsample.weight != nullptr),
                  "cdr_encoder_create: block %d: downsample present iff stride != 1 or cin != 4*planes", i);
    cin = 4 * sb.planes;
    total_stride *= sb.stride;
  }
  EncPack* e = new EncPack();
  e->kind = kind;
  e->n_blocks = spec.num_blocks;
  e->in_channels = spec.in_channels;
  e->out_channels = cin;
  e->total_stride = total_stride;
  e->blocks = new EncBlock[spec.num_blocks];
  *out = e;
  const size_t bytes = plan_encoder(*e, spec, nullptr);
  CDR_CUDA(cudaMalloc(&e->pool, bytes));
  CDR_CUDA(cudaMemsetAsync(e->pool, 0, bytes, st));       // norms start at 0 for the atomicMax
  plan_encoder(*e, spec, e->pool);
  auto pack = [&](const CdrConvBn& s, TcLayer& L, int cout, int cin_l, int taps) -> int {
    if (L.kind == kKindF16X2) {
      if (taps == 9)
        pack_rows_f16_kernel<9><<<L.n_pad, 256, 0, st>>>(s, cout, cin_l, L.k_pitch, L.n_pad, (__half*)L.w[0],
                                                                (__half*)L.w[1], L.wsi, L.bias, L.norms);
      else
        pack_rows_f16_kernel<0><<<L.n_pad, 256, 0, st>>>(s, cout, cin_l, L.k_pitch, L.n_pad, (__half*)L.w[0],
                                                                (__half*)L.w[1], L.wsi, L.bias, L.norms);
      CDR_LAUNCH_OK("pack_rows_f16_kernel");
      return layer_maps(L);
    }
    const long long total = (long long)L.n_pad * taps * cin_l;
    pack_conv_tc_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(s, cout, cin_l, taps, L.n_pad,
                                                                                    (__nv_bfloat16*)L.w[0], L.bias);
    CDR_LAUNCH_OK("pack_conv_tc_kernel");
    return layer_maps(L);
  };
  if (spec.stem.weight) {
    CDR_CHECK_ARG(spec.in_channels == 64, "cdr_encoder_create: the stem produces 64 channels");
    if (int rc = kind == kKindF16X2 ? launch_pack_stem_f16x2(spec.stem, e->stem_w, e->stem_b, st)
                                    : launch_pack_stem(spec.stem, e->stem_w, e->stem_b, st))
      return rc;
  }
  for (int i = 0; i < spec.num_blocks; ++i) {
    const CdrEncoderBlock& sb = spec.blocks[i];
    EncBlock& blk = e->blocks[i];
    int rc;
    if ((rc = pack(sb.conv1, blk.c1, blk.planes, blk.cin, 1))) return rc;
    if ((rc = pack(sb.conv2, blk.c2, blk.planes, blk.planes, 9))) return rc;
    if ((rc = pack(sb.conv3, blk.c3, 4 * blk.planes, blk.planes, 1))) return rc;
    if (blk.has_ds && (rc = pack(sb.downsample, blk.ds, 4 * blk.planes, blk.cin, 1))) return rc;
  }
  return CDR_OK;
}

void tc_encoder_destroy(void* enc) {
  EncPack* e = (EncPack*)enc;
  if (!e) return;
  if (e->pool) cudaFree(e->pool);
  delete[] e->blocks;
  delete e;
}

int tc_encoder_kind(const void* enc) { return ((const EncPack*)enc)->kind; }

// Output of an f16x2 encoder: [hi plane | lo plane | {amax, scale}] — planes of rows*channels fp16, each starting
// on a 1024-byte boundary (include/cdrhead.h: "fp16 planes")
static size_t planes_stride_bytes(size_t rows, int channels) { return round_up<size_t>(rows * channels * 2, 1024); }
static Act planes_act(const void* buf, size_t rows, int channels, ScaleSlot* sl) {
  Act a;
  a.fmt = kFmtF16P;
  const size_t stride = planes_stride_bytes(rows, channels);
  a.p[0] = const_cast<void*>(buf);
  a.p[1] = (uint8_t*)const_cast<void*>(buf) + stride;
  if (sl) {
    sl->amax = (float*)((uint8_t*)const_cast<void*>(buf) + 2 * stride);
    sl->scale = sl->amax + 1;
  }
  return a;
}
int tc_encoder_out_bytes(const void* enc, int n, int h, int w, size_t* bytes) {
  const EncPack& e = *(const EncPack*)enc;
  const size_t rows = (size_t)n * (h / e.total_stride) * (w / e.total_stride);
  *bytes = e.kind == kKindF16X2 ? 2 * planes_stride_bytes(rows, e.out_channels) + 1024 : rows * e.out_channels * 2;
  return CDR_OK;
}

struct EncWs {
  Act x[2], t1, t2, r;
  float* slots;            // f16x2: {amax, scale} pairs — 0: the input, 1 + 4*i ..: block i's t1, t2, r, out
  size_t slot_bytes, bytes;
};
static EncWs plan_enc_ws(const EncPack& e, void* base, int n, int h, int w) {
  size_t mx = 0, mt1 = 0, mt2 = 0, mr = 0;
  int H = h, W = w;
  for (int i = 0; i < e.n_blocks; ++i) {
    const EncBlock& b = e.blocks[i];
    const size_t m_in = (size_t)n * H * W;
    H /= b.stride; W /= b.stride;
    const size_t m_out = (size_t)n * H * W;
    mt1 = m_in * b.planes > mt1 ? m_in * b.planes : mt1;
    mt2 = m_out * b.planes > mt2 ? m_out * b.planes : mt2;
    if (b.has_ds) mr = m_out * 4 * b.planes > mr ? m_out * 4 * b.planes : mr;
    if (i + 1 < e.n_blocks) mx = m_out * 4 * b.planes > mx ? m_out * 4 * b.planes : mx;
  }
  Bump1K bp(base);
  EncWs ws;
  const int fmt = kind_fmt(e.kind);
  ws.slot_bytes = (size_t)(2 + 8 * e.n_blocks) * sizeof(float);
  ws.slots = (float*)bp.take(ws.slot_bytes);
  ws.x[0] = take_act(bp, mx, fmt);
  ws.x[1] = take_act(bp, mx, fmt);
  ws.t1 = take_act(bp, mt1, fmt);
  ws.t2 = take_act(bp, mt2, fmt);
  ws.r = take_act(bp, mr, fmt);
  ws.bytes = bp.off;
  return ws;
}

static int enc_check_grid(const EncPack& e, int h, int w) {
  int H = h, W = w;
  for (int i = 0; i < e.n_blocks; ++i) {
    const int s = e.blocks[i].stride;
    CDR_CHECK_ARG(H % s == 0 && W % s == 0, "cdr_encoder: %dx%d grid is not divisible by the strides", h, w);
    H /= s; W /= s;
    CDR_CHECK_ARG(W >= 8 && W <= 128 && (W & (W - 1)) == 0, "cdr_encoder: feature-map width %d (block %d) must be a "
                  "power of two in 8..128", W, i);
    const int rows = 128 / W < H ? 128 / W : H;
    CDR_CHECK_ARG(H % rows == 0 && (128 % (W * rows)) == 0, "cdr_encoder: feature map %dx%d (block %d) does not tile", H, W, i);
  }
  return CDR_OK;
}

int tc_encoder_workspace_bytes(const void* enc, int n, int h, int w, size_t* bytes) {
  const EncPack& e = *(const EncPack*)enc;
  if (int rc = enc_check_grid(e, h, w)) return rc;
  *bytes = plan_enc_ws(e, nullptr, n, h, w).bytes;
  return CDR_OK;
}

// images (n,3,H,W): [conv_out (n,H/2,W/2,64) | pooled (n,H/4,W/4,64) | layer workspace]
// (bf16: both bf16; f16x2: conv_out fp32, pooled as fp16 hi/lo planes whose scale is slot 0 of the layer workspace)
struct EncImgWs {
  void* conv_out;
  Act pooled;
  void* layers;
  size_t layer_bytes, bytes;
};
static EncImgWs plan_enc_img_ws(const EncPack& e, void* base, int n, int H, int W) {
  Bump1K bp(base);
  EncImgWs ws;
  const bool f16 = e.kind == kKindF16X2;
  ws.conv_out = bp.take((size_t)n * (H / 2) * (W / 2) * 64 * (f16 ? 4 : 2));
  ws.pooled = take_act(bp, (size_t)n * (H / 4) * (W / 4) * 64, kind_fmt(e.kind));
  ws.layer_bytes = plan_enc_ws(e, nullptr, n, H / 4, W / 4).bytes;
  ws.layers = bp.take(ws.layer_bytes);
  ws.bytes = bp.off;
  return ws;
}
int tc_encoder_workspace_bytes_images(const void* enc, int n, int H, int W, size_t* bytes) {
  const EncPack& e = *(const EncPack*)enc;
  CDR_CHECK_ARG(e.stem_w, "cdr_encoder: this handle was created without a stem");
  CDR_CHECK_ARG(H % 16 == 0 && W % 64 == 0, "cdr_encoder: image %dx%d must have H %% 16 == 0 and W %% 64 == 0", H, W);
  if (int rc = enc_check_grid(e, H / 4, W / 4)) return rc;
  *bytes = plan_enc_img_ws(e, nullptr, n, H, W).bytes;
  return CDR_OK;
}
static int enc_layers(const EncPack& e, const Act& x, bool x_scaled, int n, int h, int w, void* out_rows, void* workspace,
                      size_t workspace_bytes, cudaStream_t st);
int tc_encoder_forward_images(const void* enc, const void* images, int is_u8, const float* mean, const float* std,
                              int n, int H, int W, void* out_rows, void* workspace, size_t workspace_bytes,
                              cudaStream_t st) {
  const EncPack& e = *(const EncPack*)enc;
  CDR_CHECK_ARG(e.stem_w, "cdr_encoder_forward_images: this handle was created without a stem");
  CDR_CHECK_ARG(H % 16 == 0 && W % 64 == 0, "cdr_encoder: image %dx%d must have H %% 16 == 0 and W %% 64 == 0", H, W);
  EncImgWs ws = plan_enc_img_ws(e, workspace, n, H, W);
  if (ws.bytes > workspace_bytes) {
    set_error("cdr_encoder_forward_images: workspace %zu < required %zu bytes", workspace_bytes, ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  set_stage("enc_stem");
  if (e.kind == kKindF16X2) {
    // slot 0 of the layer workspace = {amax, scale} of the pooled tensor; every slot is zeroed here, before the stem
    EncWs lw = plan_enc_ws(e, ws.layers, n, H / 4, W / 4);
    CDR_CUDA(cudaMemsetAsync(lw.slots, 0, lw.slot_bytes, st));
    if (int rc = launch_stem_f32(images, is_u8, mean, std, n, H, W, e.stem_w, e.stem_b, (float*)ws.conv_out,
                                 ws.pooled.p[0], ws.pooled.p[1], lw.slots, st))
      return rc;
    return enc_layers(e, ws.pooled, true, n, H / 4, W / 4, out_rows, ws.layers, ws.layer_bytes, st);
  }
  if (int rc = launch_stem(images, is_u8, mean, std, n, H, W, e.stem_w, e.stem_b, ws.conv_out, ws.pooled.p[0], st)) return rc;
  return enc_layers(e, ws.pooled, false, n, H / 4, W / 4, out_rows, ws.layers, ws.layer_bytes, st);
}

int tc_encoder_out_shape(const void* enc, int h, int w, int* oh, int* ow, int* oc) {
  const EncPack& e = *(const EncPack*)enc;
  *oh = h / e.total_stride; *ow = w / e.total_stride; *oc = e.out_channels;
  return CDR_OK;
}

// H, W: the conv's OUTPUT grid.  res (optional): residual tensor with the output's shape, added before the ReLU.
static int enc_conv(const TcLayer& L, const Act& in, ScaleSlot in_slot, int cin, int n, int H, int W, int conv3, int stride,
                    const Act& out, ScaleSlot out_slot, int cout, int relu, const Act* res, ScaleSlot res_slot,
                    cudaStream_t st) {
  TcLaunch l{};
  l.A = in; l.a_pitch = cin;
  l.n_img = n; l.H = H; l.W = W; l.cin = cin; l.groups = 1;
  l.conv3 = conv3; l.stride = stride;
  l.a_rows_total = (long long)n * H * W;
  l.layer = &L; l.n = cout;
  l.C = out; l.c_pitch = cout; l.c_fill = cout; l.relu = relu; l.out_mode = kOutRows;
  l.in_slot = in_slot; l.out_slot = out_slot;
  if (res) {
    l.res = res->p[0]; l.res_lo = res->p[1]; l.res_slot = res_slot;
  }
  l.res_pitch = cout;
  // cta_group::2 pairs for the MMA-bound wide layers (conv1 / conv2 of a block: BN = 256 in bf16, every f16x2 one), as
  // on the decoder's transposed convs (layer4 conv2 38.2 -> 35.1 us, conv1 24.6 -> 23.6 us)
  l.pair2 = (L.bn == 256 || L.kind == kKindF16X2) && !res && stride <= 1;
  return launch_tc(l, st);
}

// layer1..layer4 on x (n, h, w, in_channels) in the handle's activation format.  f16x2: the workspace's slots are
// already zeroed and slot 0 holds x's {amax, scale} (x_scaled)
static int enc_layers(const EncPack& e, const Act& x, bool x_scaled, int n, int h, int w, void* out_rows, void* workspace,
                      size_t workspace_bytes, cudaStream_t st) {
  if (int rc = enc_check_grid(e, h, w)) return rc;
  EncWs ws = plan_enc_ws(e, workspace, n, h, w);
  if (ws.bytes > workspace_bytes) {
    set_error("cdr_encoder_forward: workspace %zu < required %zu bytes", workspace_bytes, ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  const bool f16 = e.kind == kKindF16X2;
  CDR_CHECK_ARG(!f16 || x_scaled, "cdr_encoder_forward: the f16x2 encoder starts from images (its stem sets the input scale)");
  Act cur = x;
  ScaleSlot cur_slot = f16 ? slot(ws.slots, 0) : ScaleSlot{};
  int H = h, W = w, pp = 0;
  char label[48];
  for (int i = 0; i < e.n_blocks; ++i) {
    const EncBlock& b = e.blocks[i];
    const int s = b.stride, Ho = H / s, Wo = W / s, o = 4 * b.planes;
    const bool last = i + 1 == e.n_blocks;
    Act out = ws.x[pp];
    ScaleSlot s_t1{}, s_t2{}, s_r{}, s_out{};
    if (f16) {
      s_t1 = slot(ws.slots, 1 + 4 * i); s_t2 = slot(ws.slots, 2 + 4 * i);
      s_r = slot(ws.slots, 3 + 4 * i); s_out = slot(ws.slots, 4 + 4 * i);
    }
    if (last) {
      if (f16) {
        out = planes_act(out_rows, (size_t)n * Ho * Wo, o, &s_out);
        CDR_CUDA(cudaMemsetAsync(s_out.amax, 0, 2 * sizeof(float), st));
      } else {
        out.p[0] = out_rows;
      }
    }
    int rc;
    auto stage = [&](const char* conv) {
      snprintf(label, sizeof(label), "enc_block%d.%s", i, conv);
      set_stage(label);
    };
    stage("conv1");
    if ((rc = enc_conv(b.c1, cur, cur_slot, b.cin, n, H, W, 0, 1, ws.t1, s_t1, b.planes, 1, nullptr, ScaleSlot{}, st))) return rc;
    stage("conv2");
    if ((rc = enc_conv(b.c2, ws.t1, s_t1, b.planes, n, Ho, Wo, 1, s, ws.t2, s_t2, b.planes, 1, nullptr, ScaleSlot{}, st))) return rc;
    Act res = cur;
    ScaleSlot res_slot = cur_slot;
    if (b.has_ds) {
      stage("downsample");
      if ((rc = enc_conv(b.ds, cur, cur_slot, b.cin, n, Ho, Wo, 0, s, ws.r, s_r, o, 0, nullptr, ScaleSlot{}, st))) return rc;
      res = ws.r;
      res_slot = s_r;
    }
    stage("conv3");
    if ((rc = enc_conv(b.c3, ws.t2, s_t2, b.planes, n, Ho, Wo, 0, 1, out, s_out, o, 1, &res, res_slot, st))) return rc;
    cur = out;
    cur_slot = s_out;
    pp ^= 1;
    H = Ho; W = Wo;
  }
  set_stage(nullptr);
  return CDR_OK;
}

// x: (n, h, w, in_channels) bf16 NHWC from the caller's own stem (bf16 handles only)
int tc_encoder_forward(const void* enc, const void* x, int n, int h, int w, void* out_rows, void* workspace,
                       size_t workspace_bytes, cudaStream_t st) {
  const EncPack& e = *(const EncPack*)enc;
  CDR_CHECK_ARG(e.kind == kKindBF16, "cdr_encoder_forward: an f16x2 encoder starts from images (cdr_encoder_forward_images)");
  Act xa;
  xa.fmt = kFmtBF16;
  xa.p[0] = const_cast<void*>(x);
  return enc_layers(e, xa, false, n, h, w, out_rows, workspace, workspace_bytes, st);
}

int tc_set_debug(unsigned int* d) {
  CDR_CUDA(cudaMemcpyToSymbol(ptx::g_cdr_debug, &d, sizeof(d)));
  return CDR_OK;
}

// ------------------------------------------------------------------------------------------
// Training convolutions at fp32 accuracy: forward, data and weight gradient on the f16x2 tap-GEMM (scaled fp16 hi/lo
// operands, 3 kind::f16 MMAs per product, main term drained every kSplitChunk K blocks).  Every op runs the same
// steps; make_train_conv says how one maps onto them:
//   forward  y  = one tap-GEMM over the x planes, the weight packed per call, planar epilogue straight into NCHW fp32
//   dgrad    dx = one tap-GEMM over the dy planes, the weight packed per call as the data-gradient operand, NCHW fp32
//   wgrad    dW = the kMN kernel: per tap a GEMM over the pixels, K split into slices -> fp32 partials ->
//               wgrad_reduce_kernel (fixed slice order: bitwise deterministic, no atomics)
//   dbias    db = bias_grad_kernel: a fixed-order fp64 sum over the pixels of every channel
// x and dy are encoded with ONE power-of-two scale per tensor (exact amax first): wgrad reduces over pixels, so
// per-pixel scales would not factor out of its sums.  The x planes and their {amax, scale} slot are what the forward
// saves; the backward encodes dy once for both of its GEMMs.

// wgrad K slices: powers of two while the `tiles` output tiles do not fill two waves of 148 SMs and a slice keeps >= 16 of
// the `kb` K blocks.  A function of the shape only, so the summation order (and the result, bit for bit) does not depend
// on the device.
static int wgrad_slices(long long kb, long long tiles) {
  int s = 1;
  while (tiles * s < 2 * 148 && kb % (2 * s) == 0 && kb / (2 * s) >= 16) s *= 2;
  return s;
}

template <int kDeconv, int kDeconvK = 4>
static void pack_rows_f16(const CdrConvBn& cb, int nout, int cin, const TcLayer& L, cudaStream_t st) {
  pack_rows_f16_kernel<kDeconv, kDeconvK><<<L.rows, 256, 0, st>>>(cb, nout, cin, L.k_pitch, L.n_pad, (__half*)L.w[0],
                                                                  (__half*)L.w[1], L.wsi, L.bias, nullptr);
}

// per TrainConvKind: the entry points' op (cdr_<op>_train_*) and the forward / backward stage labels
static const char* const kTrainConvNames[3][3] = {{"deconv", "deconv_train_fwd", "deconv_train_bwd"},
                                                  {"conv1x1", "conv1x1_train_fwd", "conv1x1_train_bwd"},
                                                  {"conv3x3", "conv3x3_train_fwd", "conv3x3_train_bwd"}};
static size_t train_rows(const TrainConv& d, const TrainPlanes& p) { return (size_t)d.n * p.h * p.w; }
static const TrainPlanes& wgrad_a(const TrainConv& d) { return d.wgrad_a_is_x ? d.x : d.dy; }
static const TrainPlanes& wgrad_b(const TrainConv& d) { return d.wgrad_a_is_x ? d.dy : d.x; }

// TrainGemm: {pack, k, bn, n_pad, groups, tap, stride, H, W, n}
TrainConv make_train_conv(int kind, int n, int cin, int cout, int h, int w, int stride) {
  TrainConv d{};
  d.kind = kind;
  d.n = n;
  const int npi = round_up(cin, 128), npo = round_up(cout, 128);
  switch (kind) {
    case kTrainDeconv:
      // ConvTranspose2d(k4, s2, p1, bias=False), x h x w -> y 2h x 2w
      //   forward  kTapDeconv (4 phases x 4 taps), weights packed unfolded, phase-scattered (planar_deconv)
      //   dgrad    kTapConv4s2 (16 taps, stride-2 box over the dy planes), B = [ci][tap*Cout + co]
      //   wgrad    M = Cin (A = x), N = Cout (B = dy through the stride-2 box), 16 taps
      d.x = {cin, h, w, cin};
      d.dy = {cout, 2 * h, 2 * w, cout};
      d.fwd = {pack_rows_f16<1>, 4 * cin, 128, npo, 4, kTapDeconv, 1, h, w, cout};
      d.dgrad = {pack_rows_f16<-16>, 16 * cout, 128, npi, 1, kTapConv4s2, 2, h, w, cin};
      d.wgrad_a_is_x = true; d.b_k = 4; d.b_stride = 2;
      break;
    case kTrainConv1x1: {
      // 1x1 Conv2d(Cin, Cout, bias optional)
      //   forward  kTapNone, weights (+ bias) packed per call
      //   dgrad    kTapNone, B = W^T packed [ci][co] (dgrad_weight<1>)
      //   wgrad    M = Cout (A = dy), N = Cin (B = x), both 2-D pixel-major maps, 1 tap
      // Channel counts need not be multiples of 64: the x and dy planes are stored with a pitch of round_up(C, 64)
      // whose pad columns the encoder writes as zeros, the packed weights' K pitch is zero-filled, and output channels
      // past Cout / Cin are masked by the epilogue.  BN = 32 for at most 32 output channels.
      const int pin = round_up(cin, 64), pout = round_up(cout, 64);
      const int bn_o = cout <= 32 ? 32 : 128, bn_i = cin <= 32 ? 32 : 128;
      d.x = {cin, h, w, pin};
      d.dy = {cout, h, w, pout};
      d.fwd = {pack_rows_f16<0>, pin, bn_o, round_up(cout, bn_o), 1, kTapNone, 1, h, w, cout};
      d.dgrad = {pack_rows_f16<-1>, pout, bn_i, round_up(cin, bn_i), 1, kTapNone, 1, h, w, cin};
      d.b_k = 1; d.b_stride = 1;
      break;
    }
    default: {   // kTrainConv3x3
      // 3x3 pad-1 Conv2d(Cin, Cout, stride s, bias=False), x h x w -> y h/s x w/s
      //   forward  kTapConv3 (s = 2: the element-strided box), weights packed unfolded (pack_rows_f16_kernel<9>)
      //   dgrad    s = 1: kTapConv3 over the dy planes, B = W^T with the taps flipped (dgrad_weight<9>)
      //            s = 2: dx = conv_transpose2d(dy, W4, stride 2, pad 1) with W4 = W zero-padded to 4x4 at index 3:
      //               the transposed-conv forward (kTapDeconv, planar_deconv) over the dy planes, W4 read by
      //               deconv_weight<3>
      //   wgrad    M = Cout (A = dy, a 2-D pixel map), N = Cin (B = x through the stride-s box shifted by
      //               (kx - 1, ky - 1)), 9 taps
      const int ho = h / stride, wo = w / stride;
      d.x = {cin, h, w, cin};
      d.dy = {cout, ho, wo, cout};
      d.fwd = {pack_rows_f16<9>, 9 * cin, 128, npo, 1, kTapConv3, stride, ho, wo, cout};
      d.dgrad = stride == 1 ? TrainGemm{pack_rows_f16<-9>, 9 * cout, 128, npi, 1, kTapConv3, 1, ho, wo, cin}
                            : TrainGemm{pack_rows_f16<1, 3>, 4 * cout, 128, npi, 4, kTapDeconv, 1, ho, wo, cin};
      d.b_k = 3; d.b_stride = stride;
      break;
    }
  }
  const TrainPlanes &a = wgrad_a(d), &b = wgrad_b(d);
  const long long tiles = (long long)ceil_div(a.c, 128) * ceil_div(b.c, 128) * d.b_k * d.b_k;
  d.slices = wgrad_slices((long long)train_rows(d, a) / 64, tiles);
  return d;
}

struct TrainConvWs {
  TcLayer L;                 // forward: the forward GEMM's packed weight; backward: the data gradient's
  void* dy_planes = nullptr; // backward: dy as an fp16 planes buffer [hi | lo | {amax, scale}]
  float* part = nullptr;     // backward: wgrad partials [slice][tap][M][round_up(N, 128)]
  size_t bytes = 0;
};
static size_t train_planes_bytes(const TrainConv& d, const TrainPlanes& p) {
  return 2 * planes_stride_bytes(train_rows(d, p), p.pitch) + 1024;
}
static TrainConvWs plan_train_conv(void* base, const TrainConv& d, bool backward) {
  TrainConvWs ws;
  Bump1K b(base);
  const TrainGemm& g = backward ? d.dgrad : d.fwd;
  plan_layer(ws.L, b, kKindF16X2, g.groups * g.n_pad, g.k, g.k, g.bn, g.n_pad, g.n_pad, false);
  if (backward) {
    ws.dy_planes = b.take(train_planes_bytes(d, d.dy));
    const size_t taps = (size_t)d.b_k * d.b_k;
    ws.part = (float*)b.take(d.slices * taps * wgrad_a(d).c * round_up(wgrad_b(d).c, 128) * sizeof(float));
  }
  ws.bytes = b.off;
  return ws;
}
size_t train_conv_saved_bytes(const TrainConv& d) { return train_planes_bytes(d, d.x); }
size_t train_conv_workspace_bytes(const TrainConv& d) {
  const size_t f = plan_train_conv(nullptr, d, false).bytes, bw = plan_train_conv(nullptr, d, true).bytes;
  return f > bw ? f : bw;
}

// NCHW fp32 -> fp16 planes with one tensor scale (exact amax pass first); columns [c, pitch) are written as zeros
static int to_planes_tensor_scale(const float* in, int n, int c, int hw, int pitch, const Act& a, ScaleSlot sl,
                                  cudaStream_t st) {
  CDR_CUDA(cudaMemsetAsync(sl.amax, 0, sizeof(float), st));
  if (int rc = launch_amax_f32(in, nullptr, (long long)n * c * hw, sl.amax, st)) return rc;
  return launch_nchw_to_rows_f16p(in, nullptr, n, c, hw, a.p[0], a.p[1], pitch, sl.amax, sl.scale, st);
}

// One forward or data-gradient GEMM: pack the weight (and bias) into L, then the tap-GEMM over the planes `a` of `in`
// into `out`, planar NCHW fp32
static int train_gemm(const TrainConv& d, const TrainGemm& g, const TrainPlanes& in, const Act& a, ScaleSlot sa,
                      const float* weight, const float* bias, TcLayer& L, float* out, cudaStream_t st) {
  CdrConvBn cb{};
  cb.weight = weight;
  cb.bias = bias;
  g.pack(cb, g.n, in.c, L, st);
  CDR_LAUNCH_OK("pack_rows_f16_kernel");
  if (int rc = layer_maps(L)) return rc;
  TcLaunch l{};
  l.A = a; l.a_pitch = in.pitch;
  l.n_img = d.n; l.H = g.H; l.W = g.W; l.cin = in.pitch; l.stride = g.stride; l.groups = g.groups;
  l.deconv = g.tap == kTapDeconv; l.conv3 = g.tap == kTapConv3; l.conv4s2 = g.tap == kTapConv4s2;
  l.a_rows_total = (long long)train_rows(d, in);
  l.layer = &L; l.b_group_rows = g.groups > 1 ? L.n_pad : 0; l.n = g.n; l.bias_group_stride = 0;
  l.C.p[0] = out; l.relu = 0; l.out_mode = kOutPlanar; l.planar_deconv = g.tap == kTapDeconv;
  l.in_slot = sa;
  return launch_tc(l, st);
}

int tc_train_conv_forward(const TrainConv& d, const float* x, const float* weight, const float* bias, float* y,
                          void* saved, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  TrainConvWs ws = plan_train_conv(workspace, d, false);
  if (workspace_bytes < ws.bytes) {
    set_error("cdr_%s_train_forward: workspace %zu < required %zu bytes", kTrainConvNames[d.kind][0], workspace_bytes,
              ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  set_stage(kTrainConvNames[d.kind][1]);
  ScaleSlot sx;
  const Act xa = planes_act(saved, train_rows(d, d.x), d.x.pitch, &sx);
  if (int rc = to_planes_tensor_scale(x, d.n, d.x.c, d.x.h * d.x.w, d.x.pitch, xa, sx, st)) return rc;
  const int rc = train_gemm(d, d.fwd, d.x, xa, sx, weight, bias, ws.L, y, st);
  set_stage(nullptr);
  return rc;
}

// dW[r][c][tap] = (sum over slices, in order, of part[slice][tap][r][c]) / (s_x * s_dy): a transposed conv's
// (Cin, Cout, 4, 4) with r = ci, c = co, 16 taps; a 1x1 conv's (Cout, Cin, 1, 1) with r = co, c = ci, 1 tap
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ part, int slices, int taps, int rows, int cols, int ldc,
                    const float* __restrict__ sx, const float* __restrict__ sdy, float* __restrict__ dw) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)rows * cols * taps) return;
  const int t = (int)(idx % taps);
  const long long r = idx / taps;
  const int c = (int)(r % cols), row = (int)(r / cols);
  const float ix = 1.f / __ldcg(sx), id = 1.f / __ldcg(sdy);      // powers of two: exact
  float s = 0.f;
  for (int sl = 0; sl < slices; ++sl) s += __ldcg(part + (((size_t)sl * taps + t) * rows + row) * ldc + c);
  dw[idx] = s * ix * id;
}
int launch_wgrad_reduce(const float* part, int slices, int taps, int rows, int cols, int ldc, const float* sx,
                        const float* sdy, float* dw, cudaStream_t st) {
  const long long total = (long long)rows * cols * taps;
  wgrad_reduce_kernel<<<(unsigned)ceil_div<long long>(total, 256), 256, 0, st>>>(part, slices, taps, rows, cols, ldc, sx,
                                                                                 sdy, dw);
  CDR_LAUNCH_OK("wgrad_reduce_kernel");
  return CDR_OK;
}

// The kMN GEMM over n*h*w pixels split into `slices` K slices: part[slice * taps + tap] (m rows, pitch round_up(nb, 128))
// = A^T B.  A: m channels of a pixel-major fp16 planes buffer (pitch a_pitch), scale slot `sa`.  B: nb channels (pitch
// b_pitch), either the same pixels through a 2-D map (b_k = 1, 1 tap), or a (b_stride*h) x (b_stride*w) map through the
// stride-b_stride box shifted by (kx - 1, ky - 1), b_k^2 taps: b_k = 4, b_stride = 2, the dy of a k4 s2 p1 transposed
// conv; b_k = 3, the x of a 3x3 pad-1 conv at stride 1 or 2.
static int launch_wgrad(int n, int h, int w, const Act& a, int m, int a_pitch, ScaleSlot sa, const Act& b, int nb,
                        int b_pitch, int b_k, int b_stride, int slices, float* part, cudaStream_t st) {
  using Cfg = TcCfg<128, kKindF16X2, kFmtF16P, 0>;
  auto kern = tap_gemm_tc_kernel<128, kKindF16X2, kFmtF16P, 0, true>;
  static DeviceOnce attr_set;
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes));
    attr_set.done();
  }
  const long long rows = (long long)n * h * w, kb = rows / 64;
  TcGemmParams p{};
  p.M = m;
  p.n_img = n; p.H = h; p.W = w;
  p.cin = (int)(kb / slices) * 64;           // pixels per K slice
  p.ntaps = 1; p.tap_mode = b_k == 4 ? kTapConv4s2 : b_k == 3 ? kTapConv3 : kTapNone; p.stride = b_stride;
  p.groups = b_k * b_k * slices;
  p.n_tiles = round_up(nb, 128) / 128;
  p.n = nb;
  p.C = part; p.c_pitch = round_up(nb, 128); p.c_fill = nb;
  p.out_mode = kOutPlanar;
  p.scale_in = sa.scale;
  p.num_tiles = ceil_div(m, 128) * p.groups * p.n_tiles;
  CUtensorMap ma[2], mb[2];
  for (int pl = 0; pl < 2; ++pl) {
    {   // A planes: (pixels, a_pitch) rows, boxes of 64 channels x 64 pixels
      const uint64_t dims[2] = {(uint64_t)a_pitch, (uint64_t)rows};
      const uint64_t strides[1] = {(uint64_t)a_pitch};
      const uint32_t box[2] = {64, 64};
      if (int rc = make_tmap(&ma[pl], a.p[pl], kFmtF16P, 2, dims, strides, box)) return rc;
    }
    if (b_k > 1) {   // B planes (n, s*h, s*w, b_pitch) seen with element stride s: 64 channels x (w x 64/w) pixels x 1 image
      const uint32_t s = (uint32_t)b_stride;
      const uint64_t iw = s * (uint64_t)w, ih = s * (uint64_t)h;
      const uint64_t dims[4] = {(uint64_t)b_pitch, iw, ih, (uint64_t)n};
      const uint64_t strides[3] = {(uint64_t)b_pitch, (uint64_t)b_pitch * iw, (uint64_t)b_pitch * iw * ih};
      const uint32_t box[4] = {64, s * (uint32_t)w, s * (uint32_t)(64 / w), 1};
      const uint32_t estr[4] = {1, s, s, 1};
      if (int rc = make_tmap(&mb[pl], b.p[pl], kFmtF16P, 4, dims, strides, box, estr)) return rc;
    } else {      // B planes: (pixels, b_pitch) rows, like A
      const uint64_t dims[2] = {(uint64_t)b_pitch, (uint64_t)rows};
      const uint64_t strides[1] = {(uint64_t)b_pitch};
      const uint32_t box[2] = {64, 64};
      if (int rc = make_tmap(&mb[pl], b.p[pl], kFmtF16P, 2, dims, strides, box)) return rc;
    }
  }
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  CDR_CUDA(launch_pdl(kern, grid, Cfg::kThreads, Cfg::kSmemBytes, false, st, ma[0], ma[1], mb[0], mb[1], ma[0], ma[0], ma[0],
                      ma[0], p));
  CDR_LAUNCH_OK("tap_gemm_tc_kernel");
  return CDR_OK;
}

// db[c] = sum over images and pixels of dy[img][c][pixel]: one block per channel, float4 element j*256 + thread of the
// channel's (image, pixel) sequence to that thread, fp64 partial sums, a fixed tree: bitwise deterministic, no atomics
__global__ void __launch_bounds__(256)
bias_grad_kernel(const float* __restrict__ dy, int n, int c, int hw, float* __restrict__ db) {
  __shared__ double red[256];
  const int ch = blockIdx.x, hw4 = hw >> 2;                 // hw is a multiple of 64
  const long long total4 = (long long)n * hw4;
  double s = 0.0;
  for (long long i = threadIdx.x; i < total4; i += 256) {
    const long long img = i / hw4;
    const float4 v = __ldg(reinterpret_cast<const float4*>(dy + (img * c + ch) * hw) + (i - img * hw4));
    s += ((double)v.x + (double)v.y) + ((double)v.z + (double)v.w);
  }
  red[threadIdx.x] = s;
  __syncthreads();
#pragma unroll
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) db[ch] = (float)red[0];
}

int tc_train_conv_backward(const TrainConv& d, const void* saved, const float* weight, const float* dy, float* dx,
                           float* dw, float* db, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  TrainConvWs ws = plan_train_conv(workspace, d, true);
  if (workspace_bytes < ws.bytes) {
    set_error("cdr_%s_train_backward: workspace %zu < required %zu bytes", kTrainConvNames[d.kind][0], workspace_bytes,
              ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  if (!dx && !dw && !db) return CDR_OK;
  set_stage(kTrainConvNames[d.kind][2]);
  if (db) {
    bias_grad_kernel<<<d.dy.c, 256, 0, st>>>(dy, d.n, d.dy.c, d.dy.h * d.dy.w, db);
    CDR_LAUNCH_OK("bias_grad_kernel");
  }
  if (dx || dw) {
    ScaleSlot sd, sx;
    const Act dya = planes_act(ws.dy_planes, train_rows(d, d.dy), d.dy.pitch, &sd);     // one copy feeds both GEMMs
    const Act xa = planes_act(saved, train_rows(d, d.x), d.x.pitch, &sx);
    if (int rc = to_planes_tensor_scale(dy, d.n, d.dy.c, d.dy.h * d.dy.w, d.dy.pitch, dya, sd, st)) return rc;
    if (dx)
      if (int rc = train_gemm(d, d.dgrad, d.dy, dya, sd, weight, nullptr, ws.L, dx, st)) return rc;
    if (dw) {
      const bool ax = d.wgrad_a_is_x;
      const TrainPlanes &a = wgrad_a(d), &b = wgrad_b(d);
      if (int rc = launch_wgrad(d.n, a.h, a.w, ax ? xa : dya, a.c, a.pitch, ax ? sx : sd, ax ? dya : xa, b.c, b.pitch,
                                d.b_k, d.b_stride, d.slices, ws.part, st))
        return rc;
      if (int rc = launch_wgrad_reduce(ws.part, d.slices, d.b_k * d.b_k, a.c, b.c, round_up(b.c, 128), sx.scale, sd.scale,
                                       dw, st))
        return rc;
    }
  }
  set_stage(nullptr);
  return CDR_OK;
}

}  // namespace cdr
