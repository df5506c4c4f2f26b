// Streaming heat-map kernels: soft-argmax (+ fused DLT + MPJPE partial sums) and the
// baseline's hard arg-max.  HBM-bound: 16 KB of logits in, 8 bytes out per heat-map.
//
// Structure (one persistent CTA per SM, 32 * (NW + 2) threads, NW = 10 by default):
//   warp 0      producer: one elected lane streams whole heat-maps (one 16 KB tile each) into a
//               NW-deep shared-memory ring with 1-D TMA bulk copies (cp.async.bulk) that
//               complete on per-stage mbarriers -> 160 KB in flight per SM with one thread.
//   warps 1..NW consumers: one warp per tile, two passes over the tile in shared memory
//               (max, then exp/sum/centre of mass) with warp-shuffle reductions; exact
//               "global max first" softmax like ATen, sums carried in fp64.
//   warp NW+1   DLT: when all 2J tiles of a pose have landed their 2D joints in shared
//               memory, lanes 0..J-1 each solve one joint's 4x4 system in fp64 registers
//               (one-sided Jacobi, jacobi.cuh) and optionally accumulate the MPJPE terms.
// Reference: models/cdrnet.py:120-149 (process_heatmap), :250 (scale), :151-179,262-266
// (dlt per joint), models/metrics.py:82-95 (MPJPE terms), tools/utils.py:30-58 (arg-max).
#include "common.cuh"
#include "jacobi.cuh"
#include <stdlib.h>

#include "ptx.cuh"

namespace cdr {

constexpr int kTileBytes = 16384;  // one 64x64 fp32 heat-map
// Consumer warps = ring stages = NW (template parameter of the kernel).  The ring depth must be a
// multiple of the consumer-warp count: tiles q and q+stages share a stage and its mbarrier, and only if
// the SAME warp consumes both (q % warps) is its wait for phase(q+stages) ordered after phase(q).  With
// 12 stages and 8 warps a starved warp could reach the barrier while it was still in the older,
// incomplete phase, whose parity test reads as "complete" — stale data, then a protocol deadlock (seen in
// the arg-max stress at 20 000 maps).  With stages == warps every warp owns one stage.
// A stage is busy for (HBM latency + one warp's two passes over the tile), so bytes in flight per SM and
// consumer parallelism both bound the stream: 8 x 16 KB reached 5.1 TB/s (78 % of the measured HBM peak)
// with the XU pipe (EX2 + fp64 conversions) at 46 %.
constexpr int kHeatWarps = 10;   // B200, 8192-pose stream: 8 -> 5.40, 10 -> 5.91, 12 -> 5.33 TB/s (12: 14 warps cap ptxas at 128 registers, the DLT warp spills)
constexpr int kHeatWarpsMin = 8;   // smallest instantiation: the fused pose hand-off needs 2J >= warps
constexpr int kPoseBufs = 4;
constexpr int kMaxTilesPerPose = 2 * kMaxJoints;

struct HeatParams {
  const void* heat[2];   // per view: (B, J, H*W)
  const float* P[2];     // per view: (B, 3, 4) or NULL (no DLT)
  float* kp[2];          // per view: (B, J, 2) or NULL
  float* xyz;            // (B, J, 3)
  const double* gt3d;    // optional MPJPE inputs
  const double* gt2d[2];
  const double* vis;
  double* pose_err;      // (B, 3)
  float* maxvals;        // arg-max mode: (B*J)
  uint8_t* pts_u8;       // arg-max mode: (B*J, 2)
  long long batch;
  int n_views, joints, H, W;
  float scale;
};

template <int NW>
struct __align__(128) HeatSmem {
  uint8_t tiles[NW][kTileBytes];
  double kps[kPoseBufs][kMaxTilesPerPose][2];
  uint64_t full[NW];
  uint64_t empty[NW];
  uint64_t pose_full[kPoseBufs];
  uint64_t pose_empty[kPoseBufs];
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// unpack 16 bytes of a tile into fp32 lanes
template <typename T>
struct Vec16;
template <>
struct Vec16<float> {
  static constexpr int kElems = 4;
  __device__ static void load(const uint8_t* tile, int i, float (&v)[4]) {
    const float4 q = reinterpret_cast<const float4*>(tile)[i];
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
};
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int kElems = 8;
  __device__ static void load(const uint8_t* tile, int i, float (&v)[8]) {
    const uint4 q = reinterpret_cast<const uint4*>(tile)[i];
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[2 * k] = __uint_as_float(w[k] << 16);
      v[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
    }
  }
};

// soft-argmax of one tile held in shared memory; result (x, y) in heat-map pixels, all lanes
template <typename T>
__device__ __forceinline__ void tile_softargmax(const uint8_t* tile, int hw, int W, int lane,
                                                double& cx, double& cy) {
  constexpr int E = Vec16<T>::kElems;
  const int nvec = hw / E;
  float m = -INFINITY;
  for (int i = lane; i < nvec; i += 32) {
    float v[E];
    Vec16<T>::load(tile, i, v);
#pragma unroll
    for (int k = 0; k < E; ++k) m = fmaxf(m, v[k]);
  }
  m = warp_max(m);
  const float kLog2e = 1.4426950408889634f;
  const float ml2 = m * kLog2e;
  double S = 0.0, SX = 0.0, SY = 0.0;
  for (int i = lane; i < nvec; i += 32) {
    float v[E];
    Vec16<T>::load(tile, i, v);
    float se = 0.f, sxl = 0.f;
#pragma unroll
    for (int k = 0; k < E; ++k) {
      const float e = exp2f(fmaf(v[k], kLog2e, -ml2));
      se += e;
      sxl = fmaf((float)k, e, sxl);
    }
    const int idx = i * E;
    const int row = idx / W;
    const int col = idx - row * W;
    const double sed = (double)se;
    S += sed;
    SX += fma((double)col, sed, (double)sxl);
    SY = fma((double)row, sed, SY);
  }
  S = warp_sum(S);
  SX = warp_sum(SX);
  SY = warp_sum(SY);
  cx = SX / S;
  cy = SY / S;
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));   // one MUFU.EX2, rel. error 2^-22
  return y;
}

// Exact fp32 -> fp64 widening of a NON-NEGATIVE float on the integer pipe (F2F.F64.F32 issues on the XU
// pipe, 4 lanes/clk/SMSP, which it would share with the EX2s: ncu had XU at 46 % with two conversions per
// step).  exponent + 896, mantissa << 29; +0 maps to 2^-127 (harmless in sums that contain e(max) = 1),
// Inf/NaN do NOT survive — the caller keeps an fp32 check sum for them.
__device__ __forceinline__ double widen_nonneg(float x) {
  const uint32_t b = __float_as_uint(x);
  return __hiloint2double((int)((b >> 3) + 0x38000000u), (int)(b << 29));
}

// Fast path for the decoder's 64x64 maps.  With 32 lanes x 16 bytes per step a lane always sits in
// the same columns (col0..col0+E-1) and walks R = 32*E/64 rows per step, so the centre of mass is
//   sum_x = col0 * S + sum(k * e),   sum_y = row0 * S + R * sum(step * S_step)
// and the inner loop carries no index arithmetic: 1 LDS.128 + E x (FFMA, EX2, FADD, FFMA) + two
// integer-pipe fp32->fp64 widenings and four fp64 adds/FMAs per step.
template <typename T>
__device__ __forceinline__ void tile_softargmax_64(const uint8_t* tile, int lane, double& cx, double& cy) {
  constexpr int E = Vec16<T>::kElems;        // 4 (fp32) / 8 (bf16)
  constexpr int IT = 4096 / E / 32;          // 32 / 16 steps
  constexpr int LPR = 64 / E;                // lanes per row
  constexpr int R = 32 / LPR;                // rows per step
  float m = -INFINITY;
#pragma unroll 8
  for (int it = 0; it < IT; ++it) {
    float v[E];
    Vec16<T>::load(tile, it * 32 + lane, v);
#pragma unroll
    for (int k = 0; k < E; ++k) m = fmaxf(m, v[k]);
  }
  m = warp_max(m);
  const float kLog2e = 1.4426950408889634f;
  const float ml2 = m * kLog2e;
  double S = 0.0, SXL = 0.0, TY = 0.0, itd = 0.0;
  float chk = 0.f;                           // fp32 shadow of S: carries Inf/NaN (see widen_nonneg)
#pragma unroll 4
  for (int it = 0; it < IT; ++it) {
    float v[E];
    Vec16<T>::load(tile, it * 32 + lane, v);
    float se = 0.f, sxl = 0.f;
#pragma unroll
    for (int k = 0; k < E; ++k) {
      const float e = ex2_approx(fmaf(v[k], kLog2e, -ml2));
      se += e;
      sxl = fmaf((float)k, e, sxl);
    }
    chk += se;
    const double sed = widen_nonneg(se);
    S += sed;
    SXL += widen_nonneg(sxl);
    TY = fma(itd, sed, TY);
    itd += 1.0;
  }
  if (!(chk <= 3.0e38f)) S = (double)chk;    // NaN / Inf logits: propagate like the reference's softmax
  const double col0 = (double)((lane % LPR) * E), row0 = (double)(lane / LPR);
  double SX = fma(col0, S, SXL);
  double SY = fma(row0, S, (double)R * TY);
  S = warp_sum(S);
  SX = warp_sum(SX);
  SY = warp_sum(SY);
  cx = SX / S;
  cy = SY / S;
}

// hard arg-max of one tile: first flat index of the maximum (np.argmax tie rule)
template <typename T>
__device__ __forceinline__ void tile_argmax(const uint8_t* tile, int hw, int lane, float& best,
                                            int& best_idx) {
  constexpr int E = Vec16<T>::kElems;
  const int nvec = hw / E;
  best = -INFINITY;
  best_idx = 0x7fffffff;
  for (int i = lane; i < nvec; i += 32) {
    float v[E];
    Vec16<T>::load(tile, i, v);
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (v[k] > best) { best = v[k]; best_idx = i * E + k; }   // strict: keeps the first
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
    if (ov > best || (ov == best && oi < best_idx)) { best = ov; best_idx = oi; }
  }
  if (best_idx == 0x7fffffff) best_idx = 0;  // all -inf / NaN map
}

template <typename T, bool kArgmax, int NW>
__global__ void __launch_bounds__(32 * (NW + 2), 1) heat_stream_kernel(const HeatParams p) {
  constexpr int kStages = NW, kConsumerWarps = NW;
  extern __shared__ uint8_t smem_raw[];
  HeatSmem<NW>& sm = *reinterpret_cast<HeatSmem<NW>*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int hw = p.H * p.W;
  const uint32_t tile_bytes = (uint32_t)hw * sizeof(T);
  const int tiles_per_pose = p.n_views * p.joints;
  const bool do_dlt = !kArgmax && p.P[0] != nullptr;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&sm.full[s], 1);
      ptx::mbar_init(&sm.empty[s], 1);
    }
    for (int s = 0; s < kPoseBufs; ++s) {
      ptx::mbar_init(&sm.pose_full[s], tiles_per_pose);
      ptx::mbar_init(&sm.pose_empty[s], 1);
    }
    ptx::fence_mbar_init();
  }
  __syncthreads();

  // poses handled by this CTA: blockIdx.x, +gridDim.x, ...
  const long long n_iter =
      (p.batch > (long long)blockIdx.x) ? (p.batch - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp == 0) {
    // ------------------------------------------------------------ producer
    if (lane == 0) {
      long long q = 0;
      for (long long it = 0; it < n_iter; ++it) {
        const long long pose = blockIdx.x + it * gridDim.x;
        for (int t = 0; t < tiles_per_pose; ++t, ++q) {
          const int stage = (int)(q % kStages);
          const uint32_t par = (uint32_t)((q / kStages) & 1);
          ptx::mbar_wait(&sm.empty[stage], par ^ 1u);
          const int v = t / p.joints, j = t - v * p.joints;
          const uint8_t* src = reinterpret_cast<const uint8_t*>(p.heat[v]) +
                               ((size_t)pose * p.joints + j) * tile_bytes;
          ptx::mbar_arrive_expect_tx(&sm.full[stage], tile_bytes);
          ptx::bulk_g2s(sm.tiles[stage], src, tile_bytes, &sm.full[stage]);
        }
      }
    }
  } else if (warp <= kConsumerWarps) {
    // ------------------------------------------------------------ consumers
    const int cw = warp - 1;
    const long long total = n_iter * tiles_per_pose;
    for (long long q = cw; q < total; q += kConsumerWarps) {
      const long long it = q / tiles_per_pose;
      const int t = (int)(q - it * tiles_per_pose);
      const long long pose = blockIdx.x + it * gridDim.x;
      const int v = t / p.joints, j = t - v * p.joints;
      const int stage = (int)(q % kStages);
      const uint32_t par = (uint32_t)((q / kStages) & 1);
      ptx::mbar_wait(&sm.full[stage], par);
      const uint8_t* tile = sm.tiles[stage];
      const size_t map = (size_t)pose * p.joints + j;
      if constexpr (kArgmax) {
        float best;
        int idx;
        tile_argmax<T>(tile, hw, lane, best, idx);
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive(&sm.empty[stage]);
          const float ok = best > 0.f ? 1.f : 0.f;   // tools/utils.py:53-57
          const float x = (float)(idx % p.W) * ok, y = (float)(idx / p.W) * ok;
          if (p.kp[v]) { p.kp[v][map * 2] = x; p.kp[v][map * 2 + 1] = y; }
          if (p.maxvals) p.maxvals[map] = best;
          if (p.pts_u8) {                                // baseline.py:52-53
            p.pts_u8[map * 2] = (uint8_t)(x * p.scale);
            p.pts_u8[map * 2 + 1] = (uint8_t)(y * p.scale);
          }
        }
      } else {
        double cx, cy;
        if (p.H == 64 && p.W == 64)
          tile_softargmax_64<T>(tile, lane, cx, cy);
        else
          tile_softargmax<T>(tile, hw, p.W, lane, cx, cy);
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive(&sm.empty[stage]);
          cx *= (double)p.scale;
          cy *= (double)p.scale;
          if (p.kp[v]) { p.kp[v][map * 2] = (float)cx; p.kp[v][map * 2 + 1] = (float)cy; }
          if (do_dlt) {
            const int buf = (int)(it % kPoseBufs);
            ptx::mbar_wait(&sm.pose_empty[buf], (uint32_t)(((it / kPoseBufs) & 1) ^ 1));
            sm.kps[buf][t][0] = cx;
            sm.kps[buf][t][1] = cy;
            ptx::mbar_arrive(&sm.pose_full[buf]);
          }
        }
      }
    }
  } else if (do_dlt) {
    // ------------------------------------------------------------ DLT / MPJPE warp
    for (long long it = 0; it < n_iter; ++it) {
      const long long pose = blockIdx.x + it * gridDim.x;
      const int buf = (int)(it % kPoseBufs);
      ptx::mbar_wait(&sm.pose_full[buf], (uint32_t)((it / kPoseBufs) & 1));
      double e0 = 0.0, e1 = 0.0, e2 = 0.0;
      for (int j = lane; j < p.joints; j += 32) {
        const double ul = sm.kps[buf][j][0], vl = sm.kps[buf][j][1];
        const double ur = sm.kps[buf][p.joints + j][0], vr = sm.kps[buf][p.joints + j][1];
        double A[4][4];
        dlt_rows(p.P[0] + pose * 12, ul, vl, A, 0);
        dlt_rows(p.P[1] + pose * 12, ur, vr, A, 2);
        double x, y, z;
        dlt_solve4(A, x, y, z);
        const size_t o = (size_t)pose * p.joints + j;
        const float fx = (float)x, fy = (float)y, fz = (float)z;
        p.xyz[o * 3] = fx;
        p.xyz[o * 3 + 1] = fy;
        p.xyz[o * 3 + 2] = fz;
        if (p.gt3d) {
          // the reference's calc_mpjpe consumes the fp32 outputs
          const double w = p.vis ? p.vis[o] : 1.0;
          double dx = ((double)(float)ul - p.gt2d[0][o * 2]) * w;
          double dy = ((double)(float)vl - p.gt2d[0][o * 2 + 1]) * w;
          e0 += sqrt(dx * dx + dy * dy);
          dx = ((double)(float)ur - p.gt2d[1][o * 2]) * w;
          dy = ((double)(float)vr - p.gt2d[1][o * 2 + 1]) * w;
          e1 += sqrt(dx * dx + dy * dy);
          dx = ((double)fx - p.gt3d[o * 3]) * w;
          dy = ((double)fy - p.gt3d[o * 3 + 1]) * w;
          const double dz = ((double)fz - p.gt3d[o * 3 + 2]) * w;
          e2 += sqrt(dx * dx + dy * dy + dz * dz);
        }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sm.pose_empty[buf]);
      if (p.gt3d) {
        e0 = warp_sum(e0);
        e1 = warp_sum(e1);
        e2 = warp_sum(e2);
        if (lane == 0) {
          p.pose_err[pose * 3] = e0;
          p.pose_err[pose * 3 + 1] = e1;
          p.pose_err[pose * 3 + 2] = e2;
        }
      }
    }
  }
}

template <typename T, bool kArgmax, int NW>
static int launch_heat_nw(const HeatParams& p, cudaStream_t st) {
  const size_t smem = sizeof(HeatSmem<NW>) + 128;
  static DeviceOnce attr_set;  // per instantiation AND per device
  if (attr_set.need()) {
    CDR_CUDA(cudaFuncSetAttribute(heat_stream_kernel<T, kArgmax, NW>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set.done();
  }
  long long grid = p.batch < num_sms() ? p.batch : num_sms();
  heat_stream_kernel<T, kArgmax, NW><<<(unsigned)grid, 32 * (NW + 2), smem, st>>>(p);
  CDR_LAUNCH_OK("heat_stream_kernel");
  return CDR_OK;
}

template <typename T, bool kArgmax>
static int launch_heat(const HeatParams& p, cudaStream_t st) {
  // the fused pose hand-off needs every consumer warp to see every pose (2J >= warps)
  const bool fused = !kArgmax && p.P[0] != nullptr;
  if (fused && 2 * p.joints < kHeatWarps) return launch_heat_nw<T, kArgmax, kHeatWarpsMin>(p, st);
  return launch_heat_nw<T, kArgmax, kHeatWarps>(p, st);
}

static int check_heat_shape(const char* who, int H, int W, int elem_bytes) {
  const long long hw = (long long)H * W;
  CDR_CHECK_ARG(H > 0 && W > 0 && hw * elem_bytes <= kTileBytes,
                "%s: heat-map %dx%d does not fit a %d-byte tile", who, H, W, kTileBytes);
  CDR_CHECK_ARG(W % (16 / elem_bytes) == 0, "%s: W=%d must be a multiple of %d", who, W,
                16 / elem_bytes);
  return CDR_OK;
}

int heat_set_debug(unsigned int* d) {
  CDR_CUDA(cudaMemcpyToSymbol(ptx::g_cdr_debug, &d, sizeof(d)));
  return CDR_OK;
}

}  // namespace cdr

using namespace cdr;

extern "C" int cdr_softargmax(const float* heat, long long n_maps, int H, int W, float scale,
                              float* kp, void* stream) {
  CDR_CHECK_ARG(heat && kp && n_maps >= 0, "cdr_softargmax: bad args");
  if (int rc = check_heat_shape("cdr_softargmax", H, W, 4)) return rc;
  CDR_CHECK_ARG(((uintptr_t)heat & 15) == 0, "cdr_softargmax: heat must be 16-byte aligned");
  if (n_maps == 0) return CDR_OK;
  HeatParams p{};
  p.heat[0] = heat;
  p.kp[0] = kp;
  p.batch = n_maps;
  p.n_views = 1;
  p.joints = 1;
  p.H = H;
  p.W = W;
  p.scale = scale;
  return launch_heat<float, false>(p, (cudaStream_t)stream);
}

extern "C" int cdr_softargmax_dlt(const void* heat_l, const void* heat_r, int heat_is_bf16,
                                  const float* P_l, const float* P_r, long long batch, int joints,
                                  int H, int W, float scale, float* kp2d_l, float* kp2d_r,
                                  float* xyz, const double* gt3d, const double* gt2d_l,
                                  const double* gt2d_r, const double* vis, double* pose_err,
                                  void* stream) {
  CDR_CHECK_ARG(heat_l && heat_r && P_l && P_r && xyz && batch >= 0, "cdr_softargmax_dlt: bad args");
  CDR_CHECK_ARG(joints > 0 && joints <= kMaxJoints, "cdr_softargmax_dlt: joints must be 1..%d",
                kMaxJoints);
  if (int rc = check_heat_shape("cdr_softargmax_dlt", H, W, heat_is_bf16 ? 2 : 4)) return rc;
  CDR_CHECK_ARG((((uintptr_t)heat_l | (uintptr_t)heat_r) & 15) == 0,
                "cdr_softargmax_dlt: heat-maps must be 16-byte aligned");
  CDR_CHECK_ARG(!gt3d || (gt2d_l && gt2d_r && pose_err),
                "cdr_softargmax_dlt: gt3d given without gt2d/pose_err");
  if (batch == 0) return CDR_OK;
  // the pose hand-off (pose_empty) assumes every consumer warp sees every pose: 2J >= #warps
  CDR_CHECK_ARG(2 * joints >= kHeatWarpsMin || !gt3d,
                "cdr_softargmax_dlt: fused MPJPE needs joints >= %d", kHeatWarpsMin / 2);
  if (2 * joints < kHeatWarpsMin) {   // tiny skeletons: unfused (two soft-argmax launches + cdr_dlt)
    CDR_CHECK_ARG(!heat_is_bf16 && kp2d_l && kp2d_r, "cdr_softargmax_dlt: joints < %d needs fp32 maps and 2D outputs",
                  kHeatWarpsMin / 2);
    if (int rc = cdr_softargmax((const float*)heat_l, batch * joints, H, W, scale, kp2d_l, stream)) return rc;
    if (int rc = cdr_softargmax((const float*)heat_r, batch * joints, H, W, scale, kp2d_r, stream)) return rc;
    CDR_CHECK_ARG(batch <= 0x7fffffff, "cdr_softargmax_dlt: batch too large for the unfused path");
    return cdr_dlt(P_l, P_r, kp2d_l, kp2d_r, (int)batch, joints, xyz, stream);
  }
  HeatParams p{};
  p.heat[0] = heat_l;
  p.heat[1] = heat_r;
  p.P[0] = P_l;
  p.P[1] = P_r;
  p.kp[0] = kp2d_l;
  p.kp[1] = kp2d_r;
  p.xyz = xyz;
  p.gt3d = gt3d;
  p.gt2d[0] = gt2d_l;
  p.gt2d[1] = gt2d_r;
  p.vis = vis;
  p.pose_err = pose_err;
  p.batch = batch;
  p.n_views = 2;
  p.joints = joints;
  p.H = H;
  p.W = W;
  p.scale = scale;
  if (heat_is_bf16) return launch_heat<__nv_bfloat16, false>(p, (cudaStream_t)stream);
  return launch_heat<float, false>(p, (cudaStream_t)stream);
}

extern "C" int cdr_argmax(const float* heat, long long n_maps, int H, int W, float scale,
                          float* preds, float* maxvals, uint8_t* pts_u8, void* stream) {
  CDR_CHECK_ARG(heat && n_maps >= 0, "cdr_argmax: bad args");
  CDR_CHECK_ARG(preds || maxvals || pts_u8, "cdr_argmax: no output requested");
  if (int rc = check_heat_shape("cdr_argmax", H, W, 4)) return rc;
  CDR_CHECK_ARG(((uintptr_t)heat & 15) == 0, "cdr_argmax: heat must be 16-byte aligned");
  if (n_maps == 0) return CDR_OK;
  HeatParams p{};
  p.heat[0] = heat;
  p.kp[0] = preds;
  p.maxvals = maxvals;
  p.pts_u8 = pts_u8;
  p.batch = n_maps;
  p.n_views = 1;
  p.joints = 1;
  p.H = H;
  p.W = W;
  p.scale = scale;
  return launch_heat<float, true>(p, (cudaStream_t)stream);
}
