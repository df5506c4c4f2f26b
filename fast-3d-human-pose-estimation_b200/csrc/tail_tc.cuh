// Fused decoder tail (included by gemm_tc.cu): deconv3 -> BN -> ReLU -> final 1x1 (+bias) -> per-tile soft-argmax
// partial sums, one kernel.  Reference: models/decoder.py:42-44 (deconv3, final_layer), models/cdrnet.py:120-149,250
// (process_heatmap) — the 256-channel 64x64 activation of deconv3 (1.07 GB per 64 stereo pairs in fp32 mode: written
// once and read once by the unfused path) never leaves the SM.
//
// Per (128-pixel block of the 32x32 input grid, output phase g) the main loop is the tap-GEMM of gemm_tc.cu (4 taps as
// shifted 4-D TMA boxes, tcgen05.mma into TMEM).  Then, instead of storing the tile:
//   convert warps (8)  TMEM -> registers, + folded-BN bias, ReLU, encode bf16 and write the tile into a 128B-swizzled
//                      shared-memory buffer "A2" laid out as the A operand of a second MMA;
//   MMA issuer         polls for A2 between K blocks of the NEXT tile and issues heat[128 x 32] (+)= A2 * Wfin^T
//                      (Wfin resident in shared memory) into TMEM columns of the accumulator the convert warps have
//                      just finished reading — no extra TMEM;
//   heat warps (4)     tcgen05.ld the 128 x 32 heat tile (one output pixel per thread, joints along columns), + bias,
//                      optionally store planar fp32 heat-maps (taps / PoseResNet), and reduce the warp's 32 pixels — one
//                      row of the phase — to a soft-argmax partial {max, sum e, sum lane*e} per joint with shuffles.
// A second, tiny kernel merges the 128 partials of every heat-map (online-softmax merge in fp64), scales to image
// pixels and runs the per-joint DLT (+ MPJPE terms) — tail_merge_dlt_kernel.
//
// This kernel runs the bf16 decoder: BN = 256 (whole channel range per tile), ring of 3 x 48 KB K-blocks, A2 = 64 KB (one
// hand-off per tile).  The f16x2 decoder runs the same tail on cta_group::2 CTA pairs (tail_pair_tc.cuh).
#pragma once

namespace cdr {

constexpr int kTailSlots = 128;   // soft-argmax partial records per heat-map: 8 pixel blocks x 4 phases x 4 warps (rows)

struct TailParams {
  int n_img;                // images (both views stacked)
  int num_units;            // (n_img * 1024 / 128) * 4 phases
  int joints;
  const float* bias;        // deconv3 folded BN bias (256)
  const float* wsi;         // f16x2: per packed deconv3 weight row (phase * 256 + n): 2^-t
  const float* scale_in;    // f16x2: s of the input tensor (d2)
  const float* amax_in;     // f16x2: max |d2|      } bound for the scale of the deconv3 activation
  const float* norms;       // f16x2: {max_row ||W||_1, max |bias|} of deconv3
  const float* bias_fin;    // final layer bias (32, zero padded)
  const float* wsi_fin;     // f16x2: per final-layer row 2^-t
  float* heat;              // optional planar (n_img, J, 64, 64) fp32 heat-maps
  float4* part;             // (n_img, J, kTailSlots) records {max, sum e, sum lane*e, -}
};

struct TailCfg {
  static constexpr int kBN = 256;
  static constexpr int kSlots = 3, kSlotBytes = kABytes + kBN * 128;     // 48 KB
  static constexpr int kA2Bytes = 4 * kABytes;          // four 64-channel K chunks
  static constexpr int kWfBytes = 4 * 32 * 128;         // 32 rows x 256 channels bf16
  static constexpr size_t kSmemBytes = (size_t)kSlots * kSlotBytes + kA2Bytes + kWfBytes + 1024 + 512;
  static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
};
constexpr int kTailThreads = 32 * 14;     // producer, MMA issuer, 8 convert warps, 4 heat warps

__device__ __forceinline__ float ptx_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));   // one MUFU.EX2, rel. error 2^-22
  return y;
}

__global__ void __launch_bounds__(kTailThreads, 1)
deconv_tail_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const __grid_constant__ CUtensorMap tmap_w, const TailParams p) {
  using Cfg = TailCfg;
  constexpr int BN = Cfg::kBN, S = Cfg::kSlots;
  constexpr int kNumKb = 16;                       // 4 taps x 256 input channels / 64
  constexpr int kW = 32, kHW = 1024;               // input grid of deconv3
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  auto slot_ptr = [&](int s) { return smem + (size_t)s * Cfg::kSlotBytes; };
  uint8_t* a2 = smem + (size_t)S * Cfg::kSlotBytes;
  uint8_t* wf = a2 + Cfg::kA2Bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(wf + Cfg::kWfBytes);
  uint64_t* full = bars;                     // [S]
  uint64_t* empty = bars + S;                // [S]
  uint64_t* tmem_full = bars + 2 * S;        // [2] tile accumulator complete
  uint64_t* tmem_empty = bars + 2 * S + 2;   // [2] heat of that accumulator read: 4 heat warps
  uint64_t* heat_full = bars + 2 * S + 4;    // [2]
  uint64_t* a2_full = bars + 2 * S + 6;      // one phase per hand-off (tile)
  uint64_t* a2_empty = bars + 2 * S + 7;     // heat MMAs of the last hand-off complete
  uint64_t* wf_full = bars + 2 * S + 8;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 9);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // provably warp-uniform (see the issuer)
  const int lane = threadIdx.x & 31;

  ptx::grid_dep_launch();
  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
    ptx::prefetch_tmap(&tmap_w);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], 4);
      ptx::mbar_init(&heat_full[a], 1);
    }
    ptx::mbar_init(a2_full, 8);
    ptx::mbar_init(a2_empty, 1);
    ptx::mbar_init(wf_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc<512>(tmem_base_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  ptx::grid_dep_wait();              // d2 is complete and visible
  const uint32_t tmem_base = *tmem_base_slot;
  // TMEM columns: [0,256) [256,512) two tile accumulators; heat of tile t in the first 32 columns of ITS accumulator
  // (written after the convert warps have drained it).

  if (warp == 0) {
    // ===================================================================== TMA producer (converged; an elected lane issues)
    {
      // final-layer weights: resident for the whole kernel
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(wf_full, Cfg::kWfBytes);
        for (int c = 0; c < 4; ++c) ptx::tma_load_2d(wf + c * 4096, &tmap_w, wf_full, 64 * c, 0);
      }
      __syncwarp();
      uint32_t pos = 0;                          // ring position (slots)
      for (int unit = blockIdx.x; unit < p.num_units; unit += gridDim.x) {
        const int g = unit & 3, m0 = (unit >> 2) * kTcBM;
        const int py = g >> 1, px = g & 1;
        const int img0 = m0 / kHW, y0 = (m0 - img0 * kHW) / kW;
        for (int kb = 0; kb < kNumKb; ++kb, ++pos) {
          const int tap = kb >> 2, k0 = (kb & 3) * 64;
          const int dy = py - (tap >> 1), dx = px - (tap & 1);
          const int brow = g * kDecC;
          const int bk = tap * kDecC + k0, ys = y0 + dy;
          const int s = pos % S;
          ptx::mbar_wait(&empty[s], ((pos / S) & 1) ^ 1u);
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(&full[s], Cfg::kSlotBytes);
            ptx::tma_load_4d(slot_ptr(s), &tmap_a, &full[s], k0, dx, ys, img0);
            ptx::tma_load_2d(slot_ptr(s) + kABytes, &tmap_b, &full[s], bk, brow);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    // The whole warp runs the loop converged and one elected lane issues (gemm_tc.cu explains why: inside an
    // `if (lane == 0)` region ptxas wraps every UTCHMMA in an ELECT / R2UR.BROADCAST loop and the kernel becomes
    // issue-bound).  Barrier polls that steer control flow are made warp-uniform with a vote.
    {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      constexpr uint32_t fmt = 1u;             // kind::f16 operand format: bf16
      constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) |
                                 ((uint32_t)(kTcBM >> 4) << 24);
      constexpr uint32_t idesc_heat = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(32 >> 3) << 17) |
                                      ((uint32_t)(kTcBM >> 4) << 24);
      constexpr uint64_t desc_hi = ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
                                   ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
      auto desc = [&](const uint8_t* ptr) { return desc_hi | (uint64_t)((ptx::smem_u32(ptr) >> 4) & 0x3FFF); };
      uint32_t pos = 0, tl = 0;
      uint32_t rounds_issued = 0;              // hand-offs (tiles) whose heat MMAs have been issued
      uint32_t rounds_due = 0;                 // tiles whose main loop has been issued
      bool wf_ready = false;
      // heat MMAs of tile t: its A2 buffer is full -> issue, release A2, publish heat
      auto issue_round = [&](uint32_t t) {
        if (!wf_ready) {
          ptx::mbar_wait(wf_full, 0);
          wf_ready = true;
        }
        ptx::tc_fence_after();
        const uint32_t acc = t & 1;
        const uint32_t d = tb + acc * BN;
        const uint64_t da0 = desc(a2), dw0 = desc(wf);
        if (ptx::elect_one()) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              ptx::umma_f16(d, da0 + (uint64_t)(c * (kABytes >> 4) + 2 * k), dw0 + (uint64_t)(c * (4096 >> 4) + 2 * k),
                            idesc_heat, (c | k) != 0);
          }
          ptx::umma_commit(a2_empty);
          ptx::umma_commit(&heat_full[acc]);
        }
        __syncwarp();
      };
      // has the next due hand-off been written?  (a vote makes the answer — and the branch — warp-uniform)
      auto round_ready = [&]() {
        return rounds_issued < rounds_due && __all_sync(0xffffffffu, ptx::mbar_test_wait(a2_full, rounds_issued & 1));
      };
      auto poll_rounds = [&]() {
        while (round_ready()) {
          issue_round(rounds_issued);
          ++rounds_issued;
        }
      };
      auto force_rounds = [&](uint32_t upto) {
        while (rounds_issued < upto) {
          ptx::mbar_wait(a2_full, rounds_issued & 1);
          issue_round(rounds_issued);
          ++rounds_issued;
        }
      };
      for (int unit = blockIdx.x; unit < p.num_units; unit += gridDim.x, ++tl) {
        const uint32_t acc = tl & 1;
        // the heat of the tile that used this accumulator must have been issued before we can wait for its readers
        if (tl >= 2) force_rounds(tl - 1);
        ptx::mbar_wait(&tmem_empty[acc], ((tl >> 1) & 1) ^ 1u);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tb + acc * BN;
        for (int kb = 0; kb < kNumKb; ++kb, ++pos) {
          poll_rounds();
          const int s = pos % S;
          ptx::mbar_wait(&full[s], (pos / S) & 1);
          ptx::tc_fence_after();
          const uint64_t da = desc(slot_ptr(s)), db = desc(slot_ptr(s) + kABytes);
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              ptx::umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
            ptx::umma_commit(&empty[s]);
          }
          __syncwarp();
        }
        if (ptx::elect_one()) ptx::umma_commit(&tmem_full[acc]);
        __syncwarp();
        ++rounds_due;
      }
      force_rounds(rounds_due);
    }
  } else if (warp < 10) {
    // ===================================================================== convert warps (2..9)
    const int q = warp & 3;                        // TMEM lane quarter
    const int ew = warp - 2;
    const int grp = ew >> 2;                       // column group: columns [grp * BN/2, (grp+1) * BN/2) of the tile
    constexpr int kCols = BN / 2;
    const int cb0 = grp * kCols;
    const int row = q * 32 + lane;                 // this thread's pixel inside the tile
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const float* __restrict__ bias = p.bias + cb0;   // first output channel of this warp
    uint32_t tl = 0;
    for (int unit = blockIdx.x; unit < p.num_units; unit += gridDim.x, ++tl) {
      const uint32_t acc = tl & 1;
      ptx::mbar_wait(&tmem_full[acc], (tl >> 1) & 1);
      ptx::tc_fence_after();
      // A2 is free once the heat MMAs of tile tl-1 have completed ("phase -1" of a fresh barrier reads as complete)
      ptx::mbar_wait(a2_empty, (tl & 1) ^ 1u);
#pragma unroll 1
      for (int c = 0; c < kCols; c += 64) {
        uint32_t r0[32], r1[32];
        ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)(acc * BN + cb0 + c), r0);
        ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)(acc * BN + cb0 + c + 32), r1);
        ptx::tmem_ld_wait();
        uint32_t w[32];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + c) + j4);
          const float4 b5 = __ldg(reinterpret_cast<const float4*>(bias + c + 32) + j4);
          const __nv_bfloat162 x0 = __floats2bfloat162_rn(fmaxf(__uint_as_float(r0[4 * j4]) + b4.x, 0.f),
                                                          fmaxf(__uint_as_float(r0[4 * j4 + 1]) + b4.y, 0.f));
          const __nv_bfloat162 x1 = __floats2bfloat162_rn(fmaxf(__uint_as_float(r0[4 * j4 + 2]) + b4.z, 0.f),
                                                          fmaxf(__uint_as_float(r0[4 * j4 + 3]) + b4.w, 0.f));
          const __nv_bfloat162 y0 = __floats2bfloat162_rn(fmaxf(__uint_as_float(r1[4 * j4]) + b5.x, 0.f),
                                                          fmaxf(__uint_as_float(r1[4 * j4 + 1]) + b5.y, 0.f));
          const __nv_bfloat162 y1 = __floats2bfloat162_rn(fmaxf(__uint_as_float(r1[4 * j4 + 2]) + b5.z, 0.f),
                                                          fmaxf(__uint_as_float(r1[4 * j4 + 3]) + b5.w, 0.f));
          w[2 * j4] = *reinterpret_cast<const uint32_t*>(&x0);
          w[2 * j4 + 1] = *reinterpret_cast<const uint32_t*>(&x1);
          w[16 + 2 * j4] = *reinterpret_cast<const uint32_t*>(&y0);
          w[16 + 2 * j4 + 1] = *reinterpret_cast<const uint32_t*>(&y1);
        }
        // K chunk (cb0 + c) / 64 of A2: row `row`, 128 bytes, 16-byte pieces XOR-swizzled by the row (SWIZZLE_128B)
        const uint32_t base = ptx::smem_u32(a2) + (uint32_t)(((cb0 + c) >> 6) * kABytes) + (uint32_t)row * 128u;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          ptx::st_shared_v4(base + (uint32_t)((j ^ (row & 7)) << 4), w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
      }
      ptx::fence_proxy_async();                    // generic-proxy writes -> visible to the tensor core's smem reads
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(a2_full);
    }
  } else {
    // ===================================================================== heat warps (10..13)
    const int q = warp & 3;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int J = p.joints;
    uint32_t tl = 0;
    const float kLog2e = 1.4426950408889634f;
    for (int unit = blockIdx.x; unit < p.num_units; unit += gridDim.x, ++tl) {
      const int g = unit & 3, m0 = (unit >> 2) * kTcBM;
      const uint32_t acc = tl & 1;
      ptx::mbar_wait(&heat_full[acc], (tl >> 1) & 1);
      ptx::tc_fence_after();
      uint32_t r[32];
      ptx::tmem_ld_32x32b_x32(lane_addr + acc * BN, r);
      ptx::tmem_ld_wait();
      float hv[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) hv[j] = __uint_as_float(r[j]);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
      // ---- one output pixel per thread: input pixel (y, x = lane) of image img, output (2y + py, 2x + px)
      const int img = m0 / kHW;
      const int y = (m0 - img * kHW) / kW + q;
      const int oy = 2 * y + (g >> 1), ox = 2 * lane + (g & 1);
      const int slot = (((m0 - img * kHW) >> 7) * 4 + g) * 4 + q;
      float rec_m = 0.f, rec_s = 0.f, rec_l = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (j < J) {                               // warp-uniform
          const float v = hv[j] + __ldg(p.bias_fin + j);
          if (p.heat) p.heat[((size_t)img * J + j) * 4096 + oy * 64 + ox] = v;
          if (p.part) {                            // warp-uniform
            float m = v;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            float e = ptx_ex2((v - m) * kLog2e);
            if (m == -INFINITY) e = 0.f;           // a row of -inf logits carries no weight (and no NaN)
            float se = e, sl = e * (float)lane;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              se += __shfl_xor_sync(0xffffffffu, se, o);
              sl += __shfl_xor_sync(0xffffffffu, sl, o);
            }
            if (lane == j) { rec_m = m; rec_s = se; rec_l = sl; }
          }
        }
      }
      if (p.part && lane < J) p.part[((size_t)img * J + lane) * kTailSlots + slot] = make_float4(rec_m, rec_s, rec_l, 0.f);
    }
  }

  // ------------------------------------------------------------------ teardown
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------
// Merge of the per-tile soft-argmax partials + DLT (+ MPJPE terms): one CTA per pose.
//   record t of a heat-map: m_t = max of its 32 logits, S_t = sum exp(h - m_t), L_t = sum lane * exp(h - m_t); its row is
//   Y_t = 2 * (8 * (t >> 4) / 2 ... ) — see slot decoding below — and its pixels sit at X = 2 * lane + px.
//   With M = max_t m_t and w_t = exp(m_t - M):  S = sum w_t S_t,  cx = sum w_t (2 L_t + px_t S_t) / S,  cy = sum w_t Y_t S_t / S
//   — the softmax of models/cdrnet.py:131-133 with its global max, evaluated in fp64 over 128 records instead of 4096 logits.
struct TailMergeParams {
  const float4* part;       // (2B, J, kTailSlots): view-major image order (left images first)
  const float* P[2];        // (B,3,4)
  float* kp[2];             // (B,J,2)
  float* xyz;               // (B,J,3)
  const double* gt3d;       // optional MPJPE inputs (as heat_stream_kernel)
  const double* gt2d[2];
  const double* vis;
  double* pose_err;         // (B,3)
  int batch, joints;
  float scale;
};

// blockDim = 32 * joints: one HALF-warp per heat-map (8 records per lane, all loads in flight at once), so the merge of
// a pose's 2J heat-maps is a single round; warp 0 then runs the J DLT solves.
__global__ void __launch_bounds__(1024) tail_merge_dlt_kernel(const TailMergeParams p) {
  __shared__ double kps[2 * kMaxJoints][2];
  ptx::grid_dep_wait();         // launched with programmatic stream serialization: the tail kernel's records are complete
  const int pose = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, l16 = lane & 15;
  const int J = p.joints;
  for (int item = 2 * warp + (lane >> 4); item < 2 * J; item += 2 * (int)(blockDim.x >> 5)) {   // uniform per half-warp
    const int v = item / J, j = item - v * J;
    const float4* rec = p.part + ((size_t)(v * p.batch + pose) * J + j) * kTailSlots;
    float4 r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = __ldg(rec + l16 + 16 * i);
    float M = -INFINITY;
#pragma unroll
    for (int i = 0; i < 8; ++i) M = fmaxf(M, r[i].x);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o));
    double S = 0.0, SX = 0.0, SY = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int t = l16 + 16 * i;                   // slot = ((pixel block * 4 + phase) * 4 + warp)
      const int blk = t >> 4, g = (t >> 2) & 3, q = t & 3;
      const double Y = (double)(2 * (blk * 4 + q) + (g >> 1));
      const double px = (double)(g & 1);
      const double w = r[i].x == -INFINITY ? 0.0 : (double)exp2f((r[i].x - M) * 1.4426950408889634f);
      const double s = w * (double)r[i].y;
      S += s;
      SX += w * (2.0 * (double)r[i].z) + px * s;
      SY += Y * s;
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      S += __shfl_xor_sync(0xffffffffu, S, o);
      SX += __shfl_xor_sync(0xffffffffu, SX, o);
      SY += __shfl_xor_sync(0xffffffffu, SY, o);
    }
    if (l16 == 0) {
      const double cx = SX / S * (double)p.scale, cy = SY / S * (double)p.scale;
      kps[item][0] = cx;
      kps[item][1] = cy;
      const size_t o = (size_t)pose * J + j;
      if (p.kp[v]) { p.kp[v][o * 2] = (float)cx; p.kp[v][o * 2 + 1] = (float)cy; }
    }
  }
  __syncthreads();
  if (warp != 0) return;
  double e0 = 0.0, e1 = 0.0, e2 = 0.0;
  for (int j = lane; j < J; j += 32) {
    const double ul = kps[j][0], vl = kps[j][1], ur = kps[J + j][0], vr = kps[J + j][1];
    double A[4][4];
    dlt_rows(p.P[0] + (size_t)pose * 12, ul, vl, A, 0);
    dlt_rows(p.P[1] + (size_t)pose * 12, ur, vr, A, 2);
    double x, y, z;
    dlt_solve4(A, x, y, z);
    const size_t o = (size_t)pose * J + j;
    const float fx = (float)x, fy = (float)y, fz = (float)z;
    p.xyz[o * 3] = fx; p.xyz[o * 3 + 1] = fy; p.xyz[o * 3 + 2] = fz;
    if (p.gt3d) {                                  // the reference's calc_mpjpe consumes the fp32 outputs
      const double w = p.vis ? p.vis[o] : 1.0;
      double dx = ((double)(float)ul - p.gt2d[0][o * 2]) * w, dy = ((double)(float)vl - p.gt2d[0][o * 2 + 1]) * w;
      e0 += sqrt(dx * dx + dy * dy);
      dx = ((double)(float)ur - p.gt2d[1][o * 2]) * w; dy = ((double)(float)vr - p.gt2d[1][o * 2 + 1]) * w;
      e1 += sqrt(dx * dx + dy * dy);
      dx = ((double)fx - p.gt3d[o * 3]) * w; dy = ((double)fy - p.gt3d[o * 3 + 1]) * w;
      const double dz = ((double)fz - p.gt3d[o * 3 + 2]) * w;
      e2 += sqrt(dx * dx + dy * dy + dz * dz);
    }
  }
  if (p.gt3d) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      e0 += __shfl_xor_sync(0xffffffffu, e0, o);
      e1 += __shfl_xor_sync(0xffffffffu, e1, o);
      e2 += __shfl_xor_sync(0xffffffffu, e2, o);
    }
    if (lane == 0) { p.pose_err[pose * 3] = e0; p.pose_err[pose * 3 + 1] = e1; p.pose_err[pose * 3 + 2] = e2; }
  }
}

}  // namespace cdr
