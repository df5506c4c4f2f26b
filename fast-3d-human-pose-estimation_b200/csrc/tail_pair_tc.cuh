// The fused decoder tail of tail_tc.cuh for the f16x2 decoder, on cta_group::2 CTA pairs (included by gemm_tc.cu after
// tail_tc.cuh).
//
// Same structure, same partial records, same merge kernel.  The operands are scaled fp16 hi/lo planes (gemm_tc.cu:
// kKindF16X2): BN = 128 (TMEM holds 2 main-chunk + 2 correction accumulators of 128 columns), the two channel halves of a
// pixel block run back to back and the heat partial of the first half waits in registers of the heat warps; A2 = 32 KB =
// one 64-channel K chunk in both planes, so a tile takes two hand-offs (column group 0, then group 1).
// What changes against tail_tc.cuh is who feeds the tensor cores: a cluster of two
// CTAs takes two consecutive 128-pixel blocks of the same output phase, every CTA stages its own A rows and HALF of
// each weight tile, the leader (cluster rank 0) issues every tcgen05.mma for both SMs (M = 256) — main loop AND the heat
// MMAs — and each CTA's convert / heat warps work on the accumulator rows in their own TMEM.  Per SM and MMA the tensor
// core then reads A + B/2 from shared memory instead of A + B, and the TMA fills shrink by the same B/2: the f16x2 main
// loop asked 213 B/clk of a 128 B/clk shared memory (gemm_tc.cu, CL = 2 comment).
//
// Shared memory per CTA: 3 stages x 48 KB [A hi | A lo | B hi (64 rows) | B lo] + A2 32 KB + final-layer tiles 24 KB.
// Final-layer operand of the pair (the B operand of a cta_group::2 MMA is split by rows between the two CTAs, at the SAME
// shared-memory offset in both):
//   N = 64 form  hi . [Wh ; Wl]: region X holds Wh (32 rows) in CTA 0 and Wl (32 rows) in CTA 1;
//   N = 32 form  lo . Wh       : region Y holds Wh rows 0-15 in CTA 0 and rows 16-31 in CTA 1.
// Barriers: the leader's instances of full[] / a2_full / chunk_empty[] / tmem_empty[] collect both CTAs (TMA bytes through
// cp.async.bulk.tensor.cta_group::2, thread arrivals through mapa + mbarrier.arrive.shared::cluster); everything the
// issuer publishes (stage release, chunk / tile / heat completion, A2 release) is a multicast commit to both CTAs.
#pragma once

namespace cdr {

struct TailPairCfg {
  static constexpr int kBN = 128, kNH = 2, kStages = 3;
  static constexpr int kBHalfBytes = (kBN / 2) * 128;                       // 8 KB per plane
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBHalfBytes;         // 48 KB
  static constexpr int kA2Bytes = 2 * kABytes;                              // one 64-channel K chunk, hi and lo planes
  static constexpr int kWxBytes = 4 * 32 * 128, kWyBytes = 4 * 16 * 128;    // (half, chunk) x 32 rows / x 16 rows
  static constexpr int kRounds = 2, kRoundWarps = 4;                        // hand-offs per tile, warps per hand-off
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + kA2Bytes + kWxBytes + kWyBytes + 1024 + 512;
  static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
};

__global__ void __launch_bounds__(kTailThreads, 1)
deconv_tail_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a_lo,
                        const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_b_lo,
                        const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_w_lo,
                        const __grid_constant__ CUtensorMap tmap_w16, const TailParams p) {
  using Cfg = TailPairCfg;
  constexpr int BN = Cfg::kBN, NH = Cfg::kNH, S = Cfg::kStages;
  constexpr int kNumKb = 16;
  constexpr int kW = 32, kHW = 1024;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // stage s: [A (hi) | A lo | B half (hi) | B half lo]
  auto st_a = [&](int s, int plane) { return smem + (size_t)s * Cfg::kStageBytes + (size_t)plane * kABytes; };
  auto st_b = [&](int s, int plane) {
    return smem + (size_t)s * Cfg::kStageBytes + (size_t)2 * kABytes + (size_t)plane * Cfg::kBHalfBytes;
  };
  uint8_t* a2 = smem + (size_t)S * Cfg::kStageBytes;
  uint8_t* wx = a2 + Cfg::kA2Bytes;              // 4 x 4 KB, index nh * 2 + j
  uint8_t* wy = wx + Cfg::kWxBytes;              // 4 x 2 KB, index nh * 2 + j
  uint64_t* bars = reinterpret_cast<uint64_t*>(wy + Cfg::kWyBytes);
  uint64_t* full = bars;                     // [S]  leader's: both CTAs' TMA bytes
  uint64_t* empty = bars + S;                // [S]  own: multicast commit
  uint64_t* tmem_full = bars + 2 * S;        // [2]  own
  uint64_t* tmem_empty = bars + 2 * S + 2;   // [2]  leader's: 4 heat warps of each CTA
  uint64_t* chunk_full = bars + 2 * S + 4;   // [2]  own
  uint64_t* chunk_empty = bars + 2 * S + 6;  // [2]  leader's: 8 convert warps of each CTA
  uint64_t* heat_full = bars + 2 * S + 8;    // [2]  own
  uint64_t* a2_full = bars + 2 * S + 10;     //      leader's: the round's warps of both CTAs
  uint64_t* a2_empty = bars + 2 * S + 11;    // [2]  own
  uint64_t* wf_full = bars + 2 * S + 13;     //      leader's: final-layer tiles of both CTAs
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 14);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  ptx::grid_dep_launch();
  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
    ptx::prefetch_tmap(&tmap_w);
    ptx::prefetch_tmap(&tmap_w16);
    ptx::prefetch_tmap(&tmap_a_lo);
    ptx::prefetch_tmap(&tmap_b_lo);
    ptx::prefetch_tmap(&tmap_w_lo);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], 2 * 4);
      ptx::mbar_init(&chunk_full[a], 1);
      ptx::mbar_init(&chunk_empty[a], 2 * 8);
      ptx::mbar_init(&heat_full[a], 1);
    }
    ptx::mbar_init(a2_full, 2 * Cfg::kRoundWarps);
    ptx::mbar_init(&a2_empty[0], 1);
    ptx::mbar_init(&a2_empty[1], 1);
    ptx::mbar_init(wf_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc_2sm<512>(tmem_base_slot);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();                 // the peer's barriers exist before any remote arrival / multicast commit
  ptx::tc_fence_after();
  const uint32_t rank = ptx::cluster_ctarank();
  ptx::grid_dep_wait();
  const uint32_t tmem_base = *tmem_base_slot;

  // pair units: (pixel-block pair, phase); this CTA's block is 2 * pair + rank
  const int pu0 = (int)(blockIdx.x >> 1), pu_step = (int)(gridDim.x >> 1);
  const int num_pu = p.num_units >> 1;
  auto unit_m0 = [&](int pu) { return (((pu >> 2) << 1) + (int)rank) * kTcBM; };
  // a thread arrival on a barrier of the MMA issuer: the leader's instance
  auto arrive_leader = [&](uint64_t* bar) {
    if (rank != 0) ptx::mbar_arrive_cluster(ptx::mapa_u32(ptx::smem_u32(bar), 0));
    else ptx::mbar_arrive(bar);
  };

  if (warp == 0) {
    // ===================================================================== TMA producer (both CTAs; converged)
    {
      const uint32_t wf_leader = ptx::mapa_u32(ptx::smem_u32(wf_full), 0);
      if (ptx::elect_one()) {
        if (rank == 0) ptx::mbar_arrive_expect_tx(wf_full, 2 * (Cfg::kWxBytes + Cfg::kWyBytes));
        for (int c = 0; c < 4; ++c) {              // c = half * 2 + chunk: channels [64c, 64c + 64)
          ptx::tma_load_2d_2sm(wx + c * 4096, rank == 0 ? &tmap_w : &tmap_w_lo, wf_leader, 64 * c, 0);
          ptx::tma_load_2d_2sm(wy + c * 2048, &tmap_w16, wf_leader, 64 * c, 16 * (int)rank);
        }
      }
      __syncwarp();
      uint32_t it = 0;
      for (int pu = pu0; pu < num_pu; pu += pu_step) {
        const int g = pu & 3, m0 = unit_m0(pu);
        const int py = g >> 1, px = g & 1;
        const int img0 = m0 / kHW, y0 = (m0 - img0 * kHW) / kW;
        for (int nh = 0; nh < NH; ++nh) {
          for (int kb = 0; kb < kNumKb; ++kb, ++it) {
            const int s = it % S;
            ptx::mbar_wait(&empty[s], ((it / S) & 1) ^ 1u);
            const int tap = kb >> 2, k0 = (kb & 3) * 64;
            const int dy = py - (tap >> 1), dx = px - (tap & 1);
            const int brow = g * kDecC + nh * BN + (int)rank * (BN / 2);
            const int bk = tap * kDecC + k0, ys = y0 + dy;
            const uint32_t full_leader = ptx::mapa_u32(ptx::smem_u32(&full[s]), 0);
            if (ptx::elect_one()) {
              if (rank == 0) ptx::mbar_arrive_expect_tx(&full[s], 2 * Cfg::kStageBytes);
              ptx::tma_load_4d_2sm(st_a(s, 0), &tmap_a, full_leader, k0, dx, ys, img0);
              ptx::tma_load_4d_2sm(st_a(s, 1), &tmap_a_lo, full_leader, k0, dx, ys, img0);
              ptx::tma_load_2d_2sm(st_b(s, 0), &tmap_b, full_leader, bk, brow);
              ptx::tma_load_2d_2sm(st_b(s, 1), &tmap_b_lo, full_leader, bk, brow);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (leader CTA only; converged)
    if (rank == 0) {
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      constexpr uint32_t fmt = 0u;             // kind::f16 operand format: f16
      constexpr uint32_t kM2 = (uint32_t)((2 * kTcBM) >> 4) << 24;          // M = 256 across the pair
      constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) | kM2;
      constexpr uint32_t idesc_n32 = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(32 >> 3) << 17) | kM2;
      constexpr uint32_t idesc_n64 = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(64 >> 3) << 17) | kM2;
      constexpr uint64_t desc_hi = ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
                                   ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
      auto desc = [&](const uint8_t* ptr) { return desc_hi | (uint64_t)((ptx::smem_u32(ptr) >> 4) & 0x3FFF); };
      uint32_t it = 0, tl = 0, ch = 0;
      uint32_t rounds_issued = 0, rounds_due = 0;
      bool wf_ready = false;
      auto issue_round = [&](uint32_t r) {
        if (!wf_ready) {
          ptx::mbar_wait(wf_full, 0);
          wf_ready = true;
        }
        ptx::tc_fence_after();
        const uint32_t t = r / Cfg::kRounds, j = r % Cfg::kRounds;
        const uint32_t acc = t & 1;
        // [hi.Wh | hi.Wl] in ONE N = 64 MMA: the hi and lo planes of the 32 final-layer rows are adjacent 32-row blocks
        // of the operand and their accumulators adjacent 32-column blocks in TMEM — the hi plane of A2 is read once
        // instead of twice (the heat MMAs are bound by their operand reads); lo.Wh then adds into the correction columns.
        const uint32_t nh = t % NH;            // tiles alternate between the two channel halves of a unit
        const uint32_t d_hm = tb + (2 + acc) * BN, d_hc = d_hm + 32;
        const uint64_t da = desc(a2), dal = desc(a2 + kABytes);
        const uint64_t dx = desc(wx) + (uint64_t)((nh * 2 + j) * (4096 >> 4));     // [Wh ; Wl] split across the pair
        const uint64_t dy = desc(wy) + (uint64_t)((nh * 2 + j) * (2048 >> 4));     // Wh split across the pair
        const uint32_t first = j != 0;
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t o = (uint64_t)(2 * k);
            ptx::umma_f16_2sm(d_hm, da + o, dx + o, idesc_n64, k ? 1u : first);      // hi * [hi ; lo]
            ptx::umma_f16_2sm(d_hc, dal + o, dy + o, idesc_n32, 1u);                 // lo * hi
          }
          ptx::umma_commit_2sm_mc(&a2_empty[j], 3);
          if (j == Cfg::kRounds - 1) ptx::umma_commit_2sm_mc(&heat_full[acc], 3);
        }
        __syncwarp();
      };
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
      for (int pu = pu0; pu < num_pu; pu += pu_step) {
        for (int nh = 0; nh < NH; ++nh, ++tl) {
          const uint32_t acc = tl & 1;
          if (tl >= 2) force_rounds((tl - 1) * Cfg::kRounds);
          ptx::mbar_wait(&tmem_empty[acc], ((tl >> 1) & 1) ^ 1u);
          ptx::tc_fence_after();
          const uint32_t d_corr = tb + (2 + acc) * BN;
          for (int kb0 = 0; kb0 < kNumKb; kb0 += kSplitChunk, ++ch) {
            const int buf = ch & 1;
            // The drain of this chunk buffer may sit behind a hand-off only this warp can complete (column group 1
            // waits for group 0's heat MMAs before it writes A2, then drains): keep serving rounds while waiting.
            {
              const long long t0 = clock64();
              while (!__all_sync(0xffffffffu, ptx::mbar_test_wait(&chunk_empty[buf], ((ch >> 1) & 1) ^ 1u))) {
                poll_rounds();
                if (clock64() - t0 > 8000000000LL) __trap();
              }
            }
            ptx::tc_fence_after();
            const uint32_t d_main = tb + (uint32_t)(buf * BN);
            const int kb1 = kb0 + kSplitChunk < kNumKb ? kb0 + kSplitChunk : kNumKb;
            for (int kb = kb0; kb < kb1; ++kb, ++it) {
              poll_rounds();
              const int s = it % S;
              ptx::mbar_wait(&full[s], (it / S) & 1);
              ptx::tc_fence_after();
              const uint64_t da = desc(st_a(s, 0)), dal = desc(st_a(s, 1));
              const uint64_t db = desc(st_b(s, 0)), dbl = desc(st_b(s, 1));
              const uint32_t first = kb != 0, first_main = kb > kb0;
              if (ptx::elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint64_t o = (uint64_t)(2 * k);
                  ptx::umma_f16_2sm(d_corr, dal + o, db + o, idesc, k ? 1u : first);        // lo*hi
                  ptx::umma_f16_2sm(d_corr, da + o, dbl + o, idesc, 1u);                    // hi*lo
                  ptx::umma_f16_2sm(d_main, da + o, db + o, idesc, k ? 1u : first_main);    // hi*hi, short chain
                }
                ptx::umma_commit_2sm_mc(&empty[s], 3);
              }
              __syncwarp();
            }
            if (ptx::elect_one()) ptx::umma_commit_2sm_mc(&chunk_full[buf], 3);
            __syncwarp();
          }
          if (ptx::elect_one()) ptx::umma_commit_2sm_mc(&tmem_full[acc], 3);
          __syncwarp();
          rounds_due += Cfg::kRounds;
        }
      }
      force_rounds(rounds_due);
    }
  } else if (warp < 10) {
    // ===================================================================== convert warps (2..9), per CTA
    const int q = warp & 3;
    const int ew = warp - 2;
    const int grp = ew >> 2;
    constexpr int kCols = BN / 2;
    const int cb0 = grp * kCols;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t tl = 0, ch = 0;
    const float a_inv = 1.f / __ldcg(p.scale_in);
    const float s_out = f16_pow2_scale(__ldcg(p.amax_in) * __ldg(p.norms) + __ldg(p.norms + 1));
    // A2 is free for this warp's hand-off of tile tl once the heat MMAs of the hand-off BEFORE it have completed:
    //   column group 0: group 1's hand-off of tile tl-1 -> a2_empty[1], phase tl-1
    //   column group 1: group 0's hand-off of tile tl   -> a2_empty[0], phase tl
    // ("phase -1" of a fresh barrier reads as complete.)  Own a2_empty[]: released for both CTAs by multicast commits.
    auto wait_a2_free = [&]() {
      if (grp == 0) ptx::mbar_wait(&a2_empty[1], (tl & 1) ^ 1u);
      else ptx::mbar_wait(&a2_empty[0], tl & 1);
    };
    auto publish_a2 = [&]() {
      ptx::fence_proxy_async();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) arrive_leader(a2_full);
    };
    for (int pu = pu0; pu < num_pu; pu += pu_step) {
      const int g = pu & 3;
      for (int nh = 0; nh < NH; ++nh, ++tl) {
        const uint32_t acc = tl & 1;
        const int n_base = nh * BN + cb0;
        const float* __restrict__ bias = p.bias + n_base;
        float sum[kCols];
#pragma unroll
        for (int j = 0; j < kCols; ++j) sum[j] = 0.f;
        for (int kb0 = 0; kb0 < kNumKb; kb0 += kSplitChunk, ++ch) {
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
          if (lane == 0) arrive_leader(&chunk_empty[buf]);
        }
        ptx::mbar_wait(&tmem_full[acc], (tl >> 1) & 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int c = 0; c < kCols; c += 32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(lane_addr + (uint32_t)((2 + acc) * BN + cb0 + c), r);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[c + j] = fmaf(__uint_as_float(r[j]), 1.f / kLoScale, sum[c + j]);
        }
        const float* __restrict__ wsi = p.wsi + (size_t)g * kDecC + n_base;
        uint32_t wh[32], wl[32];
#pragma unroll
        for (int j4 = 0; j4 < kCols / 4; ++j4) {
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(wsi) + j4);
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias) + j4);
          const float v0 = fmaxf(sum[4 * j4] * (a_inv * w4.x) + b4.x, 0.f) * s_out;
          const float v1 = fmaxf(sum[4 * j4 + 1] * (a_inv * w4.y) + b4.y, 0.f) * s_out;
          const float v2 = fmaxf(sum[4 * j4 + 2] * (a_inv * w4.z) + b4.z, 0.f) * s_out;
          const float v3 = fmaxf(sum[4 * j4 + 3] * (a_inv * w4.w) + b4.w, 0.f) * s_out;
          const __half2 h01 = __floats2half2_rn(v0, v1), h23 = __floats2half2_rn(v2, v3);
          const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
          const __half2 l01 = __floats2half2_rn((v0 - f01.x) * kLoScale, (v1 - f01.y) * kLoScale);
          const __half2 l23 = __floats2half2_rn((v2 - f23.x) * kLoScale, (v3 - f23.y) * kLoScale);
          wh[2 * j4] = *reinterpret_cast<const uint32_t*>(&h01);
          wh[2 * j4 + 1] = *reinterpret_cast<const uint32_t*>(&h23);
          wl[2 * j4] = *reinterpret_cast<const uint32_t*>(&l01);
          wl[2 * j4 + 1] = *reinterpret_cast<const uint32_t*>(&l23);
        }
        wait_a2_free();
        const uint32_t base = ptx::smem_u32(a2) + (uint32_t)row * 128u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t o = (uint32_t)((j ^ (row & 7)) << 4);
          ptx::st_shared_v4(base + o, wh[4 * j], wh[4 * j + 1], wh[4 * j + 2], wh[4 * j + 3]);
          ptx::st_shared_v4(base + kABytes + o, wl[4 * j], wl[4 * j + 1], wl[4 * j + 2], wl[4 * j + 3]);
        }
        publish_a2();
      }
    }
  } else {
    // ===================================================================== heat warps (10..13), per CTA
    const int q = warp & 3;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int J = p.joints;
    uint32_t tl = 0;
    // 1 / s(deconv3 activation)
    const float fin_scale = ldexpf(1.f, -f16_pow2_exp(__ldcg(p.amax_in) * __ldg(p.norms) + __ldg(p.norms + 1)));
    const float kLog2e = 1.4426950408889634f;
    for (int pu = pu0; pu < num_pu; pu += pu_step) {
      const int g = pu & 3, m0 = unit_m0(pu);
      float hv[32];
#pragma unroll
      for (int nh = 0; nh < NH; ++nh, ++tl) {
        const uint32_t acc = tl & 1;
        ptx::mbar_wait(&heat_full[acc], (tl >> 1) & 1);
        ptx::tc_fence_after();
        uint32_t r[32], rc[32];
        ptx::tmem_ld_32x32b_x32(lane_addr + (2 + acc) * BN, r);
        ptx::tmem_ld_32x32b_x32(lane_addr + (2 + acc) * BN + 32, rc);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float v = fmaf(__uint_as_float(rc[j]), 1.f / kLoScale, __uint_as_float(r[j]));
          hv[j] = nh == 0 ? v : hv[j] + v;       // the first half's partial waits here, in registers
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) arrive_leader(&tmem_empty[acc]);
      }
      const int img = m0 / kHW;
      const int y = (m0 - img * kHW) / kW + q;
      const int oy = 2 * y + (g >> 1), ox = 2 * lane + (g & 1);
      const int slot = (((m0 - img * kHW) >> 7) * 4 + g) * 4 + q;
      float rec_m = 0.f, rec_s = 0.f, rec_l = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (j < J) {
          float v = hv[j];
          v *= fin_scale * __ldg(p.wsi_fin + j);
          v += __ldg(p.bias_fin + j);
          if (p.heat) p.heat[((size_t)img * J + j) * 4096 + oy * 64 + ox] = v;
          if (p.part) {
            float m = v;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            float e = ptx_ex2((v - m) * kLog2e);
            if (m == -INFINITY) e = 0.f;
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
  ptx::cluster_sync();                 // the leader's last commits / the peer's last arrivals have landed
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_2sm<512>(tmem_base);
  }
}

}  // namespace cdr
