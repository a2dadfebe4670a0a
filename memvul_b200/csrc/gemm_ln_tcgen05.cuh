// Fused  x = LayerNorm(A W^T + bias + resid)  for the two residual GEMMs of a BERT layer (attention output
// projection, FFN down-projection; SURVEY.md 2.2 rows K4 and K6 in full), N = 768.
//
// A LayerNorm row needs all 768 outputs, but one CTA pair's TMEM holds only a 256-column accumulator (twice).  So a
// CLUSTER OF SIX CTAs = three cta_group::2 pairs works on one 256-row block: pair p owns columns [256p, 256p+256),
// each CTA 128 of the rows.  Per tile, in every CTA's epilogue warps:
//   pass 1  v = acc + bias + resid (residual 32x32 boxes arrive by TMA, 2 in flight); per-thread statistics of its
//           128 values, accumulated SHIFTED by a pivot piv (the mean of its first 32 values): the sums of d = v - piv
//           and d^2 give the partial's mean and centred sum of squares M2 -- never sum(v^2) - n mean^2, which cancels
//           catastrophically when |mean| >> spread; v is written BACK INTO TMEM (tcgen05.st) -- the accumulator stage
//           doubles as the stash for pass 2;
//   exchange each thread publishes its (mean, M2) for (row, column half) into the shared memory of the three CTAs
//           that own the same rows (st.shared::cluster), then a release/acquire mbarrier round at cluster scope;
//   pass 2  mean / rstd from the 6 partials by the parallel-variance (Chan et al.) combination, M2 = sum M2_p +
//           128 sum (mean_p - mean)^2; y = (v - mean) * rstd * gamma + beta is staged in swizzled smem and leaves by TMA
//           store twice: fp32 (the residual stream) and fp16 (the next GEMM's A operand).
// This removes the stand-alone LayerNorm kernels (9-13 % of the step in r01c/r01d) and the fp32 round trip of the
// pre-LN sum through HBM: 10 bytes per element instead of 18.
// Main loop, barriers and roles are those of gemm_tcgen05_2cta.cuh (warp 0 TMA, warp 1 MMA issue on even ranks,
// warp 2 TMEM alloc, warps 4-11 epilogue).
#pragma once
#include "gemm_tcgen05_2cta.cuh"

namespace mv {

struct GemmLnCfg {
  static constexpr int N = 768, PAIRS = 3, CLUSTER = 6;
  static constexpr int BM = 256, BM_CTA = 128, BN = 256, BN_CTA = 128, BK = 64;
  static constexpr int STAGES = 4;
  static constexpr int A_BYTES = BM_CTA * BK * 2, B_BYTES = BN_CTA * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TMEM_COLS = 2 * BN;
  static constexpr int THREADS = 384, EPI_WARPS = 8;
  static constexpr int STG_BYTES = 4096;                                   // 32 rows x 128 B, SWIZZLE_128B
  static constexpr int OFF_STG = STAGES * STAGE_BYTES;                     // [8 warps][2] staging buffers
  static constexpr int OFF_PRM = OFF_STG + EPI_WARPS * 2 * STG_BYTES;      // [8 warps][bias|gamma|beta][128] floats
  static constexpr int OFF_STATS = OFF_PRM + EPI_WARPS * 3 * 128 * 4;      // [2 slots][6 sources][128 rows] float2
  static constexpr int OFF_BAR = OFF_STATS + 2 * 6 * 128 * 8;
  static constexpr int SMEM_BYTES = OFF_BAR + 512;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB per-CTA shared-memory limit");
};

__global__ void __cluster_dims__(6, 1, 1) __launch_bounds__(384, 1)
gemm_ln_f16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a64,
                           const __grid_constant__ CUtensorMap tmap_b,
                           const __grid_constant__ CUtensorMap tmap_res, const __grid_constant__ CUtensorMap tmap_x32,
                           const __grid_constant__ CUtensorMap tmap_x16, int M, int K, const float* __restrict__ bias,
                           const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int a_multicast,
                           const int* __restrict__ m_dev, unsigned long long* __restrict__ trace,
                           float* __restrict__ x32_ptr, __half* __restrict__ x16_ptr, const float* resid_ptr, int pace) {
  using Cfg = GemmLnCfg;
  // debug only (MEMVUL_LN_TRACE): CTA 0 stamps clock64() at the phase boundaries of its first 8 tiles
  // (epilogue warp 0 slots 0-13, MMA warp slots 14-15; tools/ln_trace.py)
  auto stamp = [&](uint32_t it, int k) {
    if (trace != nullptr && blockIdx.x == 0 && it < 8u) trace[it * 16 + k] = static_cast<unsigned long long>(clock64());
  };
  if (m_dev) M = min(M, __ldg(m_dev));     // packed (var-len) batches: the row count lives on the device
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* empty_bar = full_bar + Cfg::STAGES;
  uint64_t* tfull_bar = empty_bar + Cfg::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* res_bar = tempty_bar + 2;                      // [EPI_WARPS][2]
  uint64_t* stats_bar = res_bar + 2 * Cfg::EPI_WARPS;      // [2 slots]
  uint64_t* xres_bar = stats_bar + 2;                      // [EPI_WARPS] third residual buffer (xbuf)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xres_bar + Cfg::EPI_WARPS);

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = static_cast<int>(threadIdx.x & 31);
  const uint32_t cta_rank = cluster_ctarank();             // 0..5
  const uint32_t pair = cta_rank >> 1;                     // column block n_blk
  const uint32_t half_m = cta_rank & 1u;                   // which 128 rows of the 256-row tile
  const uint32_t leader_rank = cta_rank & ~1u;
  const bool leader = half_m == 0;
  const int idle_tma = (a_multicast >> 4) & 3, idle_mma = (a_multicast >> 6) & 3, idle_epi = (a_multicast >> 8) & 3;   // mbar_wait_idle modes of the single-lane warps
  // epilogue variants (r02b phase trace: of a 21 k-cycle tile period at K=768, 7 k were exposed residual-load latency,
  // 5 k the fence + remote-arrive publish round, 6 k the staging buffers waiting for their TMA stores to drain):
  const bool direct_st = (a_multicast & 2) != 0;    // pass 2 writes x32 / x16 with 256-bit per-lane global stores: no staging, the
                                                    // residual buffers are free after pass 1 and the NEXT tile's first two chunks are requested then
  const bool async_stats = (a_multicast & 4) != 0;  // row statistics travel by st.async + complete_tx (no fence / arrive round)
  const bool l2_prefetch = (a_multicast & 8) != 0;  // residual chunks 2, 3 of the next tile are pulled into L2 one tile ahead
  // depth of the A/B ring actually used (<= Cfg::STAGES).  The TMA unit serves an SM's requests in order, so the epilogue's
  // residual boxes queue behind every main-loop stage in flight: a short-K problem (K = 768: 12 K-blocks per tile, the
  // kernel is epilogue / HBM bound) wants a SHALLOW ring, the K = 3072 one all four stages.
  const int nstages = ((a_multicast >> 12) & 7) ? ((a_multicast >> 12) & 7) : Cfg::STAGES;
  // residual boxes by per-lane cp.async (LDGSTS) instead of TMA: r02h showed that a residual box requested through the TMA
  // unit waits behind the four main-loop stages queued ahead of it (3.1 k + 4.1 k exposed cycles per tile at K = 768; 0.2 k
  // with a 2-deep ring, which starves the MMA instead) -- the LSU path has its own queue
  const bool res_ldgsts = ((a_multicast >> 15) & 1) != 0;
  // Third residual buffer per epilogue warp (r02o).  The exposed residual-box latency (~3 k cycles per pair of boxes, 8 k
  // of a 17.7 k-cycle tile period at K = 768) is the loaded memory-system latency of the boxes, and the two 4 KB buffers
  // per warp double as the TMA-store staging of pass 2, so the next tile's boxes can only be requested when this tile is
  // done.  A short-K problem does not need the fourth A/B stage (ring 3 measured equal), whose 32 KB become one extra 4 KB
  // buffer per warp that is NEVER used for staging: chunk 0 of the next tile is requested into it at the start of pass 2
  // (a whole pass ahead: it lands hidden), chunks 1 and 2 go to the old pair at the end of the tile, chunk 3 follows
  // chunk 0 into the extra buffer.  Three boxes instead of two are in flight when pass 1 begins.
  const bool xbuf = ((a_multicast >> 16) & 1) != 0 && nstages <= 3 && !direct_st && !res_ldgsts;
  a_multicast &= 1;

  if (warp_idx == 0 && lane == 0) {
    prefetch_tmap(&tmap_a); prefetch_tmap(&tmap_a64); prefetch_tmap(&tmap_b); prefetch_tmap(&tmap_res); prefetch_tmap(&tmap_x32); prefetch_tmap(&tmap_x16);
  }
  if (warp_idx == 1 && lane == 0) {
    // A multicast: a stage is rewritten by TMA loads issued in all three pairs, so it is free only when the MMAs of
    // all three pairs have retired (3 multicast commits); unicast: only this pair's.
    for (int i = 0; i < Cfg::STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], a_multicast ? Cfg::PAIRS : 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * Cfg::EPI_WARPS); }
    for (int i = 0; i < 2 * Cfg::EPI_WARPS; ++i) mbar_init(&res_bar[i], res_ldgsts ? 32 : 1);   // one arrival per lane / one expect_tx
    // classic exchange: 3 CTAs x 8 warps arrive; st.async exchange: one local expect_tx arrival + 6,144 bytes of complete_tx
    for (int i = 0; i < 2; ++i) mbar_init(&stats_bar[i], async_stats ? 1 : Cfg::PAIRS * Cfg::EPI_WARPS);
    for (int i = 0; i < Cfg::EPI_WARPS; ++i) mbar_init(&xres_bar[i], 1);
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_tiles = (M + Cfg::BM - 1) / Cfg::BM;       // 256-row blocks; every cluster covers all 768 columns
  const int num_kb = K / Cfg::BK;
  const int cluster_id = blockIdx.x / Cfg::CLUSTER;
  const int num_clusters = gridDim.x / Cfg::CLUSTER;
  const int row_b = static_cast<int>(pair) * Cfg::BN + static_cast<int>(half_m) * Cfg::BN_CTA;   // this CTA's W rows

  if (warp_idx == 0) {
    // ===================== TMA producer (all CTAs) =====================
    // warp-uniform loops, one elected lane issues (see gemm_tcgen05_2cta.cuh: avoids ptxas' per-instruction waterfall)
    {
      const bool issuer = elect_one();
      int stage = 0;
      uint32_t phase = 0;
      // Paced producer (MEMVUL_LN_PACE = cycles between stage requests; experiment, default off).  At K = 768 the kernel
      // is epilogue-bound (the MMA needs 6 k of a ~17.7 k-cycle tile period) and 8 k of those cycles are exposed residual
      // waits (~3 k per box pair, through TMA and LDGSTS alike).  Hypothesis: the free-running producer's 64 B/clk burst
      // for the next tile delays the residual boxes at the SM's L2 port.  Measured r02o (tools/gpu_ln_pace.sh): spreading
      // the stage requests over the tile period (600 ... 1,100 cycles apart) leaves the residual waits at 2.5-4.4 k cycles
      // and the kernel at 73.7-74.4 us; above 1,300 the MMA starves.  So the ~3 k cycles are the loaded memory-system
      // latency of the box itself (DRAM at ~50 % utilisation with mixed reads / writes), and what is missing is bytes in
      // flight for the residual (two 4 KB boxes per warp; shared memory is full), not request ordering.
      long long next_issue = pace > 0 ? clock64() : 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        const int row_a = tile * Cfg::BM + static_cast<int>(half_m) * Cfg::BM_CTA;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait_idle(&empty_bar[stage], phase ^ 1u, idle_tma);
          if (pace > 0) {
            long long now = clock64();
            while (now < next_issue) { __nanosleep(100); now = clock64(); }
            next_issue = (now - next_issue > 4 * pace ? now : next_issue) + pace;     // never bank more than 4 stages of credit
          }
          uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
          if (issuer) {
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
          if (a_multicast) {
            // The three pairs need the SAME 128 A rows per rank: pairs 0 and 1 each fetch 64 of them once and the TMA
            // multicasts the box into all three CTAs of that rank -> a third of the A traffic out of L2.
            if (pair < 2)
              tma_load_2d_pair_mc(sa + pair * (Cfg::A_BYTES / 2), &tmap_a64, &full_bar[stage], kb * Cfg::BK,
                                  row_a + static_cast<int>(pair) * 64,
                                  static_cast<uint16_t>((1u << half_m) | (1u << (2 + half_m)) | (1u << (4 + half_m))),
                                  kEvictNormal);
          } else {
            tma_load_2d_pair(sa, &tmap_a, &full_bar[stage], kb * Cfg::BK, row_a, kEvictNormal);
          }
          tma_load_2d_pair(sa + Cfg::A_BYTES, &tmap_b, &full_bar[stage], kb * Cfg::BK, row_b, kEvictLast);
          }
          if (++stage == nstages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================== MMA issuer (even rank of each pair) =====================
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_f16(Cfg::BM, Cfg::BN, false, false);
      const bool issuer = elect_one();
      const uint32_t smem_base = smem_u32(smem);
      const uint16_t pair_mask = static_cast<uint16_t>(0b11u << (pair * 2));
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        mbar_wait_idle(&tempty_bar[acc], acc_phase ^ 1u, idle_mma);
        tc_fence_after();
        if (issuer) stamp(static_cast<uint32_t>((tile - cluster_id) / num_clusters), 14);
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * Cfg::BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait_idle(&full_bar[stage], phase, idle_mma);
          tc_fence_after();
          const uint32_t sa = smem_base + static_cast<uint32_t>(stage * Cfg::STAGE_BYTES);
          const uint64_t a_desc = umma_desc_sw128(sa);
          const uint64_t b_desc = umma_desc_sw128(sa + Cfg::A_BYTES);
          if (issuer) {
#pragma unroll
            for (int k = 0; k < Cfg::BK / 16; ++k)
              umma_f16_ss_pair(d_tmem, a_desc + static_cast<uint64_t>(k * 2), b_desc + static_cast<uint64_t>(k * 2), idesc,
                               (kb | k) != 0 ? 1u : 0u);
            umma_commit_pair(&empty_bar[stage], a_multicast ? static_cast<uint16_t>(0b111111) : pair_mask);
          }
          if (++stage == nstages) { stage = 0; phase ^= 1u; }
        }
        if (issuer) umma_commit_pair(&tfull_bar[acc], pair_mask);
        if (issuer) stamp(static_cast<uint32_t>((tile - cluster_id) / num_clusters), 15);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else if (warp_idx >= 4) {
    // ===================== epilogue: bias + residual + LayerNorm =====================
    const int ew = warp_idx - 4;
    const int quarter = ew & 3;
    const int half_sel = ew >> 2;
    constexpr int NCHUNK = 4;                              // 4 x 32 columns per warp
    float* prm = reinterpret_cast<float*>(smem + Cfg::OFF_PRM) + ew * 3 * 128;
    uint8_t* buf0 = smem + Cfg::OFF_STG + ew * 2 * Cfg::STG_BYTES;       // residual ping / fp32 output staging
    uint8_t* buf1 = buf0 + Cfg::STG_BYTES;                               // residual pong / fp16 output staging
    uint64_t* my_res_bar = res_bar + 2 * ew;
    uint8_t* bufc = smem + 3 * Cfg::STAGE_BYTES + ew * Cfg::STG_BYTES;   // xbuf: this warp's slice of the unused fourth A/B stage
    uint64_t* my_xbar = xres_bar + ew;
    // chunk c of a tile -> residual buffer / its barrier.  Classic: ping-pong (c & 1).  xbuf: 0 -> C, 1 -> A, 2 -> B, 3 -> C.
    auto chunk_buf = [&](int c) -> uint8_t* {
      if (!xbuf) return (c & 1) ? buf1 : buf0;
      return (c == 0 || c == 3) ? bufc : (c == 1 ? buf0 : buf1);
    };
    auto chunk_bar = [&](int c) -> uint64_t* {
      if (!xbuf) return &my_res_bar[c & 1];
      return (c == 0 || c == 3) ? my_xbar : &my_res_bar[c - 1];
    };
    const uint32_t sw = static_cast<uint32_t>(lane & 7);
    const int col0 = static_cast<int>(pair) * Cfg::BN + half_sel * 128;  // first of this warp's 128 columns
    const int row_in_cta = quarter * 32 + lane;
    const uint32_t stats_base = smem_u32(smem + Cfg::OFF_STATS);
    const uint32_t my_src = pair * 2 + static_cast<uint32_t>(half_sel);  // 0..5: which (pair, column half) I publish
    // parameters of my 128 columns, once (the CTA's column block never changes)
    reinterpret_cast<float4*>(prm)[lane] = __ldg(reinterpret_cast<const float4*>(bias + col0) + lane);
    reinterpret_cast<float4*>(prm + 128)[lane] = __ldg(reinterpret_cast<const float4*>(gamma + col0) + lane);
    reinterpret_cast<float4*>(prm + 256)[lane] = __ldg(reinterpret_cast<const float4*>(beta + col0) + lane);
    __syncwarp();

    auto strip_row0 = [&](int tile) { return tile * Cfg::BM + static_cast<int>(half_m) * Cfg::BM_CTA + quarter * 32; };
    auto issue_res = [&](int tile, int c) {                 // residual box (rows of `tile`, chunk c) -> buffer c & 1
      uint8_t* dst = chunk_buf(c);
      if (res_ldgsts) {
        // whole warp: lane -> (row lane/8 + 4 i, 16-byte unit lane%8); four full 128 B lines per instruction, written to
        // the positions a SWIZZLE_128B TMA box would use
        const uint32_t d0 = smem_u32(dst);
        const int unit = lane & 7;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = (lane >> 3) + 4 * i;
          const int grow = min(strip_row0(tile) + r, M - 1);           // rows past M repeat the last row (never stored)
          cp_async_16B(d0 + r * 128 + ((unit ^ (r & 7)) << 4),
                       resid_ptr + static_cast<size_t>(grow) * Cfg::N + col0 + c * 32 + unit * 4);
        }
        cp_async_mbar_arrive(&my_res_bar[c & 1]);
      } else if (lane == 0) {
        mbar_arrive_expect_tx(chunk_bar(c), Cfg::STG_BYTES);
        tma_load_2d(dst, &tmap_res, chunk_bar(c), col0 + c * 32, strip_row0(tile), kEvictFirst);
      }
    };
    if (cluster_id < num_tiles) { issue_res(cluster_id, 0); issue_res(cluster_id, 1); if (xbuf) issue_res(cluster_id, 2); }

    int acc = 0;
    uint32_t acc_phase = 0, gc = 0, it = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++it) {
      const int row0 = strip_row0(tile);
      const bool tr = ew == 0 && lane == 0;
      if (tr) stamp(it, 0);
      mbar_wait_idle(&tfull_bar[acc], acc_phase, idle_epi);
      tc_fence_after();
      if (tr) stamp(it, 1);
      if (l2_prefetch && !direct_st && lane == 0 && tile + num_clusters < num_tiles) {
        // staged epilogue: the residual buffers double as the TMA-store staging of pass 2, so the next tile's residual
        // can only be requested at the very end of this tile -- pull it into L2 now, a whole tile ahead, so that those
        // requests (and the chunk 2 / 3 requests inside pass 1) find it there (r02b trace: 3.6 k + 3.7 k cycles of
        // exposed HBM latency per tile -> L2 latency)
#pragma unroll
        for (int c = 0; c < NCHUNK; ++c) tma_prefetch_l2_2d(&tmap_res, col0 + c * 32, strip_row0(tile + num_clusters));
      }
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                              static_cast<uint32_t>(acc * Cfg::BN + half_sel * 128);
      // ---------------- pass 1: v = acc + bias + resid -> TMEM, row statistics ----------------
      // shifted sums: d = v - piv with piv near the partial's mean, so s1 / s2 stay O(128 spread^2) whatever the row mean
      float s1 = 0.f, s2 = 0.f, piv = 0.f;
      uint32_t r[2][32];
      tmem_ld_32x32b_x32(t_addr, r[0]);
#pragma unroll
      for (int c = 0; c < NCHUNK; ++c) {
        tmem_wait_ld();
        if (c + 1 < NCHUNK) tmem_ld_32x32b_x32(t_addr + (c + 1) * 32, r[(c + 1) & 1]);
        const uint32_t(&a)[32] = r[c & 1];
        uint8_t* rowp = chunk_buf(c) + lane * 128;
        // n-th use of a barrier waits for parity n & 1.  Classic: each of the two barriers serves every other chunk.
        // xbuf: A / B serve one chunk per tile, C two (chunk 0: even use, chunk 3: odd use).
        const uint32_t res_parity = !xbuf ? ((gc >> 1) & 1u) : ((c == 0) ? 0u : (c == 3 ? 1u : (it & 1u)));
        mbar_wait_idle(chunk_bar(c), res_parity, idle_epi);
        ++gc;
        if (tr) stamp(it, 2 + c);
        uint32_t v[32];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const float4 x = *reinterpret_cast<const float4*>(rowp + ((static_cast<uint32_t>(u) ^ sw) << 4));
          const float4 bb = *reinterpret_cast<const float4*>(prm + c * 32 + 4 * u);
          const float v0 = __uint_as_float(a[4 * u + 0]) + bb.x + x.x;
          const float v1 = __uint_as_float(a[4 * u + 1]) + bb.y + x.y;
          const float v2 = __uint_as_float(a[4 * u + 2]) + bb.z + x.z;
          const float v3 = __uint_as_float(a[4 * u + 3]) + bb.w + x.w;
          v[4 * u + 0] = __float_as_uint(v0); v[4 * u + 1] = __float_as_uint(v1);
          v[4 * u + 2] = __float_as_uint(v2); v[4 * u + 3] = __float_as_uint(v3);
        }
        if (c == 0) {                                      // pivot = mean of the first 32 values: within O(spread / 6) of
          float q4[4] = {0.f, 0.f, 0.f, 0.f};              // the partial's mean, so s2 - s1^2 / 128 barely cancels
#pragma unroll
          for (int i = 0; i < 32; ++i) q4[i & 3] += __uint_as_float(v[i]);
          piv = ((q4[0] + q4[1]) + (q4[2] + q4[3])) * (1.0f / 32.0f);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {                      // separate sweep: folded into the loop above, ptxas spills
          const float d0 = __uint_as_float(v[4 * u + 0]) - piv, d1 = __uint_as_float(v[4 * u + 1]) - piv;
          const float d2 = __uint_as_float(v[4 * u + 2]) - piv, d3 = __uint_as_float(v[4 * u + 3]) - piv;
          s1 += (d0 + d1) + (d2 + d3);
          s2 = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, s2))));
        }
        tmem_st_32x32b_x32(t_addr + c * 32, v);            // stash for pass 2
        __syncwarp();                                      // every lane has read this residual buffer
        if (!xbuf) { if (c + 2 < NCHUNK) issue_res(tile, c + 2); }
        else if (c == 0) issue_res(tile, 3);                // chunk 3 follows chunk 0 into the extra buffer
      }
      // ---------------- exchange the row statistics with the two other column blocks ----------------
      if (tr) stamp(it, 6);
      const uint32_t slot = it & 1u;
      const int next_tile = tile + num_clusters;
      if (xbuf && next_tile < num_tiles) issue_res(next_tile, 0);   // extra buffer is free: a whole pass 2 ahead of its use
      if (direct_st && next_tile < num_tiles) {
        // both residual buffers are free (pass 2 does not stage): request the next tile's first two chunks now, a whole
        // exchange + pass 2 ahead of their use, and pull its last two chunks into L2
        issue_res(next_tile, 0);
        issue_res(next_tile, 1);
        if (l2_prefetch && lane == 0) {
          tma_prefetch_l2_2d(&tmap_res, col0 + 2 * 32, strip_row0(next_tile));
          tma_prefetch_l2_2d(&tmap_res, col0 + 3 * 32, strip_row0(next_tile));
        }
      }
      {
        // this partial's (mean, centred sum of squares) over its 128 columns
        constexpr float kInvPart = 1.0f / (NCHUNK * 32);
        const float mean_p = fmaf(s1, kInvPart, piv);
        const float m2_p = fmaxf(fmaf(-s1, s1 * kInvPart, s2), 0.f);
        const uint32_t off = ((slot * 6u + my_src) * 128u + static_cast<uint32_t>(row_in_cta)) * 8u;
        if (async_stats) {
          if (ew == 0 && lane == 0) mbar_arrive_expect_tx(&stats_bar[slot], 6u * 128u * 8u);   // what this CTA will receive
          const uint32_t bar_local = smem_u32(&stats_bar[slot]);
#pragma unroll
          for (uint32_t pp = 0; pp < 3; ++pp)
            st_async_f32x2(mapa_u32(stats_base + off, pp * 2 + half_m), mean_p, m2_p, mapa_u32(bar_local, pp * 2 + half_m));
        } else {
#pragma unroll
          for (uint32_t pp = 0; pp < 3; ++pp) st_cluster_f32x2(mapa_u32(stats_base + off, pp * 2 + half_m), mean_p, m2_p);
          fence_acq_rel_cluster();
          __syncwarp();
          if (lane == 0) {
#pragma unroll
            for (uint32_t pp = 0; pp < 3; ++pp) mbar_arrive_release_cluster(&stats_bar[slot], pp * 2 + half_m);
          }
        }
      }
      tmem_wait_st();
      if (tr) stamp(it, 7);
      if (async_stats) mbar_wait(&stats_bar[slot], (it >> 1) & 1u);
      else mbar_wait_cluster(&stats_bar[slot], (it >> 1) & 1u);
      if (tr) stamp(it, 8);
      float mean, var;
      {
        // Chan et al.: mean = sum mean_p / 6, M2 = sum M2_p + 128 sum (mean_p - mean)^2.  The partial means are taken
        // relative to partial 0 (differences of nearby values: exact), so the row mean is never rounded at 6 |mean|.
        const float2* st = reinterpret_cast<const float2*>(smem + Cfg::OFF_STATS) + (slot * 6) * 128 + row_in_cta;
        const float m0 = st[0].x;
        float dsum = 0.f, m2 = 0.f;
#pragma unroll
        for (int src = 0; src < 6; ++src) { const float2 p2 = st[src * 128]; dsum += p2.x - m0; m2 += p2.y; }
        const float dm = dsum * (1.0f / 6.0f);
        float between = 0.f;
#pragma unroll
        for (int src = 0; src < 6; ++src) { const float e = (st[src * 128].x - m0) - dm; between = fmaf(e, e, between); }
        mean = m0 + dm;
        var = fmaf(static_cast<float>(NCHUNK * 32), between, m2) * (1.0f / Cfg::N);
      }
      const float rstd = 1.0f / sqrtf(var + eps);
      // ---------------- pass 2: normalise, stage, TMA-store fp32 + fp16 ----------------
      tmem_ld_32x32b_x32(t_addr, r[0]);
#pragma unroll
      for (int c = 0; c < NCHUNK; ++c) {
        tmem_wait_ld();
        if (c + 1 < NCHUNK) tmem_ld_32x32b_x32(t_addr + (c + 1) * 32, r[(c + 1) & 1]);
        const uint32_t(&a)[32] = r[c & 1];
        if (direct_st) {
          // registers -> global: every lane owns one output row; 128 B of fp32 (4 x 256-bit stores) and 64 B of fp16 (2)
          const int grow = row0 + lane;
          uint32_t o32[32], o16[16];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float4 g = *reinterpret_cast<const float4*>(prm + 128 + c * 32 + 4 * u);
            const float4 be = *reinterpret_cast<const float4*>(prm + 256 + c * 32 + 4 * u);
            const float ox = (__uint_as_float(a[4 * u + 0]) - mean) * rstd * g.x + be.x;
            const float oy = (__uint_as_float(a[4 * u + 1]) - mean) * rstd * g.y + be.y;
            const float oz = (__uint_as_float(a[4 * u + 2]) - mean) * rstd * g.z + be.z;
            const float ow = (__uint_as_float(a[4 * u + 3]) - mean) * rstd * g.w + be.w;
            o32[4 * u + 0] = __float_as_uint(ox); o32[4 * u + 1] = __float_as_uint(oy);
            o32[4 * u + 2] = __float_as_uint(oz); o32[4 * u + 3] = __float_as_uint(ow);
            o16[2 * u + 0] = pack_half2(ox, oy);
            o16[2 * u + 1] = pack_half2(oz, ow);
          }
          if (grow < M) {
            float* p32 = x32_ptr + static_cast<size_t>(grow) * Cfg::N + col0 + c * 32;
            __half* p16 = x16_ptr + static_cast<size_t>(grow) * Cfg::N + col0 + c * 32;
#pragma unroll
            for (int q = 0; q < 4; ++q) st_global_v8(p32 + 8 * q, *reinterpret_cast<const uint32_t(*)[8]>(&o32[8 * q]));
#pragma unroll
            for (int q = 0; q < 2; ++q) st_global_v8(p16 + 16 * q, *reinterpret_cast<const uint32_t(*)[8]>(&o16[8 * q]));
          }
          if (tr) stamp(it, 9 + c);
          continue;
        }
        if (lane == 0 && c > 0) bulk_wait_read_all();      // previous boxes have left buf0 (and buf1 when c is even)
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const float4 g = *reinterpret_cast<const float4*>(prm + 128 + c * 32 + 4 * u);
          const float4 be = *reinterpret_cast<const float4*>(prm + 256 + c * 32 + 4 * u);
          float4 o;
          o.x = (__uint_as_float(a[4 * u + 0]) - mean) * rstd * g.x + be.x;
          o.y = (__uint_as_float(a[4 * u + 1]) - mean) * rstd * g.y + be.y;
          o.z = (__uint_as_float(a[4 * u + 2]) - mean) * rstd * g.z + be.z;
          o.w = (__uint_as_float(a[4 * u + 3]) - mean) * rstd * g.w + be.w;
          *reinterpret_cast<float4*>(buf0 + lane * 128 + ((static_cast<uint32_t>(u) ^ sw) << 4)) = o;
          // fp16 copy: 4 values = 8 B; two of them fill one 16 B unit of the 32 x 64 box (chunk parity = 64 B half)
          const uint32_t h_unit = static_cast<uint32_t>((c & 1) * 4 + (u >> 1));
          uint2 hv;
          hv.x = pack_half2(o.x, o.y);
          hv.y = pack_half2(o.z, o.w);
          *reinterpret_cast<uint2*>(buf1 + lane * 128 + ((h_unit ^ sw) << 4) + (u & 1) * 8) = hv;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmap_x32, buf0, col0 + c * 32, row0);
          if (c & 1) tma_store_2d(&tmap_x16, buf1, col0 + (c >> 1) * 64, row0);
          bulk_commit_group();
        }
        if (tr) stamp(it, 9 + c);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_cluster(&tempty_bar[acc], leader_rank);          // accumulator stage is free again
        if (!direct_st) bulk_wait_read_all();                        // staging buffers are free again
      }
      if (!direct_st) {
        __syncwarp();
        if (next_tile < num_tiles) {
          if (xbuf) { issue_res(next_tile, 1); issue_res(next_tile, 2); }
          else { issue_res(next_tile, 0); issue_res(next_tile, 1); }
        }
      }
      if (tr) stamp(it, 13);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
  }

  // ===================== teardown =====================
  tc_fence_before();
  cluster_sync_all();
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace mv
