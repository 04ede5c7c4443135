// tcgen05 / TMEM / TMA GEMM for sm_100a: C[m,n] = sum_k A[m,k] * W[n,k] (+bias, +residual), or the
// fused row log-sum-exp + column-pick epilogue.  Both operands K-major (nn.Linear layout).
//
// Replaces the cuBLAS calls behind nn.Linear / einsum / `x @ A` on the reference hot path
// (fairseq/models/hgt.py:320-322,347-348,401; knn/pq_wrapper.py:202;
// fairseq/modules/adaptive_softmax.py:184,197,202).
//
// Structure (persistent, warp-specialised, one CTA per SM, clusters of 2 CTAs that share the W tile through
// TMA multicast, static round-robin schedule over tile pairs):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D loads of a 128 x 128B A tile and a 256 x 128B W
//               tile (SWIZZLE_128B) per k-block into a multi-stage smem ring, mbarrier expect_tx.
//   warp 1      MMA issuer: one thread issues tcgen05.mma.cta_group::1 (M=128, N=256, K=8 tf32 / 16 bf16)
//               with smem descriptors; accumulators live in TMEM (2 x 256 columns, double buffered so the
//               epilogue of tile i overlaps the MMAs of tile i+1); tcgen05.commit frees smem stages and
//               publishes accumulators.
//   warp 2      TMEM allocator (512 columns).
//   warps 4-7   epilogue: tcgen05.ld 32x32b.x32 -> registers -> bias / residual -> global, or the
//               online (max, sum-exp, pick) reduction -- a thread owns one output row, so the LSE needs
//               no cross-thread traffic.
//   warps 8-11  (3xTF32 only) operand splitter: rewrites the fp32 A tile in smem as hi = A & ~0x1fff
//               (what kind::tf32 consumes) and writes lo = A - hi to a second tile; W is pre-split on
//               the host side once per checkpoint.  D += A_hi*W_lo + A_lo*W_hi + A_hi*W_hi recovers
//               ~2^-21 relative accuracy from three tf32 passes ("fp32 mode" of the north star).
#include "gemm_tc_common.cuh"

namespace gnnlm {

namespace tc {


template <int MODE, bool LSE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MODE == X3 ? 384 : 256, 1)
    gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                   const __grid_constant__ CUtensorMap map_blo, int64_t M_cap, const int32_t* __restrict__ m_dev, int64_t N,
                   int64_t K, EpiStore es, EpiLse el) {
  constexpr int ELEM = MODE == BF16 ? 2 : 4;
  constexpr int BLOCK_K = ROW_BYTES / ELEM;                 // 32 tf32 / 64 bf16
  constexpr int UMMA_K = 32 / ELEM;                         // 8 tf32 / 16 bf16
  constexpr int STAGE_BYTES = MODE == X3 ? 2 * (A_TILE + B_TILE) : (A_TILE + B_TILE);
  constexpr int STAGES = MODE == X3 ? 2 : 4;
  constexpr uint32_t TX_BYTES = MODE == X3 ? A_TILE + 2 * B_TILE : A_TILE + B_TILE;
  // instruction descriptor (cute InstrDescriptor): c=F32 [4,6) | a,b format [7,10),[10,13) | N>>3 [17,23) | M>>4 [24,29)
  constexpr uint32_t FMT = MODE == BF16 ? 1u : 2u;
  constexpr uint32_t IDESC = (1u << 4) | (FMT << 7) | (FMT << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) |
                             ((uint32_t)(BLOCK_M >> 4) << 24);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* epi_smem = reinterpret_cast<float*>(smem + (size_t)STAGES * STAGE_BYTES);
  __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], conv_bar[STAGES], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t M = live_rows(M_cap, m_dev);
  // A CTA pair (cluster of 2 along M) works on two vertically adjacent output tiles that share the W tile:
  // each CTA fetches half of it and multicasts to both, halving the L2 -> smem traffic of W.
  const uint32_t crank = cluster_ctarank();
  const int64_t n_m = (M + BLOCK_M - 1) / BLOCK_M, n_n = (N + BLOCK_N - 1) / BLOCK_N;
  const int64_t total = ((n_m + 1) / 2) * n_n;               // pair tiles; identical in both CTAs
  const int64_t pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;
  const int n_kb = (int)((K + BLOCK_K - 1) / BLOCK_K);

  auto sA = [&](int s) { return smem + (size_t)s * STAGE_BYTES; };
  auto sB = [&](int s) { return smem + (size_t)s * STAGE_BYTES + A_TILE; };
  auto sAlo = [&](int s) { return smem + (size_t)s * STAGE_BYTES + A_TILE + B_TILE; };
  auto sBlo = [&](int s) { return smem + (size_t)s * STAGE_BYTES + 2 * A_TILE + B_TILE; };

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    if (MODE == X3) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_blo) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 2);                         // released by the MMA warps of both CTAs
      mbar_init(&conv_bar[s], 4);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                        // peer barriers initialised before any multicast
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int half = (int)crank * (BLOCK_N / 2);             // my half of the shared W tile (rows)
      for (int64_t tile = pair0; tile < total; tile += pair_stride) {
        const int m0 = (int)(((tile / n_n) * 2 + crank) * BLOCK_M), n0 = (int)((tile % n_n) * BLOCK_N);
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);           // both CTAs have drained this stage
          mbar_expect_tx(&full_bar[stage], TX_BYTES);
          tma_load_2d(sA(stage), &map_a, kb * BLOCK_K, m0, &full_bar[stage]);
          tma_load_2d_mc(sB(stage) + half * ROW_BYTES, &map_b, kb * BLOCK_K, n0 + half, &full_bar[stage], 3);
          if (MODE == X3)
            tma_load_2d_mc(sBlo(stage) + half * ROW_BYTES, &map_blo, kb * BLOCK_K, n0 + half, &full_bar[stage], 3);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int64_t it = 0;
      for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * BLOCK_N;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(MODE == X3 ? &conv_bar[stage] : &full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = make_desc(smem_u32(sA(stage))), db = make_desc(smem_u32(sB(stage)));
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t koff = (uint64_t)((k * UMMA_K * ELEM) >> 4);     // advance inside the 128 B swizzle row
            if (MODE == X3) {
              const uint64_t dal = make_desc(smem_u32(sAlo(stage))), dbl = make_desc(smem_u32(sBlo(stage)));
              umma<1>(d_tmem, da + koff, dbl + koff, IDESC, (kb | k) > 0 ? 1u : 0u);
              umma<1>(d_tmem, dal + koff, db + koff, IDESC, 1u);
              umma<1>(d_tmem, da + koff, db + koff, IDESC, 1u);
            } else {
              umma<MODE != BF16>(d_tmem, da + koff, db + koff, IDESC, (kb | k) > 0 ? 1u : 0u);
            }
          }
          tc_commit_mc(&empty_bar[stage], 3);        // stage reusable (in BOTH CTAs) once these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit(&tmem_full[acc]);                  // accumulator complete
      }
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;                          // TMEM lane quarter this warp may access
    int64_t it = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
      const int acc = (int)(it & 1);
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      const int64_t m_blk = (tile / n_n) * 2 + crank, n_blk = tile % n_n;
      const int64_t m = m_blk * BLOCK_M + q * 32 + lane;
      const int64_t n_base = n_blk * BLOCK_N;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * BLOCK_N + ((uint32_t)(q * 32) << 16);
      epilogue_tile<LSE>(taddr, m, M, n_base, n_blk, N, es, el, epi_smem + (warp & 3) * 32 * EPI_LD);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  } else if (MODE == X3 && warp >= CONV_WARP0) {
    // ===================== operand splitter (3xTF32) =====================
    const int ct = threadIdx.x - CONV_WARP0 * 32;     // 0..127
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride) {
      for (int kb = 0; kb < n_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        float4* a = reinterpret_cast<float4*>(sA(stage));
        float4* lo = reinterpret_cast<float4*>(sAlo(stage));
#pragma unroll
        for (int i = 0; i < A_TILE / 16 / 128; ++i) {
          const int idx = ct + i * 128;
          float4 x = a[idx], h;
          h.x = __uint_as_float(__float_as_uint(x.x) & 0xffffe000u);
          h.y = __uint_as_float(__float_as_uint(x.y) & 0xffffe000u);
          h.z = __uint_as_float(__float_as_uint(x.z) & 0xffffe000u);
          h.w = __uint_as_float(__float_as_uint(x.w) & 0xffffe000u);
          a[idx] = h;
          lo[idx] = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to UMMA
        __syncwarp();
        if (lane == 0) mbar_arrive(&conv_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                        // the peer may still multicast into / arrive on this CTA
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// Single-pass (bf16 / tf32) store GEMMs are paced by the epilogue, not by the MMAs (5 us of main loop per tile against
// ~8 us of TMEM drain + stores with one warp per TMEM lane quarter): they run EIGHT epilogue warps, two per lane quarter,
// each draining half of the tile's columns, and give up one pipeline stage for the extra staging tiles.
template <int MODE, bool LSE>
__host__ __device__ constexpr bool tc2_epi8() { return MODE != X3 && !LSE; }

template <int MODE, bool LSE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__((MODE == X3 || tc2_epi8<MODE, LSE>()) ? 384 : 256, 1)
    gemm_tc2_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_blo, int64_t M_cap, const int32_t* __restrict__ m_dev, int64_t N,
                    int64_t K, EpiStore es, EpiLse el) {
  constexpr int ELEM = MODE == BF16 ? 2 : 4;
  constexpr int BLOCK_K = ROW_BYTES / ELEM;
  constexpr int UMMA_K = 32 / ELEM;
  constexpr int HALF_B = B_TILE / 2;                                   // this CTA's 128 W rows: 16 KB
  constexpr int STAGE_BYTES = MODE == X3 ? 2 * (A_TILE + HALF_B) : (A_TILE + HALF_B);
  constexpr bool EPI8 = tc2_epi8<MODE, LSE>();
  constexpr int EPI_WARPS = EPI8 ? 8 : 4;
  constexpr int STAGES = MODE == X3 ? 3 : (EPI8 ? 5 : 6);
  // bytes that land on the LEADER's w_full barrier per stage (both CTAs): W halves, plus A tiles when nobody
  // has to post-process A locally
  constexpr uint32_t W_TX = MODE == X3 ? 2u * 2u * HALF_B : 2u * (A_TILE + HALF_B);
  constexpr uint32_t FMT = MODE == BF16 ? 1u : 2u;
  constexpr uint32_t IDESC = (1u << 4) | (FMT << 7) | (FMT << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) |
                             ((uint32_t)((2 * BLOCK_M) >> 4) << 24);     // M = 256 across the pair

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* epi_smem = reinterpret_cast<float*>(smem + (size_t)STAGES * STAGE_BYTES);
  __shared__ __align__(8) uint64_t a_full[STAGES], w_full[STAGES], empty_bar[STAGES], conv_bar[STAGES], tmem_full[2],
      tmem_empty[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int64_t M = live_rows(M_cap, m_dev);
  const int64_t n_m = (M + BLOCK_M - 1) / BLOCK_M, n_n = (N + BLOCK_N - 1) / BLOCK_N;
  const int64_t total = ((n_m + 1) / 2) * n_n;
  const int64_t pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;
  const int n_kb = (int)((K + BLOCK_K - 1) / BLOCK_K);

  auto sA = [&](int s) { return smem + (size_t)s * STAGE_BYTES; };
  auto sB = [&](int s) { return smem + (size_t)s * STAGE_BYTES + A_TILE; };
  auto sAlo = [&](int s) { return smem + (size_t)s * STAGE_BYTES + A_TILE + HALF_B; };
  auto sBlo = [&](int s) { return smem + (size_t)s * STAGE_BYTES + 2 * A_TILE + HALF_B; };

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    if (MODE == X3) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_blo) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&a_full[s], 1);          // own A tile landed (3xTF32: the local splitter waits on it)
      mbar_init(&w_full[s], 1);          // leader: operands of BOTH CTAs landed
      mbar_init(&empty_bar[s], 1);       // one multicast commit per CTA
      mbar_init(&conv_bar[s], 8);        // leader: 4 splitter warps x 2 CTAs
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 2 * EPI_WARPS);      // leader: every epilogue warp of both CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int half = (int)crank * (BLOCK_N / 2);
      for (int64_t tile = pair0; tile < total; tile += pair_stride) {
        const int m0 = (int)(((tile / n_n) * 2 + crank) * BLOCK_M), n0 = (int)((tile % n_n) * BLOCK_N) + half;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_expect_tx(&w_full[stage], W_TX);
          if (MODE == X3) {
            mbar_expect_tx(&a_full[stage], A_TILE);
            tma_load_2d(sA(stage), &map_a, kb * BLOCK_K, m0, &a_full[stage]);
            tma_load_2d_2sm(sBlo(stage), &map_blo, kb * BLOCK_K, n0, &w_full[stage]);
          } else {
            tma_load_2d_2sm(sA(stage), &map_a, kb * BLOCK_K, m0, &w_full[stage]);
          }
          tma_load_2d_2sm(sB(stage), &map_b, kb * BLOCK_K, n0, &w_full[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int64_t it = 0;
      for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * BLOCK_N;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&w_full[stage], phase);
          if (MODE == X3) mbar_wait(&conv_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = make_desc(smem_u32(sA(stage))), db = make_desc(smem_u32(sB(stage)));
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t koff = (uint64_t)((k * UMMA_K * ELEM) >> 4);
            if (MODE == X3) {
              const uint64_t dal = make_desc(smem_u32(sAlo(stage))), dbl = make_desc(smem_u32(sBlo(stage)));
              umma_2sm<1>(d_tmem, da + koff, dbl + koff, IDESC, (kb | k) > 0 ? 1u : 0u);
              umma_2sm<1>(d_tmem, dal + koff, db + koff, IDESC, 1u);
              umma_2sm<1>(d_tmem, da + koff, db + koff, IDESC, 1u);
            } else {
              umma_2sm<MODE != BF16>(d_tmem, da + koff, db + koff, IDESC, (kb | k) > 0 ? 1u : 0u);
            }
          }
          tc_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit_2sm(&tmem_full[acc]);
      }
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + EPI_WARPS) {
    // ===================== epilogue (both CTAs, own 128 rows) =====================
    const int q = warp & 3;                                   // TMEM lane quarter
    const int ew = warp - EPI_WARP0;
    constexpr int COLS = EPI8 ? BLOCK_N / 2 : BLOCK_N;        // columns per epilogue warp
    const int c0 = (ew >> 2) * COLS;
    int64_t it = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
      const int acc = (int)(it & 1);
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      const int64_t m_blk = (tile / n_n) * 2 + crank, n_blk = tile % n_n;
      const int64_t m = m_blk * BLOCK_M + q * 32 + lane;
      const int64_t n_base = n_blk * BLOCK_N;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * BLOCK_N + (uint32_t)c0 + ((uint32_t)(q * 32) << 16);
      epilogue_tile<LSE>(taddr, m, M, n_base + c0, n_blk, N, es, el, epi_smem + ew * 32 * EPI_LD, 1.f, COLS);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
    }
  } else if (MODE == X3 && warp >= CONV_WARP0) {
    // ===================== operand splitter (both CTAs, own A tile) =====================
    const int ct = threadIdx.x - CONV_WARP0 * 32;
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride) {
      for (int kb = 0; kb < n_kb; ++kb) {
        mbar_wait(&a_full[stage], phase);
        float4* a = reinterpret_cast<float4*>(sA(stage));
        float4* lo = reinterpret_cast<float4*>(sAlo(stage));
#pragma unroll
        for (int i = 0; i < A_TILE / 16 / 128; ++i) {
          const int idx = ct + i * 128;
          float4 x = a[idx], h;
          h.x = __uint_as_float(__float_as_uint(x.x) & 0xffffe000u);
          h.y = __uint_as_float(__float_as_uint(x.y) & 0xffffe000u);
          h.z = __uint_as_float(__float_as_uint(x.z) & 0xffffe000u);
          h.w = __uint_as_float(__float_as_uint(x.w) & 0xffffe000u);
          a[idx] = h;
          lo[idx] = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&conv_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- 3xFP16 variant
// fp32-parity arithmetic at twice the tensor rate of 3xTF32: every fp32 operand is split into two fp16 numbers,
//   a = a_h + a_l,  a_h = fp16(a), a_l = fp16(a - a_h)            (22 significant bits, as hi/lo tf32)
//   w*S = w_h + w_l (S a power of two chosen per weight matrix so that max|w*S| = 2^13: keeps w_l normal)
// and D = a_h*w_h + a_h*w_l + a_l*w_h is accumulated in fp32 in TMEM by kind::f16 MMAs (K = 16 per
// instruction instead of 8, operand tiles half the bytes); the epilogue multiplies by 1/S (exact).
// Same cta_group::2 structure as gemm_tc2_kernel.  A arrives as fp32 (TMA, SWIZZLE_128B); the splitter warps
// rewrite it as two fp16 tiles in the SWIZZLE_64B K-major layout the MMA descriptors expect; W_h / W_l are
// pre-split fp16 matrices loaded by TMA with SWIZZLE_64B.  Operands beyond +-65504 are clamped (fp16 range).
constexpr int F16_BLOCK_K = 32;                           // k elements per stage
constexpr int F16_RAW_A = BLOCK_M * 128;                  // 16 KB fp32 tile (128 B rows)
constexpr int F16_OP_A = BLOCK_M * 64;                    // 8 KB fp16 tile (64 B rows)
constexpr int F16_OP_B = (BLOCK_N / 2) * 64;              // 8 KB: this CTA's 128 W rows
constexpr int F16_STAGE = F16_RAW_A + 2 * F16_OP_A + 2 * F16_OP_B;   // 48 KB
constexpr int F16_STAGES = 4;
constexpr int F16_CONV_WARPS = 8;                         // operand-splitter warps (conversion-throughput bound)
constexpr int F16_THREADS = (CONV_WARP0 + F16_CONV_WARPS) * 32;


template <bool LSE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F16_THREADS, 1)
    gemm_f16x3_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                      const __grid_constant__ CUtensorMap map_blo, int64_t M_cap, const int32_t* __restrict__ m_dev, int64_t N,
                      int64_t K, EpiStore es, EpiLse el, float acc_scale, int dbg) {
  constexpr int STAGES = F16_STAGES;
  constexpr uint32_t W_TX = 2u * 2u * F16_OP_B;                         // both CTAs' W_h + W_l halves -> leader
  // c = F32 | a,b = F16 (0) | N >> 3 | M >> 4 with M = 256 across the pair
  constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)((2 * BLOCK_M) >> 4) << 24);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* epi_smem = reinterpret_cast<float*>(smem + (size_t)STAGES * F16_STAGE);
  __shared__ __align__(8) uint64_t a_full[STAGES], w_full[STAGES], empty_bar[STAGES], conv_bar[STAGES], tmem_full[2],
      tmem_empty[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int64_t M = live_rows(M_cap, m_dev);
  const int64_t n_m = (M + BLOCK_M - 1) / BLOCK_M, n_n = (N + BLOCK_N - 1) / BLOCK_N;
  const int64_t total = ((n_m + 1) / 2) * n_n;
  const int64_t pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;
  const int n_kb = (int)((K + F16_BLOCK_K - 1) / F16_BLOCK_K);

  auto sRaw = [&](int s) { return smem + (size_t)s * F16_STAGE; };
  auto sAh = [&](int s) { return smem + (size_t)s * F16_STAGE + F16_RAW_A; };
  auto sAl = [&](int s) { return smem + (size_t)s * F16_STAGE + F16_RAW_A + F16_OP_A; };
  auto sBh = [&](int s) { return smem + (size_t)s * F16_STAGE + F16_RAW_A + 2 * F16_OP_A; };
  auto sBl = [&](int s) { return smem + (size_t)s * F16_STAGE + F16_RAW_A + 2 * F16_OP_A + F16_OP_B; };

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_blo) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&w_full[s], 1);
      mbar_init(&empty_bar[s], 1);
      mbar_init(&conv_bar[s], 2 * F16_CONV_WARPS);   // splitter warps of both CTAs
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {                                   // ---- TMA producer (both CTAs)
      int stage = 0;
      uint32_t phase = 0;
      const int half = (int)crank * (BLOCK_N / 2);
      for (int64_t tile = pair0; tile < total; tile += pair_stride) {
        const int m0 = (int)(((tile / n_n) * 2 + crank) * BLOCK_M), n0 = (int)((tile % n_n) * BLOCK_N) + half;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_expect_tx(&w_full[stage], (dbg & 2) ? 0u : W_TX);
          mbar_expect_tx(&a_full[stage], F16_RAW_A);
          tma_load_2d(sRaw(stage), &map_a, kb * F16_BLOCK_K, m0, &a_full[stage]);
          if (!(dbg & 2)) {
            tma_load_2d_2sm(sBh(stage), &map_b, kb * F16_BLOCK_K, n0, &w_full[stage]);
            tma_load_2d_2sm(sBl(stage), &map_blo, kb * F16_BLOCK_K, n0, &w_full[stage]);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {                         // ---- MMA issuer (leader only)
      int stage = 0;
      uint32_t phase = 0;
      int64_t it = 0;
      for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * BLOCK_N;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&w_full[stage], phase);
          mbar_wait(&conv_bar[stage], phase);
          tc_fence_after();
          const uint64_t dah = make_desc_sw64(smem_u32(sAh(stage))), dal = make_desc_sw64(smem_u32(sAl(stage)));
          const uint64_t dbh = make_desc_sw64(smem_u32(sBh(stage))), dbl = make_desc_sw64(smem_u32(sBl(stage)));
#pragma unroll
          for (int k = 0; k < ((dbg & 4) ? 0 : F16_BLOCK_K / 16); ++k) {
            const uint64_t koff = (uint64_t)(k * 2);                     // 16 fp16 = 32 B inside the 64 B row
            if (!(dbg & 8)) {
              umma_2sm<0>(d_tmem, dah + koff, dbl + koff, IDESC, (kb | k) > 0 ? 1u : 0u);
              umma_2sm<0>(d_tmem, dal + koff, dbh + koff, IDESC, 1u);
            }
            umma_2sm<0>(d_tmem, dah + koff, dbh + koff, IDESC, ((kb | k) > 0 || !(dbg & 8)) ? 1u : 0u);
          }
          tc_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit_2sm(&tmem_full[acc]);
      }
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + 4) {
    const int q = warp & 3;                            // ---- epilogue (both CTAs)
    int64_t it = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
      const int acc = (int)(it & 1);
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      const int64_t m_blk = (tile / n_n) * 2 + crank, n_blk = tile % n_n;
      const int64_t m = m_blk * BLOCK_M + q * 32 + lane;
      const int64_t n_base = n_blk * BLOCK_N;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * BLOCK_N + ((uint32_t)(q * 32) << 16);
      epilogue_tile<LSE>(taddr, m, M, n_base, n_blk, N, es, el, epi_smem + (warp & 3) * 32 * EPI_LD, acc_scale);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
    }
  } else if (warp >= CONV_WARP0) {
    // ---- operand splitter: fp32 [128 x 32] (SWIZZLE_128B) -> fp16 hi / lo [128 x 32] (SWIZZLE_64B)
    const int ct = threadIdx.x - CONV_WARP0 * 32;      // 0..32*F16_CONV_WARPS-1
    const int qd = ct & 3;                             // which 8 k-elements of the row
    constexpr int ROWS_PER_PASS = F16_CONV_WARPS * 8;  // 4 threads per row
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride) {
      for (int kb = 0; kb < n_kb; ++kb) {
        mbar_wait(&a_full[stage], phase);
        if (dbg & 1) goto conv_done;
        {
        const uint8_t* raw = sRaw(stage);
        uint8_t* oh = sAh(stage);
        uint8_t* ol = sAl(stage);
#pragma unroll
        for (int i = 0; i < BLOCK_M / ROWS_PER_PASS; ++i) {
          const int r = (ct >> 2) + ROWS_PER_PASS * i;
          const float4 x0 = *reinterpret_cast<const float4*>(raw + r * 128 + (((2 * qd) ^ (r & 7)) << 4));
          const float4 x1 = *reinterpret_cast<const float4*>(raw + r * 128 + (((2 * qd + 1) ^ (r & 7)) << 4));
          float xs[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
          float hs[8], ls[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float c = fminf(fmaxf(xs[e], -65504.f), 65504.f);
            hs[e] = __half2float(__float2half_rn(c));
            ls[e] = c - hs[e];
          }
          uint4 ph, pl;
          ph.x = pack_h2(hs[0], hs[1]); ph.y = pack_h2(hs[2], hs[3]); ph.z = pack_h2(hs[4], hs[5]); ph.w = pack_h2(hs[6], hs[7]);
          pl.x = pack_h2(ls[0], ls[1]); pl.y = pack_h2(ls[2], ls[3]); pl.z = pack_h2(ls[4], ls[5]); pl.w = pack_h2(ls[6], ls[7]);
          const int off = r * 64 + ((qd ^ ((r >> 1) & 3)) << 4);
          if (!(dbg & 16)) {
            *reinterpret_cast<uint4*>(oh + off) = ph;
            *reinterpret_cast<uint4*>(ol + off) = pl;
          } else if (ph.x == 0x12345678u && pl.y == 0x9abcdef0u) {
            *reinterpret_cast<uint4*>(oh + off) = ph;      // keeps the conversions alive in the timing experiment
          }
        }
        }
      conv_done:
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&conv_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- 3xFP16, pre-split A
// Same arithmetic as gemm_f16x3_kernel, but A arrives already in the split-fp16 activation format (GNNLM_F16X2:
// hi | lo halves of one fp16 buffer, written by the producing kernel's epilogue), so the four operand tiles
// A_h, A_l, W_h, W_l come straight from TMA (SWIZZLE_64B) and there are no splitter warps: a stage is 32 KB
// (6 stages in flight instead of 4) and the TMA -> MMA hand-off has no generic-proxy hop.
constexpr int F16S_STAGE = 2 * F16_OP_A + 2 * F16_OP_B;   // 32 KB
constexpr int F16S_STAGES = 6;

__host__ __device__ inline int64_t f16s_causal_tiles(int64_t n_p, int64_t n_n) {     // sum_{r < n_p} min(r + 1, n_n)
  const int64_t full = n_p < n_n ? n_p : n_n;
  return full * (full + 1) / 2 + (n_p - full) * n_n;
}

// The log-sum-exp epilogue (one FFMA + one MUFU.EX2 per logit, online max) paces the K = 64 tail-cluster GEMMs (ncu: a single
// epilogue warp per scheduler, 31 % issue-slot use, every other warp parked at the final barrier), so the LSE instantiation runs
// EIGHT epilogue warps -- two per TMEM lane quarter, each reducing half of the tile's columns -- and 384 threads.
// TOPK: the kNN filter epilogue (epilogue_topk) instead of a store; its MMAs are always N = 256 wide, so that a score does not
// depend on how many queries share the launch.
template <bool LSE, bool TOPK = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(LSE ? 384 : 256, 1)
    gemm_f16s_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                     const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_blo, int64_t M_cap,
                     const int32_t* __restrict__ m_dev, int64_t N, int64_t K, EpiStore es, EpiLse el, float acc_scale, int nb,
                     int64_t c_bs, int64_t r_bs, int causal, EpiTopk et) {
  constexpr int STAGES = F16S_STAGES;
  constexpr uint32_t TX = 2u * F16S_STAGE;                                // both CTAs' four operand tiles -> leader
  // N of the instruction: outputs of at most 128 columns (the P V' GEMM of the causal attention, N = d_k = 128; the narrow tail
  // projections) run N = 128 MMAs -- half the tensor work of a padded 256-column tile.  Each CTA of the pair then supplies
  // N / 2 = 64 rows of W: its TMA box starts at row crank * 64 and only the first 64 rows of its tile are read.
  const int n_mma = (!TOPK && N <= BLOCK_N / 2) ? BLOCK_N / 2 : BLOCK_N;
  const uint32_t IDESC = (1u << 4) | ((uint32_t)(n_mma >> 3) << 17) | ((uint32_t)((2 * BLOCK_M) >> 4) << 24);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* epi_smem = reinterpret_cast<float*>(smem + (size_t)STAGES * F16S_STAGE);
  __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_base_s;
  constexpr int EPI_WARPS = LSE ? 8 : 4;
  __shared__ float2 lse_pair[2][4][32];                   // [tile parity][lane quarter][row]: upper-half (max, sum)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int64_t M = live_rows(M_cap, m_dev);
  const int64_t n_m = (M + BLOCK_M - 1) / BLOCK_M, n_n = (N + BLOCK_N - 1) / BLOCK_N;
  const int64_t n_p = (n_m + 1) / 2;                             // row pairs (2 * BLOCK_M = BLOCK_N rows each)
  // causal == 1 (S = Q K'^T of causal attention): only column tiles c <= row pair r are ever read (column j <= row i),
  //   so a batch entry has sum_r min(r + 1, n_n) tiles instead of n_p * n_n;
  // causal == 2 (O = P V'): row pair r only contracts over k < (r + 1) * 2 * BLOCK_M (P is zero / unread beyond),
  //   heaviest row pairs first.
  const int64_t per_batch = causal == 1 ? f16s_causal_tiles(n_p, n_n) : n_p * n_n;   // pair tiles of one batch entry
  const int64_t total = per_batch * nb;                          // maps are 3-D: (k, row, batch)
  const int64_t pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;
  const int n_kb = (int)((K + F16_BLOCK_K - 1) / F16_BLOCK_K);
  // tile index -> (batch entry, row pair, column tile, k blocks); identical in every warp role
  auto decode = [&](int64_t tile, int& bi, int64_t& r, int64_t& c, int& kbs) {
    bi = (int)(tile / per_batch);
    int64_t rem = tile % per_batch;
    kbs = n_kb;
    if (causal == 1) {
      r = 0;
      for (int64_t cnt = 1 < n_n ? 1 : n_n; rem >= cnt; cnt = (r + 1 < n_n ? r + 1 : n_n)) { rem -= cnt; ++r; }
      c = rem;
    } else if (causal == 2) {
      r = n_p - 1 - rem / n_n;
      c = rem % n_n;
      const int64_t lim = ((r + 1) * 2 * BLOCK_M + F16_BLOCK_K - 1) / F16_BLOCK_K;
      if (lim < kbs) kbs = (int)lim;
    } else {
      r = rem / n_n;
      c = rem % n_n;
    }
  };

  auto sAh = [&](int s) { return smem + (size_t)s * F16S_STAGE; };
  auto sAl = [&](int s) { return smem + (size_t)s * F16S_STAGE + F16_OP_A; };
  auto sBh = [&](int s) { return smem + (size_t)s * F16S_STAGE + 2 * F16_OP_A; };
  auto sBl = [&](int s) { return smem + (size_t)s * F16S_STAGE + 2 * F16_OP_A + F16_OP_B; };

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ah) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_al) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_blo) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 2 * EPI_WARPS);        // every epilogue warp of both CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (lane == 0) {                                   // ---- TMA producer (both CTAs)
      int stage = 0;
      uint32_t phase = 0;
      const int half = (int)crank * (n_mma / 2);
      for (int64_t tile = pair0; tile < total; tile += pair_stride) {
        int bi, kbs;
        int64_t r, c;
        decode(tile, bi, r, c, kbs);
        const int m0 = (int)((r * 2 + crank) * BLOCK_M), n0 = (int)(c * BLOCK_N) + half;
        for (int kb = 0; kb < kbs; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_expect_tx(&full_bar[stage], TX);
          tma_load_3d_2sm(sAh(stage), &map_ah, kb * F16_BLOCK_K, m0, bi, &full_bar[stage]);
          tma_load_3d_2sm(sAl(stage), &map_al, kb * F16_BLOCK_K, m0, bi, &full_bar[stage]);
          tma_load_3d_2sm(sBh(stage), &map_b, kb * F16_BLOCK_K, n0, bi, &full_bar[stage]);
          tma_load_3d_2sm(sBl(stage), &map_blo, kb * F16_BLOCK_K, n0, bi, &full_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {                         // ---- MMA issuer (leader only)
      int stage = 0;
      uint32_t phase = 0;
      int64_t it = 0;
      for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * BLOCK_N;
        int bi, kbs;
        int64_t r, c;
        decode(tile, bi, r, c, kbs);
        for (int kb = 0; kb < kbs; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t dah = make_desc_sw64(smem_u32(sAh(stage))), dal = make_desc_sw64(smem_u32(sAl(stage)));
          const uint64_t dbh = make_desc_sw64(smem_u32(sBh(stage))), dbl = make_desc_sw64(smem_u32(sBl(stage)));
#pragma unroll
          for (int k = 0; k < F16_BLOCK_K / 16; ++k) {
            const uint64_t koff = (uint64_t)(k * 2);
            umma_2sm<0>(d_tmem, dah + koff, dbl + koff, IDESC, (kb | k) > 0 ? 1u : 0u);
            umma_2sm<0>(d_tmem, dal + koff, dbh + koff, IDESC, 1u);
            umma_2sm<0>(d_tmem, dah + koff, dbh + koff, IDESC, 1u);
          }
          tc_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit_2sm(&tmem_full[acc]);
      }
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + EPI_WARPS) {
    const int q = warp & 3;                            // ---- epilogue (both CTAs)
    const int half = (warp - EPI_WARP0) >> 2;          // LSE: 0 = lower, 1 = upper half of the tile's columns
    constexpr int COLS = LSE ? BLOCK_N / 2 : BLOCK_N;
    int64_t it = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
      const int acc = (int)(it & 1);
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      int bi, kbs;
      int64_t r, n_blk;
      decode(tile, bi, r, n_blk, kbs);
      const int64_t m_blk = r * 2 + crank;
      const int64_t m = m_blk * BLOCK_M + q * 32 + lane;
      const int64_t n_base = n_blk * BLOCK_N;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * BLOCK_N + (uint32_t)(half * COLS) + ((uint32_t)(q * 32) << 16);
      EpiStore eb = es;                                  // batch entry bi (fp32 C / residual when nb > 1)
      if (nb > 1) {
        eb.C = reinterpret_cast<float*>(es.C) + bi * c_bs;
        if (es.residual) eb.residual = reinterpret_cast<const float*>(es.residual) + bi * r_bs;
      }
      if constexpr (TOPK)
        epilogue_topk(taddr, m, M, n_base, N, et, acc_scale);
      else if constexpr (LSE)
        epilogue_tile<LSE>(taddr, m, M, n_base + half * COLS, n_blk, N, eb, el, epi_smem, acc_scale, COLS,
                           &lse_pair[it & 1][q][lane], half ? 1 : 2, 1 + q);
      else
        epilogue_tile<LSE>(taddr, m, M, n_base, n_blk, N, eb, el, epi_smem + (warp & 3) * 32 * EPI_LD, acc_scale);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- host side
// fp16 [rows, K] K-major matrix, SWIZZLE_64B boxes of 32 elements x box_rows
static int make_map_f16(CUtensorMap* map, const void* base, int64_t rows, int64_t K, int64_t ld, int box_rows) {
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)F16_BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return (int)encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// fp16 [nb, rows, K] K-major, SWIZZLE_64B boxes of 32 elements x box_rows x 1 (batch stride bs elements)
static int make_map_f16_3d(CUtensorMap* map, const void* base, int64_t rows, int64_t K, int64_t ld, int64_t nb, int64_t bs,
                           int box_rows) {
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)nb};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)(nb > 1 ? bs : rows * ld) * 2};
  cuuint32_t box[3] = {(cuuint32_t)F16_BLOCK_K, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return (int)encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

template <bool LSE>
static int32_t launch_f16x3(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mblo, int64_t M,
                            const int32_t* m_dev, int64_t N, int64_t K, const EpiStore& es, const EpiLse& el, float acc_scale,
                            cudaStream_t st);

static int make_map(CUtensorMap* map, const void* base, int bf16, int64_t rows, int64_t K, int64_t ld, int box_rows) {
  const int elem = bf16 ? 2 : 4;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * elem};
  cuuint32_t box[2] = {(cuuint32_t)(ROW_BYTES / elem), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_fn()(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                           const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return (int)r;
}

static int use_2sm() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("GNNLM_GEMM_2SM");
    v = e ? atoi(e) : 1;                    // default: cta_group::2 kernel; GNNLM_GEMM_2SM=0 -> 1-SM + W multicast
  }
  return v;
}

template <int MODE, bool LSE>
static int32_t launch(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mblo, int64_t M, const int32_t* m_dev,
                      int64_t N, int64_t K, const EpiStore& es, const EpiLse& el, cudaStream_t st) {
  const bool two = use_2sm() != 0;
  const int stage_bytes = two ? (MODE == X3 ? 2 * (A_TILE + B_TILE / 2) : (A_TILE + B_TILE / 2))
                              : (MODE == X3 ? 2 * (A_TILE + B_TILE) : (A_TILE + B_TILE));
  const bool epi8 = two && tc2_epi8<MODE, LSE>();
  const int stages = two ? (MODE == X3 ? 3 : (epi8 ? 5 : 6)) : (MODE == X3 ? 2 : 4);
  const size_t smem = (size_t)stages * stage_bytes + (epi8 ? 2 : 1) * EPI_SMEM + 1024;
  static bool attr_set[2] = {false, false};
  if (!attr_set[two]) {
    if (two) GNNLM_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<MODE, LSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    else GNNLM_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<MODE, LSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[two] = true;
  }
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    GNNLM_CUDA(cudaGetDevice(&dev));
    GNNLM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  const int64_t pairs = ceil_div(ceil_div(M, BLOCK_M), 2) * ceil_div(N, BLOCK_N);
  const int64_t max_pairs = n_sm / 2;
  const unsigned grid = 2u * (unsigned)(pairs < max_pairs ? pairs : max_pairs);     // clusters of 2 CTAs
  if (two) gemm_tc2_kernel<MODE, LSE><<<grid, (MODE == X3 || epi8) ? 384 : 256, smem, st>>>(ma, mb, mblo, M, m_dev, N, K, es, el);
  else gemm_tc_kernel<MODE, LSE><<<grid, MODE == X3 ? 384 : 256, smem, st>>>(ma, mb, mblo, M, m_dev, N, K, es, el);
  GNNLM_LAUNCH_CHECK("gemm_tcgen05");
  return 0;
}

template <bool LSE>
static int32_t launch_f16x3(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mblo, int64_t M,
                            const int32_t* m_dev, int64_t N, int64_t K, const EpiStore& es, const EpiLse& el, float acc_scale,
                            cudaStream_t st) {
  const size_t smem = (size_t)F16_STAGES * F16_STAGE + EPI_SMEM + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    GNNLM_CUDA(cudaFuncSetAttribute(gemm_f16x3_kernel<LSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    GNNLM_CUDA(cudaGetDevice(&dev));
    GNNLM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  const int64_t pairs = ceil_div(ceil_div(M, BLOCK_M), 2) * ceil_div(N, BLOCK_N);
  const int64_t max_pairs = n_sm / 2;
  const unsigned grid = 2u * (unsigned)(pairs < max_pairs ? pairs : max_pairs);
  static int dbg = -1;
  if (dbg < 0) { const char* e = getenv("GNNLM_GEMM_DEBUG"); dbg = e ? atoi(e) : 0; }   // timing experiments only
  gemm_f16x3_kernel<LSE><<<grid, F16_THREADS, smem, st>>>(ma, mb, mblo, M, m_dev, N, K, es, el, acc_scale, dbg);
  GNNLM_LAUNCH_CHECK("gemm_f16x3");
  return 0;
}

template <bool LSE, bool TOPK = false>
static int32_t launch_f16s(const CUtensorMap& mah, const CUtensorMap& mal, const CUtensorMap& mb, const CUtensorMap& mblo,
                           int64_t M, const int32_t* m_dev, int64_t N, int64_t K, const EpiStore& es, const EpiLse& el,
                           float acc_scale, cudaStream_t st, int nb = 1, int64_t c_bs = 0, int64_t r_bs = 0, int causal = 0,
                           const EpiTopk& et = EpiTopk{}) {
  const size_t smem = (size_t)F16S_STAGES * F16S_STAGE + EPI_SMEM + 1024;
  static bool attr_set[MAX_DEVICES] = {};
  bool& done = attr_set[device_slot()];
  if (!done) {
    GNNLM_CUDA(cudaFuncSetAttribute(gemm_f16s_kernel<LSE, TOPK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    done = true;
  }
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    GNNLM_CUDA(cudaGetDevice(&dev));
    GNNLM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  const int64_t n_p = ceil_div(ceil_div(M, BLOCK_M), 2), n_n = ceil_div(N, BLOCK_N);
  const int64_t pairs = (causal == 1 ? f16s_causal_tiles(n_p, n_n) : n_p * n_n) * nb;
  const int64_t max_pairs = n_sm / 2;
  const unsigned grid = 2u * (unsigned)(pairs < max_pairs ? pairs : max_pairs);
  gemm_f16s_kernel<LSE, TOPK><<<grid, LSE ? 384 : 256, smem, st>>>(mah, mal, mb, mblo, M, m_dev, N, K, es, el, acc_scale, nb, c_bs,
                                                                   r_bs, causal, et);
  GNNLM_LAUNCH_CHECK(TOPK ? "gemm_f16s_topk" : "gemm_f16s");
  return 0;
}

}  // namespace tc

int32_t gemm_tc_supported() { return tc::encode_fn() != nullptr && tc::device_is_sm100(); }
int64_t gemm_tc_lse_tile_n() { return tc::BLOCK_N; }

static int32_t tc_prepare(const char* who, const void* A, int32_t a_dtype, int64_t lda, const void* W, const void* W_lo,
                          int64_t ldw, int64_t M, int64_t N, int64_t K, int32_t math, CUtensorMap* ma, CUtensorMap* mb,
                          CUtensorMap* mblo) {
  GNNLM_CHECK_ARG(gemm_tc_supported(), GNNLM_E_UNSUPPORTED, "%s: tcgen05 path needs an sm_100 device and driver TMA support", who);
  if (math == GNNLM_MATH_F16X3) {
    GNNLM_CHECK_ARG(W_lo, GNNLM_E_ARG, "%s: MATH_F16X3 needs W_lo (gnnlm_split_f16)", who);
    GNNLM_CHECK_ARG((lda * 4) % 16 == 0 && (ldw * 2) % 16 == 0 && (uintptr_t)A % 16 == 0 && (uintptr_t)W % 16 == 0 &&
                        (uintptr_t)W_lo % 16 == 0,
                    GNNLM_E_SHAPE, "%s: TMA needs 16 B aligned bases and row strides (lda=%lld ldw=%lld)", who, (long long)lda,
                    (long long)ldw);
    int r = tc::make_map(ma, A, 0, M, K, lda, tc::BLOCK_M);                // fp32 A, SWIZZLE_128B, 32-element rows
    if (!r) r = tc::make_map_f16(mb, W, N, K, ldw, tc::BLOCK_N / 2);
    if (!r) r = tc::make_map_f16(mblo, W_lo, N, K, ldw, tc::BLOCK_N / 2);
    GNNLM_CHECK_ARG(r == 0, GNNLM_E_ARG, "%s: cuTensorMapEncodeTiled failed (%d)", who, r);
    return 0;
  }
  const int bf16 = math == GNNLM_MATH_BF16;
  const int elem = bf16 ? 2 : 4;
  GNNLM_CHECK_ARG((lda * elem) % 16 == 0 && (ldw * elem) % 16 == 0 && (uintptr_t)A % 16 == 0 && (uintptr_t)W % 16 == 0,
                  GNNLM_E_SHAPE, "%s: TMA needs 16 B aligned bases and row strides (lda=%lld ldw=%lld)", who, (long long)lda,
                  (long long)ldw);
  GNNLM_CHECK_ARG(math != GNNLM_MATH_TF32X3 || (W_lo && (uintptr_t)W_lo % 16 == 0), GNNLM_E_ARG,
                  "%s: MATH_TF32X3 needs W_lo (gnnlm_split_tf32)", who);
  int r = tc::make_map(ma, A, bf16, M, K, lda, tc::BLOCK_M);
  if (!r) r = tc::make_map(mb, W, bf16, N, K, ldw, tc::BLOCK_N / 2);       // each CTA of a pair loads half the W tile
  if (!r) r = tc::make_map(mblo, math == GNNLM_MATH_TF32X3 ? W_lo : W, bf16, N, K, ldw, tc::BLOCK_N / 2);
  GNNLM_CHECK_ARG(r == 0, GNNLM_E_ARG, "%s: cuTensorMapEncodeTiled failed (%d)", who, r);
  return 0;
}

static inline int epi_mode(int32_t dtype) { return dtype == GNNLM_BF16 ? 1 : (dtype == GNNLM_F16X2 ? 2 : 0); }

// split-fp16 A (GNNLM_F16X2): four SWIZZLE_64B maps (k, row, batch), no in-kernel operand split
static int32_t f16s_maps(const char* who, const void* A, int64_t lda, const void* W, const void* W_lo, int64_t ldw, int64_t M,
                         int64_t N, int64_t K, CUtensorMap* mah, CUtensorMap* mal, CUtensorMap* mb, CUtensorMap* mblo,
                         int64_t nb = 1, int64_t a_bs = 0, int64_t w_bs = 0) {
  GNNLM_CHECK_ARG(gemm_tc_supported(), GNNLM_E_UNSUPPORTED, "%s: tcgen05 path needs an sm_100 device and driver TMA support", who);
  GNNLM_CHECK_ARG(W_lo, GNNLM_E_ARG, "%s: MATH_F16X3 needs W_lo (gnnlm_split_f16)", who);
  GNNLM_CHECK_ARG(lda >= 2 * K && (lda * 2) % 16 == 0 && (K * 2) % 16 == 0 && (ldw * 2) % 16 == 0 && (uintptr_t)A % 16 == 0 &&
                      (uintptr_t)W % 16 == 0 && (uintptr_t)W_lo % 16 == 0 && (a_bs * 2) % 16 == 0 && (w_bs * 2) % 16 == 0,
                  GNNLM_E_SHAPE, "%s: split-fp16 A needs lda >= 2K and 16 B aligned halves (lda=%lld K=%lld)", who,
                  (long long)lda, (long long)K);
  const __half* a = reinterpret_cast<const __half*>(A);
  int r = tc::make_map_f16_3d(mah, a, M, K, lda, nb, a_bs, tc::BLOCK_M);
  if (!r) r = tc::make_map_f16_3d(mal, a + K, M, K, lda, nb, a_bs, tc::BLOCK_M);
  if (!r) r = tc::make_map_f16_3d(mb, W, N, K, ldw, nb, w_bs, tc::BLOCK_N / 2);
  if (!r) r = tc::make_map_f16_3d(mblo, W_lo, N, K, ldw, nb, w_bs, tc::BLOCK_N / 2);
  GNNLM_CHECK_ARG(r == 0, GNNLM_E_ARG, "%s: cuTensorMapEncodeTiled failed (%d)", who, r);
  return 0;
}

// nb independent products C[b] = acc_scale * A[b] W[b]^T (+ residual[b]) in one launch (per-head attention GEMMs)
int32_t gemm_tc_batched_f16x3(const void* A, int64_t lda, int64_t a_bs, const void* W_hi, const void* W_lo, int64_t ldw,
                              int64_t w_bs, float w_scale, const float* residual, int64_t ldr, int64_t r_bs, float* C,
                              int64_t ldc, int64_t c_bs, int64_t nb, int64_t M, int64_t N, int64_t K, int32_t causal,
                              cudaStream_t st) {
  if (M == 0 || nb == 0) return 0;
  tc::EpiStore es{nullptr, residual, ldr, C, ldc, 0, 0, N, N};
  tc::EpiLse el{};
  CUtensorMap mah, mal, mb, mblo;
  int32_t rc = f16s_maps("gnnlm_linear_batched_f16x3", A, lda, W_hi, W_lo, ldw, M, N, K, &mah, &mal, &mb, &mblo, nb, a_bs, w_bs);
  if (rc) return rc;
  return tc::launch_f16s<false>(mah, mal, mb, mblo, M, nullptr, N, K, es, el, 1.f / w_scale, st, (int)nb, c_bs, r_bs, causal);
}

int32_t gemm_tc_store(const void* A, int32_t a_dtype, int64_t lda, const void* W, const void* W_lo, float w_scale, int64_t ldw,
                      const float* bias, const void* residual, int32_t r_dtype, int64_t ldr, void* C, int32_t c_dtype,
                      int64_t ldc, int64_t M, const int32_t* m_dev, int64_t N, int64_t K, int32_t math, cudaStream_t st) {
  if (M == 0) return 0;
  // split-fp16 buffers keep their lo half N (resp. the residual's logical width = N) columns after the hi half
  tc::EpiStore es{bias, residual, ldr, C, ldc, epi_mode(c_dtype), epi_mode(r_dtype), N, N};
  tc::EpiLse el{};
  if (math == GNNLM_MATH_F16X3 && a_dtype == GNNLM_F16X2) {
    CUtensorMap mah, mal, mb, mblo;
    int32_t rc = f16s_maps("gnnlm_linear", A, lda, W, W_lo, ldw, M, N, K, &mah, &mal, &mb, &mblo);
    if (rc) return rc;
    return tc::launch_f16s<false>(mah, mal, mb, mblo, M, m_dev, N, K, es, el, 1.f / w_scale, st);
  }
  CUtensorMap ma, mb, mblo;
  int32_t rc = tc_prepare("gnnlm_linear", A, a_dtype, lda, W, W_lo, ldw, M, N, K, math, &ma, &mb, &mblo);
  if (rc) return rc;
  if (math == GNNLM_MATH_F16X3) return tc::launch_f16x3<false>(ma, mb, mblo, M, m_dev, N, K, es, el, 1.f / w_scale, st);
  if (math == GNNLM_MATH_TF32X3) return tc::launch<tc::X3, false>(ma, mb, mblo, M, m_dev, N, K, es, el, st);
  if (math == GNNLM_MATH_TF32) return tc::launch<tc::TF32, false>(ma, mb, mblo, M, m_dev, N, K, es, el, st);
  return tc::launch<tc::BF16, false>(ma, mb, mblo, M, m_dev, N, K, es, el, st);
}

// Top-k filter pass of the exact kNN search: scores of the keys A (split fp16 [M, 2K], rows = ids id_base ..) against the queries
// (W_hi / W_lo [N, K], scale 1), candidates above thr per query (see EpiTopk).
int32_t gemm_tc_topk(const void* A, int64_t lda, int64_t M, int64_t id_base, const void* W_hi, const void* W_lo, int64_t ldw,
                     int64_t N, int64_t K, const float* row_bias, const float* thr, float* cand_s, int32_t* cand_id,
                     int32_t* cand_cnt, int64_t cap, cudaStream_t st) {
  if (M == 0) return 0;
  tc::EpiStore es{};
  tc::EpiLse el{};
  const tc::EpiTopk et{row_bias, thr, cand_s, cand_id, cand_cnt, cap, id_base};
  CUtensorMap mah, mal, mb, mblo;
  int32_t rc = f16s_maps("gnnlm_knn_filter_f16x3", A, lda, W_hi, W_lo, ldw, M, N, K, &mah, &mal, &mb, &mblo);
  if (rc) return rc;
  return tc::launch_f16s<false, true>(mah, mal, mb, mblo, M, nullptr, N, K, es, el, 1.f, st, 1, 0, 0, 0, et);
}

int32_t gemm_tc_lse(const void* A, int32_t a_dtype, int64_t lda, const void* W, const void* W_lo, float w_scale, int64_t ldw,
                    const int32_t* pick, float* part_max, float* part_sum, float* picked, int64_t M,
                    const int32_t* m_dev, int64_t N, int64_t K, int32_t math, cudaStream_t st) {
  if (M == 0) return 0;
  tc::EpiStore es{};
  tc::EpiLse el{pick, part_max, part_sum, picked, ceil_div(N, tc::BLOCK_N)};
  if (math == GNNLM_MATH_F16X3 && a_dtype == GNNLM_F16X2) {
    CUtensorMap mah, mal, mb, mblo;
    int32_t rc = f16s_maps("gnnlm_linear_lse", A, lda, W, W_lo, ldw, M, N, K, &mah, &mal, &mb, &mblo);
    if (rc) return rc;
    return tc::launch_f16s<true>(mah, mal, mb, mblo, M, m_dev, N, K, es, el, 1.f / w_scale, st);
  }
  CUtensorMap ma, mb, mblo;
  int32_t rc = tc_prepare("gnnlm_linear_lse", A, a_dtype, lda, W, W_lo, ldw, M, N, K, math, &ma, &mb, &mblo);
  if (rc) return rc;
  if (math == GNNLM_MATH_F16X3) return tc::launch_f16x3<true>(ma, mb, mblo, M, m_dev, N, K, es, el, 1.f / w_scale, st);
  if (math == GNNLM_MATH_TF32X3) return tc::launch<tc::X3, true>(ma, mb, mblo, M, m_dev, N, K, es, el, st);
  if (math == GNNLM_MATH_TF32) return tc::launch<tc::TF32, true>(ma, mb, mblo, M, m_dev, N, K, es, el, st);
  return tc::launch<tc::BF16, true>(ma, mb, mblo, M, m_dev, N, K, es, el, st);
}

}  // namespace gnnlm
