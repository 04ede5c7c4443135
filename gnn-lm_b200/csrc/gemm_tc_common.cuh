// Shared pieces of the tcgen05 / TMEM / TMA GEMM kernels (gemm_tcgen05.cu, gemm_f16f8.cu): mbarrier / TMA / UMMA
// wrappers, shared-memory operand descriptors, the store and log-sum-exp epilogues, and the host-side tensor-map
// encoder lookup.  sm_100a only.
#pragma once
#include <cuda.h>
#include <stdlib.h>

#include <cuda_fp16.h>

#include "common.cuh"

namespace gnnlm {

namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 256;
constexpr int ROW_BYTES = 128;                       // one SWIZZLE_128B row == one k-block
constexpr int A_TILE = BLOCK_M * ROW_BYTES;          // 16 KB
constexpr int B_TILE = BLOCK_N * ROW_BYTES;          // 32 KB
constexpr int TMEM_COLS = 512;
constexpr int EPI_WARP0 = 4, CONV_WARP0 = 8;

enum Mode { X3 = 0, TF32 = 1, BF16 = 2 };

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (spin > (1u << 22)) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// multicast variant: the box lands at the same smem offset of every CTA in `mask`, each CTA's mbarrier (same
// offset) receives the complete_tx
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// commit that arrives on the mbarrier at the same offset in every CTA of `mask`
__device__ __forceinline__ void tc_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// K-major, SWIZZLE_128B smem operand descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// start>>4 [0,14) | LBO>>4 = 1 [16,30) | SBO>>4 = 64 (8 rows x 128 B) [32,46) | version 1 [46,48) | layout 2 [61,64)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

template <int KIND_TF32>
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  if constexpr (KIND_TF32) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// issue only; the registers are valid after tmem_ld_wait(v) (which names them, so that no use can be scheduled above it)
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr) : "memory");
  return r;
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct EpiStore {
  const float* bias;
  const void* residual;
  int64_t ldr;
  void* C;
  int64_t ldc;
  int c_bf16;      // C element type: 0 = f32, 1 = bf16, 2 = split-fp16 (hi | lo, lo at column offset c_lo), 3 = GNNLM_F24: 16-bit plane at C + byte plane at C8
  int r_bf16;      // residual type, same encoding (lo at column offset r_lo)
  int64_t c_lo, r_lo;
  int dbg;         // timing experiments only (GNNLM_F8_DEBUG bits 3 / 4): 1 = no global stores, 2 = no TMEM loads / staging
  uint8_t* C8;     // c_bf16 == 3 (GNNLM_F24): the byte plane, same row stride (ldc elements = ldc bytes)
};
struct EpiLse {
  const int32_t* pick;
  float* part_max;
  float* part_sum;
  float* picked;
  int64_t n_tiles;
};

// Top-k filter of the exact kNN search (gnnlm_knn_filter_f16x3): rows are datastore keys, columns queries.  Nothing is
// stored per (key, query); only scores s = acc + row_bias[m] above the query's threshold become candidates.
struct EpiTopk {
  const float* row_bias;   // [M] (-1/2 ||x||^2 for l2), nullable
  const float* thr;        // [N] per-query threshold (strict: s > thr)
  float* cand_s;           // [N, cap]
  int32_t* cand_id;        // [N, cap]
  int32_t* cand_cnt;       // [N]: counts every candidate, also past cap (overflow = cand_cnt > cap)
  int64_t cap;
  int64_t id_base;         // id of row 0
};

// One key row per thread.  The 32 thresholds of a chunk sit in one register per lane and are broadcast by shuffle; per
// column the warp ballots `s > thr`, one lane reserves the slots with a single atomicAdd, and every passing lane writes
// (s, id) at its rank.  Writes stop at cap; the count keeps growing so that the host sees the overflow.
__device__ __forceinline__ void epilogue_topk(uint32_t taddr, int64_t m, int64_t M, int64_t n_base, int64_t N, const EpiTopk& et,
                                              float acc_scale) {
  const int lane = threadIdx.x & 31;
  const bool row_ok = m < M;
  const float rb = (row_ok && et.row_bias) ? __ldg(et.row_bias + m) : 0.f;
  const int32_t id = (int32_t)(et.id_base + m);
  const uint32_t below = (1u << lane) - 1u;
  float v[32];
#pragma unroll 1
  for (int c = 0; c < BLOCK_N; c += 32) {
    const int64_t n0 = n_base + c;
    if (n0 >= N) break;                                          // warp-uniform
    const float t_l = n0 + lane < N ? __ldg(et.thr + n0 + lane) : INFINITY;
    tmem_ld32(taddr + (uint32_t)c, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float t = __shfl_sync(0xffffffffu, t_l, j);
      float s = fmaf(v[j], acc_scale, rb);
      s = s == 0.f ? 0.f : s;                                    // -0 -> +0: equal scores compare equal in the merge's ordering
      const bool p = row_ok && s > t;
      const uint32_t b = __ballot_sync(0xffffffffu, p);
      if (b) {
        int base = 0;
        if (lane == 0) base = atomicAdd(et.cand_cnt + n0 + j, __popc(b));
        base = __shfl_sync(0xffffffffu, base, 0);
        const int64_t r = base + __popc(b & below);
        if (p && r < et.cap) {
          et.cand_s[(n0 + j) * et.cap + r] = s;
          et.cand_id[(n0 + j) * et.cap + r] = id;
        }
      }
    }
  }
}

// One output row per thread: drain 32-column chunks of this warp's TMEM lane quarter and either store them
// (bias / residual fused) or fold them into the running (max, sum-exp, picked logit) of the row.
constexpr int EPI_LD = 36;                                  // padded row of the per-warp 32x32 staging tile (floats)
constexpr int EPI_SMEM = 4 * 32 * EPI_LD * 4;               // 4 epilogue warps

// Store epilogue, common case (no residual, N and every leading dimension a multiple of 4): specialised on the output
// format so that the chunk loop has no format branches, row pointers and row-valid bits computed once per tile, staging
// through 32-bit shared addresses, and the TMEM load of chunk c+1 issued before chunk c is written out.  The profile of
// the generic form showed ~400 dependent instructions per 32-column chunk at 0.11 IPC per epilogue warp -- 14 us per tile,
// three times the single-pass (bf16) main loop.
template <int CMODE>      // 0 = f32, 1 = bf16, 2 = split fp16, 3 = GNNLM_F24 (16-bit plane + byte plane)
__device__ __forceinline__ void epilogue_store_fast(uint32_t taddr, int64_t m, int64_t M, int64_t n_base, int64_t N,
                                                    const EpiStore& es, float* stage_smem, float acc_scale, int tile_cols) {
  constexpr int ES = CMODE == 0 ? 4 : 2;
  const int lane = threadIdx.x & 31;
  const int cq = (lane & 7) * 4, rsub = lane >> 3;
  const int64_t m_warp = m - lane;
  char* row0 = reinterpret_cast<char*>(es.C) + ((m_warp + rsub) * es.ldc + n_base + cq) * ES;
  const int64_t row_step = 4 * es.ldc * ES;                  // rows j*4 + rsub, j = 0..7
  const int64_t lo_bytes = es.c_lo * 2;
  uint32_t valid = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (m_warp + j * 4 + rsub < M) valid |= 1u << j;
  const uint32_t st_base = smem_u32(stage_smem);
  const uint32_t st_w = st_base + (uint32_t)lane * (EPI_LD * 4);                     // my TMEM row
  const uint32_t st_r = st_base + (uint32_t)(rsub * EPI_LD + cq) * 4;                // row rsub, my 4 columns
  const int64_t cols = N - n_base;                            // valid columns of this tile (multiple of 4)
  const int n_chunks = cols <= 0 ? 0 : (int)((cols < tile_cols ? cols : tile_cols) + 31) >> 5;
  float v[32];
  float sink = 0.f;
  const bool no_store = es.dbg & 1, no_load = es.dbg & 2;
  if (no_load) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = 0.f;
  }
  if (n_chunks > 0 && !no_load) tmem_ld32_issue(taddr, v);
#pragma unroll 1
  for (int ci = 0; ci < n_chunks; ++ci) {
    const int c = ci * 32;
    if (!no_load) {
      tmem_ld_wait(v);
#pragma unroll
      for (int j = 0; j < 8; ++j) sts128(st_w + 16 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      if (ci + 1 < n_chunks) tmem_ld32_issue(taddr + (uint32_t)(c + 32), v);           // in flight during the stores below
    }
    __syncwarp();
    const bool col_ok = c + cq < cols;                        // cols % 4 == 0: the whole quad is inside or outside
    float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
    if (es.bias && col_ok) bq = __ldg(reinterpret_cast<const float4*>(es.bias + n_base + c + cq));
    char* dst = row0 + (int64_t)c * ES;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (col_ok && (valid >> j & 1)) {
        const float4 x = no_load ? make_float4(0.f, 0.f, 0.f, 0.f) : lds128(st_r + (uint32_t)(j * 4 * EPI_LD * 4));
        const float y0 = fmaf(x.x, acc_scale, bq.x), y1 = fmaf(x.y, acc_scale, bq.y), y2 = fmaf(x.z, acc_scale, bq.z),
                    y3 = fmaf(x.w, acc_scale, bq.w);
        char* p = dst + j * row_step;
        if (no_store) { sink += y0 + y1 + y2 + y3; continue; }
        if constexpr (CMODE == 0) {
          *reinterpret_cast<float4*>(p) = make_float4(y0, y1, y2, y3);
        } else if constexpr (CMODE == 2) {
          uint2 hi, lo;
          split4_f16(y0, y1, y2, y3, hi, lo);
          *reinterpret_cast<uint2*>(p) = hi;
          *reinterpret_cast<uint2*>(p + lo_bytes) = lo;
        } else if constexpr (CMODE == 3) {
          uint2 hi;
          uint32_t lo;
          f24_pack4(y0, y1, y2, y3, hi, lo);
          *reinterpret_cast<uint2*>(p) = hi;
          *reinterpret_cast<uint32_t*>(es.C8 + ((p - reinterpret_cast<char*>(es.C)) >> 1)) = lo;
        } else {
          const __nv_bfloat162 p0 = __floats2bfloat162_rn(y0, y1), p1 = __floats2bfloat162_rn(y2, y3);
          uint2 u;
          u.x = *reinterpret_cast<const uint32_t*>(&p0);
          u.y = *reinterpret_cast<const uint32_t*>(&p1);
          *reinterpret_cast<uint2*>(p) = u;
        }
      }
    }
    __syncwarp();
  }
  if (sink == 12345.678f) *reinterpret_cast<float*>(es.C) = sink;       // keeps the no-store experiment's loads alive
}

template <bool LSE>
__device__ __forceinline__ void epilogue_tile(uint32_t taddr, int64_t m, int64_t M, int64_t n_base, int64_t n_blk, int64_t N,
                                              const EpiStore& es, const EpiLse& el, float* stage_smem, float acc_scale = 1.f,
                                              int tile_cols = BLOCK_N, float2* lse_slot = nullptr, int lse_role = 0,
                                              int lse_bar = 0) {
        if constexpr (!LSE) {
          // warp-uniform launch properties
          if (!es.residual && (N & 3) == 0 && (es.ldc & 3) == 0 && (es.c_bf16 != 2 || (es.c_lo & 3) == 0) &&
              (reinterpret_cast<uintptr_t>(es.C) & 15) == 0 && (!es.bias || (reinterpret_cast<uintptr_t>(es.bias) & 15) == 0)) {
            if (es.c_bf16 == 0) epilogue_store_fast<0>(taddr, m, M, n_base, N, es, stage_smem, acc_scale, tile_cols);
            else if (es.c_bf16 == 2) epilogue_store_fast<2>(taddr, m, M, n_base, N, es, stage_smem, acc_scale, tile_cols);
            else if (es.c_bf16 == 3) epilogue_store_fast<3>(taddr, m, M, n_base, N, es, stage_smem, acc_scale, tile_cols);
            else epilogue_store_fast<1>(taddr, m, M, n_base, N, es, stage_smem, acc_scale, tile_cols);
            return;
          }
        }
        float run_max = -INFINITY, run_sum = 0.f;
        const int32_t want = (LSE && m < M && el.pick) ? __ldg(el.pick + m) : -1;
  #pragma unroll 1
        for (int c = 0; c < tile_cols; c += 32) {
          if (n_base + c >= N) break;                  // warp-uniform
          // residual rows of this chunk in the *transposed* (coalesced) mapping, issued as one batch before the
          // TMEM load so that their DRAM latency overlaps it
          float4 res[8];
          if constexpr (!LSE) {
            const int lane_ = threadIdx.x & 31;
            const int cq_ = (lane_ & 7) * 4;
            const int64_t n0_ = n_base + c;
            const bool ok_ = es.residual && (n0_ + cq_ + 3 < N) && ((es.ldc & 3) == 0) && ((es.ldr & 3) == 0) &&
                             (es.r_bf16 != 2 || (es.r_lo & 3) == 0) && (es.c_bf16 != 2 || (es.c_lo & 3) == 0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int64_t mr = (m - lane_) + j * 4 + (lane_ >> 3);
              res[j] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (ok_ && mr < M) {
                if (!es.r_bf16) {
                  res[j] = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(es.residual) + mr * es.ldr + n0_ + cq_));
                } else if (es.r_bf16 == 2) {
                  const __half* rp = reinterpret_cast<const __half*>(es.residual) + mr * es.ldr + n0_ + cq_;
                  res[j] = join4_f16(__ldg(reinterpret_cast<const uint2*>(rp)), __ldg(reinterpret_cast<const uint2*>(rp + es.r_lo)));
                } else {
                  const uint2 t = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(es.residual) + mr * es.ldr + n0_ + cq_));
                  const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
                  const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
                  res[j] = make_float4(f0.x, f0.y, f1.x, f1.y);
                }
              }
            }
          }
          float v[32];
          tmem_ld32(taddr + (uint32_t)c, v);
          if (acc_scale != 1.f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= acc_scale;
          }
          const int64_t n0 = n_base + c;
          if constexpr (!LSE) {
            // Stage the 32x32 chunk through shared memory so that global traffic is coalesced: a thread owns
            // one accumulator ROW in TMEM, but stores / residual loads want 8 lanes on one 128 B line.
            // (Row-per-thread 16 B stores at a 12 KB stride made the epilogue slower than the MMAs.)
            float* tile = stage_smem;                                    // [32][EPI_LD] floats, private to this warp
            const int lane = threadIdx.x & 31;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<float4*>(tile + lane * EPI_LD + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            __syncwarp();
            const int cq = (lane & 7) * 4;                               // my 4 columns inside the chunk
            const bool col_ok = n0 + cq + 3 < N;                         // whole float4 inside N
            float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
            if (es.bias) {
              if (col_ok) bq = __ldg(reinterpret_cast<const float4*>(es.bias + n0 + cq));
              else {
                if (n0 + cq < N) bq.x = __ldg(es.bias + n0 + cq);
                if (n0 + cq + 1 < N) bq.y = __ldg(es.bias + n0 + cq + 1);
                if (n0 + cq + 2 < N) bq.z = __ldg(es.bias + n0 + cq + 2);
              }
            }
            const int64_t m_warp = m - lane;                             // first row of this warp's 32 rows
            const bool vec_ok = col_ok && ((es.ldc & 3) == 0) && (!es.residual || (es.ldr & 3) == 0) &&
                                (es.r_bf16 != 2 || (es.r_lo & 3) == 0) && (es.c_bf16 != 2 || (es.c_lo & 3) == 0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int r = j * 4 + (lane >> 3);
              const int64_t mr = m_warp + r;
              if (mr >= M) continue;
              float4 x = *reinterpret_cast<const float4*>(tile + r * EPI_LD + cq);
              x.x += bq.x; x.y += bq.y; x.z += bq.z; x.w += bq.w;
              float xs[4] = {x.x, x.y, x.z, x.w};
              if (vec_ok) {
                xs[0] += res[j].x; xs[1] += res[j].y; xs[2] += res[j].z; xs[3] += res[j].w;     // prefetched above
                if (!es.c_bf16) {
                  *reinterpret_cast<float4*>(reinterpret_cast<float*>(es.C) + mr * es.ldc + n0 + cq) = make_float4(xs[0], xs[1], xs[2], xs[3]);
                } else if (es.c_bf16 == 2) {
                  uint2 hi, lo;
                  split4_f16(xs[0], xs[1], xs[2], xs[3], hi, lo);
                  __half* cp = reinterpret_cast<__half*>(es.C) + mr * es.ldc + n0 + cq;
                  *reinterpret_cast<uint2*>(cp) = hi;
                  *reinterpret_cast<uint2*>(cp + es.c_lo) = lo;
                } else {
                  __nv_bfloat162 p0 = __floats2bfloat162_rn(xs[0], xs[1]), p1 = __floats2bfloat162_rn(xs[2], xs[3]);
                  uint2 u;
                  u.x = *reinterpret_cast<uint32_t*>(&p0);
                  u.y = *reinterpret_cast<uint32_t*>(&p1);
                  *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(es.C) + mr * es.ldc + n0 + cq) = u;
                }
              } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int64_t n = n0 + cq + e;
                  if (n >= N) continue;
                  float y = xs[e];
                  if (es.residual) {
                    if (es.r_bf16 == 2) {
                      const __half* rp = reinterpret_cast<const __half*>(es.residual) + mr * es.ldr + n;
                      y += __half2float(rp[0]) + __half2float(rp[es.r_lo]);
                    } else {
                      y += es.r_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(es.residual)[mr * es.ldr + n])
                                     : __ldg(reinterpret_cast<const float*>(es.residual) + mr * es.ldr + n);
                    }
                  }
                  if (!es.c_bf16) reinterpret_cast<float*>(es.C)[mr * es.ldc + n] = y;
                  else if (es.c_bf16 == 2) {
                    const float yc = fminf(fmaxf(y, -65504.f), 65504.f);
                    const __half h = __float2half_rn(yc);
                    __half* cp = reinterpret_cast<__half*>(es.C) + mr * es.ldc + n;
                    cp[0] = h;
                    cp[es.c_lo] = __float2half_rn(yc - __half2float(h));
                  } else reinterpret_cast<__nv_bfloat16*>(es.C)[mr * es.ldc + n] = __float2bfloat16(y);
                }
              }
            }
            __syncwarp();
          } else {
            // online log-sum-exp in the base-2 domain: one FFMA + one MUFU.EX2 per logit
            constexpr float L2E = 1.4426950408889634f;
            const int nv = (int)((N - n0) < 32 ? (N - n0) : 32);          // valid columns of this chunk (warp-uniform)
            if (want >= n0 && want < n0 + nv) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (n0 + j == want) el.picked[m] = v[j];
            }
            float m0 = run_max, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
            if (nv == 32) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                m0 = fmaxf(m0, v[j]); m1 = fmaxf(m1, v[j + 1]); m2 = fmaxf(m2, v[j + 2]); m3 = fmaxf(m3, v[j + 3]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < nv) m0 = fmaxf(m0, v[j]);
            }
            const float mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
            const float mxl = mx * L2E;
            float s0 = run_sum * fast_exp2(run_max * L2E - mxl), s1 = 0.f, s2 = 0.f, s3 = 0.f;
            if (nv == 32) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                s0 += fast_exp2(fmaf(v[j], L2E, -mxl)); s1 += fast_exp2(fmaf(v[j + 1], L2E, -mxl));
                s2 += fast_exp2(fmaf(v[j + 2], L2E, -mxl)); s3 += fast_exp2(fmaf(v[j + 3], L2E, -mxl));
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < nv) s0 += fast_exp2(fmaf(v[j], L2E, -mxl));
            }
            const float s = (s0 + s1) + (s2 + s3);
            run_max = mx;
            run_sum = s;
          }
        }
        if constexpr (LSE) {
          // two epilogue warps per TMEM lane quarter (lse_role 1 / 2: upper / lower half of the tile's columns) meet through
          // shared memory and a 64-thread named barrier; the lower-half warp merges and writes the tile's partial
          if (lse_role == 1) {
            *lse_slot = make_float2(run_max, run_sum);
            asm volatile("bar.sync %0, 64;" ::"r"(lse_bar) : "memory");
            return;
          }
          if (lse_role == 2) {
            asm volatile("bar.sync %0, 64;" ::"r"(lse_bar) : "memory");
            const float2 o = *lse_slot;
            const float mx = fmaxf(run_max, o.x);
            run_sum = mx > -INFINITY ? run_sum * __expf(run_max - mx) + o.y * __expf(o.x - mx) : 0.f;
            run_max = mx;
          }
          if (m < M) {
            el.part_max[m * el.n_tiles + n_blk] = run_max;
            el.part_sum[m * el.n_tiles + n_blk] = run_sum;
          }
        }
}

// ---------------------------------------------------------------------------------------------- 2-SM variant
// cta_group::2: the CTA pair of a cluster issues ONE tcgen05.mma of M = 256 (128 rows per SM), N = 256.  Each
// CTA stages its own 128-row A tile and HALF of the W tile (128 of the 256 W rows); the tensor cores read the
// peer's half over the SM-pair link.  Per CTA and k-block that is 16 KB (A) + 16 KB (W) instead of 16 + 32 KB:
// half the shared-memory operand bandwidth per MMA, half the L2 -> smem traffic for W, and 64 KB instead of
// 96 KB per 3xTF32 stage (3 stages instead of 2).  Only the even CTA (leader) issues MMAs; the peer's TMA
// loads, operand splitter and epilogue signal the leader's mbarriers through shared::cluster addresses.
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;            // clears the CTA-rank bit of a shared::cluster address

__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}
// TMA load whose complete_tx goes to the LEADER CTA's mbarrier (executed by both CTAs of the pair)
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar) {     // arrives on `bar` in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
template <int KIND_TF32>
__device__ __forceinline__ void umma_2sm(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  if constexpr (KIND_TF32) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

// K-major SWIZZLE_64B descriptor: 8-row groups are 512 B apart (SBO = 32), layout type 4
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (32ull << 32) | (1ull << 46) | (4ull << 61);
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

static int device_is_sm100() {
  static int cached = -1;
  if (cached < 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
      cudaGetLastError();
      cached = 0;
    } else {
      cached = major == 10;
    }
  }
  return cached;
}

}  // namespace tc

}  // namespace gnnlm
