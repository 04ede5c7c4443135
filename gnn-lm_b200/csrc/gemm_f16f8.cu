// fp32-parity GEMM in TWO tensor-pass equivalents (MATH_F16F8): C[m,n] = sum_k A[m,k] W[n,k] (+ bias).
//
// Replaces the three-pass 3xFP16 product for the large ntgt-side projections of the HGT layers
// (fairseq/models/hgt.py:320-322,347-348,401) and the OPQ rotation (knn/pq_wrapper.py:202).  With every fp32 operand
// split as x = hi + lo (hi = fp16(x), 11 significant bits; |lo| <= 2^-11 |x|):
//
//     a w  =  a_hi w_hi   +   a_hi w_lo  +  a_lo w_hi      (+ a_lo w_lo ~ 2^-22, dropped as in 3xFP16)
//             kind::f16       kind::f8f6f4 (e4m3 x e4m3), twice the fp16 rate
//
// the two correction products are 2^-11 of the result, so their operands only need a few bits: they are issued as FP8
// MMAs on e4m3 copies of the halves (a_hi8 = e4m3(a_hi), a_lo8 = e4m3(2^10 a_lo), w_lo8 = e4m3(w_lo), w_hi8 = e4m3(2^-10 w_hi);
// the power-of-two scales cancel inside each product), accumulating into the SAME fp32 TMEM accumulator as the fp16 main
// product.  Per-term error: 2^-11 (size of a correction) x 2^-4 (e4m3 rounding) x 2 operands ~ 2^-14 worst case -- measured
// on whole-path log-probs 4e-6 relative against the fp64 oracle (bar 1e-4), where a single fp16 / tf32 pass gives 7e-5..2.5e-4.
// Tensor time per k = 64: 4 fp16 instructions + 4 fp8 instructions of half the duration each... = 2/3 of the 3xFP16 form.
//
// The e4m3 copies of the activations are written by the PRODUCING kernels next to the split-fp16 halves (GNNLM_F16X2 buffer
// [rows, 2d] fp16 + companion [rows, 2d] bytes: hi8 | lo8), those of the weights once per checkpoint (gnnlm_quant_w8).
// A may be the concatenation along k of TWO row-aligned sources (k < K1 from A1, the rest from A2): the HGT output projection
// and the OPQ rotation of the residual are one product  [t | dec] [W_a | A^T]^T.
//
// Structure: as gemm_f16s_kernel (persistent, warp-specialised, cta_group::2 pairs, TMA producer / single-thread MMA issuer /
// four epilogue warps, double-buffered TMEM accumulators); a stage is one 64-wide k-block = 64 KB
// (fp16 tiles SWIZZLE_128B, e4m3 tiles SWIZZLE_64B), three stages.
#include <cuda_fp8.h>

#include "gemm_tc_common.cuh"

namespace gnnlm {

namespace tc {

constexpr int F8_BLOCK_K = 64;
constexpr int F8_A16 = BLOCK_M * 128;                     // 16 KB: fp16 hi tile, 128 B rows
constexpr int F8_B16 = (BLOCK_N / 2) * 128;               // 16 KB: this CTA's 128 W rows
constexpr int F8_A8 = BLOCK_M * 64;                       // 8 KB: e4m3 tile, 64 B rows
constexpr int F8_B8 = (BLOCK_N / 2) * 64;
constexpr int F8_STAGE = F8_A16 + F8_B16 + 2 * F8_A8 + 2 * F8_B8;      // 64 KB
constexpr int F8_STAGES = 3;

__device__ __forceinline__ void umma_2sm_f8(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}

struct F8Maps {
  CUtensorMap a1h, a1q_hi, a1q_lo;      // source 1: fp16 hi half, e4m3 hi8 / lo8
  CUtensorMap a2h, a2q_hi, a2q_lo;      // source 2 (k >= K1); copies of source 1 when there is none
  CUtensorMap wh, w8_lo, w8_hi;         // W fp16 hi (scaled), e4m3 lo8 / hi8
};

// Chain attention of the ntgt-intra-ntgt edges fused into the epilogue of the head-interleaved Q | K' | V' projection
// (gnnlm_linear_f16f8_nn_attn).  W rows are [Q_0 | K'_0 | Q_1 | K'_1 | ... | V'_0 .. V'_{H-1}] with d_k = 128, so N-tile h < H holds
// head h's Q and K' and N-tile H + j the V' of heads 2j, 2j + 1.  A CTA pair runs all 3H / 2 N-tiles of its two row windows in
// that order: the QK tiles leave the softmax weights alpha (3 per head: left / self / right chain neighbour) in registers, the V
// tiles mix the neighbours' V' rows and write the A-linear operand; Q | K' | V' never reach memory.
// Window j covers rows [j S - h, j S - h + 128) and owns [j S, j S + S), S = 128 - 2h, h = w - 1: a chain neighbour is at
// most h ids away, so every neighbour of an owned row is a lane of the same accumulator.
struct NnAttn {
  const int32_t* indptr;     // nn_indptr / nn_indices: [left,] self[, right] per row, in chain order
  const int32_t* indices;
  __half* out;               // [M, ld_out] fp16 hi of the attention output
  int64_t ld_out;
  uint8_t* q8;               // [M, ldq8] its e4m3 companion: hi8 at column c, lo8 at column d + c (no fp16 lo half)
  int64_t ldq8;
  int32_t* err;              // set to 1 when an owned row has a neighbour outside its window or more than three edges
  int halo;                  // h
  int heads;                 // H
};
constexpr int NN_BAR = 1;                                   // named barrier of the four epilogue warps (fused attention only)

__device__ __forceinline__ void nn_bar() { asm volatile("bar.sync %0, %1;" ::"r"(NN_BAR), "r"(4 * 32) : "memory"); }

// One window row per thread (TMEM lane L).  Per 32-column chunk every thread stages its K' (or V') row in the CTA-wide tile, and
// reads its neighbours' rows back: the rows of the warp's edges are other warps' lanes.  Rows a window does not own, and rows
// >= M, run the same instructions with themselves as their only neighbour and store nothing, so that every thread reaches every
// barrier equally often.  The arithmetic follows cluster_attn_kernel: same scores up to the summation order of the dot products,
// same softmax and mixing order.
template <class TileRC>
__device__ __forceinline__ void nn_attn_epilogue(uint32_t tmem_base, int64_t pair0, int64_t pair_stride, int64_t total, int64_t n_p,
                                                 int64_t M, int S, uint32_t crank, int q, const float* __restrict__ bias,
                                                 float acc_scale, const NnAttn& na, float* tile, uint64_t* tmem_full,
                                                 uint64_t* tmem_empty, TileRC tile_rc) {
  const int lane = threadIdx.x & 31;
  const int L = q * 32 + lane;
  const uint32_t my_row = smem_u32(tile + L * EPI_LD);
  const int H = na.heads, d = H * 128;
  float al[8], as[8], ar[8];                                // alpha of the left / self / right neighbour, per head
#pragma unroll
  for (int h = 0; h < 8; ++h) al[h] = as[h] = ar[h] = 0.f;
  int ll = L, lr = L;                                       // neighbour lanes (own lane: no such neighbour)
  bool own = false;
  int64_t g = 0;
  int64_t it = 0;
  for (int64_t t = pair0; t < total; t += pair_stride, ++it) {
    int64_t r, c;
    tile_rc(t, r, c);
    if (r >= n_p) break;
    if (c == 0) {                                           // first tile of a window
      const int64_t g0 = (r * 2 + crank) * S - na.halo;
      g = g0 + L;
      own = L >= na.halo && L < na.halo + S && g < M;
      ll = lr = L;
      if (own) {
        const int e0 = __ldg(na.indptr + g), deg = __ldg(na.indptr + g + 1) - e0;
        int64_t ml = g, mr = g;
        if (deg == 3) {
          ml = __ldg(na.indices + e0);
          mr = __ldg(na.indices + e0 + 2);
        } else if (deg == 2) {
          const int64_t a = __ldg(na.indices + e0);
          if (a == g) mr = __ldg(na.indices + e0 + 1);
          else ml = a;
        }
        const int64_t dl = ml - g0, dr = mr - g0;
        if (deg < 1 || deg > 3 || dl < 0 || dl >= BLOCK_M || dr < 0 || dr >= BLOCK_M) {
          *na.err = 1;
        } else {
          ll = (int)dl;
          lr = (int)dr;
        }
      }
    }
    const uint32_t rl = smem_u32(tile + ll * EPI_LD), rr = smem_u32(tile + lr * EPI_LD);
    const int acc = (int)(it & 1);
    const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
    mbar_wait(&tmem_full[acc], acc_phase);
    tc_fence_after();
    __syncwarp();                                           // the tcgen05.ld below are warp-collective
    const uint32_t taddr = tmem_base + (uint32_t)acc * BLOCK_N + ((uint32_t)(q * 32) << 16);
    const float* bt = bias + c * BLOCK_N;
    if (c < H) {                                            // head c: Q in columns [0, 128), K' in [128, 256)
      float s_l = 0.f, s_s = 0.f, s_r = 0.f;
#pragma unroll 1
      for (int cc = 0; cc < 128; cc += 32) {
        float qv[32], kv[32];
        tmem_ld32_issue(taddr + (uint32_t)cc, qv);
        tmem_ld32_issue(taddr + (uint32_t)(128 + cc), kv);
        tmem_ld_wait(qv);
        tmem_ld_wait(kv);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 bq = __ldg(reinterpret_cast<const float4*>(bt + cc + j));
          const float4 bk = __ldg(reinterpret_cast<const float4*>(bt + 128 + cc + j));
          qv[j] = fmaf(qv[j], acc_scale, bq.x); qv[j + 1] = fmaf(qv[j + 1], acc_scale, bq.y);
          qv[j + 2] = fmaf(qv[j + 2], acc_scale, bq.z); qv[j + 3] = fmaf(qv[j + 3], acc_scale, bq.w);
          kv[j] = fmaf(kv[j], acc_scale, bk.x); kv[j + 1] = fmaf(kv[j + 1], acc_scale, bk.y);
          kv[j + 2] = fmaf(kv[j + 2], acc_scale, bk.z); kv[j + 3] = fmaf(kv[j + 3], acc_scale, bk.w);
          sts128(my_row + 4 * j, kv[j], kv[j + 1], kv[j + 2], kv[j + 3]);
        }
        nn_bar();
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 a = lds128(rl + 4 * j), b = lds128(rr + 4 * j);
          s_s = fmaf(qv[j], kv[j], s_s); s_s = fmaf(qv[j + 1], kv[j + 1], s_s);
          s_s = fmaf(qv[j + 2], kv[j + 2], s_s); s_s = fmaf(qv[j + 3], kv[j + 3], s_s);
          s_l = fmaf(qv[j], a.x, s_l); s_l = fmaf(qv[j + 1], a.y, s_l); s_l = fmaf(qv[j + 2], a.z, s_l); s_l = fmaf(qv[j + 3], a.w, s_l);
          s_r = fmaf(qv[j], b.x, s_r); s_r = fmaf(qv[j + 1], b.y, s_r); s_r = fmaf(qv[j + 2], b.z, s_r); s_r = fmaf(qv[j + 3], b.w, s_r);
        }
        nn_bar();
      }
      if (ll == L) s_l = -INFINITY;
      if (lr == L) s_r = -INFINITY;
      const float mx = fmaxf(s_s, fmaxf(s_l, s_r));
      const float e0 = __expf(s_l - mx), e1 = __expf(s_s - mx), e2 = __expf(s_r - mx);
      const float inv = __fdividef(1.f, e0 + e1 + e2);
#pragma unroll
      for (int h = 0; h < 8; ++h)
        if (h == c) { al[h] = e0 * inv; as[h] = e1 * inv; ar[h] = e2 * inv; }
    } else {                                                // V' of heads 2 (c - H) and 2 (c - H) + 1
      const int64_t col0 = (c - H) * BLOCK_N;
#pragma unroll 1
      for (int cc = 0; cc < BLOCK_N; cc += 32) {
        const int hd = (int)(2 * (c - H)) + (cc >= 128 ? 1 : 0);
        float wl = 0.f, ws = 0.f, wr = 0.f;
#pragma unroll
        for (int h = 0; h < 8; ++h)
          if (h == hd) { wl = al[h]; ws = as[h]; wr = ar[h]; }
        float v[32];
        tmem_ld32(taddr + (uint32_t)cc, v);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 bv = __ldg(reinterpret_cast<const float4*>(bt + cc + j));
          v[j] = fmaf(v[j], acc_scale, bv.x); v[j + 1] = fmaf(v[j + 1], acc_scale, bv.y);
          v[j + 2] = fmaf(v[j + 2], acc_scale, bv.z); v[j + 3] = fmaf(v[j + 3], acc_scale, bv.w);
          sts128(my_row + 4 * j, v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
        nn_bar();
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 a = lds128(rl + 4 * j), b = lds128(rr + 4 * j);
          v[j] = fmaf(wr, b.x, fmaf(wl, a.x, ws * v[j]));
          v[j + 1] = fmaf(wr, b.y, fmaf(wl, a.y, ws * v[j + 1]));
          v[j + 2] = fmaf(wr, b.z, fmaf(wl, a.z, ws * v[j + 2]));
          v[j + 3] = fmaf(wr, b.w, fmaf(wl, a.w, ws * v[j + 3]));
        }
        nn_bar();
        if (own) {                                          // 64 B of fp16 hi + 2 x 32 B of e4m3: whole sectors per row
          uint32_t hi[16], h8[8], l8[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            uint2 h2, l2;
            split4_f16(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3], h2, l2);
            q8_from_split4(h2, l2, h8[i], l8[i]);
            hi[2 * i] = h2.x;
            hi[2 * i + 1] = h2.y;
          }
          uint4* op = reinterpret_cast<uint4*>(na.out + g * na.ld_out + col0 + cc);
          uint4* qh = reinterpret_cast<uint4*>(na.q8 + g * na.ldq8 + col0 + cc);
          uint4* ql = reinterpret_cast<uint4*>(na.q8 + g * na.ldq8 + d + col0 + cc);
#pragma unroll
          for (int i = 0; i < 4; ++i) op[i] = make_uint4(hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]);
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            qh[i] = make_uint4(h8[4 * i], h8[4 * i + 1], h8[4 * i + 2], h8[4 * i + 3]);
            ql[i] = make_uint4(l8[4 * i], l8[4 * i + 1], l8[4 * i + 2], l8[4 * i + 3]);
          }
        }
        __syncwarp();                                       // reconverge before the next chunk's tcgen05.ld and bar.sync
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
  }
}

template <bool NN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(256, 1)
    gemm_f16f8_kernel(const __grid_constant__ F8Maps maps, int64_t M_cap, const int32_t* __restrict__ m_dev, int64_t N, int64_t K,
                      int kb_split, EpiStore es, float acc_scale, int dbg, long long* __restrict__ dbg_out, NnAttn na) {
  constexpr int STAGES = F8_STAGES;
  constexpr uint32_t TX = 2u * F8_STAGE;                                  // both CTAs' six operand tiles -> leader
  const int n_mma = N <= BLOCK_N / 2 ? BLOCK_N / 2 : BLOCK_N;
  // c_format f32 | a_format / b_format 0 (F16 for kind::f16, E4M3 for kind::f8f6f4) | K-major both | N >> 3 | M >> 4
  const uint32_t IDESC = (1u << 4) | ((uint32_t)(n_mma >> 3) << 17) | ((uint32_t)((2 * BLOCK_M) >> 4) << 24);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* epi_smem = reinterpret_cast<float*>(smem + (size_t)STAGES * F8_STAGE);
  __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_base_s;
  constexpr int EPI_WARPS = 4;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int64_t M = live_rows(M_cap, m_dev);
  const int64_t pair0 = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;
  // NN: row blocks are windows of S owned rows, and a pair takes all n_n N-tiles of its windows before moving on
  const int S = NN ? BLOCK_M - 2 * na.halo : BLOCK_M;
  const int64_t n_m = (M + S - 1) / S, n_n = (N + BLOCK_N - 1) / BLOCK_N;
  const int64_t n_p = (n_m + 1) / 2;
  const int64_t total = NN ? (n_p + pair_stride - 1) / pair_stride * pair_stride * n_n : n_p * n_n;
  // (pair row block r, N-tile c) of a tile index; every role walks the same sequence and stops at r >= n_p
  auto tile_rc = [&](int64_t tile, int64_t& r, int64_t& c) {
    if (NN) {
      const int64_t k = tile / pair_stride;
      r = tile % pair_stride + k / n_n * pair_stride;
      c = k % n_n;
    } else {
      r = tile / n_n;
      c = tile % n_n;
    }
  };
  auto row0 = [&](int64_t r) { return (r * 2 + crank) * S - (NN ? na.halo : 0); };     // first A row of this CTA's block
  const int n_kb = (int)((K + F8_BLOCK_K - 1) / F8_BLOCK_K);

  auto sAh = [&](int s) { return smem + (size_t)s * F8_STAGE; };
  auto sBh = [&](int s) { return smem + (size_t)s * F8_STAGE + F8_A16; };
  auto sA8h = [&](int s) { return smem + (size_t)s * F8_STAGE + F8_A16 + F8_B16; };
  auto sA8l = [&](int s) { return smem + (size_t)s * F8_STAGE + F8_A16 + F8_B16 + F8_A8; };
  auto sB8l = [&](int s) { return smem + (size_t)s * F8_STAGE + F8_A16 + F8_B16 + 2 * F8_A8; };
  auto sB8h = [&](int s) { return smem + (size_t)s * F8_STAGE + F8_A16 + F8_B16 + 2 * F8_A8 + F8_B8; };

  if (warp == 0 && lane == 0) {
    const CUtensorMap* m = &maps.a1h;
#pragma unroll
    for (int i = 0; i < 9; ++i) asm volatile("prefetch.tensormap [%0];" ::"l"(m + i) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 2 * EPI_WARPS);
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
      long long t_wait = 0;
      for (int64_t tile = pair0; tile < total; tile += pair_stride) {
        int64_t r, c;
        tile_rc(tile, r, c);
        if (r >= n_p) break;
        const int m0 = (int)row0(r), n0 = (int)(c * BLOCK_N) + half;      // NN, window 0: m0 = -h, zero-filled by TMA
        for (int kb = 0; kb < n_kb; ++kb) {
          const long long t0 = dbg_out ? clock64() : 0;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (dbg_out) t_wait += clock64() - t0;
          if (leader) mbar_expect_tx(&full_bar[stage], TX);
          const bool first = kb < kb_split;
          const int ka = (first ? kb : kb - kb_split) * F8_BLOCK_K, kw = kb * F8_BLOCK_K;
          tma_load_2d_2sm(sAh(stage), first ? &maps.a1h : &maps.a2h, ka, m0, &full_bar[stage]);
          tma_load_2d_2sm(sBh(stage), &maps.wh, kw, n0, &full_bar[stage]);
          tma_load_2d_2sm(sA8h(stage), first ? &maps.a1q_hi : &maps.a2q_hi, ka, m0, &full_bar[stage]);
          tma_load_2d_2sm(sB8l(stage), &maps.w8_lo, kw, n0, &full_bar[stage]);
          tma_load_2d_2sm(sA8l(stage), first ? &maps.a1q_lo : &maps.a2q_lo, ka, m0, &full_bar[stage]);
          tma_load_2d_2sm(sB8h(stage), &maps.w8_hi, kw, n0, &full_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
      if (dbg_out) dbg_out[blockIdx.x * 8 + 0] = t_wait;
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {                         // ---- MMA issuer (leader only)
      int stage = 0;
      uint32_t phase = 0;
      int64_t it = 0;
      long long t_empty = 0, t_full = 0;
      const long long t_begin = dbg_out ? clock64() : 0;
      for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
        if (NN) {
          int64_t r, c;
          tile_rc(tile, r, c);
          if (r >= n_p) break;
        }
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        const long long te0 = dbg_out ? clock64() : 0;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        if (dbg_out) t_empty += clock64() - te0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * BLOCK_N;
        for (int kb = 0; kb < n_kb; ++kb) {
          const long long tf0 = dbg_out ? clock64() : 0;
          mbar_wait(&full_bar[stage], phase);
          if (dbg_out) t_full += clock64() - tf0;
          tc_fence_after();
          const uint64_t dah = make_desc(smem_u32(sAh(stage))), dbh = make_desc(smem_u32(sBh(stage)));
          const uint64_t da8h = make_desc_sw64(smem_u32(sA8h(stage))), da8l = make_desc_sw64(smem_u32(sA8l(stage)));
          const uint64_t db8l = make_desc_sw64(smem_u32(sB8l(stage))), db8h = make_desc_sw64(smem_u32(sB8h(stage)));
#pragma unroll
          for (int k = 0; k < F8_BLOCK_K / 32; ++k) {            // 32 B of k per instruction: 16 halves or 32 e4m3 bytes
            const uint64_t k16 = (uint64_t)(k * 4), k8 = (uint64_t)(k * 2);
            if (!(dbg & 1)) {                                      // (timing experiments: GNNLM_F8_DEBUG bits 0 / 1 drop a product)
              umma_2sm_f8(d_tmem, da8h + k8, db8l + k8, IDESC, (kb | k) > 0 ? 1u : 0u);
              umma_2sm_f8(d_tmem, da8l + k8, db8h + k8, IDESC, 1u);
            }
            if (!(dbg & 2)) {
              umma_2sm<0>(d_tmem, dah + k16, dbh + k16, IDESC, ((kb | k) > 0 || !(dbg & 1)) ? 1u : 0u);
              umma_2sm<0>(d_tmem, dah + k16 + 2, dbh + k16 + 2, IDESC, 1u);
            }
          }
          tc_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        tc_commit_2sm(&tmem_full[acc]);
      }
      if (dbg_out) {
        dbg_out[blockIdx.x * 8 + 1] = t_empty;
        dbg_out[blockIdx.x * 8 + 2] = t_full;
        dbg_out[blockIdx.x * 8 + 3] = clock64() - t_begin;
      }
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + EPI_WARPS) {
    const int q = warp & 3;                            // ---- epilogue (both CTAs)
    if constexpr (NN) {
      nn_attn_epilogue(tmem_base, pair0, pair_stride, total, n_p, M, S, crank, q, es.bias, acc_scale, na, epi_smem,
                       tmem_full, tmem_empty, tile_rc);
    } else {
    int64_t it = 0;
    EpiLse el{};
    long long t_epi_wait = 0, t_epi_work = 0;
    for (int64_t tile = pair0; tile < total; tile += pair_stride, ++it) {
      const int acc = (int)(it & 1);
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      const int64_t r = tile / n_n, n_blk = tile % n_n;
      const int64_t m_blk = r * 2 + crank;
      const int64_t m = m_blk * BLOCK_M + q * 32 + lane;
      const long long tw0 = dbg_out ? clock64() : 0;
      mbar_wait(&tmem_full[acc], acc_phase);
      const long long tw1 = dbg_out ? clock64() : 0;
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * BLOCK_N + ((uint32_t)(q * 32) << 16);
      if (!(dbg & 4)) epilogue_tile<false>(taddr, m, M, n_blk * BLOCK_N, n_blk, N, es, el, epi_smem + q * 32 * EPI_LD, acc_scale);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
      if (dbg_out) { t_epi_wait += tw1 - tw0; t_epi_work += clock64() - tw1; }
    }
    if (dbg_out && lane == 0) {
      dbg_out[blockIdx.x * 8 + 4 + (q & 1) * 2] = t_epi_wait;       // warps 0 / 1 of the four (2 / 3 overwrite: same order of magnitude)
      dbg_out[blockIdx.x * 8 + 5 + (q & 1) * 2] = t_epi_work;
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

// [rows, K] K-major matrix of `elem`-byte elements, boxes of 64 elements x box_rows (fp16: SWIZZLE_128B, bytes: SWIZZLE_64B)
static int make_map_k64(CUtensorMap* map, const void* base, int elem, int64_t rows, int64_t K, int64_t ld_bytes, int box_rows) {
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld_bytes};
  cuuint32_t box[2] = {(cuuint32_t)F8_BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return (int)encode_fn()(map, elem == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2,
                          const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          elem == 2 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// ---------------------------------------------------------------------------------------------- e4m3 companions
__device__ __forceinline__ uint16_t e4m3x2(__half2 v) {
  return (uint16_t)__nv_cvt_halfraw2_to_fp8x2(*reinterpret_cast<__half2_raw*>(&v), __NV_SATFINITE, __NV_E4M3);
}

// split fp16 [rows, hi | lo] -> bytes [rows, hi8 | lo8] (hi8 = e4m3(hi), lo8 = e4m3(2^10 lo)); 8 elements per thread
__global__ void __launch_bounds__(256) split_to_q8_kernel(const __half* __restrict__ x, int64_t ldx, uint8_t* __restrict__ q,
                                                           int64_t ldq, int64_t rows_cap, const int32_t* __restrict__ rows_dev,
                                                           int64_t d) {
  const int64_t rows = live_rows(rows_cap, rows_dev);
  const int64_t per_row = d / 8;
  const __half2 s = __floats2half2_rn(1024.f, 1024.f);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * per_row; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per_row, c = (i % per_row) * 8;
    const uint4 hi = __ldg(reinterpret_cast<const uint4*>(x + r * ldx + c));
    const uint4 lo = __ldg(reinterpret_cast<const uint4*>(x + r * ldx + d + c));
    const __half2* h = reinterpret_cast<const __half2*>(&hi);
    const __half2* l = reinterpret_cast<const __half2*>(&lo);
    uint2 oh, ol;
    oh.x = e4m3x2(h[0]) | ((uint32_t)e4m3x2(h[1]) << 16);
    oh.y = e4m3x2(h[2]) | ((uint32_t)e4m3x2(h[3]) << 16);
    ol.x = e4m3x2(__hmul2(l[0], s)) | ((uint32_t)e4m3x2(__hmul2(l[1], s)) << 16);
    ol.y = e4m3x2(__hmul2(l[2], s)) | ((uint32_t)e4m3x2(__hmul2(l[3], s)) << 16);
    *reinterpret_cast<uint2*>(q + r * ldq + c) = oh;
    *reinterpret_cast<uint2*>(q + r * ldq + d + c) = ol;
  }
}

// weights: (hi, lo) fp16 [N, K] (already scaled, gnnlm_split_f16) -> bytes [N, lo8 | hi8]: lo8 = e4m3(lo), hi8 = e4m3(2^-10 hi)
__global__ void __launch_bounds__(256) quant_w8_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, int64_t ldw,
                                                        uint8_t* __restrict__ q, int64_t ldq, int64_t N, int64_t K) {
  const int64_t per_row = K / 2;
  const __half2 s = __floats2half2_rn(1.f / 1024.f, 1.f / 1024.f);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N * per_row; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per_row, c = (i % per_row) * 2;
    const __half2 h = *reinterpret_cast<const __half2*>(hi + r * ldw + c);
    const __half2 l = *reinterpret_cast<const __half2*>(lo + r * ldw + c);
    *reinterpret_cast<uint16_t*>(q + r * ldq + c) = e4m3x2(l);
    *reinterpret_cast<uint16_t*>(q + r * ldq + K + c) = e4m3x2(__hmul2(h, s));
  }
}

}  // namespace tc

int32_t gemm_tc_supported();

}  // namespace gnnlm

using namespace gnnlm;

extern "C" int32_t gnnlm_split_to_q8(const void* x, int64_t ldx, void* q, int64_t ldq, int64_t rows, const int32_t* rows_dev,
                                     int64_t d, cudaStream_t stream) {
  GNNLM_CHECK_ARG(x && q && rows >= 0 && d > 0, GNNLM_E_ARG, "gnnlm_split_to_q8: null pointer / bad sizes");
  GNNLM_CHECK_ARG(d % 8 == 0 && ldx >= 2 * d && ldq >= 2 * d && ldx % 8 == 0 && ldq % 8 == 0 && (uintptr_t)x % 16 == 0 &&
                      (uintptr_t)q % 8 == 0,
                  GNNLM_E_SHAPE, "gnnlm_split_to_q8: d, ldx, ldq must be multiples of 8 with 16 B aligned rows");
  if (rows == 0) return 0;
  const int64_t work = rows * (d / 8);
  const unsigned grid = (unsigned)(work / 256 + 1 < 148 * 16 ? work / 256 + 1 : 148 * 16);
  tc::split_to_q8_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const __half*>(x), ldx, reinterpret_cast<uint8_t*>(q), ldq, rows,
                                                   rows_dev, d);
  GNNLM_LAUNCH_CHECK("gnnlm_split_to_q8");
  return 0;
}

extern "C" int32_t gnnlm_quant_w8(const void* w_hi, const void* w_lo, int64_t ldw, void* q, int64_t ldq, int64_t N, int64_t K,
                                  cudaStream_t stream) {
  GNNLM_CHECK_ARG(w_hi && w_lo && q && N > 0 && K > 0, GNNLM_E_ARG, "gnnlm_quant_w8: null pointer / bad sizes");
  GNNLM_CHECK_ARG(K % 2 == 0 && ldw % 2 == 0 && ldq >= 2 * K && ldq % 2 == 0 && (uintptr_t)w_hi % 4 == 0 && (uintptr_t)w_lo % 4 == 0 &&
                      (uintptr_t)q % 2 == 0,
                  GNNLM_E_SHAPE, "gnnlm_quant_w8: K, ldw, ldq must be even");
  const int64_t work = N * (K / 2);
  const unsigned grid = (unsigned)(work / 256 + 1 < 148 * 16 ? work / 256 + 1 : 148 * 16);
  tc::quant_w8_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const __half*>(w_hi), reinterpret_cast<const __half*>(w_lo), ldw,
                                                reinterpret_cast<uint8_t*>(q), ldq, N, K);
  GNNLM_LAUNCH_CHECK("gnnlm_quant_w8");
  return 0;
}

// operand checks and tensor maps shared by gnnlm_linear_f16f8 and gnnlm_linear_f16f8_nn_attn
static int32_t f8_maps(const char* who, tc::F8Maps& maps, const void* A1, const void* A1q, int64_t lda1, int64_t ldq1, int64_t K1,
                       const void* A2, const void* A2q, int64_t lda2, int64_t ldq2, int64_t K2, const void* W_hi, const void* W8,
                       int64_t ldw, int64_t ldw8, int64_t M, int64_t N) {
  GNNLM_CHECK_ARG(gemm_tc_supported(), GNNLM_E_UNSUPPORTED, "%s: needs an sm_100 device and driver TMA support", who);
  const int64_t K = K1 + K2;
  // k-blocks of 64 must not straddle the two sources; e4m3 halves sit K1 (resp. K2, K) bytes apart inside their rows
  GNNLM_CHECK_ARG(K1 % tc::F8_BLOCK_K == 0 && K2 % 16 == 0 && K1 % 16 == 0 && lda1 >= K1 && ldq1 >= 2 * K1 && ldw >= K &&
                      ldw8 >= 2 * K && (K2 == 0 || (lda2 >= K2 && ldq2 >= 2 * K2)),
                  GNNLM_E_SHAPE, "%s: K1 must be a multiple of 64, K1 / K2 multiples of 16 (K1=%lld K2=%lld)",
                  who, (long long)K1, (long long)K2);
  GNNLM_CHECK_ARG((lda1 * 2) % 16 == 0 && ldq1 % 16 == 0 && (ldw * 2) % 16 == 0 && ldw8 % 16 == 0 && (uintptr_t)A1 % 16 == 0 &&
                      (uintptr_t)A1q % 16 == 0 && (uintptr_t)W_hi % 16 == 0 && (uintptr_t)W8 % 16 == 0 &&
                      (K2 == 0 || ((lda2 * 2) % 16 == 0 && ldq2 % 16 == 0 && (uintptr_t)A2 % 16 == 0 && (uintptr_t)A2q % 16 == 0)),
                  GNNLM_E_SHAPE, "%s: TMA needs 16 B aligned bases and row strides", who);
  if (M == 0) return 0;
  const uint8_t* a1q = reinterpret_cast<const uint8_t*>(A1q);
  const uint8_t* w8 = reinterpret_cast<const uint8_t*>(W8);
  int r = tc::make_map_k64(&maps.a1h, A1, 2, M, K1, lda1 * 2, tc::BLOCK_M);
  if (!r) r = tc::make_map_k64(&maps.a1q_hi, a1q, 1, M, K1, ldq1, tc::BLOCK_M);
  if (!r) r = tc::make_map_k64(&maps.a1q_lo, a1q + K1, 1, M, K1, ldq1, tc::BLOCK_M);
  if (K2 > 0) {
    const uint8_t* a2q = reinterpret_cast<const uint8_t*>(A2q);
    if (!r) r = tc::make_map_k64(&maps.a2h, A2, 2, M, K2, lda2 * 2, tc::BLOCK_M);
    if (!r) r = tc::make_map_k64(&maps.a2q_hi, a2q, 1, M, K2, ldq2, tc::BLOCK_M);
    if (!r) r = tc::make_map_k64(&maps.a2q_lo, a2q + K2, 1, M, K2, ldq2, tc::BLOCK_M);
  } else {
    maps.a2h = maps.a1h;
    maps.a2q_hi = maps.a1q_hi;
    maps.a2q_lo = maps.a1q_lo;
  }
  if (!r) r = tc::make_map_k64(&maps.wh, W_hi, 2, N, K, ldw * 2, tc::BLOCK_N / 2);
  if (!r) r = tc::make_map_k64(&maps.w8_lo, w8, 1, N, K, ldw8, tc::BLOCK_N / 2);
  if (!r) r = tc::make_map_k64(&maps.w8_hi, w8 + K, 1, N, K, ldw8, tc::BLOCK_N / 2);
  GNNLM_CHECK_ARG(r == 0, GNNLM_E_ARG, "%s: cuTensorMapEncodeTiled failed (%d)", who, r);
  return 0;
}

extern "C" int32_t gnnlm_linear_f16f8(const void* A1, const void* A1q, int64_t lda1, int64_t ldq1, int64_t K1, const void* A2,
                                      const void* A2q, int64_t lda2, int64_t ldq2, int64_t K2, const void* W_hi, const void* W8,
                                      float w_scale, int64_t ldw, int64_t ldw8, const float* bias, void* C, int32_t c_dtype,
                                      int64_t ldc, int64_t M, const int32_t* m_dev, int64_t N, void* C8, cudaStream_t stream) {
  GNNLM_CHECK_ARG(A1 && A1q && W_hi && W8 && C && M >= 0 && N > 0 && K1 > 0 && K2 >= 0 && w_scale > 0.f, GNNLM_E_ARG,
                  "gnnlm_linear_f16f8: null pointer / bad sizes");
  GNNLM_CHECK_ARG(K2 == 0 || (A2 && A2q), GNNLM_E_ARG, "gnnlm_linear_f16f8: K2 > 0 needs the second source");
  GNNLM_CHECK_ARG(c_dtype == GNNLM_F32 || c_dtype == GNNLM_BF16 || c_dtype == GNNLM_F16X2 || c_dtype == GNNLM_F24, GNNLM_E_ARG,
                  "gnnlm_linear_f16f8: output dtype must be f32 / bf16 / split fp16 / f24");
  GNNLM_CHECK_ARG(c_dtype != GNNLM_F24 || (C8 && N % 4 == 0 && ldc % 4 == 0 && (uintptr_t)C % 16 == 0 && (uintptr_t)C8 % 4 == 0),
                  GNNLM_E_SHAPE, "gnnlm_linear_f16f8: GNNLM_F24 output needs the byte plane, N and ldc multiples of 4, aligned bases");
  tc::F8Maps maps;
  if (int32_t rc = f8_maps("gnnlm_linear_f16f8", maps, A1, A1q, lda1, ldq1, K1, A2, A2q, lda2, ldq2, K2, W_hi, W8, ldw, ldw8, M, N))
    return rc;
  if (M == 0) return 0;
  const int64_t K = K1 + K2;

  tc::EpiStore es{bias, nullptr, 0, C, ldc, c_dtype == GNNLM_BF16 ? 1 : (c_dtype == GNNLM_F16X2 ? 2 : (c_dtype == GNNLM_F24 ? 3 : 0)), 0, N, N};
  es.C8 = reinterpret_cast<uint8_t*>(C8);
  const size_t smem = (size_t)tc::F8_STAGES * tc::F8_STAGE + tc::EPI_SMEM + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    GNNLM_CUDA(cudaFuncSetAttribute(tc::gemm_f16f8_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    GNNLM_CUDA(cudaGetDevice(&dev));
    GNNLM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  const int64_t pairs = ceil_div(ceil_div(M, tc::BLOCK_M), 2) * ceil_div(N, tc::BLOCK_N);
  static int pair_cap = -1;
  if (pair_cap < 0) { const char* e = getenv("GNNLM_F8_MAXPAIRS"); pair_cap = e ? atoi(e) : 0; }   // timing experiments only
  const int64_t max_pairs = pair_cap > 0 && pair_cap < n_sm / 2 ? pair_cap : n_sm / 2;
  const unsigned grid = 2u * (unsigned)(pairs < max_pairs ? pairs : max_pairs);
  static int dbg = -1;
  if (dbg < 0) { const char* e = getenv("GNNLM_F8_DEBUG"); dbg = e ? atoi(e) : 0; }          // timing experiments only
  es.dbg = (dbg >> 3) & 3;
  long long* dbg_out = nullptr;
  if (dbg & 32) {                                    // per-role wait cycles (timing experiments only; synchronises)
    static long long* buf = nullptr;
    if (!buf) GNNLM_CUDA(cudaMalloc(&buf, 148 * 8 * sizeof(long long)));
    GNNLM_CUDA(cudaMemsetAsync(buf, 0, 148 * 8 * sizeof(long long), stream));
    dbg_out = buf;
  }
  tc::gemm_f16f8_kernel<false><<<grid, 256, smem, stream>>>(maps, M, m_dev, N, K, (int)(K1 / tc::F8_BLOCK_K), es, 1.f / w_scale, dbg,
                                                           dbg_out, tc::NnAttn{});
  GNNLM_LAUNCH_CHECK("gnnlm_linear_f16f8");
  if (dbg_out) {
    static long long host[148 * 8];
    GNNLM_CUDA(cudaStreamSynchronize(stream));
    GNNLM_CUDA(cudaMemcpy(host, dbg_out, sizeof(host), cudaMemcpyDeviceToHost));
    double acc[8] = {0};
    int n_lead = 0;
    for (unsigned b = 0; b < grid; ++b) {
      acc[0] += (double)host[b * 8];
      for (int i = 4; i < 8; ++i) acc[i] += (double)host[b * 8 + i];
      if (b % 2 == 0) { for (int i = 1; i < 4; ++i) acc[i] += (double)host[b * 8 + i]; ++n_lead; }
    }
    fprintf(stderr, "f16f8 M=%lld N=%lld K=%lld cycles: issuer total %.0f, wait tmem_empty %.0f, wait full %.0f | producer wait empty %.0f | "
            "epi warp0 wait %.0f work %.0f, warp1 wait %.0f work %.0f\n", (long long)M, (long long)N, (long long)K, acc[3] / n_lead,
            acc[1] / n_lead, acc[2] / n_lead, acc[0] / grid, acc[4] / grid, acc[5] / grid, acc[6] / grid, acc[7] / grid);
  }
  return 0;
}

extern "C" int32_t gnnlm_linear_f16f8_nn_attn(const void* A, const void* Aq, int64_t lda, int64_t ldq, int64_t K, const void* W_hi,
                                              const void* W8, float w_scale, int64_t ldw, int64_t ldw8, const float* bias,
                                              const int32_t* nn_indptr, const int32_t* nn_indices, int32_t max_cluster, int32_t H,
                                              void* out, int64_t ldo, void* q8, int64_t ldq8, int32_t* err, int64_t M,
                                              const int32_t* m_dev, cudaStream_t stream) {
  GNNLM_CHECK_ARG(A && Aq && W_hi && W8 && bias && nn_indptr && nn_indices && out && q8 && err && M >= 0 && K > 0 && w_scale > 0.f,
                  GNNLM_E_ARG, "gnnlm_linear_f16f8_nn_attn: null pointer / bad sizes");
  GNNLM_CHECK_ARG((max_cluster == 1 || max_cluster == 3 || max_cluster == 5 || max_cluster == 7) && H >= 2 && H <= 8 && H % 2 == 0,
                  GNNLM_E_UNSUPPORTED, "gnnlm_linear_f16f8_nn_attn: needs clusters of 1, 3, 5 or 7 nodes and an even H <= 8 (w=%d, H=%d)",
                  max_cluster, H);
  const int64_t d = (int64_t)H * 128, N = 3 * d;
  GNNLM_CHECK_ARG(ldo >= d && ldo % 8 == 0 && ldq8 >= 2 * d && ldq8 % 16 == 0 && (uintptr_t)out % 16 == 0 && (uintptr_t)q8 % 16 == 0 &&
                      (uintptr_t)bias % 16 == 0,
                  GNNLM_E_SHAPE, "gnnlm_linear_f16f8_nn_attn: output rows / bias must be 16 B aligned, ldo >= d, ldq8 >= 2d");
  tc::F8Maps maps;
  if (int32_t rc = f8_maps("gnnlm_linear_f16f8_nn_attn", maps, A, Aq, lda, ldq, K, nullptr, nullptr, 0, 0, 0, W_hi, W8, ldw, ldw8, M, N))
    return rc;
  if (M == 0) return 0;
  const int halo = max_cluster - 1, S = tc::BLOCK_M - 2 * halo;
  tc::NnAttn na{nn_indptr, nn_indices, reinterpret_cast<__half*>(out), ldo, reinterpret_cast<uint8_t*>(q8), ldq8, err, halo, H};
  tc::EpiStore es{bias, nullptr, 0, nullptr, 0, 0, 0, 0, 0};
  const size_t smem = (size_t)tc::F8_STAGES * tc::F8_STAGE + tc::EPI_SMEM + 1024;
  static bool attr_set[MAX_DEVICES] = {false};
  const int slot = device_slot();
  if (!attr_set[slot]) {
    GNNLM_CUDA(cudaFuncSetAttribute(tc::gemm_f16f8_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[slot] = true;
  }
  int dev = 0, n_sm = 0;
  GNNLM_CUDA(cudaGetDevice(&dev));
  GNNLM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  const int64_t pairs = ceil_div(ceil_div(M, S), 2);        // window pairs at capacity; the kernel walks those of the live M
  const unsigned grid = 2u * (unsigned)(pairs < n_sm / 2 ? pairs : n_sm / 2);
  tc::gemm_f16f8_kernel<true><<<grid, 256, smem, stream>>>(maps, M, m_dev, N, K, (int)(K / tc::F8_BLOCK_K), es, 1.f / w_scale, 0, nullptr,
                                                          na);
  GNNLM_LAUNCH_CHECK("gnnlm_linear_f16f8_nn_attn");
  return 0;
}
