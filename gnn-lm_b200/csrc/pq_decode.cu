// Datastore gather + product-quantisation decode.
//
// Replaces `quant_neighbor_feats[offset]` / `neighbor_tokens[offset]` of new_build_graph
// (reference: fairseq/data/token_block_dataset.py:369-371,392-394) and the centroid gather of
// TorchPQCodec.decode (knn/pq_wrapper.py:169-196; `x -= b` of :200-201 fused).  The OPQ rotation
// `x @ A` (:202) is a GEMM and lives in gemm_*.cu.
//
// Layout / roofline.  HBM-bound byte work: per node M code bytes are read (one 128 B line at
// M=128) and M*dsub*4 B (4 KB at d=1024) are written.  The codebook [M,256,dsub] fp32 (1 MB at
// d=1024) does not fit in shared memory, so the grid is 2-D: blockIdx.x (fastest, so that the CTAs
// writing the pieces of one output row are resident together and the row's lines fill up in L2 within a short
// window) picks a chunk of MC subspaces whose centroids (MC*256*dsub*4 B = 128 KB) are staged ONCE per CTA into shared memory
// with TMA bulk copies (cp.async.bulk + mbarrier expect_tx), and the CTA then streams over many
// nodes: each warp takes one node at a time, each lane owns 4 consecutive output floats
// (one float4 smem read indexed by the code byte, one coalesced 16 B global store; a warp writes
// 512 contiguous bytes).  Code bytes are read with one 32-bit load per 4 subspaces.
#include <type_traits>

#include "common.cuh"

namespace gnnlm {

constexpr int PQ_THREADS = 1024;    // 32 warps x 8 nodes in flight: the kernel is latency-bound, not ALU-bound
constexpr int PQ_CHUNK_FLOATS = 128;     // output floats per node per chunk == 32 lanes * float4
constexpr int PQ_NODES_PER_CTA = 4096;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(phase)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <typename OutT>
__device__ __forceinline__ void store4(OutT* p, float4 v, int lo_off = 0);
template <>
__device__ __forceinline__ void store4<float>(float* p, float4 v, int) {
  *reinterpret_cast<float4*>(p) = v;
}
template <>
__device__ __forceinline__ void store4<__half>(__half* p, float4 v, int lo_off) {       // split-fp16: hi | lo
  uint2 hi, lo;
  split4_f16(v.x, v.y, v.z, v.w, hi, lo);
  *reinterpret_cast<uint2*>(p) = hi;
  *reinterpret_cast<uint2*>(p + lo_off) = lo;
}
template <>
__device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16* p, float4 v, int) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}

// dsub % 4 == 0 path.  MC subspaces per chunk, MC * dsub == chunk_floats <= 128.
template <typename OutT>
__global__ void __launch_bounds__(PQ_THREADS, 1)
    pq_decode_smem_kernel(const uint8_t* __restrict__ codes, int M, const float* __restrict__ centroids, int dsub,
                          const float* __restrict__ bias, const int64_t* __restrict__ rows,
                          const int32_t* __restrict__ row_ids, int64_t n_cap, const int32_t* __restrict__ n_dev,
                          OutT* __restrict__ out, int64_t ld_out, int mc, int nodes_per_cta) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  float* cb = reinterpret_cast<float*>(smem_raw);                   // [mc][256][dsub]
  __shared__ __align__(8) uint64_t bar;

  const int64_t n = live_rows(n_cap, n_dev);
  const int64_t node0 = (int64_t)blockIdx.y * nodes_per_cta;
  if (node0 >= n) return;
  const int m0 = blockIdx.x * mc;
  const int mc_here = min(mc, M - m0);
  const uint32_t chunk_bytes = (uint32_t)mc_here * 256u * (uint32_t)dsub * 4u;

  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar, chunk_bytes);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(centroids + (size_t)m0 * 256 * dsub);
    for (uint32_t off = 0; off < chunk_bytes; off += 32768u) {
      uint32_t sz = min(32768u, chunk_bytes - off);
      bulk_g2s(smem_raw + off, src + off, sz, &bar);
    }
  }
  mbar_wait(&bar, 0);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int f4_per_sub = dsub >> 2;                                  // float4 per centroid
  const int n_f4 = mc_here * f4_per_sub;                             // float4 per node in this chunk (<= 32)
  const int sub = lane / f4_per_sub, part = lane % f4_per_sub;       // lane -> (subspace, float4 within)
  const bool active = lane < n_f4;
  float4 bsub = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias && active) bsub = __ldg(reinterpret_cast<const float4*>(bias + (size_t)(m0 + sub) * dsub) + part);
  const int64_t node_end = min(n, node0 + nodes_per_cta);
  const float4* cb4 = reinterpret_cast<const float4*>(cb);

  // PQ_INFLIGHT nodes in flight per warp per iteration to overlap the dependent (row -> code -> centroid)
  // chain: the kernel is latency-bound otherwise
  constexpr int PQ_INFLIGHT = 8;
  for (int64_t i = node0 + warp * PQ_INFLIGHT; i < node_end; i += (PQ_THREADS / 32) * PQ_INFLIGHT) {
    int64_t r[PQ_INFLIGHT];
    uint32_t c[PQ_INFLIGHT];
#pragma unroll
    for (int u = 0; u < PQ_INFLIGHT; ++u) {
      int64_t node = i + u;
      bool ok = node < node_end;
      int64_t nid = ok ? (row_ids ? (int64_t)__ldg(row_ids + node) : node) : 0;
      r[u] = ok ? __ldg(rows + nid) : -1;
    }
#pragma unroll
    for (int u = 0; u < PQ_INFLIGHT; ++u)
      c[u] = (r[u] >= 0 && active) ? (uint32_t)__ldg(codes + (size_t)r[u] * M + m0 + sub) : 0u;
#pragma unroll
    for (int u = 0; u < PQ_INFLIGHT; ++u) {
      if (r[u] >= 0 && active) {
        float4 v = cb4[((size_t)sub * 256 + c[u]) * f4_per_sub + part];
        v.x -= bsub.x; v.y -= bsub.y; v.z -= bsub.z; v.w -= bsub.w;
        store4<OutT>(out + (size_t)(i + u) * ld_out + (size_t)(m0 + sub) * dsub + part * 4, v, M * dsub);
      }
    }
  }
}

// Split-fp16 output from a codebook that is ALREADY split (hi / lo fp16 halves of `centroid - bias`, prepared once per
// quantizer): with dsub == 8 a centroid is one 16 B quad per half, so a lane moves one (node, subspace) pair with two 16 B
// shared-memory reads and two 16 B global stores and no arithmetic at all -- the fp32 form above spends ~25 instructions
// per 16 B on the split and was issue-bound at 60 % of the HBM roofline.  16 subspaces per chunk (64 KB hi + 64 KB lo in
// shared memory): a half-warp owns a node, a warp two.
constexpr int PQS_MC = 16;
constexpr int PQS_INFLIGHT = 8;     // x 2 nodes per warp in flight

// HIQ8: the second codebook holds the e4m3 companion of every centroid (8 B hi8 | 8 B lo8) instead of its fp16 lo half, and a
// row is written as fp16 hi [ld_out >= M*8] + companion bytes [ldq >= 2*M*8] only -- the operand set of gnnlm_linear_f16f8,
// same bytes per node as the plain hi | lo form and no conversion instructions.
template <bool HIQ8>
__global__ void __launch_bounds__(PQ_THREADS, 1)
    pq_decode_presplit_kernel(const uint8_t* __restrict__ codes, int M, const uint4* __restrict__ cb_hi,
                              const uint4* __restrict__ cb_lo, const int64_t* __restrict__ rows,
                              const int32_t* __restrict__ row_ids, int64_t n_cap, const int32_t* __restrict__ n_dev,
                              __half* __restrict__ out, int64_t ld_out, int nodes_per_cta, uint8_t* __restrict__ q8,
                              int64_t ldq) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint4* s_hi = reinterpret_cast<uint4*>(smem_raw);                  // [PQS_MC][256] quads
  uint4* s_lo = s_hi + PQS_MC * 256;
  __shared__ __align__(8) uint64_t bar;

  const int64_t n = live_rows(n_cap, n_dev);
  const int64_t node0 = (int64_t)blockIdx.y * nodes_per_cta;
  if (node0 >= n) return;
  const int m0 = blockIdx.x * PQS_MC;
  const int mc_here = min(PQS_MC, M - m0);
  const uint32_t half_bytes = (uint32_t)mc_here * 256u * 16u;

  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar, 2 * half_bytes);
    for (uint32_t off = 0; off < half_bytes; off += 32768u) {
      const uint32_t sz = min(32768u, half_bytes - off);
      bulk_g2s(reinterpret_cast<uint8_t*>(s_hi) + off, reinterpret_cast<const uint8_t*>(cb_hi + (size_t)m0 * 256) + off, sz, &bar);
      bulk_g2s(reinterpret_cast<uint8_t*>(s_lo) + off, reinterpret_cast<const uint8_t*>(cb_lo + (size_t)m0 * 256) + off, sz, &bar);
    }
  }
  mbar_wait(&bar, 0);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & (PQS_MC - 1), half = lane >> 4;             // lane -> (subspace, which of the warp's two nodes)
  const bool active = sub < mc_here;
  const int64_t node_end = min(n, node0 + nodes_per_cta);
  const int64_t lo_off = (int64_t)M * 8;                              // lo half of the row, in fp16 elements
  // HIQ8: 16-byte companion stores need an even subspace count here and 16 B aligned companion rows
  const bool pair16 = HIQ8 && (mc_here % 2 == 0) && ldq % 16 == 0 && lo_off % 16 == 0 && ((uintptr_t)q8 % 16 == 0);
  for (int64_t i = node0 + warp * (2 * PQS_INFLIGHT); i < node_end; i += (PQ_THREADS / 32) * (2 * PQS_INFLIGHT)) {
    int64_t r[PQS_INFLIGHT];
    uint32_t c[PQS_INFLIGHT];
#pragma unroll
    for (int u = 0; u < PQS_INFLIGHT; ++u) {
      const int64_t node = i + 2 * u + half;
      const bool ok = node < node_end;
      const int64_t nid = ok ? (row_ids ? (int64_t)__ldg(row_ids + node) : node) : 0;
      r[u] = ok ? __ldg(rows + nid) : -1;
    }
#pragma unroll
    for (int u = 0; u < PQS_INFLIGHT; ++u)
      c[u] = (r[u] >= 0 && active) ? (uint32_t)__ldg(codes + (size_t)r[u] * M + m0 + sub) : 0u;
#pragma unroll
    for (int u = 0; u < PQS_INFLIGHT; ++u) {
      if constexpr (HIQ8) {
        if (pair16) {
          // companion bytes as ONE 16-byte store per lane: neighbouring subspaces swap halves, the even lane writes hi8 of both,
          // the odd lane lo8 of both (8-byte stores at two offsets made this form 20 % slower than the hi | lo one)
          const bool ok = r[u] >= 0 && active;
          const uint4 vl = s_lo[sub * 256 + c[u]];                // (x, y) = hi8, (z, w) = lo8 of this subspace's 8 elements
          const bool odd = sub & 1;
          const uint32_t rx = __shfl_xor_sync(0xffffffffu, odd ? vl.x : vl.z, 1), ry = __shfl_xor_sync(0xffffffffu, odd ? vl.y : vl.w, 1);
          if (ok) {
            __half* dst = out + (size_t)(i + 2 * u + half) * ld_out + (size_t)(m0 + sub) * 8;
            *reinterpret_cast<uint4*>(dst) = s_hi[sub * 256 + c[u]];
            uint8_t* qd = q8 + (size_t)(i + 2 * u + half) * ldq + (size_t)(m0 + (sub & ~1)) * 8 + (odd ? lo_off : 0);
            *reinterpret_cast<uint4*>(qd) = odd ? make_uint4(rx, ry, vl.z, vl.w) : make_uint4(vl.x, vl.y, rx, ry);
          }
          continue;
        }
      }
      if (r[u] >= 0 && active) {
        __half* dst = out + (size_t)(i + 2 * u + half) * ld_out + (size_t)(m0 + sub) * 8;
        const uint4 vh = s_hi[sub * 256 + c[u]], vl = s_lo[sub * 256 + c[u]];
        *reinterpret_cast<uint4*>(dst) = vh;
        if constexpr (HIQ8) {
          uint8_t* qd = q8 + (size_t)(i + 2 * u + half) * ldq + (size_t)(m0 + sub) * 8;
          *reinterpret_cast<uint2*>(qd) = make_uint2(vl.x, vl.y);
          *reinterpret_cast<uint2*>(qd + lo_off) = make_uint2(vl.z, vl.w);
          continue;
        }
        *reinterpret_cast<uint4*>(dst + lo_off) = vl;
        if (q8) {                                        // e4m3 companion (hi8 | lo8): 8 B per (node, subspace) and half
          uint2 h8, l8;
          q8_from_split4(make_uint2(vh.x, vh.y), make_uint2(vl.x, vl.y), h8.x, l8.x);
          q8_from_split4(make_uint2(vh.z, vh.w), make_uint2(vl.z, vl.w), h8.y, l8.y);
          uint8_t* qd = q8 + (size_t)(i + 2 * u + half) * ldq + (size_t)(m0 + sub) * 8;
          *reinterpret_cast<uint2*>(qd) = h8;
          *reinterpret_cast<uint2*>(qd + lo_off) = l8;
        }
      }
    }
  }
}

// generic fallback (any dsub): one thread per (node, subspace); codebook through L1/L2
template <typename OutT>
__global__ void __launch_bounds__(256) pq_decode_generic_kernel(const uint8_t* __restrict__ codes, int M,
                                                                const float* __restrict__ centroids, int dsub,
                                                                const float* __restrict__ bias,
                                                                const int64_t* __restrict__ rows,
                                                                const int32_t* __restrict__ row_ids, int64_t n_cap,
                                                                const int32_t* __restrict__ n_dev, OutT* __restrict__ out,
                                                                int64_t ld_out) {
  const int64_t n = live_rows(n_cap, n_dev);
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n * M) return;
  const int64_t node = g / M;
  const int m = (int)(g % M);
  const int64_t nid = row_ids ? (int64_t)__ldg(row_ids + node) : node;
  const int64_t r = __ldg(rows + nid);
  const uint32_t c = __ldg(codes + (size_t)r * M + m);
  const float* src = centroids + ((size_t)m * 256 + c) * dsub;
  for (int j = 0; j < dsub; ++j) {
    float v = __ldg(src + j) - (bias ? __ldg(bias + m * dsub + j) : 0.f);
    if constexpr (sizeof(OutT) == 4) out[(size_t)node * ld_out + m * dsub + j] = v;
    else if constexpr (std::is_same<OutT, __half>::value) {
      const float c_ = fminf(fmaxf(v, -65504.f), 65504.f);
      const __half h = __float2half_rn(c_);
      out[(size_t)node * ld_out + m * dsub + j] = h;
      out[(size_t)node * ld_out + (size_t)M * dsub + m * dsub + j] = __float2half_rn(c_ - __half2float(h));
    } else out[(size_t)node * ld_out + m * dsub + j] = __float2bfloat16(v);
  }
}

__global__ void __launch_bounds__(256) pq_gather_side_kernel(const uint8_t* __restrict__ codes, int M,
                                                             const int64_t* __restrict__ rows,
                                                             const int32_t* __restrict__ row_ids, int64_t n_cap,
                                                             const int32_t* __restrict__ n_dev,
                                                             const void* __restrict__ labels_table, int label_bytes,
                                                             int64_t* __restrict__ labels_out,
                                                             uint8_t* __restrict__ codes_out) {
  const int64_t n = live_rows(n_cap, n_dev);
  const int lane = threadIdx.x & 31;
  int64_t node = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (node >= n) return;
  const int64_t nid = row_ids ? (int64_t)__ldg(row_ids + node) : node;
  const int64_t r = __ldg(rows + nid);
  if (labels_out && lane == 0) {
    int64_t v = label_bytes == 2 ? (int64_t)__ldg(reinterpret_cast<const int16_t*>(labels_table) + r)
                                 : (int64_t)__ldg(reinterpret_cast<const int32_t*>(labels_table) + r);
    labels_out[node] = v;
  }
  if (codes_out)
    for (int j = lane; j < M; j += 32) codes_out[(size_t)node * M + j] = __ldg(codes + (size_t)r * M + j);
}

}  // namespace gnnlm

using namespace gnnlm;

extern "C" int32_t gnnlm_pq_gather_decode(const uint8_t* codes, int64_t n_datastore, int32_t M, const float* centroids,
                                          int32_t dsub, const float* bias, const int64_t* rows, const int32_t* row_ids,
                                          int64_t n_cap, const int32_t* n_dev, void* out, int32_t out_dtype,
                                          int64_t ld_out, const void* labels_table, int32_t label_bytes,
                                          int64_t* labels_out, uint8_t* codes_out, gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(codes && rows, GNNLM_E_ARG, "gnnlm_pq_gather_decode: null pointer");
  GNNLM_CHECK_ARG(M > 0 && dsub > 0 && n_cap >= 0 && n_datastore > 0, GNNLM_E_SHAPE, "gnnlm_pq_gather_decode: bad sizes");
  GNNLM_CHECK_ARG(out_dtype == GNNLM_F32 || out_dtype == GNNLM_BF16 || out_dtype == GNNLM_F16X2, GNNLM_E_UNSUPPORTED,
                  "gnnlm_pq_gather_decode: out dtype must be F32, BF16 or F16X2");
  GNNLM_CHECK_ARG(!labels_out || (labels_table && (label_bytes == 2 || label_bytes == 4)), GNNLM_E_ARG,
                  "gnnlm_pq_gather_decode: labels_table/label_bytes");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_cap == 0) return 0;
  if (out) {
    GNNLM_CHECK_ARG(centroids, GNNLM_E_ARG, "gnnlm_pq_gather_decode: centroids null");
    GNNLM_CHECK_ARG(ld_out >= (int64_t)M * dsub * (out_dtype == GNNLM_F16X2 ? 2 : 1), GNNLM_E_SHAPE,
                    "gnnlm_pq_gather_decode: ld_out too small");
    const bool vec = (dsub % 4 == 0) && (PQ_CHUNK_FLOATS % dsub == 0) && (ld_out % 4 == 0) &&
                     ((uintptr_t)out % 16 == 0) && ((uintptr_t)centroids % 16 == 0) &&
                     (!bias || (uintptr_t)bias % 16 == 0);
    if (vec) {
      int mc = PQ_CHUNK_FLOATS / dsub;
      if (mc > M) mc = M;
      const size_t smem = (size_t)mc * 256 * dsub * 4;
      int nodes_per_cta = PQ_NODES_PER_CTA;
      // keep at least ~2 waves of CTAs on small inputs
      while (nodes_per_cta > 64 && ceil_div(n_cap, nodes_per_cta) * ceil_div(M, mc) < 296) nodes_per_cta >>= 1;
      dim3 grid((unsigned)ceil_div(M, mc), (unsigned)ceil_div(n_cap, nodes_per_cta));
      if (out_dtype == GNNLM_F32) {
        GNNLM_CUDA(cudaFuncSetAttribute(pq_decode_smem_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        pq_decode_smem_kernel<float><<<grid, PQ_THREADS, smem, st>>>(codes, M, centroids, dsub, bias, rows, row_ids, n_cap,
                                                                     n_dev, (float*)out, ld_out, mc, nodes_per_cta);
      } else if (out_dtype == GNNLM_F16X2) {
        GNNLM_CUDA(cudaFuncSetAttribute(pq_decode_smem_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        pq_decode_smem_kernel<__half><<<grid, PQ_THREADS, smem, st>>>(codes, M, centroids, dsub, bias, rows, row_ids, n_cap,
                                                                      n_dev, (__half*)out, ld_out, mc, nodes_per_cta);
      } else {
        GNNLM_CUDA(cudaFuncSetAttribute(pq_decode_smem_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        pq_decode_smem_kernel<__nv_bfloat16><<<grid, PQ_THREADS, smem, st>>>(
            codes, M, centroids, dsub, bias, rows, row_ids, n_cap, n_dev, (__nv_bfloat16*)out, ld_out, mc, nodes_per_cta);
      }
    } else {
      unsigned blocks = (unsigned)ceil_div(n_cap * M, 256);
      if (out_dtype == GNNLM_F32)
        pq_decode_generic_kernel<float><<<blocks, 256, 0, st>>>(codes, M, centroids, dsub, bias, rows, row_ids, n_cap, n_dev,
                                                                 (float*)out, ld_out);
      else if (out_dtype == GNNLM_F16X2)
        pq_decode_generic_kernel<__half><<<blocks, 256, 0, st>>>(codes, M, centroids, dsub, bias, rows, row_ids, n_cap, n_dev,
                                                                  (__half*)out, ld_out);
      else
        pq_decode_generic_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(codes, M, centroids, dsub, bias, rows, row_ids, n_cap,
                                                                         n_dev, (__nv_bfloat16*)out, ld_out);
    }
    GNNLM_LAUNCH_CHECK("gnnlm_pq_gather_decode");
  }
  if (labels_out || codes_out) {
    pq_gather_side_kernel<<<(unsigned)ceil_div(n_cap * 32, 256), 256, 0, st>>>(codes, M, rows, row_ids, n_cap, n_dev,
                                                                                labels_table, label_bytes, labels_out,
                                                                                codes_out);
    GNNLM_LAUNCH_CHECK("gnnlm_pq_gather_side");
  }
  return 0;
}

extern "C" int32_t gnnlm_pq_gather_decode_presplit(const uint8_t* codes, int64_t n_datastore, int32_t M, const void* cb_hi,
                                                   const void* cb_lo, int32_t dsub, const int64_t* rows,
                                                   const int32_t* row_ids, int64_t n_cap, const int32_t* n_dev, void* out,
                                                   int64_t ld_out, gnnlm_stream_t stream) {
  return gnnlm_pq_gather_decode_presplit_q8(codes, n_datastore, M, cb_hi, cb_lo, dsub, rows, row_ids, n_cap, n_dev, out, ld_out,
                                            nullptr, 0, stream);
}

extern "C" int32_t gnnlm_pq_gather_decode_presplit_q8(const uint8_t* codes, int64_t n_datastore, int32_t M, const void* cb_hi,
                                                      const void* cb_lo, int32_t dsub, const int64_t* rows,
                                                      const int32_t* row_ids, int64_t n_cap, const int32_t* n_dev, void* out,
                                                      int64_t ld_out, void* q8v, int64_t ldq, gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(codes && rows && cb_hi && cb_lo && out, GNNLM_E_ARG, "gnnlm_pq_gather_decode_presplit: null pointer");
  uint8_t* q8 = reinterpret_cast<uint8_t*>(q8v);
  GNNLM_CHECK_ARG(!q8 || (ldq >= 2 * (int64_t)M * 8 && ldq % 8 == 0 && (uintptr_t)q8 % 8 == 0), GNNLM_E_SHAPE,
                  "gnnlm_pq_gather_decode_presplit_q8: the e4m3 companion needs ldq >= 2*M*8, 8 B aligned rows");
  GNNLM_CHECK_ARG(M > 0 && n_cap >= 0 && n_datastore > 0, GNNLM_E_SHAPE, "gnnlm_pq_gather_decode_presplit: bad sizes");
  GNNLM_CHECK_ARG(dsub == 8, GNNLM_E_UNSUPPORTED, "gnnlm_pq_gather_decode_presplit: dsub must be 8 (use gnnlm_pq_gather_decode)");
  GNNLM_CHECK_ARG(ld_out >= 2 * (int64_t)M * 8 && ld_out % 8 == 0 && (uintptr_t)out % 16 == 0 && (uintptr_t)cb_hi % 16 == 0 &&
                      (uintptr_t)cb_lo % 16 == 0,
                  GNNLM_E_SHAPE, "gnnlm_pq_gather_decode_presplit: out / codebooks must be 16 B aligned, ld_out >= 2*M*8");
  if (n_cap == 0) return 0;
  const size_t smem = (size_t)2 * PQS_MC * 256 * 16;
  static bool attr_set[MAX_DEVICES] = {};
  bool& done = attr_set[device_slot()];
  if (!done) {
    GNNLM_CUDA(cudaFuncSetAttribute(pq_decode_presplit_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GNNLM_CUDA(cudaFuncSetAttribute(pq_decode_presplit_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    done = true;
  }
  int nodes_per_cta = PQ_NODES_PER_CTA;
  while (nodes_per_cta > 64 && ceil_div(n_cap, nodes_per_cta) * ceil_div(M, PQS_MC) < 296) nodes_per_cta >>= 1;
  dim3 grid((unsigned)ceil_div(M, PQS_MC), (unsigned)ceil_div(n_cap, nodes_per_cta));
  pq_decode_presplit_kernel<false><<<grid, PQ_THREADS, smem, (cudaStream_t)stream>>>(
      codes, M, (const uint4*)cb_hi, (const uint4*)cb_lo, rows, row_ids, n_cap, n_dev, (__half*)out, ld_out, nodes_per_cta, q8, ldq);
  GNNLM_LAUNCH_CHECK("gnnlm_pq_gather_decode_presplit");
  return 0;
}

extern "C" int32_t gnnlm_pq_gather_decode_hiq8(const uint8_t* codes, int64_t n_datastore, int32_t M, const void* cb_hi,
                                               const void* cb_q8, int32_t dsub, const int64_t* rows, const int32_t* row_ids,
                                               int64_t n_cap, const int32_t* n_dev, void* out_hi, int64_t ld_out, void* q8v,
                                               int64_t ldq, gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(codes && rows && cb_hi && cb_q8 && out_hi && q8v, GNNLM_E_ARG, "gnnlm_pq_gather_decode_hiq8: null pointer");
  GNNLM_CHECK_ARG(M > 0 && n_cap >= 0 && n_datastore > 0, GNNLM_E_SHAPE, "gnnlm_pq_gather_decode_hiq8: bad sizes");
  GNNLM_CHECK_ARG(dsub == 8, GNNLM_E_UNSUPPORTED, "gnnlm_pq_gather_decode_hiq8: dsub must be 8");
  GNNLM_CHECK_ARG(ld_out >= (int64_t)M * 8 && ld_out % 8 == 0 && ldq >= 2 * (int64_t)M * 8 && ldq % 8 == 0 && (uintptr_t)out_hi % 16 == 0 &&
                      (uintptr_t)q8v % 8 == 0 && (uintptr_t)cb_hi % 16 == 0 && (uintptr_t)cb_q8 % 16 == 0,
                  GNNLM_E_SHAPE, "gnnlm_pq_gather_decode_hiq8: 16 B aligned rows, ld_out >= M*8, ldq >= 2*M*8");
  if (n_cap == 0) return 0;
  const size_t smem = (size_t)2 * PQS_MC * 256 * 16;
  static bool attr_set = false;
  if (!attr_set) {
    GNNLM_CUDA(cudaFuncSetAttribute(pq_decode_presplit_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  int nodes_per_cta = PQ_NODES_PER_CTA;
  while (nodes_per_cta > 64 && ceil_div(n_cap, nodes_per_cta) * ceil_div(M, PQS_MC) < 296) nodes_per_cta >>= 1;
  dim3 grid((unsigned)ceil_div(M, PQS_MC), (unsigned)ceil_div(n_cap, nodes_per_cta));
  pq_decode_presplit_kernel<true><<<grid, PQ_THREADS, smem, (cudaStream_t)stream>>>(
      codes, M, (const uint4*)cb_hi, (const uint4*)cb_q8, rows, row_ids, n_cap, n_dev, (__half*)out_hi, ld_out, nodes_per_cta,
      reinterpret_cast<uint8_t*>(q8v), ldq);
  GNNLM_LAUNCH_CHECK("gnnlm_pq_gather_decode_hiq8");
  return 0;
}
