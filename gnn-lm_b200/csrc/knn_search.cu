// Exact k-nearest-neighbour search over the datastore (the faiss index search of knn/find_knn.py:29-71 and of
// KNNModel.get_knns, knn/knn_model.py:87-101), without faiss:
//   score s(q, x) = q.x + bias(x)   (bias = -1/2 ||x||^2 for l2, 0 for ip), ranked by score descending, ties by smaller id.
// The scores come from the 3xFP16 tcgen05 GEMM with the top-k filter epilogue (gemm_tcgen05.cu, gemm_tc_topk): keys are the
// A operand, queries W, and only scores above each query's running k-th score leave the SM, as candidates.  This file holds the
// rest: the per-query merge of the running top-k with a span's candidates, and the per-key bias.
#include "common.cuh"

namespace gnnlm {

int32_t gemm_tc_topk(const void* A, int64_t lda, int64_t M, int64_t id_base, const void* W_hi, const void* W_lo, int64_t ldw,
                     int64_t N, int64_t K, const float* row_bias, const float* thr, float* cand_s, int32_t* cand_id,
                     int32_t* cand_cnt, int64_t cap, cudaStream_t st);

namespace {

constexpr int MERGE_THREADS = 512;
constexpr int MAX_K = 2048, MAX_CAP = 4096;

// (score, id) -> one 64-bit key whose ascending order is (score descending, id ascending); empty slots sort last
__device__ __forceinline__ uint64_t rank_key(float s, int32_t id) {
  if (id < 0) return ~0ull;
  const uint32_t u = __float_as_uint(s);
  const uint32_t ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);        // ascending with s
  return ((uint64_t)(~ord) << 32) | (uint32_t)id;
}
__device__ __forceinline__ float key_score(uint64_t key) {
  const uint32_t ord = ~(uint32_t)(key >> 32);
  return __uint_as_float((ord & 0x80000000u) ? (ord & 0x7fffffffu) : ~ord);
}

// One CTA per query: running top-k (sorted) + min(cnt, cap) candidates -> bitonic sort in shared memory -> new top-k, threshold
// (k-th score, -inf while fewer than k are held), cand_cnt reset to 0.  A query whose count exceeds cap is left untouched (the
// host re-runs its span in pieces that cannot overflow).
__global__ void __launch_bounds__(MERGE_THREADS) topk_merge_kernel(float* __restrict__ top_s, int32_t* __restrict__ top_id, int k,
                                                                   const float* __restrict__ cand_s,
                                                                   const int32_t* __restrict__ cand_id, int32_t* cand_cnt,
                                                                   int64_t cap, float* __restrict__ thr) {
  extern __shared__ uint64_t keys[];
  const int64_t q = blockIdx.x;
  const int cnt = cand_cnt[q];
  if (cnt == 0 || cnt > cap) return;                           // block-uniform
  int P = 1;
  while (P < k + cnt) P <<= 1;
  float* ts = top_s + q * k;
  int32_t* ti = top_id + q * k;
  for (int i = threadIdx.x; i < P; i += MERGE_THREADS) {
    uint64_t key = ~0ull;
    if (i < k) key = rank_key(ts[i], ti[i]);
    else if (i < k + cnt) key = rank_key(cand_s[q * cap + (i - k)], cand_id[q * cap + (i - k)]);
    keys[i] = key;
  }
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < P / 2; i += MERGE_THREADS) {
        const int lo = 2 * stride * (i / stride) + (i % stride), hi = lo + stride;
        const bool asc = (lo & size) == 0;
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a > b) == asc) {
          keys[lo] = b;
          keys[hi] = a;
        }
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < k; i += MERGE_THREADS) {
    const uint64_t key = keys[i];
    const bool held = key != ~0ull;
    ts[i] = held ? key_score(key) : -INFINITY;
    ti[i] = held ? (int32_t)(uint32_t)key : -1;
  }
  if (threadIdx.x == 0) {
    thr[q] = keys[k - 1] != ~0ull ? key_score(keys[k - 1]) : -INFINITY;
    cand_cnt[q] = 0;
  }
}

// out[i] = -1/2 ||x_i||^2 in fp32, one warp per row, a fixed summation order (lane-strided partial sums, butterfly)
template <typename T>
__global__ void key_bias_rows_kernel(const T* __restrict__ x, int64_t ld, int64_t n, int64_t d, float* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const T* p = x + row * ld;
  float acc = 0.f;
  for (int64_t c = lane; c < d; c += 32) {
    const float v = (float)p[c];
    acc = fmaf(v, v, acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[row] = -0.5f * acc;
}

// out[i] = -1/2 sum_m norm2[m, codes[i, m]]: ||x_i||^2 of a PQ-decoded key from the per-centroid table
__global__ void key_bias_pq_kernel(const uint8_t* __restrict__ codes, int64_t n, int M, const float* __restrict__ norm2,
                                   float* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  float acc = 0.f;
  for (int m = lane; m < M; m += 32) acc += __ldg(norm2 + m * 256 + codes[row * M + m]);
  acc = warp_sum(acc);
  if (lane == 0) out[row] = -0.5f * acc;
}

}  // namespace

}  // namespace gnnlm

using namespace gnnlm;

extern "C" int32_t gnnlm_knn_filter_f16x3(const void* keys, int64_t ldk, int64_t n_keys, int64_t id_base, const void* q_hi,
                                          const void* q_lo, int64_t ldq, int64_t n_q, int64_t d, const float* key_bias,
                                          const float* thr, float* cand_s, int32_t* cand_id, int32_t* cand_cnt, int64_t cap,
                                          gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(keys && q_hi && q_lo && thr && cand_s && cand_id && cand_cnt, GNNLM_E_ARG, "gnnlm_knn_filter_f16x3: null pointer");
  GNNLM_CHECK_ARG(cap >= 1 && cap <= MAX_CAP, GNNLM_E_ARG, "gnnlm_knn_filter_f16x3: cap must be in [1, %d]", MAX_CAP);
  GNNLM_CHECK_ARG(n_keys >= 0 && n_q >= 0 && d > 0 && d % 8 == 0 && ldk >= 2 * d && ldq >= d, GNNLM_E_SHAPE,
                  "gnnlm_knn_filter_f16x3: bad shape (n_keys=%lld n_q=%lld d=%lld ldk=%lld ldq=%lld)", (long long)n_keys,
                  (long long)n_q, (long long)d, (long long)ldk, (long long)ldq);
  GNNLM_CHECK_ARG(id_base >= 0 && id_base + n_keys <= INT32_MAX, GNNLM_E_SHAPE,
                  "gnnlm_knn_filter_f16x3: ids must stay below 2^31 (id_base=%lld n_keys=%lld)", (long long)id_base,
                  (long long)n_keys);
  if (n_keys == 0 || n_q == 0) return 0;
  return gemm_tc_topk(keys, ldk, n_keys, id_base, q_hi, q_lo, ldq, n_q, d, key_bias, thr, cand_s, cand_id, cand_cnt, cap,
                      (cudaStream_t)stream);
}

extern "C" int32_t gnnlm_topk_merge(float* top_s, int32_t* top_id, int64_t n_q, int32_t k, const float* cand_s,
                                    const int32_t* cand_id, int32_t* cand_cnt, int64_t cap, float* thr, gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(top_s && top_id && cand_s && cand_id && cand_cnt && thr, GNNLM_E_ARG, "gnnlm_topk_merge: null pointer");
  GNNLM_CHECK_ARG(k >= 1 && k <= MAX_K, GNNLM_E_ARG, "gnnlm_topk_merge: k must be in [1, %d]", MAX_K);
  GNNLM_CHECK_ARG(cap >= 1 && cap <= MAX_CAP, GNNLM_E_ARG, "gnnlm_topk_merge: cap must be in [1, %d]", MAX_CAP);
  GNNLM_CHECK_ARG(n_q >= 0 && n_q <= INT32_MAX, GNNLM_E_SHAPE, "gnnlm_topk_merge: bad n_q");
  if (n_q == 0) return 0;
  int P = 1;
  while (P < k + cap) P <<= 1;
  const size_t smem = (size_t)P * sizeof(uint64_t);
  static size_t configured[MAX_DEVICES] = {};
  size_t& done = configured[device_slot()];
  if (smem > done) {
    GNNLM_CUDA(cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    done = smem;
  }
  topk_merge_kernel<<<(unsigned)n_q, MERGE_THREADS, smem, (cudaStream_t)stream>>>(top_s, top_id, k, cand_s, cand_id, cand_cnt, cap,
                                                                                    thr);
  GNNLM_LAUNCH_CHECK("gnnlm_topk_merge");
  return 0;
}

extern "C" int32_t gnnlm_knn_key_bias(const void* x, int32_t dtype, int64_t ld, int64_t n, int64_t d, float* out,
                                      gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(x && out, GNNLM_E_ARG, "gnnlm_knn_key_bias: null pointer");
  GNNLM_CHECK_ARG(dtype == GNNLM_F32 || dtype == GNNLM_F16, GNNLM_E_UNSUPPORTED, "gnnlm_knn_key_bias: rows must be fp32 or fp16");
  GNNLM_CHECK_ARG(n >= 0 && d > 0 && ld >= d, GNNLM_E_SHAPE, "gnnlm_knn_key_bias: bad shape");
  if (n == 0) return 0;
  const unsigned grid = (unsigned)ceil_div(n, 8);
  if (dtype == GNNLM_F16)
    key_bias_rows_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>((const __half*)x, ld, n, d, out);
  else
    key_bias_rows_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)x, ld, n, d, out);
  GNNLM_LAUNCH_CHECK("gnnlm_knn_key_bias");
  return 0;
}

extern "C" int32_t gnnlm_knn_key_bias_pq(const uint8_t* codes, int64_t n, int32_t M, const float* norm2, float* out,
                                         gnnlm_stream_t stream) {
  GNNLM_CHECK_ARG(codes && norm2 && out, GNNLM_E_ARG, "gnnlm_knn_key_bias_pq: null pointer");
  GNNLM_CHECK_ARG(n >= 0 && M > 0, GNNLM_E_SHAPE, "gnnlm_knn_key_bias_pq: bad shape");
  if (n == 0) return 0;
  key_bias_pq_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, (cudaStream_t)stream>>>(codes, n, M, norm2, out);
  GNNLM_LAUNCH_CHECK("gnnlm_knn_key_bias_pq");
  return 0;
}
