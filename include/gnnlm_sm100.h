/*
 * libgnnlm_sm100.so -- C ABI of the B200-native GNN-LM evaluation hot path.
 *
 * The reference (ShannonAI/GNN-LM) has no FFI: its boundary is fairseq's Python plugin API and its
 * hot-path arithmetic lives in DGL / ATen / cuBLAS calls made from Python.  This header is the
 * boundary a maintainer binds with ctypes (see INTEGRATION.md); every entry point cites the
 * reference call it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - extern "C", POD arguments only: device pointers, int64 sizes, int32 enums, cudaStream_t last.
 *   - Every function returns int32: 0 = ok, >0 = cudaError_t, <0 = argument/shape error
 *     (GNNLM_E_*).  gnnlm_last_error() returns a thread-local message for the last failure.
 *   - No allocation, no ownership transfer, no hidden synchronisation: the caller owns every buffer
 *     (workspaces are sized by the *_workspace_bytes queries) and every launch goes to `stream`.
 *   - Row counts that are only known on the device after graph assembly (number of ntgt nodes,
 *     number of valid neighbours, rows per adaptive-softmax cluster) are passed twice: a host-side
 *     capacity `*_cap` used to size grids, and an optional device pointer `*_dev` (int32) holding
 *     the true count; kernels process min(cap, *dev) rows.  Pass NULL when the host count is exact.
 *   - All matrices are row-major with an explicit leading dimension in ELEMENTS.
 */
#ifndef GNNLM_SM100_H
#define GNNLM_SM100_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* gnnlm_stream_t; /* == cudaStream_t */

/* element types */
#define GNNLM_F32 0
#define GNNLM_BF16 1
#define GNNLM_F16 2
/* "split fp16": an fp32 matrix [rows, d] stored as two fp16 halves in ONE [rows, 2d] fp16 buffer, hi = fp16(x) in
 * columns [0, d), lo = fp16(x - hi) in columns [d, 2d) (22 significant bits, |x| clamped to 65504).  Same bytes as
 * fp32; it is the activation format of GNNLM_MATH_F16X3: GEMMs consume it straight through TMA (no in-kernel
 * operand split) and the producing kernels (PQ decode, GEMM epilogue, LayerNorm, cluster attention) emit it.
 * Leading dimensions of F16X2 buffers are in fp16 elements (>= 2d). */
#define GNNLM_F16X2 3
/* An fp32 value rounded to its top three bytes (15 mantissa bits, 2^-16 relative): a 16-bit plane [rows, ld] (bytes 3, 2 of the
 * value: its bf16 truncation) + a byte plane (byte 1) with the same row stride in elements.  Output of gnnlm_linear_f16f8 / input of
 * gnnlm_hgt_cluster_attn_hq: the ntgt-side Q | K' | V' of MATH_F16F8 in 3 bytes per element instead of 4, decoded by byte permutes. */
#define GNNLM_F24 4

/* argument errors */
#define GNNLM_E_ARG (-1)
#define GNNLM_E_SHAPE (-2)
#define GNNLM_E_UNSUPPORTED (-3)
#define GNNLM_E_WORKSPACE (-4)

/* GEMM arithmetic modes (gnnlm_linear*, `math` argument) */
#define GNNLM_MATH_FP32_SIMT 0  /* fp32 FMA on CUDA cores: strict-parity / validation mode      */
#define GNNLM_MATH_TF32X3 1     /* tcgen05 kind::tf32, 3-pass split (hi*hi + hi*lo + lo*hi)      */
#define GNNLM_MATH_TF32 2       /* tcgen05 kind::tf32, single pass                              */
#define GNNLM_MATH_BF16 3       /* tcgen05 kind::f16 with bf16 operands, fp32 accumulate        */
#define GNNLM_MATH_F16X3 4      /* tcgen05 kind::f16, fp32 operands split into 2 x fp16, 3 passes   */

int32_t gnnlm_version(void);
const char* gnnlm_last_error(void);
/* 1 when the library was built with the tcgen05/TMA GEMM and the device is sm_100. */
int32_t gnnlm_has_tcgen05(void);

/* ------------------------------------------------------------------------------------------------
 * (1) Graph assembly -- replaces GraphTokenBlockDataset.new_build_graph
 *     (fairseq/data/token_block_dataset.py:338-412), build_ntgt_edges (:545-584),
 *     auto_regressive_edges (:586-594) and dgl.batch (fairseq/data/monolingual_dataset.py:261).
 *
 *  nbr      [T, k] int64  neighbour datastore rows per target token, -1 = missing
 *                         (= neighbor_offsets[offsets], token_block_dataset.py:309)
 *  tgt_pos  [T]    int64  stream position of each target token (`offsets`); only read when
 *                         invalid_ctx > 0 (token_block_dataset.py:361), may be NULL otherwise
 *  Node numbering is the reference's: tgt id = b*L + t; ntgt ids in creation order (tgt-major,
 *  neighbour-rank-major, centre, then left context ascending, then right context ascending).
 * ---------------------------------------------------------------------------------------------- */

/* Pass 1: per (token, neighbour) cluster sizes and their exclusive scans.
 *  node_base  [T*k + 1] int32  first ntgt id of each cluster; node_base[T*k]  = n_ntgt
 *  valid_base [T*k + 1] int32  #valid clusters before;        valid_base[T*k] = n_valid
 *  workspace: gnnlm_graph_workspace_bytes(T*k) bytes. */
int64_t gnnlm_graph_workspace_bytes(int64_t n_clusters);
int32_t gnnlm_graph_count(const int64_t* nbr, const int64_t* tgt_pos, int64_t T, int64_t k,
                          int64_t n_datastore, int32_t left_ctx, int32_t right_ctx, int64_t invalid_ctx,
                          int32_t* node_base, int32_t* valid_base, void* workspace, int64_t workspace_bytes,
                          gnnlm_stream_t stream);

/* Pass 2: node tables and the canonical CSRs (COO in reference insertion order, stable-sorted by
 * destination).  Capacity of the per-node outputs is node_cap = T*k*(1+left_ctx+right_ctx).
 *  ntgt_row     [node_cap]   int64  datastore row of every ntgt node
 *  ntgt_owner   [node_cap]   int32  tgt id whose neighbour produced the node        (nullable)
 *  ntgt_dist    [node_cap]   int32  |sorted position - centre position| in cluster  (nullable)
 *  nn_indptr    [node_cap+1] int32, nn_indices [3*node_cap] int32   ('ntgt','intra','ntgt')
 *  inter_indptr [T+1] int32,        inter_indices [T*k] int32       ('ntgt','inter','tgt'); the
 *               indices are exactly the centre-node ids in creation order.
 *  cluster_nl   [T*k] int32  number of left-context nodes of each (token, neighbour) cluster, -1 when
 *               the neighbour is invalid (nullable; consumed by gnnlm_hgt_cluster_attn). */
int32_t gnnlm_graph_fill(const int64_t* nbr, const int64_t* tgt_pos, int64_t T, int64_t k,
                         int64_t n_datastore, int32_t left_ctx, int32_t right_ctx, int64_t invalid_ctx,
                         const int32_t* node_base, const int32_t* valid_base, int64_t* ntgt_row,
                         int32_t* ntgt_owner, int32_t* ntgt_dist, int32_t* nn_indptr, int32_t* nn_indices,
                         int32_t* inter_indptr, int32_t* inter_indices, int32_t* cluster_nl, gnnlm_stream_t stream);

/* ('tgt','intra','tgt') CSR, materialised only for parity checks (the attention kernel treats it as
 * implicit causal).  n_edges = B * sum_v min(v+1, intra_ctx or inf).  indptr [B*L+1], indices [E]. */
int64_t gnnlm_graph_tt_num_edges(int64_t B, int64_t L, int64_t intra_ctx);
int32_t gnnlm_graph_tt_csr(int64_t B, int64_t L, int64_t intra_ctx, int32_t* indptr, int32_t* indices,
                           gnnlm_stream_t stream);

/* Distinct centre rows of a batch (cluster-level reuse).  new_build_graph creates a fresh cluster for every (token, neighbour)
 * pair (token_block_dataset.py:355,363-374), and an ntgt node only ever receives messages from inside its cluster, so clusters
 * with the same centre row carry identical features in every layer: the ntgt side can run once per DISTINCT centre.
 *  nbr [n] neighbour ids (n = T*k), valid_base [n + 1] from gnnlm_graph_count
 *  uniq [n]      out: the distinct ids of the valid pairs, -1 padded (a k = 1 neighbour array for gnnlm_graph_count / _fill);
 *                order unspecified (first inserter into a hash table)
 *  inv  [n]      out: inv[valid_base[i]] = index into uniq of pair i's id, for every valid pair
 *  n_unique [1]  out (device): number of distinct ids
 *  workspace: gnnlm_unique_workspace_bytes(n) bytes, 8 B aligned. */
int64_t gnnlm_unique_workspace_bytes(int64_t n);
int32_t gnnlm_unique_centres(const int64_t* nbr, const int32_t* valid_base, int64_t n, int64_t* uniq, int32_t* inv,
                             int32_t* n_unique, void* workspace, int64_t workspace_bytes, gnnlm_stream_t stream);

/* `--deprecated` graph assembly (GraphTokenBlockDataset.deprecated_build_graph, token_block_dataset.py:414-479): ONE ntgt
 * node per distinct datastore row of a block, numbered by first appearance (centre, left context ascending, right context
 * ascending, neighbour by neighbour, token by token); ntgt-ntgt edges between rows at distance <= 1 wherever they came
 * from (+ self loops); blocks of a batch share no nodes.  T = B * L tokens, block length L.
 *  valid_base   [T*k + 1] from gnnlm_graph_count (same contexts / invalid_ctx)
 *  ntgt_row     [T*k*w] int64 datastore row per node; n_ntgt [1] live node count (device)
 *  nn_indptr [T*k*w + 1], nn_indices [3*T*k*w]: canonical CSR by destination, sources in row order (o-1, o, o+1)
 *  inter_indptr [T + 1], inter_indices [T*k]: the centre node of every valid (token, neighbour), in that order
 *  workspace: gnnlm_graph_dedup_workspace_bytes(T, k, w) bytes, 256 B aligned. */
int64_t gnnlm_graph_dedup_workspace_bytes(int64_t T, int64_t k, int32_t w);
int32_t gnnlm_graph_dedup(const int64_t* nbr, const int64_t* tgt_pos, int64_t T, int64_t L, int64_t k, int64_t n_datastore,
                          int32_t left_ctx, int32_t right_ctx, int64_t invalid_ctx, const int32_t* valid_base,
                          int64_t* ntgt_row, int32_t* n_ntgt, int32_t* nn_indptr, int32_t* nn_indices, int32_t* inter_indptr,
                          int32_t* inter_indices, void* workspace, int64_t workspace_bytes, gnnlm_stream_t stream);

/* Host-side slice copy of a batch's inputs: dst <- src (bytes) over n_threads native threads (one blocking call, no interpreter
 * lock), optionally checking that the range -- int64 neighbour ids, token_block_dataset.py:309 -- lies in [lo, hi): *bad = 1
 * otherwise (the reference raises IndexError at quant_neighbor_feats[o], :369-370).  dst == NULL: check only. */
int32_t gnnlm_host_copy(void* dst, const void* src, int64_t bytes, int32_t check_i64, int64_t lo, int64_t hi, int32_t n_threads,
                        int32_t* bad);

/* ------------------------------------------------------------------------------------------------
 * (2) Datastore gather + PQ decode -- replaces `quant_neighbor_feats[offset]` /
 *     `neighbor_tokens[offset]` (token_block_dataset.py:369-371,392-394) and the centroid gather of
 *     TorchPQCodec.decode (knn/pq_wrapper.py:169-196).  `x -= b` (:200-201) is fused when bias != NULL;
 *     the OPQ rotation `x @ A` (:202) is a gnnlm_linear call with W = A^T.
 *
 *  codes      [n_datastore, M] uint8 (quantized-keys.npy), centroids [M, 256, dsub] fp32
 *  rows       [n_cap] int64 datastore rows (ntgt_row), optionally indirected through
 *             row_ids [n_cap] int32 (process rows[row_ids[i]]; e.g. centre nodes only)
 *  out        [n_cap, M*dsub] out_dtype, leading dimension ld_out
 *  labels_table [n_datastore] int16/int32 (vals.npy; label_bytes = 2|4) -> labels_out [n_cap] int64
 *             (nullable pair; `ntgt.labels`, token_block_dataset.py:410)
 *  codes_out  [n_cap, M] uint8 gathered code rows (nullable; `ntgt.h`, :408-409) */
int32_t gnnlm_pq_gather_decode(const uint8_t* codes, int64_t n_datastore, int32_t M, const float* centroids,
                               int32_t dsub, const float* bias, const int64_t* rows, const int32_t* row_ids,
                               int64_t n_cap, const int32_t* n_dev, void* out, int32_t out_dtype,
                               int64_t ld_out, const void* labels_table, int32_t label_bytes,
                               int64_t* labels_out, uint8_t* codes_out, gnnlm_stream_t stream);

/* Same gather + decode for the split-fp16 activation format from a codebook that is already split: cb_hi / cb_lo
 * [M, 256, 8] fp16 = hi / lo halves of (centroid - bias) (prepared once per quantizer; dsub == 8 only, i.e. one 16 B quad per
 * centroid half).  out [n_cap, 2*M*8] split fp16 (leading dimension ld_out, in fp16 elements).  Pure byte movement. */
int32_t gnnlm_pq_gather_decode_presplit(const uint8_t* codes, int64_t n_datastore, int32_t M, const void* cb_hi,
                                        const void* cb_lo, int32_t dsub, const int64_t* rows, const int32_t* row_ids,
                                        int64_t n_cap, const int32_t* n_dev, void* out, int64_t ld_out,
                                        gnnlm_stream_t stream);

/* ..._q8: additionally writes the e4m3 companion q8 [n_cap, 2*M*8] bytes (ldq; hi8 = e4m3(hi) | lo8 = e4m3(2^10 lo)) that
 * gnnlm_linear_f16f8 reads; q8 == NULL is the plain call. */
int32_t gnnlm_pq_gather_decode_presplit_q8(const uint8_t* codes, int64_t n_datastore, int32_t M, const void* cb_hi,
                                           const void* cb_lo, int32_t dsub, const int64_t* rows, const int32_t* row_ids,
                                           int64_t n_cap, const int32_t* n_dev, void* out, int64_t ld_out, void* q8,
                                           int64_t ldq, gnnlm_stream_t stream);

/* The operand set of gnnlm_linear_f16f8 only: out_hi [n_cap, M*8] fp16 (ld_out >= M*8) + q8 [n_cap, 2*M*8] bytes, from cb_hi
 * [M, 256, 8] fp16 and cb_q8 [M, 256, 16] bytes = the e4m3 companion (8 B hi8 | 8 B lo8) of every centroid, prepared once per
 * quantizer (gnnlm_split_to_q8 over the split codebook).  Same bytes per node as the plain form, no conversions. */
int32_t gnnlm_pq_gather_decode_hiq8(const uint8_t* codes, int64_t n_datastore, int32_t M, const void* cb_hi, const void* cb_q8,
                                    int32_t dsub, const int64_t* rows, const int32_t* row_ids, int64_t n_cap,
                                    const int32_t* n_dev, void* out_hi, int64_t ld_out, void* q8, int64_t ldq,
                                    gnnlm_stream_t stream);

/* PQ encode (the producer of quantized-keys.npy; knn/pq_wrapper.py:51-68,131-167, knn/quantize_features.py:115-152):
 *  codes[n, m] = argmin_c (norm2[m, c] - 2 <x[n, m*dsub:(m+1)*dsub], centroids[m, c]>), first minimum wins.
 *  x fp32 [n, M*dsub] (ldx) must already carry the OPQ pre-rotation `x @ A.T (+ b)` (a gnnlm_linear call);
 *  norm2 [M, 256] = ||centroid||^2 (`norm2_centroids_torch`).  dsub in {1, 2, 4, 8, 16}. */
int32_t gnnlm_pq_encode(const float* x, int64_t ldx, int64_t n, int32_t M, int32_t dsub, const float* centroids,
                        const float* norm2, uint8_t* codes, gnnlm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (3) Dense projections -- replace the nn.Linear / einsum calls of HGTLayer.forward
 *     (fairseq/models/hgt.py:320-322,347-348,401), the OPQ rotation (knn/pq_wrapper.py:202) and the
 *     adaptive-softmax projections (fairseq/modules/adaptive_softmax.py:184,197,202).
 *
 *  C[m, n] = sum_k A[m, k] * W[n, k] + bias[n] (+ residual[m, n])          (nn.Linear layout)
 *  A [M, K] a_dtype lda; W [N, K] (same dtype as A; fp16 hi/lo pair for MATH_F16X3, whose A is fp32) ldw; bias fp32 [N] nullable; residual [M, N] of
 *  r_dtype (F32, or BF16 on the tensor-core path) ldr nullable; C c_dtype ldc.  For GNNLM_MATH_TF32X3, W_lo is the low half of the split
 *  (W - tf32(W)), prepared once by gnnlm_split_tf32; NULL otherwise. */
int32_t gnnlm_split_tf32(const float* w, float* w_hi, float* w_lo, int64_t n, gnnlm_stream_t stream);
/* MATH_F16X3 weight preparation: w_hi = fp16(w * scale), w_lo = fp16(w * scale - w_hi) (both fp16 arrays of n
 * elements); `scale` must be a power of two with max|w * scale| <= 2^15; pass it as w_scale to gnnlm_linear*
 * (the epilogue multiplies by 1 / w_scale).  w_scale is ignored by every other math mode. */
int32_t gnnlm_split_f16(const float* w, float scale, void* w_hi, void* w_lo, int64_t n, gnnlm_stream_t stream);
int32_t gnnlm_linear(const void* A, int32_t a_dtype, int64_t lda, const void* W, const void* W_lo, float w_scale, int64_t ldw,
                     const float* bias, const void* residual, int32_t r_dtype, int64_t ldr, void* C,
                     int32_t c_dtype, int64_t ldc, int64_t M, const int32_t* m_dev, int64_t N, int64_t K,
                     int32_t math, gnnlm_stream_t stream);

/* nb independent products in ONE launch (the per-head GEMMs of the tensor-core causal attention):
 *   C[b] = (1 / w_scale) * A[b] W[b]^T (+ residual[b]),  b = 0..nb-1,   MATH_F16X3 arithmetic.
 * A[b] split-fp16 [M, 2K] at A + b*a_bs (fp16 elements, lda >= 2K); W_hi[b], W_lo[b] fp16 [N, K] at + b*w_bs;
 * C[b], residual[b] fp32 at + b*c_bs / b*r_bs (elements; a column offset when the heads share rows).
 * causal: 0 = plain; 1 = scores of causal attention: 256 x 256 output tiles entirely above the diagonal (first column >
 *   last row) are skipped and left unwritten; 2 = probabilities x values: rows [256 r, 256 (r+1)) contract over
 *   k < 256 (r+1) only (the caller guarantees A is zero -- or never meant to be read -- beyond that). */
int32_t gnnlm_linear_batched_f16x3(const void* A, int64_t lda, int64_t a_bs, const void* W_hi, const void* W_lo, int64_t ldw,
                                   int64_t w_bs, float w_scale, const float* residual, int64_t ldr, int64_t r_bs, float* C,
                                   int64_t ldc, int64_t c_bs, int64_t nb, int64_t M, int64_t N, int64_t K, int32_t causal,
                                   gnnlm_stream_t stream);

/* fp32-parity product in TWO tensor-pass equivalents (the large ntgt-side projections of hgt.py:320-322,347-348,401 and the
 * rotation of pq_wrapper.py:202): the fp16 main product a_hi w_hi (kind::f16) plus the two 2^-11-sized correction products
 * a_hi w_lo + a_lo w_hi as FP8 MMAs (kind::f8f6f4, e4m3 x e4m3, twice the fp16 rate) into the same fp32 accumulator.
 *   C[m, n] = (1 / w_scale) * sum_k A[m, k] W[n, k] + bias[n],   A = [A1 | A2] along k (K = K1 + K2; K2 = 0: one source)
 * A1 / A2: split-fp16 buffers (GNNLM_F16X2; only the hi half [., 0:Ki) is read, so lda >= Ki suffices), lda in fp16 elements;
 * A1q / A2q: their e4m3 companions [M, 2*Ki] bytes (ldq >= 2*Ki): hi8 = e4m3(hi) in [0, Ki), lo8 = e4m3(2^10 * lo) in [Ki, 2Ki)
 *   -- written by the producing kernels (gnnlm_layernorm_q8 / gnnlm_hgt_cluster_attn_q8 / gnnlm_pq_gather_decode_presplit_q8)
 *   or by gnnlm_split_to_q8;
 * W_hi fp16 [N, K] from gnnlm_split_f16 (scaled by w_scale), W8 [N, 2K] bytes from gnnlm_quant_w8: lo8 = e4m3(w_lo) in [0, K),
 *   hi8 = e4m3(2^-10 * w_hi) in [K, 2K).  K1 must be a multiple of 64, K2 of 16; C F32 / BF16 / F16X2. */
int32_t gnnlm_split_to_q8(const void* x, int64_t ldx, void* q, int64_t ldq, int64_t rows, const int32_t* rows_dev, int64_t d,
                          gnnlm_stream_t stream);
int32_t gnnlm_quant_w8(const void* w_hi, const void* w_lo, int64_t ldw, void* q, int64_t ldq, int64_t N, int64_t K,
                       gnnlm_stream_t stream);
int32_t gnnlm_linear_f16f8(const void* A1, const void* A1q, int64_t lda1, int64_t ldq1, int64_t K1, const void* A2,
                           const void* A2q, int64_t lda2, int64_t ldq2, int64_t K2, const void* W_hi, const void* W8,
                           float w_scale, int64_t ldw, int64_t ldw8, const float* bias, void* C, int32_t c_dtype, int64_t ldc,
                           int64_t M, const int32_t* m_dev, int64_t N, void* C8, gnnlm_stream_t stream);

/* Same contraction, but instead of storing C the epilogue keeps, per row and per column tile,
 * (max, sum exp(x - max)) and the single column `pick[m]` -- the [rows, vocab] tensor of
 * AdaptiveSoftmax.get_log_prob (adaptive_softmax.py:184-203) is never written.
 *  pick [M] int32 column to extract per row (-1: none); part_max / part_sum [M, n_tiles] fp32 with
 *  n_tiles = gnnlm_lse_num_tiles(N, math); picked [M] fp32. */
int64_t gnnlm_lse_num_tiles(int64_t N, int32_t math);
int32_t gnnlm_linear_lse(const void* A, int32_t a_dtype, int64_t lda, const void* W, const void* W_lo,
                         float w_scale, int64_t ldw, const int32_t* pick, float* part_max, float* part_sum, float* picked,
                         int64_t M, const int32_t* m_dev, int64_t N, int64_t K, int32_t math,
                         gnnlm_stream_t stream);
/* out[row_map ? row_map[m] : m] (+)= picked[m] - logsumexp_m   (log-softmax at the picked column). */
int32_t gnnlm_lse_finish(const float* part_max, const float* part_sum, const float* picked, int64_t n_tiles,
                         const int32_t* row_map, float* out, int32_t accumulate, int64_t M,
                         const int32_t* m_dev, gnnlm_stream_t stream);

/* Row utilities used between stages. */
/* dst[i, :] = src[ids[i], :]  (n x d elements of `dtype`) */
int32_t gnnlm_gather_rows(const void* src, int64_t ld_src, const int32_t* ids, void* dst, int64_t ld_dst,
                          int64_t n_cap, const int32_t* n_dev, int64_t d, int32_t dtype, gnnlm_stream_t stream);
/* --reinit-nfeat (fairseq/models/transformer.py:1046-1048; fairseq/data/token_block_dataset.py:371,394): ntgt features are
 * `embed_tokens(labels)` instead of decoded keys.  dst[i, :] = table[labels[rows[node(i)]], :], node(i) = row_ids ? row_ids[i] : i;
 * table fp32 [vocab, d] = the (projected) input-embedding table, labels = the datastore values (int16 / int32, vals.npy),
 * rows = datastore row of every ntgt node (int64).  labels_out (nullable) receives the int64 token of every node (`ntgt.labels`);
 * *err (nullable) is set to 1 if a value falls outside [0, vocab) (that row is zero-filled). */
int32_t gnnlm_embed_gather(const float* table, int64_t ld_table, int64_t vocab, const void* labels, int32_t label_bytes,
                           int64_t n_datastore, const int64_t* rows, const int32_t* row_ids, float* dst, int64_t ld_dst,
                           int64_t n_cap, const int32_t* n_dev, int64_t d, int64_t* labels_out, int32_t* err,
                           gnnlm_stream_t stream);
/* y = LayerNorm(x + residual) * gamma + beta over the last dim (hgt.py:403-405; eps as nn.LayerNorm, 1e-5).
 * x fp32 [n, d]; residual nullable, [n, d] of r_dtype (F32 / BF16 / F16X2), added in fp32 before the
 * statistics -- the `trans_out + h[ntype]` of hgt.py:403 fused here rather than in the GEMM epilogue;
 * y out_dtype (F32 / BF16 / F16X2).  In-place (y == x) allowed when out_dtype == F32. */
int32_t gnnlm_layernorm(const float* x, int64_t ldx, const void* residual, int32_t r_dtype, int64_t ldr,
                        const float* gamma, const float* beta, float eps, void* y, int32_t out_dtype, int64_t ldy,
                        int64_t n_cap, const int32_t* n_dev, int64_t d, gnnlm_stream_t stream);
/* gnnlm_layernorm with a split-fp16 output plus its e4m3 companion q8 [n, 2d] bytes (ldq) for gnnlm_linear_f16f8
 * (d in {128, 256, 512, 1024}); q8 == NULL is the plain call. */
int32_t gnnlm_layernorm_q8(const float* x, int64_t ldx, const void* residual, int32_t r_dtype, int64_t ldr, const float* gamma,
                           const float* beta, float eps, void* y, int32_t out_dtype, int64_t ldy, void* q8, int64_t ldq,
                           int64_t n_cap, const int32_t* n_dev, int64_t d, gnnlm_stream_t stream);
/* fp16 / fp32 rows [rows, d] (ld_src elements) -> split-fp16 [rows, 2d] (GNNLM_F16X2, ld_dst >= 2d fp16 elements). */
int32_t gnnlm_to_split_f16(const void* src, int32_t src_dtype, int64_t ld_src, void* dst, int64_t ld_dst, int64_t rows,
                           const int32_t* rows_dev, int64_t d, gnnlm_stream_t stream);
/* The same of scale * src (fp32 source): a gradient operand scaled into the fp16 range by a power of two on its way into the operand
 * format (the training products divide it out) -- instead of a scaled fp32 copy first. */
int32_t gnnlm_scale_split_f16(const float* src, int64_t ld_src, float scale, void* dst, int64_t ld_dst, int64_t rows,
                              const int32_t* rows_dev, int64_t d, gnnlm_stream_t stream);
/* y = gelu(x), exact erf form -- the activation of HGT's input adapters `gelu(adapt_ws[t](h))` (hgt.py:505-507), used when
 * --decoder_gcn_dim differs from the embedding width.  x fp32 [rows, d]; y F32 / BF16 / F16X2. */
int32_t gnnlm_gelu(const float* src, int64_t ld_src, void* dst, int32_t dst_dtype, int64_t ld_dst, int64_t rows,
                   const int32_t* rows_dev, int64_t d, gnnlm_stream_t stream);
/* Convert fp16/fp32 rows (keys.npy slices, token_block_dataset.py:327-329) to fp32/bf16. */
int32_t gnnlm_convert(const void* src, int32_t src_dtype, void* dst, int32_t dst_dtype, int64_t n,
                      gnnlm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (4) HGT edge attention -- replaces, per edge type, apply_edges(fn.v_dot_u) (hgt.py:354), the
 *     relation_pri / sqrt(d_k) scaling (:355; folded into K' by the caller), dgl.ops.edge_softmax
 *     (:356), and multi_update_all(u_mul_e, sum, cross_reducer='mean') (:383-386).
 *     One warp per destination: shuffle reductions, online segmented softmax, no atomics.
 *
 *  out[dst] (+)= out_scale * sum_{e -> dst} softmax_dst(<q[dst,h,:], k[src_e,h,:]>)_e * v[src_e,h,:]
 *  q [n_dst, H*d_k] ldq; k, v [n_src, H*d_k] ldk, ldv; dtype F32 or BF16 for q/k/v; out fp32 ldo.
 *  CSR by destination: indptr [n_rows+1], indices [E] (NULL indices => source id = edge id, i.e.
 *  contiguous ranges); dst_ids [n_dst] nullable: the CSR row (node id) of the i-th processed
 *  destination (q and out rows are then compact, i = 0..n_dst).  Zero in-degree => contributes 0. */
int32_t gnnlm_hgt_edge_attn(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                            int32_t dtype, const int32_t* indptr, const int32_t* indices,
                            const int32_t* dst_ids, int64_t n_dst_cap, const int32_t* n_dst_dev, int32_t H,
                            int32_t d_k, float* out, int64_t ldo, float out_scale, int32_t accumulate,
                            gnnlm_stream_t stream);

/* ('ntgt','intra','ntgt') without the CSR indirection: every valid (token, neighbour) pair owns a cluster
 * of w contiguous node ids (creation order: centre, left ascending, right ascending) whose intra edges
 * are a chain with self loops (build_ntgt_edges(context=1, bidirect=True), token_block_dataset.py:395-400),
 * so the node at sorted position p attends to positions p-1, p, p+1.  One warp owns one
 * (cluster, 128 B feature slice): Q / K' / V' rows of the cluster are read exactly once, all of them in
 * flight together, and the w outputs are produced from registers -- the same arithmetic as
 * gnnlm_hgt_edge_attn over nn_indptr / nn_indices (tests compare the two).
 *  k, v [n_ntgt, H*d_k] indexed by node id.  centre_only == 0: q and out are indexed by node id too and
 *  every node of every cluster is produced.  centre_only == 1: only the centre node of each cluster is
 *  produced; q and out rows are compact, indexed by valid_base[cluster] (layer n_layers-1 of the
 *  decoder's tgt-only mode).  node_base / valid_base / cluster_nl come from gnnlm_graph_count / _fill.
 *  out is F32 or BF16 (out_dtype).  Supports cluster sizes up to 7 (neighbour context <= 3 per side). */
int32_t gnnlm_hgt_cluster_attn(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                               int32_t dtype, const int32_t* node_base, const int32_t* valid_base,
                               const int32_t* cluster_nl, int64_t n_clusters, int32_t max_cluster, int32_t centre_only,
                               int32_t H, int32_t d_k, void* out, int32_t out_dtype, int64_t ldo,
                               gnnlm_stream_t stream);
/* Split-fp16 output plus its e4m3 companion q8 ([rows, hi8 | lo8] bytes, row stride ldq8 >= 2d) for gnnlm_linear_f16f8;
 * write_lo == 0: only the fp16 hi half is stored (ldo >= d) -- hi + companion is everything that product reads.
 * q8 == NULL (write_lo = 1) is the plain call. */
int32_t gnnlm_hgt_cluster_attn_q8(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                                  int32_t dtype, const int32_t* node_base, const int32_t* valid_base,
                                  const int32_t* cluster_nl, int64_t n_clusters, int32_t max_cluster, int32_t centre_only,
                                  int32_t H, int32_t d_k, void* out, int32_t out_dtype, int64_t ldo, void* q8, int64_t ldq8,
                                  int32_t write_lo, gnnlm_stream_t stream);

/* The same with GNNLM_F24 inputs (the 3-byte form the MATH_F16F8 projection writes: 25 % fewer bytes in and out of HBM than
 * fp32 Q | K' | V'): q / k / v point at the 16-bit planes (row strides ldq / ldk / ldv in elements), q_lo8 / k_lo8 / v_lo8 at the
 * byte of the byte planes that belongs to the same element (the planes share the row stride in elements).  Split-fp16 output
 * (+ e4m3 companion, write_lo) as gnnlm_hgt_cluster_attn_q8.  Clusters of at most 7 nodes; d % 128 == 0.
 *  kv_stats (nullable, centre-only form): the k / v rows are RAW products of a deferred LayerNorm (gnnlm_rowstats_q8): K'[m] =
 *  rs_m (k_raw[m] - mean_m k_c) + k_b, V' likewise, with kv_stats [n_ntgt] = (mean, rs) per node and per-column vectors [H*d_k]. */
int32_t gnnlm_hgt_cluster_attn_hq(const void* q, const void* q_lo8, int64_t ldq, const void* k, const void* k_lo8, int64_t ldk,
                                  const void* v, const void* v_lo8, int64_t ldv, const int32_t* node_base,
                                  const int32_t* valid_base, const int32_t* cluster_nl, int64_t n_clusters, int32_t max_cluster,
                                  int32_t centre_only, int32_t H, int32_t d_k, void* out, int64_t ldo, void* q8, int64_t ldq8,
                                  int32_t write_lo, const float* kv_stats, const float* k_c, const float* k_b, const float* v_c,
                                  const float* v_b, gnnlm_stream_t stream);

/* Deferred LayerNorm of HGT layer 0 when the OPQ rotation is folded (hgt.py:401-405 with h = x rot^T, rot orthonormal): the
 * pre-norm sum is kept in the UN-rotated basis, z' = o + x (o = A-linear(t) rot, a K = d product; x the decoded features as fp16 hi
 * [rows, d] + e4m3 companion [rows, hi8 | lo8]), and the statistics of the rotated sum z = z' rot^T follow from z' alone:
 * mean = <z', u> with u = rot^T 1 / d, var = |z' - mean d u|^2 / d.  Writes z' as a gnnlm_linear_f16f8 operand (y_hi fp16 [rows, d],
 * y_q8 [rows, hi8 | lo8]) and stats [rows] = (mean, 1 / sqrt(var + eps)).  The consumers apply the normalisation as a per-row
 * affine, so the residual is never rotated (half of the output projection's flops) and the normalised rows of the non-centre nodes
 * are never materialised. */
int32_t gnnlm_rowstats_q8(const float* o, int64_t ldo, const void* x_hi, int64_t ldxh, const void* x_q8, int64_t ldxq, const float* u,
                          float eps, void* y_hi, int64_t ldy, void* y_q8, int64_t ldq, float* stats, int64_t n_cap,
                          const int32_t* n_dev, int64_t d, gnnlm_stream_t stream);

/* ('tgt','intra','tgt') as implicit causal attention inside each of B blocks of L tokens
 * (edges u -> v for u <= v, v - u < intra_ctx when intra_ctx > 0; token_block_dataset.py:586-594). */
int32_t gnnlm_hgt_causal_attn(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v,
                              int64_t ldv, int32_t dtype, int64_t B, int64_t L, int64_t intra_ctx, int32_t H,
                              int32_t d_k, float* out, int64_t ldo, float out_scale, int32_t accumulate,
                              gnnlm_stream_t stream);

/* The same attention as ONE flash kernel on the tensor cores at fp32 parity (three-pass fp16 split on mma.sync, fp32
 * accumulation, online softmax; S and P never leave the SM): replaces the heads_split / batched-GEMM / causal_softmax_split
 * sequence below for d_k in {64, 128}.  Reference: fairseq/models/hgt.py:350-358 over the edges of
 * fairseq/data/token_block_dataset.py:586-594.
 *  q        fp32 [B*L, >= H*d_k] (row stride ldq)
 *  k_split, v_split  K' / V' as split fp16 (GNNLM_F16X2): hi at [t, h*d_k + j], lo at [t, lo_off + h*d_k + j], row stride ldkv
 *           (elements) -- e.g. column slices of a projection written with c_dtype = GNNLM_F16X2
 *  out      fp32 [B*L, >= H*d_k]: out (+)= out_scale * attention (accumulate != 0 adds to what is there)
 *  out_split  optional: the final value is written as split fp16 (hi at column c, lo at os_lo + c, row stride ldos) INSTEAD of
 *           to `out`, which is then only read (accumulate != 0) -- the operand format of the output projection. */
int32_t gnnlm_hgt_causal_flash(const float* q, int64_t ldq, const void* k_split, const void* v_split, int64_t ldkv,
                               int64_t lo_off, int64_t B, int64_t L, int64_t intra_ctx, int32_t H, int32_t d_k, float* out,
                               int64_t ldo, void* out_split, int64_t ldos, int64_t os_lo, float out_scale, int32_t accumulate,
                               gnnlm_stream_t stream);

/* tcgen05 form of the same flash attention (d_k = 128): both products on tcgen05.mma with TMEM accumulators, operands by TMA.
 *  qk_split  [B*L, ldqk] fp16: Q hi | K' hi | Q lo | K' lo, each d = H*d_k columns wide (gnnlm_to_split_f16 of the Q | K' columns)
 *  vt        [2][B*H*d_k][ldvt] fp16: V'^T hi, then lo -- row (b*H + h)*d_k + j holds V'[b*L + 0 .. L, h*d_k + j]
 *            (gnnlm_heads_transpose_split_f16 per block); ldvt >= L, a multiple of 8
 *  out / out_split / out_scale / accumulate as gnnlm_hgt_causal_flash. */
int32_t gnnlm_hgt_causal_flash_tc(const void* qk_split, int64_t ldqk, int64_t d, const void* vt, int64_t ldvt, int64_t B, int64_t L,
                                  int64_t intra_ctx, int32_t H, int32_t d_k, float* out, int64_t ldo, void* out_split,
                                  int64_t ldos, int64_t os_lo, float out_scale, int32_t accumulate, gnnlm_stream_t stream);

/* ('ntgt','inter','tgt') attention with the K' / V' projections moved from the ~k*T centre nodes to the T target tokens
 * (every centre row is used by exactly one (token, neighbour) pair): with q~[t,h] = W_k'[h]^T q[t,h] in R^d (a per-head GEMM
 * of the caller) this kernel computes, per token and head, alpha = softmax_c <h_c, q~[t,h]> over the token's centre rows and
 * a[t,h] = sum_c alpha_c h_c; the caller finishes with out[t,h] = W_v'[h] a[t,h] (+ b_v' when the token has a neighbour).
 * Same value as hgt.py:339-358 for this edge type up to fp32 re-association (b_k' cancels inside the softmax).
 *  q_tilde [H, n_all, d] fp32 (head stride q_head_stride, row stride d), rows t0 .. t0 + n_tokens are processed
 *  hc      compact centre features, row i = i-th inter edge (F32 [*, d] / BF16 [*, d] / F16X2 [*, 2d]; ldh elements)
 *  inter_indptr [n_tokens + 1]: token t0 + i owns rows [indptr[i], indptr[i+1]) of hc
 *  a_out   [H, n_all, 2d] split fp16 (head stride a_head_stride, row stride lda): zero rows for tokens without neighbours
 *  t_agg   [n_all, d] fp32 (ldt): row t := out_scale * b_v' if the token has a neighbour else 0 (the caller's final
 *          per-head GEMM accumulates out_scale * W_v' a on top).  H in {4, 8, 12, 16}, d % 4 == 0, d <= 1024. */
int32_t gnnlm_hgt_inter_fused(const float* q_tilde, int64_t q_head_stride, const void* hc, int32_t hc_dtype, int64_t ldh,
                              const int32_t* inter_indptr, int64_t t0, int64_t n_tokens, int32_t H, int64_t d, void* a_out,
                              int64_t a_head_stride, int64_t lda, const float* bias_v, float out_scale, float* t_agg,
                              int64_t ldt, gnnlm_stream_t stream);

/* Tensor-core form of the same causal attention for MATH_F16X3 (fp32 parity): per block and head,
 * S = Q K'^T and O = softmax_causal(S) V' are two gnnlm_linear calls on split-fp16 operands; these three
 * streaming kernels produce the operands.
 *  gnnlm_heads_split_f16: src fp32 [L, H*d_k] (row stride ld) -> a_style = 1: hi = split-fp16 [H, L, 2*d_k]
 *    (A operands, lo unused); a_style = 0: hi, lo fp16 [H, L, d_k] each (W operands, scale 1).
 *  gnnlm_heads_transpose_split_f16: src fp32 [L, H*d_k] -> hi, lo fp16 [H, d_k, L] (W operands of P V').
 *  gnnlm_causal_softmax_split: S fp32 [H, L, L] -> P split-fp16 [H, L, 2L]; row i = softmax over
 *    j in [max(0, i - intra_ctx + 1), i] (all j <= i when intra_ctx == 0), zeros elsewhere -- written for
 *    j < (i / k_tile + 1) * k_tile only when k_tile > 0 (256 for a `causal = 2` consumer), the whole row when 0;
 *    S entries with j > i are never read (a `causal = 1` producer leaves tiles above the diagonal unwritten). */
int32_t gnnlm_heads_split_f16(const float* src, int64_t ld, int64_t L, int32_t H, int32_t d_k, int32_t a_style, void* hi,
                              void* lo, gnnlm_stream_t stream);
int32_t gnnlm_heads_transpose_split_f16(const float* src, int64_t ld, int64_t L, int32_t H, int32_t d_k, void* hi, void* lo,
                                        gnnlm_stream_t stream);
int32_t gnnlm_causal_softmax_split(const float* S, int64_t L, int64_t intra_ctx, int32_t H, int64_t k_tile, void* P,
                                   gnnlm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (5) Adaptive-softmax bookkeeping + kNN-LM interpolation + NLL -- replaces adapt_target
 *     (adaptive_softmax.py:122-145), KNNModel.get_knn_prob minus the faiss search
 *     (knn/knn_model.py:187-217), combine_knn_and_vocab_probs (fairseq/sequence_scorer.py:55-68),
 *     combinetow_probs (fairseq/models/transformer.py:1055-1062) and the score accumulation of
 *     fairseq_cli/eval_lm.py:273-274.
 * ---------------------------------------------------------------------------------------------- */

/* cutoff [n_cut] int64 on the HOST (n_cut = 1 + #tails, last = vocab). For every token:
 *  head_pick [T] = target if target < cutoff[0] else cutoff[0] + cluster;
 *  for tail i: rows_i = tokens whose target is in [cutoff[i], cutoff[i+1]) in ascending order,
 *  tail_rows [(n_cut-1), T] int32, tail_pick [(n_cut-1), T] int32 (= target - cutoff[i]),
 *  tail_count [n_cut-1] int32.  Order inside a cluster is ascending token id (deterministic). */
int32_t gnnlm_adapt_target(const int64_t* target, int64_t T, const int64_t* cutoff_host, int32_t n_cut,
                           int32_t* head_pick, int32_t* tail_rows, int32_t* tail_pick, int32_t* tail_count,
                           gnnlm_stream_t stream);

/* Per token: p_knn = sum_j softmax(sims/T)_j [vals[ids_j] == target] with ids == -1 masked
 * (sims = dists * sim_sign: +1 do_not_recomp_ip, -1 do_not_recomp_l2); recall = #matches;
 * lp = logsumexp(lm_lp + ln(1-lambda), ln(p_knn + 1e-10) + ln(lambda)).  lambda == 0 or dists == NULL
 * => lp = lm_lp.  Optional orig-LM mixing first: lm_lp = logsumexp(orig_lp + ln(a), lm_lp + ln(1-a)).
 * Accumulates sum(lp * w) and sum(w) into nll_acc[0..1] (fp64, device) when non-NULL, where
 * w = weight[t] (fp32, nullable => 1) and w = 0 for pad targets (pad_id >= 0; strip_pad,
 * sequence_scorer.py:159) and for positions t % L < loss_start[t / L] (loss_start int32 [T/L] nullable;
 * start_indices of --gcn-context-window, sequence_scorer.py:156-162).
 *  vals: int16/int32 table (val_bytes = 2|4). */
int32_t gnnlm_knn_mix_nll(const float* lm_lp, const float* orig_lp, float orig_ratio, const float* dists,
                          const int64_t* ids, int64_t k_nn, const void* vals, int32_t val_bytes,
                          int64_t n_datastore, const int64_t* target, float sim_sign, float temperature,
                          float lambda, const float* weight, int64_t pad_id, const int32_t* loss_start, int64_t L,
                          float* out_lp, float* out_knn_prob, int32_t* out_recall, double* nll_acc, int64_t T,
                          gnnlm_stream_t stream);

/* Full-vocabulary kNN distribution (knn_model.py:202-208): probs [T, V] fp32, zero-filled by the
 * callee, += softmax weights at vals[ids]; kept for API parity with get_knn_prob(targets=None). */
int32_t gnnlm_knn_full_prob(const float* dists, const int64_t* ids, int64_t k_nn, const void* vals,
                            int32_t val_bytes, int64_t n_datastore, float sim_sign, float temperature,
                            float* probs, int64_t V, int64_t T, gnnlm_stream_t stream);

/* Similarity recompute -- metric_type `l2` / `ip` of KNNModel.get_knn_prob (knn/knn_model.py:159-177), for pipelines
 * that keep only the neighbour ids (knn/find_knn.py:65-66).  metric: 0 = l2 (sims = -||q - key||^2), 1 = ip.
 * sims [T, k_nn] fp32 feed gnnlm_knn_mix_nll / gnnlm_knn_full_prob as `dists` with sim_sign = +1.  ids == -1 wrap to
 * the last datastore row like numpy indexing (:163,:169); the consumer masks them (:193).
 *
 *  _keys: keys [n_datastore, d] fp32 / fp16 (GNNLM_F32 / GNNLM_F16; the datastore's keys.npy), d % 8 == 0.
 *         normalise bit 0: L2-normalise the gathered keys (cosine index, `ip`, :171-172);
 *         bit 1: L2-normalise the queries first (cosine index, :181-184).
 *  _pq:   keys only as PQ codes [n_datastore, M] uint8 + centroids [M, 256, dsub] (+ OPQ bias [M*dsub], nullable):
 *         similarity to the DECODED key x^ = (y - b) A (knn/pq_wrapper.py:169-203) by asymmetric distance computation.
 *         rotated [T, M*dsub] = queries A^T (a gnnlm_linear call; pass the queries themselves when there is no OPQ
 *         transform).  l2 assumes A A^T = I (OPQ rotations are orthonormal).  M % 4 == 0, M*(256+dsub)*4 B <= 220 KB.
 *         normalise as above (an extension: the reference needs the raw keys for a cosine index); bit 0 reads
 *         key_norm2 [M, 256] = ||centroid[m, c] - b_m||^2, the squared norm of a decoded key being the sum over m (A A^T = I). */
int32_t gnnlm_knn_sims_keys(const float* queries, int64_t ldq, const void* keys, int32_t key_dtype, int64_t n_datastore,
                            int32_t d, const int64_t* ids, int64_t k_nn, int32_t metric, int32_t normalise, float* sims,
                            int64_t T, gnnlm_stream_t stream);
int32_t gnnlm_knn_sims_pq(const float* queries, int64_t ldq, int32_t d_q, const float* rotated, int64_t ldr,
                          const uint8_t* codes, int64_t n_datastore, int32_t M, int32_t dsub, const float* centroids,
                          const float* bias, const int64_t* ids, int64_t k_nn, int32_t metric, const float* key_norm2,
                          int32_t normalise, float* sims, int64_t T, gnnlm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (9) Training backward of the HGT fine-tuning step (SURVEY.md 8f rank 4: `--freeze` trains decoder.hgt_decoder.* only,
 *     fairseq/models/transformer_lm.py:183-186, under fairseq/criterions/adaptive_loss.py:31-83).  The reference obtains these
 *     from autograd over DGL's SDDMM / edge_softmax / SpMM (hgt.py:350-358,383-386), F.layer_norm (hgt.py:405) and
 *     F.cross_entropy; here they are explicit kernels (fp32), driven by torch.autograd.Function wrappers in train.py.
 *
 * gnnlm_hgt_edge_attn_bwd: backward of gnnlm_hgt_edge_attn / gnnlm_hgt_causal_attn for fp32 q / k / v and out = scale * attention.
 *   dq [n_dst, d] is written; dk, dv [n_src, d] are ACCUMULATED with atomics (zero them first).  Edges: the CSR of the forward
 *   (indptr / indices / dst_ids), or -- causal_L > 0 -- the implicit causal edges inside blocks of causal_L tokens.
 * gnnlm_layernorm_bwd: y = LayerNorm(o + residual) * gamma + beta; dx = d o = d residual is written, dgamma / dbeta accumulated.
 * gnnlm_xent_fwd_bwd: one adaptive-softmax cluster: loss += sum_r -log softmax(logits[r])[target[r]] (fp64 accumulate) and
 *   logits[r] <- grad_scale * (softmax(logits[r]) - onehot(target[r])) in place; target < 0 rows are ignored.
 * gnnlm_transpose_f32 (rows past the live count / up to rows_pad are written as zeros: k-padding of dW = dY^T X),
 * gnnlm_colsum_f32 (out += column sums: bias gradients), gnnlm_axpy_f32 (y += a x), gnnlm_scatter_add_rows
 * (dst[ids[r]] += src[r]: backward of gnnlm_gather_rows). */
/* gnnlm_transpose_split_f16: (scale * src)^T as split fp16 in one pass -- the operands of dW = dY^T X for the 3xFP16 products straight
 * from the row-major fp32 tensors: src [rows, cols] -> a_style != 0: hi [cols, 2 * rows_pad], hi | lo in one row (A operand);
 * a_style == 0: hi, lo [cols, rows_pad] (W operand).  Columns rows .. rows_pad are zeros; rows_pad even. */
int32_t gnnlm_transpose_split_f16(const float* src, int64_t ld_src, int64_t rows, int64_t cols, float scale, int64_t rows_pad,
                                  int32_t a_style, void* hi, void* lo, gnnlm_stream_t stream);
int32_t gnnlm_hgt_edge_attn_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                                const float* dout, int64_t ldo, const int32_t* indptr, const int32_t* indices,
                                const int32_t* dst_ids, int64_t n_dst_cap, const int32_t* n_dst_dev, int64_t causal_L,
                                int64_t intra_ctx, int32_t H, int32_t d_k, float scale, float* dq, int64_t lddq, float* dk,
                                int64_t lddk, float* dv, int64_t lddv, float p_drop, uint64_t seed, gnnlm_stream_t stream);
/* A CSR edge type whose edge set is SYMMETRIC (u -> v iff v -> u, equal multiplicities; n_dst == n_src == n -- the ntgt-intra-ntgt
 * chains of build_ntgt_edges(bidirect=True), token_block_dataset.py:395-400) without atomics: the by-destination pass writes dq and
 * `stats` [n*H*3], a by-source pass over the SAME CSR rows writes dk, dv (NOT accumulated).  (gnnlm_hgt_edge_attn_bwd itself uses
 * plain stores instead of atomics when indices == NULL: source id = edge id, no two edges share a source.) */
int32_t gnnlm_hgt_edge_attn_bwd_sym(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                                    const float* dout, int64_t ldo, const int32_t* indptr, const int32_t* indices, int64_t n,
                                    int32_t H, int32_t d_k, float scale, float* dq, int64_t lddq, float* dk, int64_t lddk, float* dv,
                                    int64_t lddv, float* stats, float p_drop, uint64_t seed, gnnlm_stream_t stream);
/* Backward of gnnlm_hgt_cluster_attn (all-nodes form, fp32): the ntgt-intra-ntgt chains of the non-deduplicating builder, one warp per
 * (cluster, head) walking the chain with a three-row window in registers -- every row read / written once, no atomics.  dq, dk, dv
 * [n_ntgt, H*d_k] are written for every node of a valid cluster (NOT accumulated).  d_k in {32, 64, 128}. */
int32_t gnnlm_hgt_cluster_attn_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                                   const float* dout, int64_t ldo, const int32_t* node_base, const int32_t* cluster_nl,
                                   int64_t n_clusters, int32_t H, int32_t d_k, float scale, float* dq, int64_t lddq, float* dk,
                                   int64_t lddk, float* dv, int64_t lddv, float p_drop, uint64_t seed, gnnlm_stream_t stream);
/* The implicit causal edges without atomics: a by-destination pass writes dq and the softmax statistics {max, 1 / sum, D} per
 * (destination, head) into `stats` [B*L*H*3] floats; a by-source pass writes dk, dv (NOT accumulated). */
int32_t gnnlm_hgt_causal_attn_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                                  const float* dout, int64_t ldo, int64_t B, int64_t L, int64_t intra_ctx, int32_t H, int32_t d_k,
                                  float scale, float* dq, int64_t lddq, float* dk, int64_t lddk, float* dv, int64_t lddv,
                                  float* stats, float p_drop, uint64_t seed, gnnlm_stream_t stream);
/* The same backward in GEMM form (tensor cores at fp32 parity): S = Q K'^T and G = dOut V'^T come from gnnlm_linear_batched_f16x3
 * (causal = 1), this entry turns them into the split-fp16 A operands [H, L, 2L] of the three closing products -- dS row-major
 * (dQ = dS K', causal = 2), W^T (dV' = W^T dOut) and dS^T (dK' = dS^T Q) -- with P = softmax_causal(S), D_i = sum_j P_ij beta_ij G_ij,
 * W_ij = scale beta_ij P_ij, dS_ij = scale P_ij (beta_ij G_ij - D_i), beta the attention-dropout multiplier of edge
 * (row0 + i, row0 + j, head).  S, G fp32 [H, L, L] (entries above the diagonal are never read); stats [H, L, 3] scratch.
 * Only the 64 x 64 tiles on or below the diagonal are written: dS / WT / dST must be zero above it (allocate them zeroed once
 * and reuse them).  L % 64 == 0. */
int32_t gnnlm_causal_softmax_bwd_split(const float* S, const float* G, int64_t L, int64_t intra_ctx, int32_t H, int64_t row0,
                                       float scale, float p_drop, uint64_t seed, float* stats, void* dS, void* WT, void* dST,
                                       gnnlm_stream_t stream);
/* Dropout in training (hgt.py:74-75: `drop` on the output projection :401, `attn_drop` on the edge-softmax weights :356; the
 * adaptive softmax's input / tail dropouts, adaptive_softmax.py:156,101).  A mask is a pure function of (seed, element): splitmix64
 * of seed + index * 0x9E3779B97F4A7C15, keep iff its top 24 bits >= floor(p * 2^24), kept values scaled by 1 / (1 - p); element
 * index = row * cols + col (gnnlm_dropout_f32) or (dst << 38) ^ (src << 6) ^ head (attention; `p_drop` / `seed` of the two
 * backward entries above and of the training forward below).  Forward and backward regenerate the mask; nothing is stored.
 * gnnlm_hgt_edge_attn_train_fwd: out (+)= scale * sum_e dropout(alpha)_e V'[src_e] for fp32 q / k / v, CSR or implicit causal
 * edges (the evaluation kernels have no dropout). */
int32_t gnnlm_hgt_edge_attn_train_fwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                                      const int32_t* indptr, const int32_t* indices, int64_t n_dst, int64_t causal_L,
                                      int64_t intra_ctx, int32_t H, int32_t d_k, float scale, int32_t accumulate, float* out,
                                      int64_t ldo, float p_drop, uint64_t seed, gnnlm_stream_t stream);
/* Fast forms of the training forward (the generic kernel above handles any CSR; it also takes the contiguous-source case
 * indices == NULL in one pass per (destination, head) when d_k is 32 / 64 / 128):
 *   gnnlm_causal_softmax_drop_split: gnnlm_causal_softmax_split with the dropout multiplier of edge (row0 + i, row0 + j, head) on
 *     the softmax weights -- the middle of the GEMM form of the causal edges (S from gnnlm_linear_batched_f16x3 causal = 1, P~ V'
 *     with causal = 2);
 *   gnnlm_hgt_cluster_attn_train_fwd: the ntgt-intra-ntgt chains, one warp per (cluster, head); out [n_ntgt, H*d_k] fp32 written
 *     for every node of a valid cluster. */
int32_t gnnlm_causal_softmax_drop_split(const float* S, int64_t L, int64_t intra_ctx, int32_t H, int64_t k_tile, int64_t row0,
                                        float p_drop, uint64_t seed, void* P, gnnlm_stream_t stream);
int32_t gnnlm_hgt_cluster_attn_train_fwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                                         const int32_t* node_base, const int32_t* cluster_nl, int64_t n_clusters, int32_t H,
                                         int32_t d_k, float scale, float* out, int64_t ldo, float p_drop, uint64_t seed,
                                         gnnlm_stream_t stream);
int32_t gnnlm_dropout_f32(const float* x, int64_t ldx, float* y, int64_t ldy, int64_t rows, int64_t cols, float p_drop,
                          uint64_t seed, gnnlm_stream_t stream);
int32_t gnnlm_layernorm_bwd(const float* o, int64_t ldo, const float* residual, int64_t ldr, const float* gamma, float eps,
                            const float* dy, int64_t ldy, int64_t rows, const int32_t* rows_dev, int64_t d, float* dx,
                            int64_t ldx, float* dgamma, float* dbeta, gnnlm_stream_t stream);
int32_t gnnlm_xent_fwd_bwd(float* logits, int64_t ld, const int64_t* target, int64_t rows, int64_t C, float grad_scale,
                           double* loss, gnnlm_stream_t stream);
int32_t gnnlm_transpose_f32(const float* src, int64_t ld_src, int64_t rows, const int32_t* rows_dev, int64_t cols, float* dst,
                            int64_t ld_dst, int64_t rows_pad, gnnlm_stream_t stream);
int32_t gnnlm_colsum_f32(const float* x, int64_t ld, int64_t rows, const int32_t* rows_dev, int64_t cols, float* out,
                         gnnlm_stream_t stream);
int32_t gnnlm_axpy_f32(float* y, int64_t ldy, const float* x, int64_t ldx, int64_t rows, const int32_t* rows_dev, int64_t cols,
                       float a, gnnlm_stream_t stream);
int32_t gnnlm_scatter_add_rows(float* dst, int64_t ld_dst, const float* src, int64_t ld_src, const int32_t* ids, int64_t rows,
                               const int32_t* rows_dev, int64_t cols, gnnlm_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (10) Exact k-nearest-neighbour search over the datastore -- replaces the faiss index search that writes the neighbour-id files
 *      (knn/find_knn.py:29-71) and KNNModel.get_knns (knn/knn_model.py:87-101).  For every query q the k rows x with the highest
 *      score s(q, x) = q.x + bias(x), ties by smaller id; bias = -1/2 ||x||^2 ranks like squared L2 (faiss METRIC_L2), bias = 0 is
 *      inner product.  The datastore is scanned in spans of increasing ids; per span:
 *
 * gnnlm_knn_filter_f16x3: the 3xFP16 tcgen05 product of the span's keys [n_keys, 2d] (split fp16, GNNLM_F16X2, ldk >= 2d; row r has
 *   id id_base + r, id_base + n_keys < 2^31) with the queries q_hi / q_lo [n_q, d] fp16 (gnnlm_split_f16 with scale 1, ldq >= d),
 *   plus key_bias [n_keys] fp32 (nullable = 0).  Nothing per (key, query) is stored: a score with s > thr[q] is appended to
 *   cand_s / cand_id [n_q, cap] (order within a span unspecified) and counted in cand_cnt[q] (zero it before the first span).  Past cap
 *   the writes stop and the count keeps growing: cand_cnt[q] > cap flags an overflowed query.  1 <= cap <= 4096, d % 8 == 0.
 * gnnlm_topk_merge: per query, merge the running top_s / top_id [n_q, k] (sorted, id -1 = empty, score -inf) with its min(cnt, cap)
 *   candidates into the new sorted top-k, write thr[q] = its k-th score (-inf while fewer than k are held) and reset cand_cnt[q]
 *   to 0.  Queries with cand_cnt[q] > cap are left untouched (count included).  1 <= k <= 2048, 1 <= cap <= 4096.  Deterministic.
 * gnnlm_knn_key_bias: out[i] = -1/2 ||x_i||^2 (fp32, fixed summation order) of fp32 / fp16 rows x [n, d] (ld elements).
 * gnnlm_knn_key_bias_pq: the same for PQ-decoded keys: out[i] = -1/2 sum_m norm2[m, codes[i, m]], norm2 [M, 256] fp32 =
 *   ||centroid[m, c] - b_m||^2, codes [n, M] uint8. */
int32_t gnnlm_knn_filter_f16x3(const void* keys, int64_t ldk, int64_t n_keys, int64_t id_base, const void* q_hi, const void* q_lo,
                               int64_t ldq, int64_t n_q, int64_t d, const float* key_bias, const float* thr, float* cand_s,
                               int32_t* cand_id, int32_t* cand_cnt, int64_t cap, gnnlm_stream_t stream);
int32_t gnnlm_topk_merge(float* top_s, int32_t* top_id, int64_t n_q, int32_t k, const float* cand_s, const int32_t* cand_id,
                         int32_t* cand_cnt, int64_t cap, float* thr, gnnlm_stream_t stream);
int32_t gnnlm_knn_key_bias(const void* x, int32_t dtype, int64_t ld, int64_t n, int64_t d, float* out, gnnlm_stream_t stream);
int32_t gnnlm_knn_key_bias_pq(const uint8_t* codes, int64_t n, int32_t M, const float* norm2, float* out, gnnlm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNNLM_SM100_H */
