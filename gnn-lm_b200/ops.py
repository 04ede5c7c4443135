"""Thin torch-tensor wrappers over the C ABI (include/gnnlm_sm100.h).

torch is plumbing here: it owns device memory and the current stream; every computation below is
a call into libgnnlm_sm100.so.  No function in this file has a CPU or torch-op fallback.
"""
from typing import Optional

import torch

from . import _lib as L

_I32 = torch.int32
SPLIT = "split"          # out_dtype selector for the split-fp16 activation format (GNNLM_F16X2)
SPLIT_Q8 = "split+q8"    # the same with the e4m3 companion (Split.q8) written by the producing kernel (MATH_F16F8 GEMM operands)
HI_Q8 = "hi+q8"          # fp16 hi half + companion only (no lo half): for matrices that only feed gnnlm_linear_f16f8
HILO8 = "f24"            # GNNLM_F24: 16-bit plane + byte plane (3 bytes per element): Q | K' | V' of the ntgt side in MATH_F16F8


class HiLo8:
    """An fp32 matrix [rows, d] rounded to its top three bytes (GNNLM_F24): `hi` [rows, d] bfloat16 (bytes 3, 2 of every value: its
    bf16 truncation) + `lo8` [rows, d] uint8 (byte 1).  Written by gnnlm_linear_f16f8, read by gnnlm_hgt_cluster_attn_hq.  Column
    slices keep the two planes aligned."""

    def __init__(self, hi: torch.Tensor, lo8: torch.Tensor):
        assert hi.dtype == torch.bfloat16 and lo8.dtype == torch.uint8 and hi.shape == lo8.shape and hi.stride(0) == lo8.stride(0)
        self.hi, self.lo8 = hi, lo8

    @staticmethod
    def empty(rows: int, d: int, device) -> "HiLo8":
        return HiLo8(torch.empty((rows, d), device=device, dtype=torch.bfloat16), torch.empty((rows, d), device=device, dtype=torch.uint8))

    @property
    def shape(self):
        return self.hi.shape

    @property
    def device(self):
        return self.hi.device

    def __getitem__(self, idx):
        return HiLo8(self.hi[idx], self.lo8[idx])

    def float(self) -> torch.Tensor:
        """fp32 reconstruction (tests / API boundary; torch ops)."""
        bits = ((self.hi.contiguous().view(torch.int16).to(torch.int32) & 0xFFFF) << 16) | (self.lo8.to(torch.int32) << 8)
        return bits.view(torch.float32)


class Split:
    """An fp32 matrix [rows, d] stored as split fp16 (GNNLM_F16X2): `.data` is [rows, 2d] float16 with
    hi = fp16(x) in columns [0, d) and lo = fp16(x - hi) in [d, 2d).  Activation format of MATH_F16X3.

    `.q8` (optional): the e4m3 companion [rows, 2d] bytes (hi8 = e4m3(hi) | lo8 = e4m3(2^10 lo)) -- the operands of the FP8
    correction MMAs of gnnlm_linear_f16f8 (MATH_F16F8), written by the kernel that produced `data` (or by to_q8).
    A matrix that only ever feeds that product may drop its lo half: `.data` is then [rows, d] (hi only, `has_lo` False) and
    nothing but linear_f16f8 accepts it."""

    def __init__(self, data: torch.Tensor, d: int, q8: Optional[torch.Tensor] = None):
        assert data.dtype == torch.float16 and data.dim() == 2 and data.shape[1] in (d, 2 * d) and data.stride(1) == 1
        assert q8 is None or (q8.dtype == torch.uint8 and q8.shape == (data.shape[0], 2 * d) and q8.stride(1) == 1)
        self.data, self.d, self.q8 = data, d, q8
        self.has_lo = data.shape[1] == 2 * d
        assert self.has_lo or q8 is not None

    @staticmethod
    def empty(rows: int, d: int, device, q8: bool = False, lo: bool = True) -> "Split":
        return Split(torch.empty((rows, 2 * d if lo else d), device=device, dtype=torch.float16), d,
                     torch.empty((rows, 2 * d), device=device, dtype=torch.uint8) if q8 else None)

    @property
    def shape(self):
        return (self.data.shape[0], self.d)

    @property
    def device(self):
        return self.data.device

    def float(self) -> torch.Tensor:
        """fp32 reconstruction (API-boundary convenience, torch ops)."""
        assert self.has_lo, "hi + e4m3 companion only: not reconstructible to fp32"
        return self.data[:, :self.d].float() + self.data[:, self.d:].float()


def empty_act(rows: int, d: int, act, device):
    if act == HILO8:
        return HiLo8.empty(rows, d, device)
    if act in (SPLIT, SPLIT_Q8, HI_Q8):
        return Split.empty(rows, d, device, q8=act != SPLIT, lo=act != HI_Q8)
    return torch.empty((rows, d), device=device, dtype=act)


def _mat(x):
    """(pointer, dtype code, leading dimension, logical columns) of a Tensor or Split."""
    if isinstance(x, Split):
        assert x.has_lo, "this kernel reads / writes both fp16 halves"
        return L.ptr(x.data), L.F16X2, x.data.stride(0), x.d
    assert x.dim() == 2 and x.stride(1) == 1
    return L.ptr(x), L.dtype_code(x.dtype), x.stride(0), x.shape[1]


def to_split(x: torch.Tensor, rows_dev=None, scale: float = 1.0) -> Split:
    """fp16 / fp32 [rows, d] -> split fp16 (of scale * x when scale != 1: fp32 sources, gnnlm_scale_split_f16)."""
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype in (torch.float16, torch.float32)
    out = Split.empty(x.shape[0], x.shape[1], x.device)
    if scale != 1.0:
        assert x.dtype == torch.float32
        L.call("gnnlm_scale_split_f16", L.ptr(x), x.stride(0), float(scale), L.ptr(out.data), out.data.stride(0), x.shape[0],
               L.ptr(rows_dev), x.shape[1], L.stream_ptr())
        return out
    L.call("gnnlm_to_split_f16", L.ptr(x), L.dtype_code(x.dtype), x.stride(0), L.ptr(out.data), out.data.stride(0), x.shape[0],
           L.ptr(rows_dev), x.shape[1], L.stream_ptr())
    return out


def _dev_count(t: Optional[torch.Tensor]):
    return L.ptr(t)


def linear(A, W: torch.Tensor, bias: Optional[torch.Tensor] = None, *, W_lo: Optional[torch.Tensor] = None,
           residual=None, out=None, out_dtype=None, m_dev: Optional[torch.Tensor] = None, math: int = L.MATH_FP32_SIMT,
           tag=None, w_scale: float = 1.0):
    """C = A @ W^T + bias (+ residual).  A [M,K] Tensor or Split, W [N,K]; out_dtype a torch dtype or ops.SPLIT."""
    a_ptr, a_code, lda, K = _mat(A)
    M = A.shape[0]
    N = W.shape[0]
    math = L.base_math(math)
    assert W.dim() == 2 and W.stride(1) == 1 and W.shape[1] == K, (A.shape, W.shape)
    dev = W.device
    if out is None:
        out = empty_act(M, N, out_dtype or torch.float32, dev)
    c_ptr, c_code, ldc, n_out = _mat(out)
    assert n_out == N and out.shape[0] == M
    r_ptr, r_code, ldr = None, 0, 0
    if residual is not None:
        r_ptr, r_code, ldr, n_r = _mat(residual)
        assert n_r == N
    L.call("gnnlm_linear", a_ptr, a_code, lda, L.ptr(W), L.ptr(W_lo), float(w_scale), W.stride(0), L.ptr(bias), r_ptr, r_code,
           ldr, c_ptr, c_code, ldc, M, _dev_count(m_dev), N, K, math, L.stream_ptr(), tag=tag or f"linear[{N}x{K}]", work=(M, N, K))
    return out


def to_q8(x: Split, rows_dev=None) -> Split:
    """Attach the e4m3 companion to a split-fp16 matrix (standalone pass; the big producers write it themselves)."""
    if x.q8 is None:
        q = torch.empty(x.data.shape, device=x.data.device, dtype=torch.uint8)
        L.call("gnnlm_split_to_q8", L.ptr(x.data), x.data.stride(0), L.ptr(q), q.stride(0), x.data.shape[0], L.ptr(rows_dev), x.d,
               L.stream_ptr())
        x.q8 = q
    return x


def quant_w8(w_hi: torch.Tensor, w_lo: torch.Tensor) -> torch.Tensor:
    """fp16 (hi, lo) halves of a scaled weight [N, K] -> e4m3 bytes [N, 2K] (lo8 | 2^-10 hi8) for gnnlm_linear_f16f8."""
    N, K = w_hi.shape
    q = torch.empty((N, 2 * K), device=w_hi.device, dtype=torch.uint8)
    L.call("gnnlm_quant_w8", L.ptr(w_hi), L.ptr(w_lo), w_hi.stride(0), L.ptr(q), q.stride(0), N, K, L.stream_ptr())
    return q


def f16f8_supported(K1: int, K2: int = 0) -> bool:
    return K1 % 64 == 0 and K2 % 16 == 0


def linear_f16f8(A1: Split, W_hi, W8, bias=None, *, A2: Optional[Split] = None, w_scale=1.0, out=None, out_dtype=None,
                 m_dev=None, tag=None):
    """C = [A1 | A2] @ W^T + bias in two tensor-pass equivalents (fp16 main product + FP8 corrections, MATH_F16F8).
    A1 / A2 split fp16 with e4m3 companions; W_hi fp16 [N, K1 + K2] (scaled), W8 = quant_w8(W_hi, W_lo)."""
    M, K1 = A1.shape
    K2 = 0 if A2 is None else A2.shape[1]
    N = W_hi.shape[0]
    assert A1.q8 is not None and (A2 is None or (A2.q8 is not None and A2.shape[0] == M))
    assert W_hi.shape[1] == K1 + K2 and W8.shape == (N, 2 * (K1 + K2)) and W_hi.dtype == torch.float16
    if out is None:
        out = empty_act(M, N, out_dtype or torch.float32, W_hi.device)
    if isinstance(out, HiLo8):
        c_ptr, c_code, ldc, n_out, c8 = L.ptr(out.hi), L.F24, out.hi.stride(0), out.hi.shape[1], L.ptr(out.lo8)
    else:
        (c_ptr, c_code, ldc, n_out), c8 = _mat(out), None
    assert n_out == N and out.shape[0] == M
    a2 = (None, None, 0, 0) if A2 is None else (L.ptr(A2.data), L.ptr(A2.q8), A2.data.stride(0), A2.q8.stride(0))
    L.call("gnnlm_linear_f16f8", L.ptr(A1.data), L.ptr(A1.q8), A1.data.stride(0), A1.q8.stride(0), K1, a2[0], a2[1], a2[2], a2[3],
           K2, L.ptr(W_hi), L.ptr(W8), float(w_scale), W_hi.stride(0), W8.stride(0), L.ptr(bias), c_ptr, c_code, ldc, M,
           _dev_count(m_dev), N, c8, L.stream_ptr(), tag=tag or f"linear_f16f8[{N}x{K1 + K2}]", work=(M, N, K1 + K2))
    return out


def linear_lse(A, W, pick, *, W_lo=None, m_dev=None, math=L.MATH_FP32_SIMT, w_scale=1.0):
    """Row log-sum-exp partials + picked column of A @ W^T without materialising it."""
    a_ptr, a_code, lda, K = _mat(A)
    M = A.shape[0]
    N = W.shape[0]
    dev = W.device
    math = L.base_math(math)
    nt = L.load().gnnlm_lse_num_tiles(N, math)
    pmax = torch.empty((M, nt), device=dev, dtype=torch.float32)
    psum = torch.empty((M, nt), device=dev, dtype=torch.float32)
    picked = torch.zeros((M,), device=dev, dtype=torch.float32)
    L.call("gnnlm_linear_lse", a_ptr, a_code, lda, L.ptr(W), L.ptr(W_lo), float(w_scale), W.stride(0), L.ptr(pick), L.ptr(pmax),
           L.ptr(psum), L.ptr(picked), M, _dev_count(m_dev), N, K, math, L.stream_ptr(), work=(M, N, K))
    return pmax, psum, picked, nt


def lse_finish(pmax, psum, picked, nt, out, *, row_map=None, accumulate=False, m_dev=None):
    L.call("gnnlm_lse_finish", L.ptr(pmax), L.ptr(psum), L.ptr(picked), nt, L.ptr(row_map), L.ptr(out),
           int(accumulate), pmax.shape[0], _dev_count(m_dev), L.stream_ptr())
    return out


def gather_rows(src, ids, n_cap=None, n_dev=None, out=None):
    if isinstance(src, Split):      # a row gather of the [rows, 2d] fp16 buffer (and of its e4m3 companion)
        q8 = None if src.q8 is None else gather_rows(src.q8.view(torch.float16), ids, n_cap, n_dev).view(torch.uint8)   # bytes moved as 2-byte words
        return Split(gather_rows(src.data, ids, n_cap, n_dev), src.d, q8)
    n = ids.shape[0] if n_cap is None else n_cap
    d = src.shape[1]
    if out is None:
        out = torch.empty((n, d), device=src.device, dtype=src.dtype)
    L.call("gnnlm_gather_rows", L.ptr(src), src.stride(0), L.ptr(ids), L.ptr(out), out.stride(0), n,
           _dev_count(n_dev), d, L.dtype_code(src.dtype), L.stream_ptr())
    return out


def embed_gather(table, labels_table, rows, *, row_ids=None, n_cap=None, n_dev=None, want_labels=False, err=None):
    """`embed_tokens(neighbor_tokens[rows])` (--reinit-nfeat): table fp32 [V, d], labels_table int16/int32 [N_d], rows int64."""
    n = (row_ids.shape[0] if row_ids is not None else rows.shape[0]) if n_cap is None else n_cap
    V, d = table.shape
    out = torch.empty((n, d), device=table.device, dtype=torch.float32)
    labels = torch.empty((n,), device=table.device, dtype=torch.int64) if want_labels else None
    lb = {torch.int16: 2, torch.int32: 4}[labels_table.dtype]
    L.call("gnnlm_embed_gather", L.ptr(table), table.stride(0), V, L.ptr(labels_table), lb, labels_table.numel(), L.ptr(rows),
           L.ptr(row_ids), L.ptr(out), out.stride(0), n, _dev_count(n_dev), d, L.ptr(labels), L.ptr(err), L.stream_ptr())
    return out, labels


def layernorm(x, gamma, beta, eps=1e-5, out=None, out_dtype=None, n_dev=None, residual=None):
    """LayerNorm(x + residual); residual a Tensor (fp32 / bf16) or Split."""
    n, d = x.shape
    if out is None:
        out = empty_act(n, d, out_dtype or torch.float32, x.device)
    o_ptr, o_code, ldy, _ = _mat(out)
    r_ptr, r_code, ldr = (None, 0, 0) if residual is None else _mat(residual)[:3]
    if isinstance(out, Split) and out.q8 is not None:
        L.call("gnnlm_layernorm_q8", L.ptr(x), x.stride(0), r_ptr, r_code, ldr, L.ptr(gamma), L.ptr(beta), float(eps), o_ptr, o_code,
               ldy, L.ptr(out.q8), out.q8.stride(0), n, _dev_count(n_dev), d, L.stream_ptr(), tag="layernorm")
        return out
    L.call("gnnlm_layernorm", L.ptr(x), x.stride(0), r_ptr, r_code, ldr, L.ptr(gamma), L.ptr(beta), float(eps), o_ptr, o_code,
           ldy, n, _dev_count(n_dev), d, L.stream_ptr())
    return out


def convert(src, dst_dtype):
    src = src.contiguous()
    out = torch.empty_like(src, dtype=dst_dtype)
    L.call("gnnlm_convert", L.ptr(src), L.dtype_code(src.dtype), L.ptr(out), L.dtype_code(dst_dtype), src.numel(),
           L.stream_ptr())
    return out


def split_tf32(w):
    w = w.contiguous()
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    L.call("gnnlm_split_tf32", L.ptr(w), L.ptr(hi), L.ptr(lo), w.numel(), L.stream_ptr())
    return hi, lo


def split_f16(w, scale: Optional[float] = None):
    """fp32 [N, K] -> (fp16 hi, fp16 lo, power-of-two scale) for MATH_F16X3; `scale` given: that one instead of the one that
    brings max|w| to 2^13."""
    import math
    w = w.contiguous()
    if scale is None:
        amax = float(w.abs().max().item()) if w.numel() else 1.0
        scale = 2.0 ** math.floor(math.log2(8192.0 / amax)) if amax > 0 else 1.0
    hi = torch.empty(w.shape, device=w.device, dtype=torch.float16)
    lo = torch.empty(w.shape, device=w.device, dtype=torch.float16)
    L.call("gnnlm_split_f16", L.ptr(w), float(scale), L.ptr(hi), L.ptr(lo), w.numel(), L.stream_ptr())
    return hi, lo, scale


def edge_attn(q, k, v, indptr, indices, H, out, *, dst_ids=None, n_dst=None, n_dst_dev=None, out_scale=1.0,
              accumulate=False, tag=None):
    d = q.shape[1]
    n = q.shape[0] if n_dst is None else n_dst
    assert q.dtype == k.dtype == v.dtype and out.dtype == torch.float32
    L.call("gnnlm_hgt_edge_attn", L.ptr(q), q.stride(0), L.ptr(k), k.stride(0), L.ptr(v), v.stride(0),
           L.dtype_code(q.dtype), L.ptr(indptr), L.ptr(indices), L.ptr(dst_ids), n, _dev_count(n_dst_dev), H, d // H,
           L.ptr(out), out.stride(0), float(out_scale), int(accumulate), L.stream_ptr(), tag=tag)
    return out


def cluster_attn_hq_supported(d: int, H: int, w: int) -> bool:
    """Shape envelope of gnnlm_hgt_cluster_attn_hq (GNNLM_F24 inputs)."""
    dk = d // H
    return d % 128 == 0 and dk % 4 == 0 and dk // 4 <= 32 and 32 % (dk // 4) == 0 and w <= 7


def cluster_attn_supported(d: int, H: int, dtype, w: int) -> bool:
    """Shape envelope of gnnlm_hgt_cluster_attn (else use edge_attn over the CSR)."""
    cs = 4 if dtype == torch.float32 else 8
    dk = d // H
    return d % (32 * cs) == 0 and dk % cs == 0 and dk // cs <= 32 and 32 % (dk // cs) == 0       # any H


def rowstats_q8(o: torch.Tensor, x: "Split", u: torch.Tensor, eps: float, n_dev=None):
    """Deferred LayerNorm (gnnlm_rowstats_q8): z' = o + x as fp16 hi + e4m3 companion and (mean, 1 / std) per row of the ROTATED sum.
    o fp32 [rows, d]; x: hi + companion (Split without a lo half or with one); u fp32 [d] = rot^T 1 / d."""
    rows, d = o.shape
    assert x.q8 is not None and x.shape == (rows, d) and u.shape == (d,)
    z = Split.empty(rows, d, o.device, q8=True, lo=False)
    stats = torch.empty((rows, 2), device=o.device, dtype=torch.float32)
    L.call("gnnlm_rowstats_q8", L.ptr(o), o.stride(0), L.ptr(x.data), x.data.stride(0), L.ptr(x.q8), x.q8.stride(0), L.ptr(u), float(eps),
           L.ptr(z.data), z.data.stride(0), L.ptr(z.q8), z.q8.stride(0), L.ptr(stats), rows, _dev_count(n_dev), d, L.stream_ptr(),
           tag="rowstats")
    return z, stats


def cluster_attn(q, k, v, G, H, out, *, centre_only=False, tag=None, kv_affine=None):
    """ntgt-intra-ntgt chain attention per (token, neighbour) cluster; G is a TokenGraph.  kv_affine = (stats, k_c, k_b, v_c, v_b):
    k / v are raw products under a deferred LayerNorm (rowstats_q8) -- GNNLM_F24 inputs, centre-only form."""
    d = k.shape[1]
    if isinstance(q, HiLo8):       # the 3-byte Q | K' | V' of MATH_F16F8
        assert isinstance(k, HiLo8) and isinstance(v, HiLo8) and isinstance(out, Split) and G.w <= 7
        q8p, ldq8 = (None, 0) if out.q8 is None else (L.ptr(out.q8), out.q8.stride(0))
        L.call("gnnlm_hgt_cluster_attn_hq", L.ptr(q.hi), L.ptr(q.lo8), q.hi.stride(0), L.ptr(k.hi), L.ptr(k.lo8), k.hi.stride(0),
               L.ptr(v.hi), L.ptr(v.lo8), v.hi.stride(0), L.ptr(G.node_base), L.ptr(G.valid_base), L.ptr(G.cluster_nl), G.T * G.k, G.w,
               int(centre_only), H, d // H, L.ptr(out.data), out.data.stride(0), q8p, ldq8, int(out.has_lo),
               *([None] * 5 if kv_affine is None else [L.ptr(t) for t in kv_affine]), L.stream_ptr(), tag=tag)
        return out
    assert kv_affine is None
    if isinstance(out, Split) and out.q8 is not None:
        L.call("gnnlm_hgt_cluster_attn_q8", L.ptr(q), q.stride(0), L.ptr(k), k.stride(0), L.ptr(v), v.stride(0),
               L.dtype_code(q.dtype), L.ptr(G.node_base), L.ptr(G.valid_base), L.ptr(G.cluster_nl), G.T * G.k, G.w,
               int(centre_only), H, d // H, L.ptr(out.data), L.F16X2, out.data.stride(0), L.ptr(out.q8), out.q8.stride(0),
               int(out.has_lo), L.stream_ptr(), tag=tag)
        return out
    o_ptr, o_code, ldo, _ = _mat(out)
    L.call("gnnlm_hgt_cluster_attn", L.ptr(q), q.stride(0), L.ptr(k), k.stride(0), L.ptr(v), v.stride(0),
           L.dtype_code(q.dtype), L.ptr(G.node_base), L.ptr(G.valid_base), L.ptr(G.cluster_nl), G.T * G.k, G.w,
           int(centre_only), H, d // H, o_ptr, o_code, ldo, L.stream_ptr(), tag=tag)
    return out


def inter_fused_supported(d: int, H: int) -> bool:
    dk = d // H
    return H in (4, 8, 12, 16) and d % 8 == 0 and d <= 1024 and dk % 8 == 0 and (16 * (d + 4) + H * d + 19 * H) * 4 <= 220 * 1024


def inter_attn_fused(q, hc_chunks, H, t_agg, wk_t, wv, bias_v, out_scale=0.5):
    """('ntgt','inter','tgt') attention with the K' / V' projections on the token side (gnnlm_hgt_inter_fused).
    q fp32 [T, d] (column slice ok); hc_chunks: [(t0, n_tokens, inter_indptr, hc)] covering all T tokens; t_agg fp32 [T, d] is
    OVERWRITTEN with out_scale * inter.  wk_t / wv: (hi, lo, scale) fp16 splits of W_k'[h]^T [H, d, d_k] and W_v'[h] [H, d_k, d]."""
    T, d = q.shape
    dk = d // H
    dev = q.device
    st = L.stream_ptr
    qs = torch.empty((H, T, 2 * dk), device=dev, dtype=torch.float16)
    L.call("gnnlm_heads_split_f16", L.ptr(q), q.stride(0), T, H, dk, 1, L.ptr(qs), None, st())
    qt = torch.empty((H, T, d), device=dev, dtype=torch.float32)
    L.call("gnnlm_linear_batched_f16x3", L.ptr(qs), 2 * dk, T * 2 * dk, L.ptr(wk_t[0]), L.ptr(wk_t[1]), dk, d * dk, float(wk_t[2]),
           None, 0, 0, L.ptr(qt), d, T * d, H, T, d, dk, 0, st(), tag="inter_q")
    a = torch.empty((H, T, 2 * d), device=dev, dtype=torch.float16)
    for t0, n_tok, indptr, hc in hc_chunks:
        h_ptr, h_code, ldh, _ = _mat(hc)
        L.call("gnnlm_hgt_inter_fused", L.ptr(qt), T * d, h_ptr, h_code, ldh, L.ptr(indptr), t0, n_tok, H, d, L.ptr(a), T * 2 * d,
               2 * d, L.ptr(bias_v), float(out_scale), L.ptr(t_agg), t_agg.stride(0), st(), tag="inter_fused")
    L.call("gnnlm_linear_batched_f16x3", L.ptr(a), 2 * d, T * 2 * d, L.ptr(wv[0]), L.ptr(wv[1]), d, dk * d, float(wv[2]) / out_scale,
           L.ptr(t_agg), t_agg.stride(0), dk, L.ptr(t_agg), t_agg.stride(0), dk, H, T, dk, d, 0, st(), tag="inter_v")
    return t_agg


def causal_attn(q, k, v, B, Lb, intra_ctx, H, out, *, out_scale=1.0, accumulate=False):
    d = q.shape[1]
    L.call("gnnlm_hgt_causal_attn", L.ptr(q), q.stride(0), L.ptr(k), k.stride(0), L.ptr(v), v.stride(0),
           L.dtype_code(q.dtype), B, Lb, intra_ctx, H, d // H, L.ptr(out), out.stride(0), float(out_scale),
           int(accumulate), L.stream_ptr())
    return out


def causal_flash_supported(d: int, H: int) -> bool:
    return d % H == 0 and d // H in (64, 128)


def causal_attn_flash(q, kv: Split, B, Lb, intra_ctx, H, out, *, out_scale=1.0, accumulate=False, out_split: Optional[Split] = None):
    """tgt-intra-tgt attention as one flash kernel (gnnlm_hgt_causal_flash): q fp32 [B*Lb, d] (column slice ok), kv = K' | V' as
    one split-fp16 matrix [B*Lb, 2d]; out fp32 [B*Lb, d] (+)= out_scale * attention, or -- with out_split -- the final value as
    split fp16 (out is then only read when accumulating)."""
    d = q.shape[1]
    assert kv.has_lo and kv.d == 2 * d and q.dtype == torch.float32 and q.stride(1) == 1
    os_ptr, ldos, os_lo = (None, 0, 0) if out_split is None else (L.ptr(out_split.data), out_split.data.stride(0), out_split.d)
    kd = kv.data
    L.call("gnnlm_hgt_causal_flash", L.ptr(q), q.stride(0), L.ptr(kd), L.ptr(kd[:, d:]), kd.stride(0), 2 * d, B, Lb, intra_ctx, H, d // H,
           L.ptr(out), out.stride(0), os_ptr, ldos, os_lo, float(out_scale), int(accumulate), L.stream_ptr(), tag="causal_flash")
    return out if out_split is None else out_split


def causal_flash_tc_supported(d: int, H: int, Lb: int) -> bool:
    return d % H == 0 and d // H == 128 and Lb % 8 == 0


def causal_attn_flash_tc(qkv, B, Lb, intra_ctx, H, out, *, out_scale=1.0, accumulate=False, out_split: Optional[Split] = None):
    """tgt-intra-tgt attention on tcgen05 (gnnlm_hgt_causal_flash_tc): qkv fp32 [B*Lb, 3d] (Q | K' | V' of the projection)."""
    d = qkv.shape[1] // 3
    dk = d // H
    dev = qkv.device
    qk = to_split(qkv[:, :2 * d])                                                     # Q hi | K' hi | Q lo | K' lo
    vt = torch.empty((2, B * H * dk, Lb), device=dev, dtype=torch.float16)
    for b in range(B):
        vb = qkv[b * Lb:(b + 1) * Lb, 2 * d:]
        L.call("gnnlm_heads_transpose_split_f16", L.ptr(vb), vb.stride(0), Lb, H, dk, L.ptr(vt[0, b * H * dk:]), L.ptr(vt[1, b * H * dk:]),
               L.stream_ptr())
    os_ptr, ldos, os_lo = (None, 0, 0) if out_split is None else (L.ptr(out_split.data), out_split.data.stride(0), out_split.d)
    L.call("gnnlm_hgt_causal_flash_tc", L.ptr(qk.data), qk.data.stride(0), d, L.ptr(vt), Lb, B, Lb, intra_ctx, H, dk, L.ptr(out),
           out.stride(0), os_ptr, ldos, os_lo, float(out_scale), int(accumulate), L.stream_ptr(), tag="causal_flash_tc")
    return out if out_split is None else out_split


CAUSAL_K_TILE = 256      # rows per tile pair of the batched GEMM (2 * BLOCK_M): the contraction limit of `causal = 2`


def causal_attn_gemm_supported(d: int, H: int, Lb: int) -> bool:
    dk = d // H
    return Lb % 8 == 0 and dk % 8 == 0 and Lb >= 256


def causal_attn_gemm(q, k, v, B, Lb, intra_ctx, H, out, *, out_scale=1.0, accumulate=False, drop=None):
    """tgt-intra-tgt attention on the tensor cores at fp32 parity (MATH_F16X3): per block and head two 3xFP16 GEMMs
    (S = Q K'^T, O = softmax_causal(S) V') with split-fp16 operands; q / k / v fp32 [B*Lb, d] (column slices ok)."""
    d = q.shape[1]
    dk = d // H
    dev = q.device
    f16 = dict(device=dev, dtype=torch.float16)
    st = L.stream_ptr
    for b in range(B):
        rows = slice(b * Lb, (b + 1) * Lb)
        qb, kb, vb = q[rows], k[rows], v[rows]
        qs = torch.empty((H, Lb, 2 * dk), **f16)
        kh, kl = torch.empty((H, Lb, dk), **f16), torch.empty((H, Lb, dk), **f16)
        vh, vl = torch.empty((H, dk, Lb), **f16), torch.empty((H, dk, Lb), **f16)
        L.call("gnnlm_heads_split_f16", L.ptr(qb), qb.stride(0), Lb, H, dk, 1, L.ptr(qs), None, st())
        L.call("gnnlm_heads_split_f16", L.ptr(kb), kb.stride(0), Lb, H, dk, 0, L.ptr(kh), L.ptr(kl), st())
        L.call("gnnlm_heads_transpose_split_f16", L.ptr(vb), vb.stride(0), Lb, H, dk, L.ptr(vh), L.ptr(vl), st())
        S = torch.empty((H, Lb, Lb), device=dev, dtype=torch.float32)
        # all heads in one launch each: S[h] = Q_h K'_h^T, then O[:, h] (+)= out_scale * P_h V'_h
        L.call("gnnlm_linear_batched_f16x3", L.ptr(qs), 2 * dk, Lb * 2 * dk, L.ptr(kh), L.ptr(kl), dk, Lb * dk, 1.0, None, 0, 0,
               L.ptr(S), Lb, Lb * Lb, H, Lb, Lb, dk, 1, st(), tag="attn_qk")      # causal = 1: tiles above the diagonal skipped
        P = torch.empty((H, Lb, 2 * Lb), **f16)
        if drop is not None and drop[0] > 0:      # training: (p, seed) -- the attention dropout on the softmax weights (hgt.py:356)
            L.call("gnnlm_causal_softmax_drop_split", L.ptr(S), Lb, intra_ctx, H, CAUSAL_K_TILE, b * Lb, float(drop[0]), drop[1], L.ptr(P), st())
        else:
            L.call("gnnlm_causal_softmax_split", L.ptr(S), Lb, intra_ctx, H, CAUSAL_K_TILE, L.ptr(P), st())
        ob = out[rows]
        L.call("gnnlm_linear_batched_f16x3", L.ptr(P), 2 * Lb, Lb * 2 * Lb, L.ptr(vh), L.ptr(vl), Lb, dk * Lb, 1.0 / out_scale,
               L.ptr(ob) if accumulate else None, ob.stride(0), dk, L.ptr(ob), ob.stride(0), dk, H, Lb, dk, Lb, 2, st(),
               tag="attn_pv")                                                     # causal = 2: k < 256 (r + 1) per row pair
    return out


def pq_gather_decode(codes, centroids, rows, *, bias=None, row_ids=None, n_cap=None, n_dev=None, out_dtype=torch.float32,
                     labels_table=None, want_codes=False, decode=True):
    n_d, M = codes.shape
    dsub = centroids.shape[2]
    n = (row_ids.shape[0] if row_ids is not None else rows.shape[0]) if n_cap is None else n_cap
    dev = codes.device
    out = empty_act(n, M * dsub, out_dtype, dev) if decode else None
    o_ptr, o_code, ld_out = (None, L.F32, M * dsub) if out is None else _mat(out)[:3]
    labels = torch.empty((n,), device=dev, dtype=torch.int64) if labels_table is not None else None
    codes_out = torch.empty((n, M), device=dev, dtype=torch.uint8) if want_codes else None
    lb = 0
    if labels_table is not None:
        lb = {torch.int16: 2, torch.int32: 4}[labels_table.dtype]
    L.call("gnnlm_pq_gather_decode", L.ptr(codes), n_d, M, L.ptr(centroids), dsub,
           L.ptr(bias) if bias is not None and bias.numel() else None, L.ptr(rows), L.ptr(row_ids), n, _dev_count(n_dev),
           o_ptr, o_code, ld_out, L.ptr(labels_table), lb, L.ptr(labels), L.ptr(codes_out),
           L.stream_ptr())
    return out, labels, codes_out


def gelu(x, out_dtype=torch.float32, n_dev=None):
    """gelu(x) (erf form) of fp32 rows into an activation format (torch dtype or SPLIT)."""
    n, d = x.shape
    assert x.dtype == torch.float32 and x.stride(1) == 1
    out = empty_act(n, d, out_dtype, x.device)
    o_ptr, o_code, ldo, _ = _mat(out)
    L.call("gnnlm_gelu", L.ptr(x), x.stride(0), o_ptr, o_code, ldo, n, _dev_count(n_dev), d, L.stream_ptr())
    return out


def pq_gather_decode_hiq8(codes, cb_hi, cb_q8, rows, *, row_ids=None, n_cap=None, n_dev=None):
    """Gather + decode into the operand set of linear_f16f8 only (fp16 hi + e4m3 companion) from pre-quantised codebooks."""
    n_d, M = codes.shape
    assert cb_hi.dtype == torch.float16 and cb_hi.shape == (M, 256, 8) and cb_q8.dtype == torch.uint8 and cb_q8.shape == (M, 256, 16)
    n = (row_ids.shape[0] if row_ids is not None else rows.shape[0]) if n_cap is None else n_cap
    out = empty_act(n, M * 8, HI_Q8, codes.device)
    L.call("gnnlm_pq_gather_decode_hiq8", L.ptr(codes), n_d, M, L.ptr(cb_hi), L.ptr(cb_q8), 8, L.ptr(rows), L.ptr(row_ids), n,
           _dev_count(n_dev), L.ptr(out.data), out.data.stride(0), L.ptr(out.q8), out.q8.stride(0), L.stream_ptr(),
           tag="pq_gather_decode")
    return out


def pq_gather_decode_presplit(codes, cb_hi, cb_lo, rows, *, row_ids=None, n_cap=None, n_dev=None, q8=False):
    """Gather + decode straight into the split-fp16 format from a pre-split codebook (dsub == 8); q8: also the e4m3 companion."""
    n_d, M = codes.shape
    assert cb_hi.dtype == torch.float16 and cb_hi.shape == cb_lo.shape == (M, 256, 8) and cb_hi.is_contiguous()
    n = (row_ids.shape[0] if row_ids is not None else rows.shape[0]) if n_cap is None else n_cap
    out = empty_act(n, M * 8, SPLIT_Q8 if q8 else SPLIT, codes.device)
    o_ptr, _, ld_out, _ = _mat(out)
    if q8:
        L.call("gnnlm_pq_gather_decode_presplit_q8", L.ptr(codes), n_d, M, L.ptr(cb_hi), L.ptr(cb_lo), 8, L.ptr(rows), L.ptr(row_ids),
               n, _dev_count(n_dev), o_ptr, ld_out, L.ptr(out.q8), out.q8.stride(0), L.stream_ptr(), tag="pq_gather_decode")
        return out
    L.call("gnnlm_pq_gather_decode_presplit", L.ptr(codes), n_d, M, L.ptr(cb_hi), L.ptr(cb_lo), 8, L.ptr(rows), L.ptr(row_ids),
           n, _dev_count(n_dev), o_ptr, ld_out, L.stream_ptr(), tag="pq_gather_decode")
    return out


def adapt_target(target, cutoff):
    """target [T] int64 (device), cutoff: python list ending with vocab size."""
    T = target.numel()
    nt = len(cutoff) - 1
    dev = target.device
    head_pick = torch.empty((T,), device=dev, dtype=_I32)
    tail_rows = torch.empty((max(nt, 1), T), device=dev, dtype=_I32)
    tail_pick = torch.empty((max(nt, 1), T), device=dev, dtype=_I32)
    tail_count = torch.zeros((max(nt, 1),), device=dev, dtype=_I32)
    import ctypes as C
    arr = (C.c_int64 * len(cutoff))(*cutoff)
    L.call("gnnlm_adapt_target", L.ptr(target), T, C.cast(arr, C.c_void_p), len(cutoff), L.ptr(head_pick),
           L.ptr(tail_rows), L.ptr(tail_pick), L.ptr(tail_count), L.stream_ptr())
    return head_pick, tail_rows, tail_pick, tail_count


def knn_mix_nll(lm_lp, *, target=None, dists=None, ids=None, vals=None, n_datastore=0, sim_sign=1.0, temperature=1.0,
                lmbda=0.0, orig_lp=None, orig_ratio=0.0, weight=None, nll_acc=None, want_knn=False, pad_id=-1,
                loss_start=None, block_len=0):
    T = lm_lp.numel()
    dev = lm_lp.device
    out_lp = torch.empty((T,), device=dev, dtype=torch.float32)
    use_knn = dists is not None and lmbda > 0
    knn_p = torch.empty((T,), device=dev, dtype=torch.float32) if (use_knn and want_knn) else None
    recall = torch.empty((T,), device=dev, dtype=_I32) if (use_knn and want_knn) else None
    vb = 0
    if use_knn:
        vb = {torch.int16: 2, torch.int32: 4}[vals.dtype]
        assert dists.dtype == torch.float32 and ids.dtype == torch.int64 and dists.is_contiguous() and ids.is_contiguous()
    L.call("gnnlm_knn_mix_nll", L.ptr(lm_lp), L.ptr(orig_lp), float(orig_ratio), L.ptr(dists) if use_knn else None,
           L.ptr(ids) if use_knn else None, dists.shape[1] if use_knn else 0, L.ptr(vals) if use_knn else None, vb,
           n_datastore, L.ptr(target), float(sim_sign), float(temperature), float(lmbda), L.ptr(weight),
           int(pad_id), L.ptr(loss_start), int(block_len), L.ptr(out_lp), L.ptr(knn_p), L.ptr(recall), L.ptr(nll_acc), T, L.stream_ptr())
    return out_lp, knn_p, recall


def knn_full_prob(dists, ids, vals, vocab, n_datastore, sim_sign=1.0, temperature=1.0):
    T, k = dists.shape
    probs = torch.empty((T, vocab), device=dists.device, dtype=torch.float32)
    vb = {torch.int16: 2, torch.int32: 4}[vals.dtype]
    L.call("gnnlm_knn_full_prob", L.ptr(dists), L.ptr(ids), k, L.ptr(vals), vb, n_datastore, float(sim_sign),
           float(temperature), L.ptr(probs), vocab, T, L.stream_ptr())
    return probs


METRICS = {"l2": 0, "ip": 1}


def knn_sims_keys(queries, keys, ids, metric: str, cosine: bool = False):
    """sims [T, k] from the datastore's own key rows (knn_model.py:159-177); keys [N_d, d] fp16 / fp32 on the device."""
    T, d = queries.shape
    assert queries.dtype == torch.float32 and queries.stride(1) == 1 and ids.dtype == torch.int64 and ids.is_contiguous()
    assert keys.is_contiguous() and keys.shape[1] == d and keys.dtype in (torch.float16, torch.float32)
    sims = torch.empty(ids.shape, device=queries.device, dtype=torch.float32)
    norm = (3 if metric == "ip" else 2) if cosine else 0
    L.call("gnnlm_knn_sims_keys", L.ptr(queries), queries.stride(0), L.ptr(keys), L.F16 if keys.dtype == torch.float16 else L.F32,
           keys.shape[0], d, L.ptr(ids), ids.shape[1], METRICS[metric], norm, L.ptr(sims), T, L.stream_ptr())
    return sims


def knn_sims_pq(queries, rotated, codes, centroids, bias, ids, metric: str, *, key_norm2=None, cosine: bool = False):
    """sims [T, k] against the PQ-decoded keys by asymmetric distance computation; rotated = queries @ A.T.
    cosine: normalised queries (and, for `ip`, normalised decoded keys: key_norm2 [M, 256] = ||centroid - b_m||^2)."""
    T = queries.shape[0]
    M, ksub, dsub = centroids.shape
    assert ksub == 256 and codes.dtype == torch.uint8 and codes.is_contiguous() and codes.shape[1] == M
    assert rotated.shape == (T, M * dsub) and rotated.stride(1) == 1 and queries.stride(1) == 1
    sims = torch.empty(ids.shape, device=queries.device, dtype=torch.float32)
    L.call("gnnlm_knn_sims_pq", L.ptr(queries), queries.stride(0), queries.shape[1], L.ptr(rotated), rotated.stride(0),
           L.ptr(codes), codes.shape[0], M, dsub, L.ptr(centroids), L.ptr(bias), L.ptr(ids), ids.shape[1], METRICS[metric],
           L.ptr(key_norm2), (3 if metric == "ip" else 2) if cosine else 0, L.ptr(sims), T, L.stream_ptr())
    return sims


def knn_filter(keys: Split, id_base: int, q_hi, q_lo, key_bias, thr, cand_s, cand_id, cand_cnt):
    """Top-k filter pass of the exact kNN search over one span of keys (gnnlm_knn_filter_f16x3): appends (score, id) of every
    score above thr[q] to cand_s / cand_id [n_q, cap] and counts it in cand_cnt (counts past cap flag an overflow)."""
    n_q, d = q_hi.shape
    assert keys.has_lo and keys.d == d and q_lo.shape == q_hi.shape and q_hi.stride(0) == q_lo.stride(0)
    cap = cand_s.shape[1]
    L.call("gnnlm_knn_filter_f16x3", L.ptr(keys.data), keys.data.stride(0), keys.data.shape[0], int(id_base), L.ptr(q_hi),
           L.ptr(q_lo), q_hi.stride(0), n_q, d, L.ptr(key_bias), L.ptr(thr), L.ptr(cand_s), L.ptr(cand_id), L.ptr(cand_cnt), cap,
           L.stream_ptr(), tag="knn_filter", work=(keys.data.shape[0], n_q, d))


def topk_merge(top_s, top_id, cand_s, cand_id, cand_cnt, thr):
    """Running top-k [n_q, k] (+) a span's candidates, in place; new thresholds; counts reset except for overflowed queries."""
    n_q, k = top_s.shape
    L.call("gnnlm_topk_merge", L.ptr(top_s), L.ptr(top_id), n_q, k, L.ptr(cand_s), L.ptr(cand_id), L.ptr(cand_cnt),
           cand_s.shape[1], L.ptr(thr), L.stream_ptr(), tag="topk_merge")


def knn_key_bias(x):
    """-1/2 ||x_i||^2 [n] fp32 of fp16 / fp32 rows."""
    assert x.dim() == 2 and x.stride(1) == 1
    out = torch.empty((x.shape[0],), device=x.device, dtype=torch.float32)
    L.call("gnnlm_knn_key_bias", L.ptr(x), L.dtype_code(x.dtype), x.stride(0), x.shape[0], x.shape[1], L.ptr(out), L.stream_ptr())
    return out


def knn_key_bias_pq(codes, norm2):
    """-1/2 ||x_i||^2 [n] of PQ-decoded keys: codes [n, M] uint8, norm2 [M, 256] = ||centroid - b_m||^2."""
    assert codes.dtype == torch.uint8 and codes.is_contiguous() and norm2.shape == (codes.shape[1], 256) and norm2.is_contiguous()
    out = torch.empty((codes.shape[0],), device=codes.device, dtype=torch.float32)
    L.call("gnnlm_knn_key_bias_pq", L.ptr(codes), codes.shape[0], codes.shape[1], L.ptr(norm2), L.ptr(out), L.stream_ptr())
    return out
