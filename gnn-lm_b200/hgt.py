"""Heterogeneous Graph Transformer over the kNN token graph -- host-side mirror of the reference's
fairseq/models/hgt.py (HGTLayer :22-79,299-420; HGT :459-513) with identical constructor arguments,
parameter names and state_dict keys, executing on libgnnlm_sm100.so kernels only.

B200-first restructuring (results identical up to fp rounding, see tests/test_gpu_parity.py):
  * the per-relation d_k x d_k transforms (hgt.py:347-348) and the relation_pri / sqrt(d_k) score
    scale (:355) are folded into the K/V projection weights once per checkpoint, and the
    projections that share an input are concatenated, so one GEMM emits Q | K' | V' directly;
  * score, segmented softmax, weighted sum and the cross-edge-type mean are one fused kernel per
    edge type (no [E,H] / [E,H,d_k] intermediates);
  * tgt-intra-tgt is executed as implicit causal attention (no 4.7M-edge COO);
  * ntgt nodes only ever receive messages from ntgt nodes, so the ntgt side of all layers is run
    first and only the compact centre-node features each tgt layer needs are kept; in the
    decoder's tgt-only mode the last layer skips the ntgt side and the one before computes centre
    rows only (dead-work elimination, SURVEY.md 7.6).
"""
import math
from typing import Dict, List, Optional

import os

import torch
import torch.nn as nn

from . import _lib as L
from . import ops
from .graph import TokenGraph
from . import hetero
from .hetero import HeteroGraph


def _fold(W: torch.Tensor, b: torch.Tensor, R: torch.Tensor, scale: Optional[torch.Tensor]):
    """K' = (h W^T + b) @ blockdiag(R)  ==  h W'^T + b'   (fp64 fold, returned as fp32)."""
    H, dk, _ = R.shape
    d_in = W.shape[1]
    W3 = W.detach().double().view(H, dk, d_in)
    Rd = R.detach().double()
    Wf = torch.einsum("ijk,ijd->ikd", Rd, W3)
    bf = torch.einsum("ij,ijk->ik", b.detach().double().view(H, dk), Rd)
    if scale is not None:
        Wf = Wf * scale.double()[:, None, None]
        bf = bf * scale.double()[:, None]
    return Wf.reshape(H * dk, d_in).float(), bf.reshape(H * dk).float()


class _Weight:
    """A prepared [N,K] weight in the layout/precision the selected GEMM math wants."""

    def __init__(self, W: torch.Tensor, b: Optional[torch.Tensor], math_mode: int):
        W = W.contiguous().float()
        self.b = None if b is None else b.contiguous().float()
        self.lo = None
        self.scale = 1.0
        self._q8 = None
        self.f8 = math_mode == L.MATH_F16F8
        if math_mode == L.MATH_TF32X3:
            self.W, self.lo = ops.split_tf32(W)
        elif math_mode in (L.MATH_F16X3, L.MATH_F16F8):
            self.W, self.lo, self.scale = ops.split_f16(W)
        elif math_mode == L.MATH_BF16:
            self.W = ops.convert(W, torch.bfloat16)
        else:
            self.W = W

    def w8(self) -> torch.Tensor:
        """e4m3 companion [N, 2K] of the fp16 halves (MATH_F16F8), built on first use."""
        if self._q8 is None:
            self._q8 = ops.quant_w8(self.W, self.lo)
        return self._q8

    def permuted(self, perm: torch.Tensor) -> "_Weight":
        """The same prepared weight with its rows (and bias entries) in the order `perm`."""
        v = object.__new__(_Weight)
        v.f8 = self.f8
        v._q8 = self.w8()[perm].contiguous() if self.f8 else None
        v.W = self.W[perm].contiguous()
        v.lo = None if self.lo is None else self.lo[perm].contiguous()
        v.b = None if self.b is None else self.b[perm].contiguous()
        v.scale = self.scale
        return v

    def rows(self, a: int, b_: int) -> "_Weight":
        v = object.__new__(_Weight)
        v.f8 = self.f8
        v._q8 = self.w8()[a:b_] if self.f8 else None
        v.W = self.W[a:b_]
        v.lo = None if self.lo is None else self.lo[a:b_]
        v.b = None if self.b is None else self.b[a:b_]
        v.scale = self.scale
        return v


def head_interleave(H: int, dk: int) -> torch.Tensor:
    """Row order [Q_0 | K'_0 | Q_1 | K'_1 | ... | Q_{H-1} | K'_{H-1} | V'_0 .. V'_{H-1}] of a [Q | K' | V'] projection: with d_k = 128
    every 256-row tile of the first 2 d rows holds one head's Q and K', every one of the last d rows the V' of two heads
    (the N-tiles of gnnlm_linear_f16f8_nn_attn)."""
    d = H * dk
    qk = torch.arange(d).view(H, dk)
    return torch.cat([torch.stack([qk, qk + d], 1).reshape(-1), torch.arange(2 * d, 3 * d)])


FUSED_INTER_MODES = (L.MATH_F16X3, L.MATH_F16F8, L.MATH_BF16, L.MATH_TF32)     # modes whose operands are already fp16-range on tensor cores


def _lin(x, w: _Weight, math_mode, x2=None, **kw):
    """x @ W^T + b; `x2`: second row-aligned source, W = [W1 | W2] along k (MATH_F16F8 only)."""
    if math_mode == L.MATH_F16F8 and isinstance(x, ops.Split) and x.q8 is not None and "residual" not in kw and \
            ops.f16f8_supported(x.d, 0 if x2 is None else x2.d):
        return ops.linear_f16f8(x, w.W, w.w8(), w.b, A2=x2, w_scale=w.scale, **kw)
    assert x2 is None
    return ops.linear(x, w.W, w.b, W_lo=w.lo, w_scale=w.scale, math=math_mode, **kw)


F16F8_MIN_ROWS = 0          # rows below which a split operand is not given an e4m3 companion (0: always in MATH_F16F8)


def with_q8(x, math_mode: int, n_dev=None):
    """MATH_F16F8: make sure a large split-fp16 GEMM operand carries its e4m3 companion (a standalone pass when the
    producing kernel did not write it)."""
    if math_mode == L.MATH_F16F8 and isinstance(x, ops.Split) and x.q8 is None and x.shape[0] >= F16F8_MIN_ROWS and \
            ops.f16f8_supported(x.d):
        ops.to_q8(x, n_dev)
    return x


def gemm_act(math_mode: int, rows: int, d: int, lo: bool = True):
    """Output format for an activation that feeds a GEMM: split fp16, with the e4m3 companion in MATH_F16F8 (lo=False: and
    without the fp16 lo half, for an activation that feeds NOTHING but that product)."""
    act = act_dtype(math_mode)
    if math_mode == L.MATH_F16F8 and rows >= F16F8_MIN_ROWS and ops.f16f8_supported(d) and d in (128, 256, 512, 1024):
        return ops.SPLIT_Q8 if lo else ops.HI_Q8
    return act


def act_dtype(math_mode: int):
    """Activation storage type of a math mode: bf16 end to end in MATH_BF16, split fp16 (same bytes as fp32, consumed
    by the GEMMs without an operand-split pass) in MATH_F16X3, fp32 otherwise."""
    if math_mode == L.MATH_BF16:
        return torch.bfloat16
    return ops.SPLIT if math_mode in (L.MATH_F16X3, L.MATH_F16F8) else torch.float32


def as_act(x, math_mode: int):
    dt = act_dtype(math_mode)
    if dt == ops.SPLIT:
        if isinstance(x, ops.Split):
            return x
        if x.dtype not in (torch.float16, torch.float32):
            x = x.float()
        return ops.to_split(x if x.stride(-1) == 1 else x.contiguous())
    if isinstance(x, ops.Split):
        x = x.float()
    if x.dtype == dt:
        return x if x.is_contiguous() else x.contiguous()
    return ops.convert(x, dt)


def _attn_in_dtype(math_mode: int, hq: bool = False):
    """Q | K' | V' storage: bf16 in MATH_BF16, fp32 otherwise (the attention kernels read fp32 / bf16); `hq`: the 3-byte
    GNNLM_F24 form (the value's top three bytes) when the MATH_F16F8 projection feeds the cluster kernel."""
    if hq and math_mode == L.MATH_F16F8:
        return ops.HILO8
    return torch.bfloat16 if math_mode == L.MATH_BF16 else torch.float32


def as_float(x) -> torch.Tensor:
    return x.float() if isinstance(x, ops.Split) or x.dtype != torch.float32 else x


class HGTLayer(hetero.IncrementalState, nn.Module):
    """Same parameters as the reference layer (hgt.py:27-79; @with_incremental_state, :21)."""

    def __init__(self, in_dim: int, out_dim: int, ntype2idx: Dict[str, int], etype2idx: Dict[str, int], n_heads: int,
                 dropout=0.2, use_norm=True, two_stream=False, attn_drop=0.2):
        super().__init__()
        self.init_incremental_state()
        self.in_dim, self.out_dim = in_dim, out_dim
        self.ntype2idx, self.etype2idx = ntype2idx, etype2idx
        self.num_types, self.num_relations = len(ntype2idx), len(etype2idx)
        self.n_heads = n_heads
        assert out_dim % n_heads == 0
        self.d_k = out_dim // n_heads
        self.sqrt_dk = math.sqrt(self.d_k)
        self.use_norm = use_norm
        self.two_stream = two_stream
        self.k_linears, self.q_linears = nn.ModuleList(), nn.ModuleList()
        self.v_linears, self.a_linears = nn.ModuleList(), nn.ModuleList()
        self.norms = nn.ModuleList()
        for _ in range(self.num_types):
            self.k_linears.append(nn.Linear(in_dim, out_dim))
            self.q_linears.append(nn.Linear(in_dim, out_dim))
            self.v_linears.append(nn.Linear(in_dim, out_dim))
            self.a_linears.append(nn.Linear(out_dim, out_dim))
            if use_norm:
                self.norms.append(nn.LayerNorm(out_dim))
        self.relation_pri = nn.Parameter(torch.ones(self.num_relations, n_heads))
        self.relation_att = nn.Parameter(torch.Tensor(self.num_relations, n_heads, self.d_k, self.d_k))
        self.relation_msg = nn.Parameter(torch.Tensor(self.num_relations, n_heads, self.d_k, self.d_k))
        self.skip = nn.Parameter(torch.ones(self.num_types))      # unused by the reference forward (:399)
        self.drop = nn.Dropout(dropout)
        self.attn_drop = nn.Dropout(attn_drop)
        nn.init.xavier_uniform_(self.relation_att)
        nn.init.xavier_uniform_(self.relation_msg)
        self._prep = None
        self._prep_key = None
        self.use_cluster_kernel = True     # False: always go through the generic CSR kernel (tests compare both)
        self.use_fused_inter = True        # False: project every centre node to K' / V' and use the CSR kernel
        self.use_gemm_attention = True     # MATH_F16X3, long blocks: tgt-intra-tgt attention as tensor-core GEMMs
        # tensor-core modes, d_k in {64, 128}: one flash kernel instead (gnnlm_hgt_causal_flash); GNNLM_FLASH=0 for A/B timing
        self.use_flash_attention = os.environ.get("GNNLM_FLASH", "1") != "0"
        self.use_flash_tc = os.environ.get("GNNLM_FLASH", "1") != "mma"      # d_k = 128: the tcgen05 form (GNNLM_FLASH=mma: mma.sync form)
        # MATH_F16F8: Q | K' | V' of the ntgt side rounded to three bytes (GNNLM_F24) instead of fp32 (GNNLM_HQ=0: fp32, for A/B)
        self.use_hq_attention = {"0": False, "all": "all"}.get(os.environ.get("GNNLM_HQ", "1"), True)
        # layer 0 with the rotation folded, followed by the centre-only layer: LayerNorm deferred into its consumers (HGT._ntgt_side)
        self.use_deferred_ln = os.environ.get("GNNLM_DEFER_LN", "1") != "0"
        # MATH_F16F8, d_k = 128: the all-nodes chain attention in the epilogue of its Q|K'|V' projection (GNNLM_FUSED_NN=0: two kernels, for A/B)
        self.use_fused_nn = os.environ.get("GNNLM_FUSED_NN", "1") != "0"

    # ------------------------------------------------------------------ weight preparation
    def prepare(self, math_mode: int, rot: Optional[torch.Tensor] = None, prev_ln=None):
        """`rot` [d, d_dec] (layer 0, MATH_F16F8): the ntgt input features are given UN-rotated, h = x @ rot^T (the OPQ inverse
        rotation `x @ A` of pq_wrapper.py:202, rot = A^T), and the rotation is folded into this layer's ntgt-side weights in
        fp64 -- Q|K'|V' = x (W rot)^T, the inter K' / V' likewise, and the residual of hgt.py:403 inside the output projection:
        A-linear(t) + h = [t | x] [W_a | rot]^T -- so the rotated features are never materialised."""
        # `prev_ln` = (gamma, beta, rot) of the PREVIOUS layer when that layer defers its ntgt LayerNorm (HGT._prepare_layers): this
        # layer's ntgt K' | V' projection is then prepared for the un-normalised, un-rotated input z' as well ("kv_deferred")
        key = (math_mode, self.relation_pri.device, tuple(int(p._version) for p in self.parameters()),
               None if rot is None else (rot.data_ptr(), int(rot._version)),
               None if prev_ln is None else tuple((t.data_ptr(), int(t._version)) for t in prev_ln))
        if self._prep is not None and self._prep_key == key:
            return self._prep
        if not self.use_norm:
            raise NotImplementedError("use_norm=False is never used by the reference decoder")
        t, n = self.ntype2idx["tgt"], self.ntype2idx["ntgt"]
        intra, inter = self.etype2idx["intra"], self.etype2idx["inter"]
        d = self.out_dim
        pri = self.relation_pri.detach()

        def kv(tau, rel):
            Wk, bk = _fold(self.k_linears[tau].weight, self.k_linears[tau].bias, self.relation_att[rel],
                           pri[rel] / self.sqrt_dk)
            Wv, bv = _fold(self.v_linears[tau].weight, self.v_linears[tau].bias, self.relation_msg[rel], None)
            return Wk, bk, Wv, bv

        rot64 = None if rot is None else rot.detach().double()
        through = lambda W: W if rot64 is None else (W.double() @ rot64).float()        # x (W rot)^T == (x rot^T) W^T

        def qkv(tau):
            Wk, bk, Wv, bv = kv(tau, intra)
            W = torch.cat([self.q_linears[tau].weight.detach().float(), Wk, Wv], 0)
            b = torch.cat([self.q_linears[tau].bias.detach().float(), bk, bv], 0)
            return _Weight(through(W) if tau == n else W, b, math_mode)

        Wk, bk, Wv, bv = kv(n, inter)
        Wk, Wv = through(Wk), through(Wv)
        fused = None
        if math_mode in FUSED_INTER_MODES and ops.inter_fused_supported(d, self.n_heads):
            # token-side form of the inter projections (inter_attn.cu): W_k'[h]^T [H, d, d_k] and W_v'[h] [H, d_k, d] as
            # fp16 splits; b_k' drops out of the softmax, b_v' is added once per token
            Hh, dk = self.n_heads, d // self.n_heads
            fused = {"wk_t": ops.split_f16(Wk.view(Hh, dk, d).transpose(1, 2).contiguous().view(Hh * d, dk)),
                     "wv": ops.split_f16(Wv.contiguous()), "bv": bv.contiguous().float()}
        P = {
            "tgt_qkv": qkv(t), "ntgt_qkv": qkv(n),
            "ntgt_kv_inter": _Weight(torch.cat([Wk, Wv], 0), torch.cat([bk, bv], 0), math_mode),
            "a": {tau: _Weight(self.a_linears[tau].weight.detach(), self.a_linears[tau].bias.detach(), math_mode)
                  for tau in (t, n)},
            "ln": {tau: (self.norms[tau].weight.detach().float().contiguous(),
                         self.norms[tau].bias.detach().float().contiguous(), self.norms[tau].eps) for tau in (t, n)},
            "math": math_mode, "d": d, "t": t, "n": n, "inter_fused": fused,
            # [W_a | rot]: output projection and rotation of the residual as one product over [t | x]
            "a_rot": None if rot is None else _Weight(torch.cat([self.a_linears[n].weight.detach().float(), rot.detach().float()], 1),
                                                      self.a_linears[n].bias.detach(), math_mode),
        }
        H = self.n_heads
        if math_mode == L.MATH_F16F8 and d == 128 * H and H % 2 == 0 and H <= 8:
            P["ntgt_qkv_heads"] = P["ntgt_qkv"].permuted(head_interleave(H, 128).to(P["ntgt_qkv"].W.device))
        if rot is not None and self.use_deferred_ln and math_mode == L.MATH_F16F8 and rot.shape[0] == rot.shape[1]:
            r64 = rot.detach().double()
            eye = torch.eye(r64.shape[0], dtype=r64.dtype, device=r64.device)
            if torch.allclose(r64.T @ r64, eye, atol=1e-5) and torch.allclose(r64 @ r64.T, eye, atol=1e-5):     # orthonormal rotation
                Wa, ba = self.a_linears[n].weight.detach().double(), self.a_linears[n].bias.detach().double()
                P["defer"] = {
                    "a": _Weight((r64.T @ Wa).float(), (ba @ r64).float(), math_mode),        # z' = t (rot^T W_a)^T + b_a rot (+ x)
                    "u": (r64.sum(0) / r64.shape[0]).float().contiguous(),                      # mean(z) = <z', rot^T 1 / d>
                    "rot": _Weight(rot.detach().float(), None, math_mode),                      # z = z' rot^T
                }
        if prev_ln is not None and math_mode == L.MATH_F16F8:
            g64, b64, r64 = (t.detach().double() for t in prev_ln)
            Wk, bk, Wv, bv = kv(n, intra)
            W = torch.cat([Wk, Wv], 0).double()
            bias = torch.cat([bk, bv], 0).double()
            c = (W @ g64).float()
            bt = (W @ b64 + bias).float()
            P["kv_deferred"] = {"w": _Weight(((W * g64[None, :]) @ r64).float(), None, math_mode),   # raw = z' (W diag(gamma) rot)^T
                                "k_c": c[:d].contiguous(), "k_b": bt[:d].contiguous(), "v_c": c[d:].contiguous(), "v_b": bt[d:].contiguous()}
        self._prep, self._prep_key = P, key
        return P

    # ------------------------------------------------------------------ building blocks
    def _out(self, P, tau, t_agg, h_in, n_dev, feeds_gemm: bool = False):
        """LayerNorm(A-linear(t) + h) (hgt.py:401-405).  The residual add is fused into the LayerNorm kernel (fp32 sum
        before the statistics) instead of the GEMM epilogue.  Measured on the wiki103 shape: moving it into the epilogue
        halves LayerNorm (1.0 -> 0.5 ms per step) but makes the epilogue the GEMM's bottleneck (a split-fp16 residual
        turns the 1.3 ms A-linear into 3.4 ms, an fp32 one into 1.7 ms; profiles/gemm_probe_split.py)."""
        if tau == P["n"] and P["a_rot"] is not None:      # rotation folded: h_in is un-rotated, the product adds the residual
            o = _lin(with_q8(t_agg, P["math"], n_dev), P["a_rot"], P["math"], x2=with_q8(h_in, P["math"], n_dev), m_dev=n_dev)
            h_in = None
        else:
            o = _lin(with_q8(t_agg, P["math"], n_dev), P["a"][tau], P["math"], m_dev=n_dev)
        g, b, eps = P["ln"][tau]
        act = gemm_act(P["math"], o.shape[0], o.shape[1]) if feeds_gemm else act_dtype(P["math"])
        if act == torch.float32:
            return ops.layernorm(o, g, b, eps, out=o, n_dev=n_dev, residual=h_in)
        return ops.layernorm(o, g, b, eps, out_dtype=act, n_dev=n_dev, residual=h_in)       # bf16 or split fp16 (+ e4m3 companion)

    def _hq(self, G, h_n, centre: bool) -> bool:
        """Q | K' | V' of the ntgt side as GNNLM_F24 (3 bytes per element instead of 4): when the f16f8 product writes them (the
        operand carries its e4m3 companion) and the centre-only cluster kernel reads them.  The all-nodes cluster kernel is faster on
        fp32 rows (cluster_attn.cu), so only the centre-only layer uses the format unless GNNLM_HQ=all."""
        d, H = self.in_dim, self.n_heads
        return ((centre or self.use_hq_attention == "all") and bool(self.use_hq_attention) and isinstance(h_n, ops.Split)
                and self.use_cluster_kernel and not G.dedup and ops.cluster_attn_hq_supported(d, H, G.w) and ops.f16f8_supported(d))

    def _nn_attn(self, P, G, q, k, v, rows, *, centre: bool, n_dev, c_dev, kv_affine=None):
        """ntgt-intra-ntgt attention -> [rows, d] in the activation dtype."""
        d, H = P["d"], self.n_heads
        act = act_dtype(P["math"])
        tag = "nn_centre" if centre else "nn_full"
        if isinstance(q, ops.HiLo8) or (self.use_cluster_kernel and not G.dedup and ops.cluster_attn_supported(d, H, q.dtype, G.w)):
            t_agg = ops.empty_act(rows, d, gemm_act(P["math"], rows, d, lo=False), q.device)   # feeds the A-linear and nothing else
            ops.cluster_attn(q, k, v, G, H, t_agg, centre_only=centre, tag=tag, kv_affine=kv_affine)
            return t_agg
        assert kv_affine is None
        t_agg = torch.empty((rows, d), device=q.device, dtype=torch.float32)
        if centre:
            ops.edge_attn(q, k, v, G.nn_indptr, G.nn_indices, H, t_agg, dst_ids=G.inter_indices, n_dst_dev=c_dev, tag=tag)
        else:
            ops.edge_attn(q, k, v, G.nn_indptr, G.nn_indices, H, t_agg, n_dst_dev=n_dev, tag=tag)
        return as_act(t_agg, P["math"])

    def _full_attn(self, P, G: TokenGraph, h_n, n_dev):
        """Q|K'|V' of all ntgt nodes -> chain attention -> the A-linear operand.  One kernel (ops.linear_f16f8_nn_attn) where it
        applies: MATH_F16F8, d_k = 128, clusters of 1, 3, 5 or 7 nodes and an fp32 Q|K'|V'."""
        d = P["d"]
        x = with_q8(h_n, P["math"], n_dev)
        hq = self._hq(G, h_n, centre=False)
        if ("ntgt_qkv_heads" in P and self.use_fused_nn and self.use_cluster_kernel and not G.dedup and G.w in (1, 3, 5, 7) and not hq
                and isinstance(x, ops.Split) and x.q8 is not None and ops.f16f8_supported(x.d)
                and gemm_act(P["math"], x.shape[0], d, lo=False) == ops.HI_Q8):
            W = P["ntgt_qkv_heads"]
            return ops.linear_f16f8_nn_attn(x, W.W, W.w8(), W.b, G, self.n_heads, w_scale=W.scale)
        qkv = _lin(x, P["ntgt_qkv"], P["math"], m_dev=n_dev, out_dtype=_attn_in_dtype(P["math"], hq))
        return self._nn_attn(P, G, qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], h_n.shape[0], centre=False, n_dev=n_dev, c_dev=None)

    def ntgt_full(self, P, G: TokenGraph, h_n, n_dev):
        """All ntgt nodes: Q|K'|V' -> chain attention -> A-linear + residual + LN."""
        t_agg = self._full_attn(P, G, h_n, n_dev)
        return self._out(P, P["n"], t_agg, h_n, n_dev, feeds_gemm=True)        # h of the next layer: a GEMM operand

    def ntgt_full_deferred(self, P, G: TokenGraph, x_n, n_dev):
        """ntgt_full of layer 0 with the rotation folded and the LayerNorm DEFERRED: returns (z', stats) -- the pre-norm sum in the
        un-rotated basis as a GEMM operand and (mean, 1 / std) of its rotation per node (ops.rowstats_q8) -- instead of h1.  The
        residual x is added un-rotated (z' = A-linear(t) rot + x), which halves the output projection (K = d instead of 2 d)."""
        D = P["defer"]
        t_agg = self._full_attn(P, G, x_n, n_dev)
        o = _lin(with_q8(t_agg, P["math"], n_dev), D["a"], P["math"], m_dev=n_dev)
        return ops.rowstats_q8(o, x_n, D["u"], P["ln"][P["n"]][2], n_dev)

    def deferred_centres(self, P, G: TokenGraph, z, n_dev, c_dev):
        """h1 of the centre nodes from the deferred sum: LayerNorm(z'_c rot^T) -- what the inter edges and the next layer's Q /
        residual read (compact rows)."""
        zc = ops.gather_rows(z, G.inter_indices, n_dev=c_dev)
        o = _lin(zc, P["defer"]["rot"], P["math"], m_dev=c_dev)
        g, b, eps = P["ln"][P["n"]]
        return ops.layernorm(o, g, b, eps, out_dtype=gemm_act(P["math"], o.shape[0], o.shape[1]), n_dev=c_dev)

    def ntgt_centre(self, P, G: TokenGraph, h_n, n_dev, hc, c_dev, deferred=None):
        """Centre nodes only (compact rows): K'|V' for every node, Q / A-linear / LN for centres.  `deferred` = stats of
        ntgt_full_deferred: h_n is then the un-normalised z' and K' | V' are its raw products, normalised inside the attention
        kernel (P["kv_deferred"])."""
        d = P["d"]
        act = _attn_in_dtype(P["math"], self._hq(G, h_n, centre=True))
        kv_affine = None
        if deferred is not None:
            KD = P["kv_deferred"]
            assert act == ops.HILO8
            kv = _lin(h_n, KD["w"], P["math"], m_dev=n_dev, out_dtype=act)
            kv_affine = (deferred, KD["k_c"], KD["k_b"], KD["v_c"], KD["v_b"])
        else:
            kv = _lin(with_q8(h_n, P["math"], n_dev), P["ntgt_qkv"].rows(d, 3 * d), P["math"], m_dev=n_dev, out_dtype=act)
        qc = _lin(with_q8(hc, P["math"], c_dev), P["ntgt_qkv"].rows(0, d), P["math"], m_dev=c_dev, out_dtype=act)
        t_agg = self._nn_attn(P, G, qc, kv[:, :d], kv[:, d:], hc.shape[0], centre=True, n_dev=n_dev, c_dev=c_dev, kv_affine=kv_affine)
        return self._out(P, P["n"], t_agg, hc, c_dev)

    def tgt(self, P, G: TokenGraph, h_t, hc, c_dev, chunks=None):
        """tgt nodes: mean of (centre ntgt -> tgt) attention and causal tgt -> tgt attention.  Q/K'/V' of this
        (small) side are kept in fp32 in every mode.  `chunks`: [(t0, t1, chunk_graph, hc_chunk)] when the ntgt side
        was run in token chunks -- the inter attention is then applied chunk by chunk (hc / c_dev unused)."""
        d, H = P["d"], self.n_heads
        gemm_modes = (L.MATH_F16X3, L.MATH_F16F8, L.MATH_BF16, L.MATH_TF32)
        flash = (P["math"] in gemm_modes and self.use_flash_attention and ops.causal_flash_supported(d, H)
                 and L.load().gnnlm_has_tcgen05())
        qkv = _lin(h_t, P["tgt_qkv"], P["math"])
        flash_tc = flash and self.use_flash_tc and ops.causal_flash_tc_supported(d, H, G.L)      # tcgen05 form (d_k = 128)
        if flash and not flash_tc:   # Q stays fp32 (the inter path and the mma.sync kernel split it themselves); K' | V' as split fp16
            kv = ops.to_split(qkv[:, d:])
        t_agg = torch.empty((h_t.shape[0], d), device=qkv.device, dtype=torch.float32)
        # inter edges in compact centre numbering are the contiguous ranges of inter_indptr
        if P["inter_fused"] is not None and self.use_fused_inter:
            F_ = P["inter_fused"]
            parts = [(0, G.T, G.inter_indptr, hc)] if chunks is None else [(t0, t1 - t0, g_c.inter_indptr, hc_c)
                                                                          for t0, t1, g_c, hc_c in chunks]
            ops.inter_attn_fused(qkv[:, :d], parts, H, t_agg, F_["wk_t"], F_["wv"], F_["bv"], out_scale=0.5)
        elif chunks is None:
            kvi = _lin(hc, P["ntgt_kv_inter"], P["math"], m_dev=c_dev)
            ops.edge_attn(qkv[:, :d], kvi[:, :d], kvi[:, d:], G.inter_indptr, None, H, t_agg, out_scale=0.5, tag="inter")
        else:
            for t0, t1, g_c, hc_c in chunks:
                kvi = _lin(hc_c, P["ntgt_kv_inter"], P["math"], m_dev=g_c.n_valid_dev)
                ops.edge_attn(qkv[t0:t1, :d], kvi[:, :d], kvi[:, d:], g_c.inter_indptr, None, H, t_agg[t0:t1], out_scale=0.5,
                              tag="inter")
        # tensor-core form (3xFP16 GEMMs on the fp32 Q / K' / V', fp32-level accuracy) in every mode that already puts fp16-range
        # operands on the tensor cores; tf32x3 / fp32 keep the CUDA-core kernel (no fp16 range limit on Q / K' / V')
        if flash:
            act = act_dtype(P["math"])
            t_split = ops.Split.empty(h_t.shape[0], d, qkv.device) if act == ops.SPLIT else None    # the output projection's operand
            if flash_tc:
                ops.causal_attn_flash_tc(qkv, G.B, G.L, G.intra_ctx, H, t_agg, out_scale=0.5, accumulate=True, out_split=t_split)
            else:
                ops.causal_attn_flash(qkv[:, :d], kv, G.B, G.L, G.intra_ctx, H, t_agg, out_scale=0.5, accumulate=True, out_split=t_split)
            if t_split is not None:
                return self._out(P, P["t"], t_split, h_t, None)
        elif P["math"] in gemm_modes and self.use_gemm_attention and ops.causal_attn_gemm_supported(d, H, G.L) and G.L >= 1024:
            ops.causal_attn_gemm(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], G.B, G.L, G.intra_ctx, H, t_agg, out_scale=0.5,
                                 accumulate=True)
        else:
            ops.causal_attn(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], G.B, G.L, G.intra_ctx, H, t_agg, out_scale=0.5,
                            accumulate=True)
        return self._out(P, P["t"], as_act(t_agg, P["math"]), h_t, None)

    def forward(self, G: TokenGraph, h: Dict[str, torch.Tensor], etypes=None, incremental_state=None,
                math_mode: int = L.MATH_FP32_SIMT) -> Dict[str, torch.Tensor]:
        """Full layer, every node of both types (hgt.py:299-420).  A general heterograph (hetero.HeteroGraph: any node / edge
        types, `two_stream`) and incremental decoding (`incremental_state`, hgt.py:308-310 -> infer) run in hetero.py."""
        if incremental_state is not None:
            return hetero.layer_infer(self, G, h, etypes, incremental_state, math_mode)
        if isinstance(G, HeteroGraph):
            return hetero.layer_forward(self, G, h, etypes, math_mode)
        if self.two_stream:
            raise KeyError(("src", "intra", "tgt"))      # the token graph has no 'src' node type (hgt.py:390-393 would raise)
        P = self.prepare(math_mode)
        n_valid = G.counts()[1]
        h_t, h_n = as_act(h["tgt"], math_mode), as_act(h["ntgt"], math_mode)
        hc = ops.gather_rows(h_n, G.inter_indices, n_cap=n_valid)
        new_t = self.tgt(P, G, h_t, hc, None)
        new_n = self.ntgt_full(P, G, h_n, None)
        return {"tgt": new_t, "ntgt": new_n}       # activation format of the math mode (HGT.forward converts back)


    def reorder_incremental_state(self, incremental_state, new_order):
        """hgt.py:422-438."""
        return hetero.reorder_incremental_state(self, incremental_state, new_order)


class HGT(nn.Module):
    """Same constructor / keys as the reference (hgt.py:459-492)."""

    def __init__(self, ntype2idx, etype2idx, in_dim, hidden_dim, out_dim, n_layers, n_heads, use_norm=True,
                 dropout=0.0, two_stream=False, attn_drop=0.0):
        super().__init__()
        self.ntype2idx, self.etype2idx = ntype2idx, etype2idx
        self.in_dim, self.hidden_dim, self.out_dim, self.n_layers = in_dim, hidden_dim, out_dim, n_layers
        self.adapt_ws = nn.ModuleList()                       # hgt.py:482-492: only when --decoder_gcn_dim != embedding width
        if in_dim != hidden_dim:
            for _ in range(len(ntype2idx)):
                self.adapt_ws.append(nn.Linear(in_dim, hidden_dim))
        if hidden_dim != out_dim:
            self.out = nn.Linear(hidden_dim, out_dim)
        self._io_prep, self._io_key = None, None
        self.gcs = nn.ModuleList(HGTLayer(hidden_dim, hidden_dim, ntype2idx, etype2idx, n_heads, use_norm=use_norm,
                                          dropout=dropout, two_stream=two_stream, attn_drop=attn_drop)
                                 for _ in range(n_layers))
        self.math_mode = L.MATH_FP32_SIMT

    def set_math(self, mode):
        self.math_mode = L.MATH_NAMES[mode] if isinstance(mode, str) else int(mode)
        return self

    def _io(self):
        """Prepared weights of the input adapters / output projection for the current math mode."""
        mode = self.math_mode
        ws = list(self.adapt_ws) + ([self.out] if self.hidden_dim != self.out_dim else [])
        key = (mode,) + tuple((w.weight.device, int(w.weight._version), int(w.bias._version)) for w in ws)
        if self._io_prep is None or self._io_key != key:
            mk = lambda lin: _Weight(lin.weight.detach(), lin.bias.detach(), mode)
            self._io_prep = {"adapt": [mk(w) for w in self.adapt_ws],
                             "out": mk(self.out) if self.hidden_dim != self.out_dim else None}
            self._io_key = key
        return self._io_prep

    def adapt(self, x, ntype: str, n_dev=None):
        """h = gelu(adapt_ws[t](x)) when in_dim != hidden_dim (hgt.py:505-507), in the activation format; else x."""
        if self.in_dim == self.hidden_dim or x is None:
            return x
        w = self._io()["adapt"][self.ntype2idx[ntype]]
        y = _lin(as_act(x, self.math_mode), w, self.math_mode, m_dev=n_dev)                 # fp32 pre-activation
        return ops.gelu(y, act_dtype(self.math_mode), n_dev=n_dev)

    def project_out(self, h, n_dev=None):
        """self.out(h) when hidden_dim != out_dim (hgt.py:513)."""
        if self.hidden_dim == self.out_dim:
            return h
        return _lin(as_act(h, self.math_mode), self._io()["out"], self.math_mode, m_dev=n_dev)

    def forward(self, G: TokenGraph, features: Dict[str, torch.Tensor] = None, etypes=None, incremental_state=None):
        """Reference-shaped call (hgt.py:494-513): returns features of every node of every type."""
        h = {}
        if incremental_state is not None and not isinstance(G, HeteroGraph):
            raise TypeError("incremental decoding runs over a hetero.HeteroGraph with max_len tgt nodes per block (hgt.py:93)")
        for ntype in (G.ntypes if isinstance(G, HeteroGraph) else ("tgt", "ntgt")):
            x = None if not features else features.get(ntype)
            if x is None:
                x = G.nodes[ntype].data["h"]
            x = x if x.dtype == torch.bfloat16 else x.float().contiguous()
            h[ntype] = self.adapt(x, ntype)
        for layer in self.gcs:
            h = layer(G, h, etypes=etypes, incremental_state=incremental_state, math_mode=self.math_mode)
        return {k_: as_float(self.project_out(v)) for k_, v in h.items()}

    @torch.no_grad()
    def forward_tgt(self, G: TokenGraph, h_tgt: torch.Tensor, h_ntgt: Optional[torch.Tensor],
                    hc0: Optional[torch.Tensor] = None, rot: Optional[torch.Tensor] = None) -> torch.Tensor:
        """tgt features only (what the decoder consumes, transformer.py:1053), capacity-sized ntgt
        arrays + device-side row counts: no host synchronisation anywhere.

        h_ntgt [node_cap, d] decoded features of every ntgt node (may be None when n_layers == 1 and
        hc0, the decoded centre rows [T*k, d], is given)."""
        mode = self.math_mode
        prep = self._prepare_layers(rot)
        hc = self._ntgt_side(prep, G, h_ntgt, hc0)
        h_t = as_act(self.adapt(h_tgt, "tgt"), mode)
        for l in range(self.n_layers):
            h_t = self.gcs[l].tgt(prep[l], G, h_t, hc[l], G.n_valid_dev)
        return self.project_out(h_t)

    @torch.no_grad()
    def forward_tgt_shared(self, G: TokenGraph, h_tgt, decode, rot=None):
        """Same result as forward_tgt with the ntgt side run once per DISTINCT centre row (graph.unique_centre_graph): clusters
        that share a centre are identical in every layer, so their compact centre features are computed on the graph of the
        distinct rows and gathered back per (token, neighbour) pair.  `decode(graph, centre_only)` as in forward_tgt_chunked."""
        from .graph import unique_centre_graph
        mode = self.math_mode
        prep = self._prepare_layers(rot)
        G_u, inv, _ = unique_centre_graph(G)
        if self.n_layers == 1:
            hc_u = self._ntgt_side(prep, G_u, None, hc0=decode(G_u, True))
        else:
            hc_u = self._ntgt_side(prep, G_u, decode(G_u, False), hc0=decode(G_u, True) if rot is not None else None)
        hc = [ops.gather_rows(x, inv, n_dev=G.n_valid_dev) for x in hc_u]
        h_t = as_act(self.adapt(h_tgt, "tgt"), mode)
        for l in range(self.n_layers):
            h_t = self.gcs[l].tgt(prep[l], G, h_t, hc[l], G.n_valid_dev)
        return self.project_out(h_t)

    def can_fold_rotation(self, d_dec: int) -> bool:
        """MATH_F16F8 with no input adapters: the OPQ rotation of the ntgt features can be folded into layer 0
        (HGTLayer.prepare `rot`); needs the two-source f16f8 product (k-blocks of 64) and the fused inter kernel."""
        d = self.hidden_dim
        return (self.math_mode == L.MATH_F16F8 and self.in_dim == self.hidden_dim and d_dec == d and d in (128, 256, 512, 1024)
                and ops.f16f8_supported(d, d) and ops.inter_fused_supported(d, self.gcs[0].n_heads) and self.gcs[0].use_fused_inter)

    def _prepare_layers(self, rot=None):
        """`rot`: ntgt input features (h_ntgt / hc0 and whatever `decode` returns) are un-rotated; folded into layer 0."""
        assert rot is None or self.can_fold_rotation(rot.shape[1])
        prep = []
        for l, layer in enumerate(self.gcs):
            prev_ln = None
            if l == 1 and rot is not None and self.n_layers == 3 and "defer" in prep[0]:      # layer 0 may defer its ntgt LayerNorm
                n = self.gcs[0].ntype2idx["ntgt"]
                prev_ln = (self.gcs[0].norms[n].weight, self.gcs[0].norms[n].bias, rot)
            prep.append(layer.prepare(self.math_mode, rot if l == 0 else None, prev_ln))
        return prep

    def _ntgt_side(self, prep, G: TokenGraph, h_ntgt, hc0=None) -> List:
        """All layers of the ntgt side of one (chunk) graph -> compact centre features entering each layer."""
        n_dev, c_dev = G.n_ntgt_dev, G.n_valid_dev
        NL, mode = self.n_layers, self.math_mode
        hc: List = []
        if h_ntgt is not None:
            h_ntgt = as_act(self.adapt(h_ntgt, "ntgt", n_dev), mode)
        elif hc0 is not None:
            hc0 = self.adapt(hc0, "ntgt", c_dev)
        # (rotation folded into layer 0: the caller passes both, un-rotated -- h_ntgt as fp16 hi + e4m3 companion only, hc0 as a
        # full split matrix, because the inter kernel reads both fp16 halves of the centre rows)
        if hc0 is None:
            hc0 = ops.gather_rows(h_ntgt, G.inter_indices, n_dev=c_dev)
        hc.append(hc0)
        h_n = h_ntgt
        if (NL == 3 and "defer" in prep[0] and "kv_deferred" in prep[1] and isinstance(h_n, ops.Split) and h_n.q8 is not None
                and self.gcs[1]._hq(G, h_n, centre=True)):
            # layer 0's LayerNorm deferred into its consumers: no rotation of the residual, no normalised non-centre rows
            z, stats = self.gcs[0].ntgt_full_deferred(prep[0], G, h_n, n_dev)
            hc.append(self.gcs[0].deferred_centres(prep[0], G, z, n_dev, c_dev))
            hc.append(self.gcs[1].ntgt_centre(prep[1], G, z, n_dev, hc[1], c_dev, deferred=stats))
            return hc
        for l in range(NL - 1):
            if l < NL - 2:
                h_n = self.gcs[l].ntgt_full(prep[l], G, h_n, n_dev)
                hc.append(ops.gather_rows(h_n, G.inter_indices, n_dev=c_dev))
            else:
                hc.append(self.gcs[l].ntgt_centre(prep[l], G, h_n, n_dev, hc[l], c_dev))
        return hc

    @torch.no_grad()
    def forward_tgt_chunked(self, G: TokenGraph, h_tgt, decode, chunk_tokens: int, rot=None):
        """Same result as forward_tgt with the ntgt side run in chunks of `chunk_tokens` target tokens, so that the
        ntgt activations (T*k*w rows per buffer) never exceed a memory budget: ntgt clusters belong to exactly one
        token and only ever exchange messages inside their cluster (SURVEY.md 7.4).  `decode(chunk_graph, centre_only)`
        returns the decoded ntgt features of a chunk graph (all nodes, or compact centre rows)."""
        from .graph import token_chunk_graph
        mode = self.math_mode
        prep = self._prepare_layers(rot)
        chunks = []
        for t0 in range(0, G.T, chunk_tokens):
            t1 = min(G.T, t0 + chunk_tokens)
            g_c = token_chunk_graph(G, t0, t1)
            if self.n_layers == 1:
                hc_c = self._ntgt_side(prep, g_c, None, hc0=decode(g_c, True))
            else:
                hc_c = self._ntgt_side(prep, g_c, decode(g_c, False), hc0=decode(g_c, True) if rot is not None else None)
            chunks.append((t0, t1, g_c, hc_c))
        h_t = as_act(self.adapt(h_tgt, "tgt"), mode)
        for l in range(self.n_layers):
            h_t = self.gcs[l].tgt(prep[l], G, h_t, None, None, chunks=[(t0, t1, g_c, hc_c[l]) for t0, t1, g_c, hc_c in chunks])
        return self.project_out(h_t)
