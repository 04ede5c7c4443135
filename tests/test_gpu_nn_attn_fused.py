"""gnnlm_linear_f16f8_nn_attn (the all-nodes chain attention in the epilogue of its Q|K'|V' projection) against the two-kernel
path it replaces: gnnlm_linear_f16f8 into fp32 Q|K'|V', then gnnlm_hgt_cluster_attn_q8 into the same fp16 hi + e4m3 operand."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _graph(dev, T, k, c, n_d, seed):
    """Random neighbours with invalid ones (-1) and rows at both ends of the datastore (truncated clusters)."""
    from gnnlm_b200.graph import build_token_graph
    rng = np.random.RandomState(seed)
    nbr = rng.randint(0, n_d, size=(1, T, k)).astype(np.int64)
    nbr[rng.rand(1, T, k) < 0.05] = -1
    ends = rng.rand(1, T, k) < 0.05
    nbr[ends] = rng.choice([0, 1, n_d - 2, n_d - 1], size=int(ends.sum()))
    nbr[0, 0, 0] = n_d // 2                                  # at least one cluster
    return build_token_graph(torch.from_numpy(nbr).to(dev), n_d, c, c)


def _operands(g, K, H, seed, dev):
    from gnnlm_b200 import _lib as L, ops
    from gnnlm_b200.hgt import _Weight, head_interleave
    gen = torch.Generator(device="cpu").manual_seed(seed)
    d = 128 * H
    x = ops.to_q8(ops.to_split(torch.randn(g.node_cap, K, generator=gen).to(dev)))
    W = torch.randn(3 * d, K, generator=gen) / K ** 0.5
    W[d:2 * d] /= 128 ** 0.5                                 # K' carries 1 / sqrt(d_k) (HGTLayer.prepare): scores of order one
    W = W.to(dev)
    b = (0.1 * torch.randn(3 * d, generator=gen)).to(dev)
    w = _Weight(W, b, L.MATH_F16F8)
    return x, w, w.permuted(head_interleave(H, 128).to(dev))


def _reconstruct(t):
    """fp32 value of an fp16 hi + e4m3 companion operand: hi + lo8 / 2^10."""
    return t.data.float() + t.q8[:, t.d:].view(torch.float8_e4m3fn).float() / 1024.0


def _two_kernels(x, w, g, H):
    from gnnlm_b200 import ops
    d = 128 * H
    qkv = ops.linear_f16f8(x, w.W, w.w8(), w.b, w_scale=w.scale, m_dev=g.n_ntgt_dev, out_dtype=torch.float32)
    out = ops.empty_act(x.shape[0], d, ops.HI_Q8, x.data.device)
    ops.cluster_attn(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], g, H, out)
    return out


def _check(dev, T, k, c, n_d, H, K, seed):
    from gnnlm_b200 import ops
    g = _graph(dev, T, k, c, n_d, seed)
    n = g.counts()[0]
    x, w, wp = _operands(g, K, H, seed, dev)
    err = ops.nn_attn_error(dev)
    err.zero_()
    ref = _two_kernels(x, w, g, H)
    out = ops.linear_f16f8_nn_attn(x, wp.W, wp.w8(), wp.b, g, H, w_scale=wp.scale)
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    a, r = _reconstruct(out)[:n].double(), _reconstruct(ref)[:n].double()
    assert torch.isfinite(a).all()
    row_max = r.abs().amax(1, keepdim=True)
    diff = (a - r).abs()
    strict = 2e-6 * row_max
    # The GEMM accumulators are identical; the score dot products are summed in another order, which moves the fp32 results by
    # ~1e-7 of the row.  The output keeps fp16 hi + an e4m3 lo8 (3 bits): where such a difference crosses a rounding boundary of
    # either, the two reconstructions are one companion step (<= 2^-14 |x|) apart -- a fraction of a percent of the elements.
    beyond = float((diff > strict).double().mean())
    hi_same = float((out.data[:n] == ref.data[:n]).double().mean())
    info = f"max diff / row max {float((diff / row_max).max()):.3e}, beyond 2e-6: {beyond:.2e}, fp16 hi equal: {hi_same:.6f}"
    assert (diff <= strict + 2.0 ** -14 * r.abs()).all(), info
    assert beyond < 1e-2, info
    assert hi_same > 0.995, info
    return n


@pytest.mark.parametrize("c", [0, 1, 2])
def test_fused_matches_two_kernels(c, dev):
    """w = 1, 3, 5; thousands of rows: clusters straddle warp (32-row) and window boundaries; live rows below capacity."""
    n = _check(dev, T=96, k=16, c=c, n_d=4096, H=2, K=256, seed=11 + c)
    assert n > 4 * 128


def test_fused_wiki103_width(dev):
    """d = 1024, H = 8 (the Wiki103 model): every QK tile and both heads of every V tile."""
    _check(dev, T=64, k=8, c=1, n_d=1 << 20, H=8, K=1024, seed=5)


@pytest.mark.parametrize("T,k", [(1, 1), (1, 4), (2, 20)])
def test_fused_fewer_rows_than_a_window(T, k, dev):
    """M below one window (S = 124 at w = 3), window 0 starting at row -h (zero-filled by TMA), a single window pair."""
    _check(dev, T=T, k=k, c=1, n_d=64, H=2, K=128, seed=T * 100 + k)


def test_fused_flags_neighbours_outside_the_window(dev):
    """A graph whose chains are longer than the w the kernel is told: rows at window edges have neighbours beyond the halo.  The
    kernel sets the error word instead of reading outside its accumulator."""
    from types import SimpleNamespace
    from gnnlm_b200 import ops
    g = _graph(dev, T=64, k=16, c=1, n_d=4096, seed=3)
    x, _, wp = _operands(g, 128, 2, 3, dev)
    err = ops.nn_attn_error(dev)
    err.zero_()
    bad = SimpleNamespace(nn_indptr=g.nn_indptr, nn_indices=g.nn_indices, w=1, n_ntgt_dev=g.n_ntgt_dev)
    ops.linear_f16f8_nn_attn(x, wp.W, wp.w8(), wp.b, bad, 2, w_scale=wp.scale)
    torch.cuda.synchronize()
    assert int(err.item()) == 1
    err.zero_()


def test_hgt_layer_uses_fused_path(dev, monkeypatch):
    """HGTLayer.ntgt_full takes the fused kernel in MATH_F16F8 at d_k = 128 and gives the two-kernel result."""
    from gnnlm_b200 import _lib as L, ops
    from gnnlm_b200.hgt import HGTLayer
    torch.manual_seed(0)
    g = _graph(dev, T=32, k=8, c=1, n_d=4096, seed=9)
    n = g.counts()[0]
    layer = HGTLayer(256, 256, {"tgt": 0, "ntgt": 1}, {"intra": 0, "inter": 1}, n_heads=2).to(dev)
    h = ops.to_q8(ops.to_split(torch.randn(g.node_cap, 256, device=dev)))
    calls = []
    real = ops.linear_f16f8_nn_attn
    monkeypatch.setattr(ops, "linear_f16f8_nn_attn", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    P = layer.prepare(L.MATH_F16F8)
    fused = layer.ntgt_full(P, g, h, g.n_ntgt_dev).float()[:n]
    assert calls
    layer.use_fused_nn = False
    plain = layer.ntgt_full(P, g, h, g.n_ntgt_dev).float()[:n]
    assert len(calls) == 1
    torch.testing.assert_close(fused, plain, rtol=0, atol=1e-4)
