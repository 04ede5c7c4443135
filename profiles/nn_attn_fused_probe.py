"""The all-nodes ntgt-intra-ntgt attention of layer 0 at the Wiki103 shape (c3: 3072 tokens x 32 neighbours x w = 3, d = 1024,
H = 8): the fused projection + attention (gnnlm_linear_f16f8_nn_attn) against the two kernels it replaces (gnnlm_linear_f16f8
into fp32 Q|K'|V', then gnnlm_hgt_cluster_attn_q8), CUDA events over many back-to-back launches of each, alternated.
  python profiles/nn_attn_fused_probe.py [reps] [rounds]"""
import subprocess, sys, torch
sys.path.insert(0, '.')
from gnnlm_b200 import _lib as L, ops, synth
from gnnlm_b200.graph import build_token_graph
from gnnlm_b200.hgt import _Weight, head_interleave

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
dev = torch.device('cuda')
print(subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip(), flush=True)
cfg = synth.CONFIGS['c3']
d, H = cfg['d'], cfg['H']
tables = synth.make_tables(cfg, device=dev)
batch = synth.make_batch(cfg, tables, device=dev)
g = build_token_graph(batch['nbr'], tables['n_d'], cfg['c'], cfg['c'])
n, _ = g.counts()
gen = torch.Generator(device='cpu').manual_seed(0)
x = ops.to_q8(ops.to_split(torch.randn(g.node_cap, d, generator=gen).to(dev)))
W = torch.randn(3 * d, d, generator=gen) / d ** 0.5
W[d:2 * d] /= 128 ** 0.5                                     # K' carries 1 / sqrt(d_k), as folded by HGTLayer.prepare
w = _Weight(W.to(dev), (0.1 * torch.randn(3 * d, generator=gen)).to(dev), L.MATH_F16F8)
wp = w.permuted(head_interleave(H, 128).to(dev))
qkv = torch.empty(g.node_cap, 3 * d, device=dev)
out_ref = ops.empty_act(g.node_cap, d, ops.HI_Q8, dev)


def two_kernels():
    ops.linear_f16f8(x, w.W, w.w8(), w.b, w_scale=w.scale, m_dev=g.n_ntgt_dev, out=qkv)
    ops.cluster_attn(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], g, H, out_ref)


def fused():
    return ops.linear_f16f8_nn_attn(x, wp.W, wp.w8(), wp.b, g, H, w_scale=wp.scale)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


for fn in (two_kernels, fused):
    for _ in range(3):
        fn()
torch.cuda.synchronize()
out = fused()
two_kernels()
torch.cuda.synchronize()
same = float((out.data[:n] == out_ref.data[:n]).double().mean())
print(f"rows {n} (capacity {g.node_cap}), K = N / 3 = {d}; fp16 hi equal to the two-kernel output: {same:.6f}; "
      f"error word {int(ops.nn_attn_error(dev).item())}", flush=True)
flops = 2.0 * n * 3 * d * d
for r in range(rounds):
    a, b = timed(two_kernels), timed(fused)
    print(f"round {r}: linear_f16f8 + cluster_attn {a:.3f} ms   fused {b:.3f} ms ({flops / b / 1e9:.0f} useful TFLOP/s)   "
          f"saved {a - b:.3f} ms", flush=True)
