"""Exact kNN search at the Wiki103 shape: d = 1024, a 103 M-row OPQ-PQ datastore (M = 128, dsub = 8: 13.2 GB of random codes,
resident), 16 384 queries, k = 1024, metric l2.  Prints (and writes as JSON with --out):
  - the GPU's name and power limit (read in the same run);
  - queries/s of one end-to-end search (no per-call events);
  - the time split decode / filter GEMM / merge / key bias from a second, instrumented search (CUDA events around every C-ABI
    call), candidates per query per span and the overflow re-runs;
  - useful TFLOP/s of the filter GEMM (2 n_q N_d d over its time);
  - the same GEMM shape (65 536 keys x 16 384 queries x 1024) through gnnlm_linear with an fp32 store, timed alternately with the
    filter GEMM, to price the epilogue;
  - a raw-fp16-keys search streamed from host memory (device budget forced to zero, so every span crosses PCIe) against the same
    keys resident, and the bare H2D time of those bytes: the overlap of copy and search.
    python profiles/knn_search_probe.py [--n-d 103000000] [--stream-keys 4000000] [--out FILE]"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from gnnlm_b200 import _lib as L, ops  # noqa: E402
from gnnlm_b200.knn_search import KNNSearcher, PQKeys, RawKeys  # noqa: E402
from gnnlm_b200.pq_codec import TorchPQCodec  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
    return out


def timed_search(searcher, q):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d, i = searcher.search(q)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, d, i


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-d", type=int, default=103_000_000)
    ap.add_argument("--n-q", type=int, default=16384)
    ap.add_argument("--k", type=int, default=1024)
    ap.add_argument("--span-keys", type=int, default=1 << 19)
    ap.add_argument("--stream-keys", type=int, default=4_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda")
    res = {"gpu": gpu_info(), "n_d": a.n_d, "n_q": a.n_q, "k": a.k, "d": 1024, "M": 128}
    print("GPU (name, power limit, max SM clock):", res["gpu"], flush=True)
    g = torch.Generator(device=dev).manual_seed(0)
    rng = np.random.RandomState(0)
    cen = rng.randn(128, 256, 8).astype(np.float32)
    A = np.linalg.qr(rng.randn(1024, 1024))[0].astype(np.float32)
    codec = TorchPQCodec(centroids=cen, A=A, b=(0.1 * rng.randn(1024)).astype(np.float32))
    codes = torch.randint(0, 256, (a.n_d, 128), generator=g, device=dev, dtype=torch.uint8)
    q = torch.randn((a.n_q, 1024), generator=g, device=dev) * 3.0
    s = KNNSearcher(PQKeys(codes, codec), "l2", a.k, span_keys=a.span_keys, device=dev)
    res["spans"] = len(s.schedule)
    s.search(q[:256])                                         # warm-up: module load, every kernel once
    t, d, i = timed_search(s, q)
    res["search_s"], res["queries_per_s"] = t, a.n_q / t
    print(f"end-to-end: {t:.2f} s for {a.n_q} queries over {a.n_d} keys ({len(s.schedule)} spans) -> {a.n_q / t:.0f} queries/s",
          flush=True)

    # instrumented pass: events around every C-ABI call, candidates counted before each merge (on the device)
    cand = torch.zeros((), dtype=torch.int64, device=dev)
    merges = [0]
    merge = ops.topk_merge

    def counting_merge(top_s, top_id, cs, ci, cc, thr):
        if cc.shape[0] == a.n_q:
            cand.add_(cc.clamp(max=cs.shape[1]).sum())
            merges[0] += 1
        merge(top_s, top_id, cs, ci, cc, thr)
    ops.topk_merge = counting_merge
    s.reruns = 0
    L.TIMING = []
    t2, d2, i2 = timed_search(s, q)
    torch.cuda.synchronize()
    split = {}
    for name, tag, e0, e1, work in L.TIMING:
        split[tag or name] = split.get(tag or name, 0.0) + e0.elapsed_time(e1) / 1e3
    L.TIMING = None
    ops.topk_merge = merge
    assert torch.equal(d2, d) and torch.equal(i2, i)
    res["instrumented_s"], res["split_s"] = t2, split
    res["candidates_per_query_per_span"] = float(cand) / a.n_q / max(merges[0], 1)
    res["overflow_reruns"] = s.reruns
    flop = 2.0 * a.n_q * a.n_d * 1024
    res["filter_tflops_useful"] = flop / split["knn_filter"] / 1e12
    print("time split (s): " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(split.items(), key=lambda kv: -kv[1])), flush=True)
    print(f"filter GEMM: {res['filter_tflops_useful']:.0f} TFLOP/s useful; candidates per query per span "
          f"{res['candidates_per_query_per_span']:.1f}; overflow re-runs {s.reruns}", flush=True)

    # the filter epilogue against a plain fp32 store on one shape (thresholds: the final ones of the search above)
    m = 65536
    keys = ops.pq_gather_decode_presplit(codes, *codec.to(dev)._split_codebook(), torch.arange(m, device=dev))
    qr = ops.linear(q, codec.A.to(dev).contiguous(), None, math=0)
    q_hi, q_lo, _ = ops.split_f16(qr, scale=1.0)
    bias = ops.knn_key_bias_pq(codes[:m], s.source.norm2)
    thr = (-0.5 * d[:, -1] - ops.knn_key_bias(q)).contiguous()          # k-th score: d_k = ||q||^2 - 2 s_k
    cs = torch.empty((a.n_q, 4096), device=dev)
    ci = torch.empty((a.n_q, 4096), device=dev, dtype=torch.int32)
    cc = torch.zeros((a.n_q,), device=dev, dtype=torch.int32)
    C = torch.empty((m, a.n_q), device=dev)

    def run_filter():
        cc.zero_()
        ops.knn_filter(keys, 0, q_hi, q_lo, bias, thr, cs, ci, cc)

    def run_store():
        ops.linear(keys, q_hi, None, W_lo=q_lo, out=C, math=L.MATH_F16X3, w_scale=1.0)

    times = {"filter": [], "store": []}
    for _ in range(2):
        run_filter(), run_store()
    for _ in range(5):
        for name, f in (("filter", run_filter), ("store", run_store)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                f()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / 3)
    fl = 2.0 * m * a.n_q * 1024
    res["same_shape_ms"] = {k: float(np.median(v)) for k, v in times.items()}
    res["same_shape_tflops_useful"] = {k: fl / (v * 1e-3) / 1e12 for k, v in res["same_shape_ms"].items()}
    print(f"same shape {m} x {a.n_q} x 1024: filter {res['same_shape_ms']['filter']:.2f} ms, fp32 store "
          f"{res['same_shape_ms']['store']:.2f} ms (medians of 5; useful TFLOP/s {res['same_shape_tflops_useful']['filter']:.0f} / "
          f"{res['same_shape_tflops_useful']['store']:.0f})", flush=True)
    del C, keys, codes, s
    torch.cuda.empty_cache()

    # raw fp16 keys streamed from host memory vs resident
    n_s = a.stream_keys
    host = np.empty((n_s, 1024), np.float16)
    for c0 in range(0, n_s, 1 << 20):
        host[c0:c0 + (1 << 20)] = torch.randn((min(1 << 20, n_s - c0), 1024), generator=g, device=dev).half().cpu().numpy()
    out = {}
    for name, budget in (("resident", None), ("streamed", 0)):
        sr = KNNSearcher(RawKeys(host, device_bytes=budget), "l2", a.k, span_keys=a.span_keys, device=dev)
        sr.search(q[:256])
        t, ds, is_ = timed_search(sr, q)
        out[name] = (t, ds, is_)
    assert torch.equal(out["resident"][1], out["streamed"][1]) and torch.equal(out["resident"][2], out["streamed"][2])
    pinned = torch.empty((a.span_keys, 1024), dtype=torch.float16).pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for c0 in range(0, n_s, a.span_keys):
        c1 = min(n_s, c0 + a.span_keys)
        np.copyto(pinned[:c1 - c0].numpy(), host[c0:c1])
        pinned[:c1 - c0].to(dev, non_blocking=True)
        torch.cuda.synchronize()
    t_copy = time.perf_counter() - t0
    res["raw_fp16"] = {"keys": n_s, "resident_s": out["resident"][0], "streamed_s": out["streamed"][0], "host_to_device_only_s": t_copy}
    print(f"raw fp16 keys ({n_s} x 1024, {n_s * 2048 / 1e9:.1f} GB): resident {out['resident'][0]:.2f} s, streamed "
          f"{out['streamed'][0]:.2f} s, host read + H2D alone {t_copy:.2f} s (identical results)", flush=True)
    if a.out:
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
