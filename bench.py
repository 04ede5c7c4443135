#!/usr/bin/env python
"""bench.py -- eval tokens/s of the GNN-LM hot path (graph assembly + PQ gather/decode -> HGT ->
adaptive-softmax log-probs -> kNN-LM mix -> NLL) on synthetic data of the Wiki103 shape
(BASELINE.json configs[2]: d=1024, H=8, V=267,744, cutoffs 20000/60000, L=3072, k=32, c=1, M=128, 3 HGT
layers, k_nn=1024), one process per GPU.

  python bench.py [--gpus N --steps K --warmup W] [--config c3] [--math f16f8|f16x3|tf32x3|fp32|tf32|bf16]
  python bench.py --impl reference ...      # the CPU restatement of the reference path (oracle/) on host cores

A "step" is one pass of the hot path over one batch (B blocks x L tokens).  `value` is measured with all
inputs resident in HBM; `e2e` goes through the same public call with pinned HOST inputs (H2D inside the
timed region, 16 B result read back per step); `e2e_evaluate` is eval_lm.evaluate() -- the call a user makes -- over a
reference-layout data directory in tmpfs (mmap slicing, collater, staging, scoring).  Prints ONE JSON line on rank 0.

  python bench.py --gpus N --scaling strong   # a fixed corpus sharded over the ranks through evaluate() (extra evidence)
  python bench.py ... --dump-outputs DIR      # also write the last timed step's outputs as DIR/*.npy (compare two builds)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=8)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", default="c3")
    p.add_argument("--math", default="auto")
    p.add_argument("--n-datastore", type=int, default=0, help="override datastore rows (default: the config's)")
    p.add_argument("--deprecated", action="store_true", help="--deprecated (de-duplicating) graph builder, general CSR attention")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-full-block", action="store_true", help="--impl reference: skip the single pass over a full block")
    p.add_argument("--cpu-tokens", type=int, default=768, help="tokens in the CPU-baseline sample block")
    p.add_argument("--also-modes", default="f16x3,tf32x3,tf32,bf16",
                   help="extra arithmetic modes timed briefly (resident inputs) and reported under `other_modes`")
    p.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false",
                   help="launch the step's kernels one by one instead of replaying the captured whole-step CUDA graph")
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                   help="weak: one block per step per rank (the headline line).  strong: ONE fixed corpus of --strong-blocks blocks "
                        "(+ a ragged tail) through eval_lm.evaluate(rank, world_size): contiguous block shards, replicated datastore, "
                        "one NCCL all-reduce of {sum log p, n_tokens}")
    p.add_argument("--strong-blocks", type=int, default=128)
    p.add_argument("--eval-blocks", type=int, default=32, help="blocks of the e2e_evaluate leg (0: skip it)")
    p.add_argument("--locality", default="0.5,1048576",
                   help="p_continue,n_hot of the realistic-duplication leg (synth.local_neighbours); empty: skip the leg")
    p.add_argument("--no-train-leg", dest="train_leg", action="store_false",
                   help="skip the fine-tuning-step leg (`train_step` in the line; information only, after the timed regions)")
    p.add_argument("--ncu-range", action="store_true",
                   help="after warm-up run ONE resident step inside cudaProfilerStart/Stop and exit "
                        "(use with `ncu --profile-from-start off`); prints no bench line")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps write what the last one returned as DIR/<name>.npy (rank 0): logprob [B, L] and "
                        "gcn_feat [B, L, d] in float32, nll_acc (sum log p, tokens over every step so far) in float64.  The "
                        "inputs are seeded, so two builds run with the same arguments can be compared output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


DUMP_LIMIT = (64 << 20) - (64 << 10)          # 64 MB in all, with room for the .npy headers


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor, written smallest first as <out_dir>/<name>.npy.  An array that would take the total past
    DUMP_LIMIT is written as a fixed, seeded sample (in order) of its rows over the last dimension, [n_sampled, last_dim]."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_LIMIT
    for name, t in sorted(arrays.items(), key=lambda kv: kv[1].numel()):
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > left:
            a = a.reshape(-1, a.shape[-1])
            keep = np.random.RandomState(0).choice(a.shape[0], left // (a.itemsize * a.shape[1]), replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        left -= a.nbytes


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU legs
def cpu_sample(cfg_name, n_tokens, n_d=1 << 22):
    """Bounded sample of the same workload for the CPU oracle: one block of n_tokens tokens with the
    config's d / V / k / c / M / layers / k_nn and a 2^22-row datastore (the CPU cost per token does not
    depend on the datastore size)."""
    from gnnlm_b200 import synth
    cfg = dict(synth.CONFIGS[cfg_name])
    n_tokens = min(n_tokens, cfg["B"] * cfg["L"])                # never more than the workload's own block
    cfg.update(B=1, L=n_tokens, n_d=min(cfg["n_d"], n_d))
    model = synth.make_model(cfg)
    data = synth.make_data(cfg, seed=0, device="cpu")
    return cfg, model, data


def time_oracle(prob, steps, warmup):
    from tests.synth import run_oracle
    torch.set_num_threads(os.cpu_count())
    try:        # torchrun exports OMP_NUM_THREADS=1: give numpy's BLAS (the oracle's PQ rotation) every host core back
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass
    for _ in range(warmup):
        run_oracle(prob)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = run_oracle(prob)
        ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)), out


def bench_config(cfg_name, world, scaling="weak"):
    """The `config` object of BOTH arms (the reference arm runs on our arm's config; what it actually times per step is stated
    in its cpu_baseline.sample)."""
    return {"workload": workload_name(cfg_name),
            "parallelism": f"dp{world} (contiguous block shards, replicated datastore, one 16 B all-reduce)",
            "l2_policy": "inputs larger than L2 (datastore + activations are GBs); 4 distinct batches rotated",
            "scaling_mode": scaling}


def sample_note(cfg, args):
    full = __import__("gnnlm_b200").synth.CONFIGS[args.config]["L"]
    return (f"CPU oracle port (torch fp32, {torch.get_num_threads()} threads): each step scores ONE block of {cfg['L']} tokens -- "
            f"a bounded sample, {cfg['L']}/{full} of the workload's {full}-token block -- at the {args.config} shape (d={cfg['d']}, "
            f"V={cfg['V']}, k={cfg['k']}, c={cfg['c']}, M={cfg['M']}, {cfg['NL']} HGT layers, k_nn={cfg['k_nn']}), datastore "
            f"2^22 rows; the CPU cost per token GROWS with the block length (tgt-intra-tgt attention is quadratic), so the "
            f"sample understates the CPU time of the full block")


def run_reference(args):
    """--impl reference: the reference's own CPU implementation cannot run here (needs dgl + faiss; DESIGN.md), so this times
    the oracle port of it on all host cores.  Same `config` as our arm; each step is a bounded sample of that workload (a
    768-token block instead of the 3072-token one, stated in cpu_baseline.sample and `sample_tokens`), and one pass over a
    FULL block is timed once beside it (`full_block`) so that the two can be compared."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gnnlm_b200 import synth
    cfg, model, data = cpu_sample(args.config, args.cpu_tokens)
    sec, out = time_oracle((cfg, model, data), max(1, args.steps), max(0, min(args.warmup, 1)))
    tps = cfg["L"] / sec
    full = None
    L_full = synth.CONFIGS[args.config]["L"] * synth.CONFIGS[args.config]["B"]
    if not args.no_full_block and L_full != cfg["L"]:
        fcfg, fmodel, fdata = cpu_sample(args.config, L_full)
        fsec, _ = time_oracle((fcfg, fmodel, fdata), 1, 0)
        full = {"tokens": L_full, "seconds": fsec, "tokens_per_s": L_full / fsec, "passes": 1,
                "note": "one un-warmed pass over a full block of the workload (dense-causal oracle form)"}
    line = {"impl": "reference", "metric": "eval tokens/s (HGT+kNN-LM fwd)", "value": tps, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args.config, args.gpus), "sample_tokens": cfg["L"], "full_block": full,
            "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": sample_note(cfg, args)},
            "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def committed_ncu(kernel_key):
    """Per-launch counters of a kernel from the committed `ncu --set full` captures of this workload (profiles/*ncu_traffic.json,
    written by profiles/ncu_metrics.py from captures taken under gpurun -- NOT measured by this run)."""
    for name in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            db = json.load(open(path))
            if kernel_key in db:
                return dict(db[kernel_key], file=f"profiles/{name}")
    return None


def workload_name(cfg_name):
    from gnnlm_b200 import synth
    c = synth.CONFIGS[cfg_name]
    names = {"c1": "tiny", "c2": "enwik8-shape", "c3": "wiki103-shape", "c4": "one-billion-word-shape",
             "c3e": "wiki103-shape at the reference eval script's setting"}
    return f"{cfg_name}: {names.get(cfg_name, cfg_name)} GNN+kNN eval" + \
        f" d={c['d']} H={c['H']} V={c['V']} B={c['B']}xL={c['L']} k={c['k']} c={c['c']} M={c['M']} layers={c['NL']} k_nn={c['k_nn']}"


# ----------------------------------------------------------------------------------------------- evaluate() legs
def build_eval(cfg, model, dev, math, root, n_blocks, tail, seed=0, write=True):
    """A reference-layout data directory under `root` (tmpfs) + everything eval_lm.evaluate() needs, through the same loaders
    eval_lm.main uses (formats.load_graph_lm_dataset, DeviceDatastore.from_dir, KNNModel over the neighbour memmaps)."""
    from argparse import Namespace
    from gnnlm_b200 import synth
    from gnnlm_b200.dataset import DeviceDatastore, neighbor_path
    from gnnlm_b200.formats import MmapDataset, load_graph_lm_dataset
    from gnnlm_b200.knn_model import KNNModel
    from gnnlm_b200.sequence_scorer import SequenceScorer
    if write:
        info = synth.write_data_dir(root, cfg, n_blocks, tail_tokens=tail, seed=seed, device=dev)
    else:
        info = {"n_tokens": n_blocks * cfg["L"] + tail, "n_blocks": n_blocks + (1 if tail else 0),
                "dists_file": os.path.join(root, "valid_dstore", f"dists.{cfg['k_nn']}")}
    n = info["n_tokens"]
    knn_ids = MmapDataset(neighbor_path(root, "valid", cfg["k_nn"]), (n, cfg["k_nn"]), np.int64).array()
    knn_dists = MmapDataset(info["dists_file"], (n, cfg["k_nn"]), np.float32).array()
    ds, dictionary = load_graph_lm_dataset(root, "valid", tokens_per_sample=cfg["L"], gcn_k=cfg["k"], neighbor_context=cfg["c"],
                                           knn_dists=knn_dists, knn_ids=knn_ids)
    dstore = DeviceDatastore.from_dir(root, len(dictionary), dev)
    knn = KNNModel(dstore.vals, vocab_size=cfg["V"], metric_type="do_not_recomp_ip", k=cfg["k_nn"])
    scorer = SequenceScorer(dictionary, args=Namespace(lmbda=cfg["lmbda"], knn_keytype=None))
    return ds, dstore, knn, scorer, info


def run_evaluate(model, ds, dstore, knn, scorer, cfg, dev, rank=0, world=1, cache=None):
    """`cache`: kept by the caller between the warm-up and the timed call (captured graphs + activation pool are reused)."""
    from gnnlm_b200.eval_lm import evaluate
    return evaluate(model, ds, dstore, scorer, knn_dstore=knn, temperature=cfg["temp"], max_sentences=cfg["B"], device=dev,
                    rank=rank, world_size=world, cuda_graph=True, graph_cache=cache)


def tmp_root(tag):
    import tempfile
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    return tempfile.mkdtemp(prefix=f"gnnlm_bench_{tag}_", dir=base)


def run_strong(args, world, rank, dev, dist, math):
    """Strong scaling through the product API: ONE corpus of --strong-blocks blocks + a ragged tail (not divisible by 2 / 4 / 8),
    every rank holds the whole data directory and the replicated datastore, evaluates its contiguous block range
    (eval_lm.shard_range) and joins the single NCCL all-reduce.  Timed: evaluate() on every rank between two barriers, max
    over ranks.  The combined score_sum must not depend on N."""
    import shutil
    from gnnlm_b200 import synth
    cfg = dict(synth.CONFIGS[args.config])
    cfg["n_d"] = args.n_datastore or min(cfg["n_d"], 1 << 24)
    model = synth.make_model(cfg).to(dev).set_math(math)
    # ONE data directory for the node (rank 0 writes it, every rank maps it), as a shared dataset would be
    name = [tmp_root("strong") if rank == 0 else None]
    if dist is not None:
        dist.broadcast_object_list(name, src=0)
    root = name[0]
    try:
        if rank == 0:
            build_eval(cfg, model, dev, math, root, args.strong_blocks, tail=1000, seed=0)
        if dist is not None:
            dist.barrier()
        ds, dstore, knn, scorer, info = build_eval(cfg, model, dev, math, root, args.strong_blocks, tail=1000, seed=0, write=False)
        cache = {}
        run_evaluate(model, ds, dstore, knn, scorer, cfg, dev, rank, world, cache)     # warm-up pass (graph capture, weight preparation)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        res = run_evaluate(model, ds, dstore, knn, scorer, cfg, dev, rank, world, cache)
        torch.cuda.synchronize(dev)
        sec = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(sec, op=dist.ReduceOp.MAX)
            dist.barrier()
        sec = float(sec.item())
    finally:
        if dist is not None:
            dist.barrier()
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)
    line = {"metric": "eval tokens/s (HGT+kNN-LM fwd)", "value": res["count"] / sec, "unit": "tokens/s", "n_gpus": world,
            "steps": 1, "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": math, "data": "synthetic", "impl": "ours",
            "config": dict(bench_config(args.config, world, "strong"), n_datastore=cfg["n_d"], math=math,
                           corpus=f"{info['n_blocks']} blocks = {info['n_tokens']} tokens ({args.strong_blocks} x {cfg['L']} + a "
                                  f"1000-token tail), reference-layout data directory in tmpfs, eval_lm.evaluate(cuda_graph=True)"),
            "score_sum": repr(res["score_sum"]), "count": res["count"], "ppl": res["ppl"],
            "blocks_this_rank": list(__import__("gnnlm_b200").eval_lm.shard_range(len(ds), rank, world)),
            "seconds_max_over_ranks": sec}
    if rank == 0:
        print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- GPU arm
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from gnnlm_b200 import _lib as L
    from gnnlm_b200 import synth
    lib = L.load()
    math = args.math
    if math == "auto":
        math = "f16f8" if lib.gnnlm_has_tcgen05() else "fp32"      # fp32-parity mode with the fewest tensor cycles
    if args.scaling == "strong":
        run_strong(args, world, rank, dev, dist, math)
        if dist is not None:
            dist.destroy_process_group()
        return
    cfg = dict(synth.CONFIGS[args.config])
    if args.n_datastore:
        cfg["n_d"] = args.n_datastore
    if args.deprecated:
        cfg["deprecated"] = True
    T = cfg["B"] * cfg["L"]

    model = synth.make_model(cfg)
    tables = synth.make_tables(cfg, seed=rank, device=dev)          # replicated datastore, per-rank stream
    NB = 4                                                          # distinct resident batches, rotated
    dev_batches = [synth.make_batch(cfg, tables, seed=1000 * rank + i, device=dev) for i in range(NB)]
    host_batches = [{k: v.cpu().pin_memory() for k, v in b.items() if k != "positions"} for b in dev_batches]
    runner = synth.Runner(cfg, model, tables, dev, math)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    eager = lambda i: runner.step_resident(dev_batches[i % NB])
    last = {}

    def resident(i):
        last["out"] = runner.step_resident(dev_batches[i % NB], cuda_graph=args.cuda_graph)

    host = lambda i: runner.step_host(host_batches[i % NB], cuda_graph=args.cuda_graph)

    eager(0)                                                         # one-time weight preparation (folds, fp16 splits) happens here
    l0 = L.launches
    eager(1)
    launches_per_step = L.launches - l0                              # kernels of ONE step; graph replays launch the same kernels
    for i in range(max(3, args.warmup)):
        resident(i)
    if args.ncu_range:
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        eager(0)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return
    clocks = ClockSampler(local)
    clocks.start()
    ms = timed(resident, args.steps)
    launches = launches_per_step * args.steps
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:         # before the host leg: it replays the same CUDA graph into the same buffers
        lp, _, _, (feat, _) = last["out"]
        dump_outputs(args.dump_outputs, {"logprob": lp, "gcn_feat": feat, "nll_acc": runner.acc})
    for i in range(2):
        host(i)
    # e2e: K steps through the runner's host-input loop -- per step: H2D of that step's pinned inputs (double-buffered on a
    # copy stream), the scoring step, and a D2H read of the accumulated result
    ms_e2e = timed(lambda i: runner.run_host(host_batches, args.steps, cuda_graph=args.cuda_graph) if i == 0 else None,
                   args.steps)

    # the path's only collective: {sum log p, n_tokens}
    acc = runner.acc.clone()
    if dist is not None:
        dist.all_reduce(acc)
    score_sum, count = acc.tolist()

    # ---- per-kernel pass (CUDA events around every C-ABI launch, same workload, separately timed region)
    L.TIMING = []
    for i in range(args.steps):
        eager(i)
    torch.cuda.synchronize(dev)
    g = synth.build_token_graph(dev_batches[0]["nbr"], tables["n_d"], cfg["c"], cfg["c"], reach=cfg["NL"] - 1)
    n_ntgt, n_valid = g.counts()
    live = {g.node_cap: n_ntgt, T * cfg["k"]: n_valid}              # capacity-sized launches -> live rows of batch 0
    per, gemm = {}, {}
    for name, tag, a, b, work in L.TIMING:
        base = name.replace("gnnlm_", "").replace("_q8", "").replace("_hiq8", "").replace("_presplit", "").replace("cluster_attn_hq", "cluster_attn")
        key = base + (f":{tag}" if tag else "")
        dt = a.elapsed_time(b)
        d_ = per.setdefault(key, [0.0, 0])
        d_[0] += dt
        d_[1] += 1
        if work is not None and base in ("linear", "linear_f16f8", "linear_lse"):
            M_, N_, K_ = work
            w_ = gemm.setdefault(base, [0.0, 0.0, 0])
            w_[0] += dt
            w_[1] += 2.0 * live.get(M_, M_) * N_ * K_
            w_[2] += 1
    L.TIMING = None
    step_ms_instr = sum(v[0] for v in per.values()) / args.steps
    kernels = {k: {"ms_per_launch": v[0] / v[1], "launches_per_step": v[1] / args.steps,
                   "share": v[0] / args.steps / step_ms_instr} for k, v in sorted(per.items(), key=lambda kv: -kv[1][0])}

    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    tf_peak, tf_src = (peaks["bf16_tflops_sustained"], "measured (cuBLAS bf16, sustained)") if "bf16_tflops_sustained" in peaks \
        else (1400.0, "fallback")

    # ---- roofline of the DOMINANT kernel: the projection GEMM family of the mode (share of the step in `share_of_step`)
    passes = {"tf32x3": 3, "f16x3": 3, "f16f8": 2, "fp32": 1, "tf32": 1, "bf16": 1}[math]
    fam = max(gemm, key=lambda k_: gemm[k_][0]) if gemm else None
    roof = None
    if fam is not None:
        ms_f, flops_f, n_f = gemm[fam]
        useful = flops_f / (ms_f * 1e-3) / 1e12
        kname = {"linear_f16f8": "gemm_f16f8_kernel", "linear": "gemm_f16s_kernel<0> (3xFP16)" if math in ("f16x3", "f16f8")
                 else "gnnlm_linear"}.get(fam, fam)
        ncu = committed_ncu(kname.split(" ")[0])
        roof = {"kernel": kname, "bound": "tensor", "achieved": useful, "unit": "TFLOP/s", "peak": tf_peak, "peak_source": tf_src,
                "frac": useful / tf_peak, "achieved_useful": useful, "passes": passes if fam != "linear" or math != "f16f8" else 3,
                "launches_per_step": n_f / args.steps, "ms_per_step": ms_f / args.steps, "share_of_step": ms_f / args.steps / step_ms_instr,
                "algorithmic_flops_per_step": flops_f / args.steps,
                "note": "achieved = useful flops (2 M N K over the live rows) / device time of every launch of the kernel in the "
                        "step; achieved_executed counts the tensor-pass equivalents the parity arithmetic issues (fp16 main "
                        "product = 1, the two FP8 correction products = 0.5 each; 3xFP16 = 3)",
                "traffic": None if ncu is None else ncu.get("dram_bytes"),
                "traffic_source": None if ncu is None else f"committed ncu capture ({ncu['file']}), largest launch; not measured by this run"}
        roof["achieved_executed"] = useful * roof["passes"]
        roof["frac_executed"] = roof["achieved_executed"] / tf_peak

    # ---- edge-aggregation kernels (the metric's second half): algorithmic bytes (SURVEY.md 8d) / device time, vs the HBM peak
    d, s = cfg["d"], (2 if math == "bf16" else 4)          # bytes per activation element (bf16 mode: Q | K' | V' and outputs in bf16)
    out_b = {"f16f8": 3}.get(math, s)                       # f16f8: cluster attention writes fp16 hi + 2 companion bytes per element
    hq_env = os.environ.get("GNNLM_HQ", "1")
    in_c = 3 if (math == "f16f8" and hq_env != "0") else s        # f16f8: Q | K' | V' of the centre-only layer rounded to three bytes (GNNLM_F24)
    in_b = 3 if (math == "f16f8" and hq_env == "all") else s      # (the all-nodes layers keep fp32 rows unless GNNLM_HQ=all)

    def _edge_bytes(key):
        if key.endswith("nn_full"):
            return n_ntgt * 2 * d * in_b + n_ntgt * d * in_b + n_ntgt * d * out_b + (3 * n_ntgt - 2 * n_valid) * 4 + (n_ntgt + 1) * 4
        if key.endswith("nn_centre"):
            return min(n_ntgt, 3 * n_valid) * 2 * d * in_c + n_valid * d * in_c + n_valid * d * out_b + 3 * n_valid * 4 + 2 * n_valid * 4
        return n_valid * 2 * d * s + T * d * s + T * d * 4 + (T + 1) * 4
    edge_all = {key: {"GB/s": _edge_bytes(key) / (kv["ms_per_launch"] * 1e-3) / 1e9,
                      "frac": _edge_bytes(key) / (kv["ms_per_launch"] * 1e-3) / 1e9 / hbm_peak,
                      "algorithmic_bytes": _edge_bytes(key), "ms_per_launch": kv["ms_per_launch"], "share_of_step": kv["share"]}
                for key, kv in kernels.items() if key.startswith(("hgt_cluster_attn", "hgt_edge_attn"))}
    if "hgt_inter_fused:inter_fused" in kernels:
        # token-side form of the inter edges (inter_attn.cu): centre rows once + H transformed queries in + H weighted row sums out
        Hh = cfg["H"]
        ib = n_valid * d * s + T * Hh * d * 4 + T * Hh * d * 4 + T * d * 4 + (T + 1) * 4
        kv = kernels["hgt_inter_fused:inter_fused"]
        edge_all["hgt_inter_fused:inter"] = {"GB/s": ib / (kv["ms_per_launch"] * 1e-3) / 1e9,
                                             "frac": ib / (kv["ms_per_launch"] * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": ib,
                                             "ms_per_launch": kv["ms_per_launch"], "share_of_step": kv["share"],
                                             "note": "token-side form: replaces the K'|V' projection of every centre (2 d^2 MACs each)"}
    pq_keys = [k_ for k_ in kernels if k_.startswith("pq_gather_decode")]
    if pq_keys:
        pq_ms = sum(kernels[k_]["ms_per_launch"] * kernels[k_]["launches_per_step"] for k_ in pq_keys)
        pq_bytes = n_ntgt * (cfg["M"] + 8 + d * s) + (n_valid * (cfg["M"] + 8 + d * s) if math == "f16f8" else 0)
        edge_all["pq_gather_decode"] = {"GB/s": pq_bytes / (pq_ms * 1e-3) / 1e9, "frac": pq_bytes / (pq_ms * 1e-3) / 1e9 / hbm_peak,
                                        "algorithmic_bytes": pq_bytes, "ms_per_step": pq_ms}
    roof_edge = None
    for key in ("hgt_cluster_attn:nn_full", "hgt_edge_attn:nn_full", "hgt_cluster_attn:nn_centre", "hgt_edge_attn:nn_centre"):
        if key in edge_all:
            e = edge_all[key]
            kn = "cluster_attn_kernel<float, __half, 4, 3, 32>" if key == "hgt_cluster_attn:nn_full" else key
            ncu = committed_ncu(kn) if (cfg["L"], cfg["k"], cfg["c"]) == (3072, 32, 1) else None
            roof_edge = {"kernel": key, "bound": "hbm", "achieved": e["GB/s"], "peak": hbm_peak, "peak_source": hbm_src, "unit": "GB/s",
                         "frac": e["frac"], "algorithmic_bytes": e["algorithmic_bytes"], "nominal_peak": 7700.0,
                         "frac_of_nominal": e["GB/s"] / 7700.0, "ms_per_launch": e["ms_per_launch"], "share_of_step": e["share_of_step"],
                         "peak_note": "peak = driver-measured copy bandwidth (1:1 read:write); this kernel reads 3 bytes per "
                                      "byte written and can exceed it -- nominal HBM3e is 7.7 TB/s",
                         "traffic": None if ncu is None else ncu.get("dram_bytes"),
                         "traffic_source": None if ncu is None else f"committed ncu capture ({ncu['file']}); not measured by this run"}
            break

    tokens_all = world * args.steps * T
    line = {
        "metric": "eval tokens/s (HGT+kNN-LM fwd)", "value": tokens_all / (ms * 1e-3), "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "tf32x3": "f32 (3xTF32 tensor-core split)",
                                                           "f16x3": "f32 (3xFP16 tensor-core split, fp32 accumulate)",
                                                           "f16f8": "f32 (fp16 main product + FP8 e4m3 correction products, fp32 accumulate)",
                                                           "tf32": "tf32", "bf16": "bf16"}[math],
        "data": "synthetic", "impl": "ours",
        "config": bench_config(args.config, world),
        "run": {"math": math, "n_datastore": tables["n_d"], "cuda_graph": bool(args.cuda_graph),
                "graph_builder": "deprecated (dedup)" if args.deprecated else "new", "n_ntgt": n_ntgt, "n_valid_neighbours": n_valid},
        "e2e": {"value": tokens_all / (ms_e2e * 1e-3), "unit": "tokens/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host_batches[0].values())),
                "d2h_bytes_per_step": 16,
                "api": "synth.Runner.run_host: pinned host inputs of one block per step, double-buffered H2D, scoring step, 16 B read-back"},
        "gpu_launches": launches, "clocks": clk, "roofline": roof, "roofline_edge": roof_edge, "hbm_kernels": edge_all,
        "kernels": kernels, "score_sum": score_sum, "count": count,
    }
    # ---- the public call end to end: eval_lm.evaluate() over a reference-layout data directory (rank 0, N = 1 only)
    if world == 1 and args.eval_blocks > 0:
        import shutil
        ecfg = dict(cfg, n_d=min(cfg["n_d"], 1 << 24))
        root = tmp_root("eval")
        try:
            emodel = runner.model                                   # same weights, already prepared
            ds, dstore_e, knn_e, scorer_e, info = build_eval(ecfg, emodel, dev, math, root, args.eval_blocks, tail=0, seed=3)
            ecache = {}
            run_evaluate(emodel, ds, dstore_e, knn_e, scorer_e, ecfg, dev, cache=ecache)    # warm-up pass: page cache, graph capture
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            res = run_evaluate(emodel, ds, dstore_e, knn_e, scorer_e, ecfg, dev, cache=ecache)
            torch.cuda.synchronize(dev)
            sec = time.perf_counter() - t0
            line["e2e_evaluate"] = {
                "value": res["count"] / sec, "unit": "tokens/s", "seconds": sec, "blocks": info["n_blocks"], "tokens": int(res["count"]),
                "ppl": res["ppl"], "loss_base2": res["loss_base2"], "n_datastore": ecfg["n_d"],
                "api": "eval_lm.evaluate(cuda_graph=True) over formats.load_graph_lm_dataset(<tmpfs data dir>): mmap slicing "
                       "(dataset.__getitem__), collater, pinned staging + H2D, graph assembly .. NLL, one read-back at the end; "
                       "wall clock around the call"}
            del ds, dstore_e, knn_e
        finally:
            shutil.rmtree(root, ignore_errors=True)
    # ---- realistic duplication: neighbour ids with the locality of real kNN graphs (repeated centres, overlapping clusters)
    # through (a) the default path, (b) the ntgt side once per distinct centre row (share_centres), (c) the --deprecated builder
    if world == 1 and args.locality and not args.deprecated:
        import copy
        p_c, n_hot = args.locality.split(",")
        loc = (float(p_c), int(n_hot))
        lb = [synth.make_batch(cfg, tables, seed=5000 + i, device=dev, locality=loc) for i in range(2)]
        flat = lb[0]["nbr"].reshape(-1)
        ok = flat >= 0
        n_pairs, n_cent = int(ok.sum()), int(torch.unique(flat[ok]).numel())
        leg = {"p_continue": loc[0], "n_hot_rows": loc[1], "valid_pairs": n_pairs, "distinct_centres": n_cent,
               "duplicate_rate": 1.0 - n_cent / max(n_pairs, 1),
               "note": "synth.local_neighbours: neighbour j of token t continues neighbour j of token t-1 (row + 1) with probability "
                       "p_continue, else a fresh retrieval from n_hot popular rows with 1/rank popularity; same model / datastore "
                       "as the headline; results of (a) and (b) are identical (tested against the oracle)"}
        for name, kw in (("new_builder", {}), ("new_builder_share_centres", {"share": True}), ("deprecated_builder", {"dep": True})):
            c2 = dict(cfg, deprecated=True) if kw.get("dep") else cfg
            m2 = copy.deepcopy(model)
            m2.decoder.share_centres = bool(kw.get("share"))
            r3 = synth.Runner(c2, m2, tables, dev, math)
            f3 = lambda i: r3.step_resident(lb[i % 2], cuda_graph=args.cuda_graph)
            for i in range(3):
                f3(i)
            ms3 = timed(f3, args.steps)
            leg[name] = {"value": args.steps * T / (ms3 * 1e-3), "unit": "tokens/s", "ms_per_step": ms3 / args.steps,
                         "score_sum": float(r3.acc[0].item())}
            del r3, m2
        line["locality"] = leg
    # secondary arithmetic modes (same workload, resident inputs, short timed loop) -- information only; the
    # headline stays the fp32-parity mode
    other = {}
    for m in [x for x in args.also_modes.split(",") if x and x != math]:
        if m != "fp32" and not lib.gnnlm_has_tcgen05():
            continue
        r2 = synth.Runner(cfg, model, tables, dev, m)
        f2 = lambda i: r2.step_resident(dev_batches[i % NB])
        for i in range(3):
            f2(i)
        ms2 = timed(f2, args.steps)
        other[m] = {"value": world * args.steps * T / (ms2 * 1e-3), "unit": "tokens/s", "ms_per_step": ms2 / args.steps,
                    "cuda_graph": False,        # launched kernel by kernel; `--math <mode>` times it like the headline
                    "parity": {"tf32": "single-pass tf32: log-probs ~1e-3 of fp32 (not a parity mode)",
                               "bf16": "log-probs within 1e-2 of fp32 (tested)",
                               "tf32x3": "log-probs within 1e-4 of fp32 (tested); no fp16 range limit on operands",
                               "f16x3": "log-probs within 1e-4 of fp32 (tested)", "fp32": "fp32 FMA",
                               "f16f8": "log-probs within 1e-4 of fp32 (tested)"}.get(m, "")}
        del r2
    line["other_modes"] = other
    # the fine-tuning step of the same shape (SURVEY.md 8f rank 4) -- information only, outside every timed region above: forward +
    # backward of train.train_step_loss on one block with the dropout rates of transformer_lm_wiki103, 3xFP16 projections
    if world == 1 and args.train_leg and lib.gnnlm_has_tcgen05() and not args.deprecated:
        try:
            import copy
            from gnnlm_b200 import train
            tm = copy.deepcopy(model).train()
            for n_, p_ in tm.named_parameters():
                p_.requires_grad_("hgt" in n_)
            for layer in tm.decoder.hgt_decoder.gcs:
                layer.drop.p, layer.attn_drop.p = 0.3, 0.1
            if tm.decoder.adaptive_softmax is not None:
                tm.decoder.adaptive_softmax.dropout = 0.2
            tr = synth.Runner(cfg, tm, tables, dev, "fp32", prune_unreachable=False)
            tm.train()
            b0 = dev_batches[0]
            ts = tr.sample_from(b0["nbr"], b0["feats"], b0["target"], b0["knn_dists"], b0["knn_ids"])
            best = None
            for it in range(3):
                tm.zero_grad(set_to_none=True)
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record()
                loss = train.train_step_loss(tm, ts, "f16x3", seed=it)
                e1.record()
                loss.backward()
                e2.record()
                torch.cuda.synchronize()
                fw, bw = e0.elapsed_time(e1), e1.elapsed_time(e2)
                if it and (best is None or fw + bw < best[0] + best[1]):
                    best = (fw, bw)
            line["train_step"] = {"value": T / ((best[0] + best[1]) * 1e-3), "unit": "tokens/s", "forward_ms": best[0], "backward_ms": best[1],
                                  "math": "f16x3", "dropout": [0.3, 0.1, 0.2],
                                  "api": "train.train_step_loss(model, sample).backward() on one block, --freeze parameter set; best of 2 after 1 warm-up"}
            del tm, tr, ts, loss
            torch.cuda.empty_cache()
        except Exception as e:                                    # never let the extra leg take the bench line down
            line["train_step"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if world == 1 and not args.no_cpu_baseline:
        ccfg, cmodel, cdata = cpu_sample(args.config, args.cpu_tokens)
        sec, _ = time_oracle((ccfg, cmodel, cdata), 2, 1)       # ~10 s of CPU work: one warm-up + two timed passes
        line["cpu_baseline"] = {
            "value": ccfg["L"] / sec, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port",
            "sample": sample_note(ccfg, args) + f"; mean of 2 timed passes after 1 warm-up, {sec:.1f} s per pass"}
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
