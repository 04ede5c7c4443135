"""Exact kNN search on the GPU (gnnlm_knn_filter_f16x3 / gnnlm_topk_merge / gnnlm_knn_key_bias*, knn_search.KNNSearcher,
find_knn): the merge against numpy's lexsort, the filter GEMM against fp64 scores, the searcher against an fp64 brute force,
bit-identical output across schedules, and the neighbour files feeding eval_lm."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ranked(s, ids):
    """(score descending, id ascending) order of one row."""
    return np.lexsort((ids, -s.astype(np.float64)))


@pytest.mark.parametrize("k", [1, 32, 1000, 1024, 2048])
def test_topk_merge_matches_lexsort(dev, k):
    from gnnlm_b200 import ops
    rng = np.random.RandomState(k)
    cap = 4096 if k >= 1000 else 256
    n_q = 24
    held_n = rng.randint(0, k + 1, n_q)
    held_n[:3] = [0, k, max(k - 1, 0)]
    cnt = rng.randint(0, cap + 1, n_q)
    cnt[:6] = [0, cap, cap + 7, 1, cap, 0]                    # row 2 overflowed: left untouched
    top_s = np.full((n_q, k), -np.inf, np.float32)
    top_id = np.full((n_q, k), -1, np.int32)
    cand_s = rng.randn(n_q, cap).astype(np.float32)          # garbage past the count
    cand_id = rng.randint(0, 1 << 30, (n_q, cap)).astype(np.int32)
    for i in range(n_q):
        ids = rng.choice(1 << 24, held_n[i] + min(cnt[i], cap), replace=False).astype(np.int32)
        s = (rng.randint(-12, 12, ids.size) / 4.0).astype(np.float32)        # many ties
        h = held_n[i]
        o = _ranked(s[:h], ids[:h])
        top_s[i, :h], top_id[i, :h] = s[:h][o], ids[:h][o]
        c = min(cnt[i], cap)
        cand_s[i, :c], cand_id[i, :c] = s[h:], ids[h:]
    thr = rng.randn(n_q).astype(np.float32)
    t = {n: torch.from_numpy(a).to(dev) for n, a in dict(top_s=top_s, top_id=top_id, cand_s=cand_s, cand_id=cand_id,
                                                          cnt=cnt.astype(np.int32), thr=thr).items()}
    ops.topk_merge(t["top_s"], t["top_id"], t["cand_s"], t["cand_id"], t["cnt"], t["thr"])
    got = {n: v.cpu().numpy() for n, v in t.items()}
    for i in range(n_q):
        if cnt[i] == 0 or cnt[i] > cap:
            assert (got["top_s"][i] == top_s[i]).all() and (got["top_id"][i] == top_id[i]).all()
            assert got["cnt"][i] == cnt[i] and got["thr"][i] == thr[i]
            continue
        h, c = held_n[i], cnt[i]
        s = np.concatenate([top_s[i, :h], cand_s[i, :c]])
        ids = np.concatenate([top_id[i, :h], cand_id[i, :c]])
        o = _ranked(s, ids)[:k]
        assert (got["top_id"][i, :o.size] == ids[o]).all() and (got["top_s"][i, :o.size] == s[o]).all(), i
        assert (got["top_id"][i, o.size:] == -1).all() and (got["top_s"][i, o.size:] == -np.inf).all()
        assert got["thr"][i] == (s[o[k - 1]] if o.size == k else -np.inf) and got["cnt"][i] == 0


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_filter_gemm_candidates(dev, metric):
    """Candidates = {x : s(q, x) > thr[q]} against fp64 scores (up to entries within 1e-5 * scale of the threshold); counts and
    overflow with a small cap; M, N, d not tile multiples; a nonzero id base."""
    from gnnlm_b200 import ops
    g = torch.Generator().manual_seed(3)
    M, N, d, base = 1000, 300, 200, 123457
    x = torch.randn(M, d, generator=g)
    q = torch.randn(N, d, generator=g)
    s64 = q.double() @ x.double().T
    if metric == "l2":
        s64 = s64 - 0.5 * (x.double() ** 2).sum(1)[None]
    scale = (q.double().norm(dim=1) * x.double().norm(dim=1).max() + 0.5 * (x.double() ** 2).sum(1).max()).numpy()
    thr = torch.quantile(s64, 0.9, dim=1).float()
    thr[:5] = -np.inf                                          # every key a candidate
    keys = ops.to_split(x.to(dev))
    bias = ops.knn_key_bias(x.to(dev)) if metric == "l2" else None
    q_hi, q_lo, _ = ops.split_f16(q.to(dev), scale=1.0)
    for cap in (1024, 40):
        cs = torch.empty((N, cap), device=dev)
        ci = torch.empty((N, cap), device=dev, dtype=torch.int32)
        cc = torch.zeros((N,), device=dev, dtype=torch.int32)
        ops.knn_filter(keys, base, q_hi, q_lo, bias, thr.to(dev), cs, ci, cc)
        cs, ci, cc = cs.cpu().numpy(), ci.cpu().numpy(), cc.cpu().numpy()
        s, t = s64.numpy(), thr.double().numpy()
        for i in range(N):
            want = set(np.nonzero(s[i] > t[i])[0] + base)
            near = set(np.nonzero(np.abs(s[i] - t[i]) <= 1e-5 * scale[i])[0] + base)
            lo, hi = len(want - near), len(want | near)
            assert lo <= cc[i] <= hi, (i, cc[i], lo, hi)
            n_w = min(cc[i], cap)
            got = ci[i, :n_w]
            assert len(set(got)) == n_w and set(got) <= (want | near)
            if cc[i] <= cap:
                assert (want - near) <= set(got)
            np.testing.assert_allclose(cs[i, :n_w], s[i, got - base], rtol=0, atol=1e-5 * scale[i])
        if cap == 40:
            assert (cc > cap).any() and (cc[:5] == M).all()


def _pq_problem(n_d, M, dsub, opq, with_b, seed, ortho=True):
    from gnnlm_b200.pq_codec import TorchPQCodec
    rng = np.random.RandomState(seed)
    d = M * dsub
    cen = rng.randn(M, 256, dsub).astype(np.float32)
    A = np.linalg.qr(rng.randn(d, d))[0] if ortho else rng.randn(d, d) / np.sqrt(d)
    A = A.astype(np.float32)
    b = (0.1 * rng.randn(d)).astype(np.float32) if with_b else np.zeros(0, np.float32)
    codes = rng.randint(0, 256, (n_d, M)).astype(np.uint8)
    y = cen[np.arange(M)[None, :], codes].reshape(n_d, d).astype(np.float64)
    x = (y - (b.astype(np.float64) if with_b else 0.0)) @ A.astype(np.float64) if opq else y
    codec = TorchPQCodec(centroids=cen, A=A if opq else None, b=b if opq else None)
    return codes, codec, x


def _check(dists, ids, q, x, k, metric):
    """ids = fp64 oracle up to swaps of entries within 1e-5 * scale; distances within 1e-5 of the fp64 recompute."""
    q64 = q.double().cpu().numpy()
    x = np.asarray(x, np.float64)
    s = q64 @ x.T
    xn = (x ** 2).sum(1)
    if metric == "l2":
        s = s - 0.5 * xn[None]
    n, n_d = s.shape
    kk = min(k, n_d)
    ids, dists = ids.cpu().numpy(), dists.cpu().numpy()
    assert ids.shape == dists.shape == (n, k) and ids.dtype == np.int64 and dists.dtype == np.float32
    assert (ids[:, kk:] == -1).all() and (dists[:, kk:] == (np.inf if metric == "l2" else -np.inf)).all()
    qn = (q64 ** 2).sum(1)
    scale = np.sqrt(qn) * np.sqrt(xn.max()) + (0.5 * xn.max() if metric == "l2" else 0.0)
    got = ids[:, :kk]
    assert (got >= 0).all() and all(len(set(r)) == kk for r in got)
    want = np.stack([_ranked(s[i], np.arange(n_d))[:kk] for i in range(n)])
    gs, ws = np.take_along_axis(s, got, 1), np.take_along_axis(s, want, 1)
    diff = got != want
    assert (np.abs(gs - ws) <= 1e-5 * scale[:, None])[diff].all(), f"{diff.sum()} ids differ beyond near-ties"
    if metric == "l2":
        true = qn[:, None] - 2 * q64.dot(x.T)[np.arange(n)[:, None], got] + xn[got]
        tol = 1e-5 * (qn[:, None] + xn[got])
    else:
        true, tol = gs, 1e-5 * scale[:, None]
    assert (np.abs(dists[:, :kk] - true) <= tol).all()
    return diff.sum()


PQ_CASES = [  # (opq, with_b, metric, k)
    (True, True, "l2", 8), (True, False, "ip", 1024), (False, False, "l2", 1), (False, False, "ip", 8), (True, True, "ip", 1)]


@pytest.mark.parametrize("opq,with_b,metric,k", PQ_CASES)
def test_searcher_pq(dev, opq, with_b, metric, k):
    from gnnlm_b200.knn_search import KNNSearcher, PQKeys
    codes, codec, x = _pq_problem(23457, 16, 8, opq, with_b, seed=k)
    q = torch.from_numpy(np.random.RandomState(1).randn(70, 128).astype(np.float32))
    s = KNNSearcher(PQKeys(codes, codec), metric, k, cap=2048 if k > 8 else 4096, span_keys=5000, device=dev)
    assert len(s.schedule) > 3 and s.schedule[-1][1] - s.schedule[-1][0] != s.schedule[-2][1] - s.schedule[-2][0]
    dists, ids = s.search(q)
    _check(dists, ids, q, x, k, metric)


def test_searcher_pq_non_orthonormal(dev):
    """ip holds for any OPQ matrix (q A^T . (y - b) = q . x); l2 needs ||y - b|| = ||x|| and refuses otherwise."""
    from gnnlm_b200.knn_search import KNNSearcher, PQKeys
    codes, codec, x = _pq_problem(3000, 8, 8, True, True, seed=5, ortho=False)
    q = torch.randn(20, 64, generator=torch.Generator().manual_seed(2))
    _check(*KNNSearcher(PQKeys(codes, codec), "ip", 16, device=dev).search(q), q, x, 16, "ip")
    with pytest.raises(NotImplementedError, match="orthonormal"):
        KNNSearcher(PQKeys(codes, codec), "l2", 16, device=dev)


@pytest.mark.parametrize("dtype,streamed,metric,k", [(np.float16, False, "l2", 8), (np.float32, False, "ip", 1024),
                                                      (np.float16, True, "ip", 1), (np.float32, True, "l2", 1024)])
def test_searcher_raw_keys(dev, dtype, streamed, metric, k):
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    rng = np.random.RandomState(7)
    keys = rng.randn(20011, 96).astype(dtype)
    q = torch.from_numpy(rng.randn(65, 96).astype(np.float32))
    src = RawKeys(keys, device_bytes=1 if streamed else None)
    s = KNNSearcher(src, metric, k, cap=2048, span_keys=3000, device=dev)
    assert src.resident == (not streamed) and len(s.schedule) > 3
    _check(*s.search(q), q, keys, k, metric)


def test_searcher_fewer_keys_than_k(dev):
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    keys = np.random.RandomState(0).randn(300, 32).astype(np.float32)
    q = torch.randn(9, 32, generator=torch.Generator().manual_seed(0))
    for metric in ("l2", "ip"):
        _check(*KNNSearcher(RawKeys(keys), metric, 1024, device=dev).search(q), q, keys, 1024, metric)


def test_search_invariance(dev):
    """Bit-identical ids and distances across span lengths, cap (one small enough to force overflow re-runs), query batches and
    1 vs 2 ranks (contiguous query ranges)."""
    from gnnlm_b200.eval_lm import shard_range
    from gnnlm_b200.knn_search import KNNSearcher, PQKeys, RawKeys
    codes, codec, _ = _pq_problem(30000, 16, 8, True, True, seed=11)
    q = torch.from_numpy(np.random.RandomState(3).randn(301, 128).astype(np.float32))
    keys = np.random.RandomState(4).randn(30000, 128).astype(np.float16)
    for make in (lambda: PQKeys(codes, codec), lambda: RawKeys(keys)):
        ref = KNNSearcher(make(), "l2", 32, device=dev).search(q)
        small = KNNSearcher(make(), "l2", 32, cap=64, span_keys=20000, query_batch=50, device=dev)
        out = small.search(q)
        assert small.reruns > 0
        spans = KNNSearcher(make(), "l2", 32, span_keys=4096, query_batch=77, device=dev)
        outs = [out, spans.search(q)]
        ranked = [spans.search(q[lo:hi]) for lo, hi in (shard_range(301, r, 2) for r in range(2))]
        outs.append((torch.cat([r[0] for r in ranked]), torch.cat([r[1] for r in ranked])))
        for d, i in outs:
            assert torch.equal(i, ref[1]) and torch.equal(d, ref[0])


def test_find_knn_feeds_eval_lm(dev, tmp_path):
    """find_knn on a data directory in the reference layout: neighbors.mmap.{k} = the fp64 oracle's ids; eval_lm --knnlm with
    --knn-dists-file <dists.{k}> --knn-sim-func do_not_recomp_l2 scores as the same run fed the oracle's ids and distances."""
    import json
    from argparse import Namespace
    from gnnlm_b200 import synth
    from gnnlm_b200.eval_lm import main
    from gnnlm_b200.find_knn import find_knn
    from gnnlm_b200.formats import write_faiss_quantizer
    from tests.test_formats import write_mmap_indexed
    cfg = dict(synth.CONFIGS["c1"], NL=2, k=4, n_d=1 << 14, V=1000, cutoff=[200, 600], k_nn=8)
    model = synth.make_model(cfg)
    tables = synth.make_tables(cfg, device="cpu")
    rng = np.random.RandomState(12)
    lens = [64, 64, 40]
    sents = [np.concatenate([rng.randint(4, cfg["V"], size=n - 1), [2]]).astype(np.int64) for n in lens]
    n_tok, k_nn = sum(lens), cfg["k_nn"]
    root = str(tmp_path / "data-bin")
    for sub in ("valid_dstore", "train_dstore"):
        os.makedirs(os.path.join(root, sub))
    with open(os.path.join(root, "dict.txt"), "w") as f:
        f.write("".join(f"w{i} {cfg['V'] - i}\n" for i in range(4, cfg["V"])))
    write_mmap_indexed(os.path.join(root, "valid"), sents, np.uint16)
    rng.randint(1, cfg["n_d"] - 1, size=(n_tok, cfg["k"])).astype(np.int64).tofile(os.path.join(root, "valid_dstore", f"neighbors.mmap.{cfg['k']}"))
    feats = rng.randn(n_tok, cfg["d"]).astype(np.float16)
    feats.tofile(os.path.join(root, "valid_dstore", "keys.npy"))
    info = {"hidden_size": cfg["d"], "vocab_size": cfg["V"], "dstore_fp16": True, "val_size": 1}
    json.dump(dict(info, dstore_size=n_tok), open(os.path.join(root, "valid_dstore", "info.json"), "w"))
    json.dump(dict(info, dstore_size=cfg["n_d"]), open(os.path.join(root, "train_dstore", "info.json"), "w"))
    tables["vals"].numpy().astype(np.int16).reshape(-1, 1).tofile(os.path.join(root, "train_dstore", "vals.npy"))
    codes = tables["codes"].numpy()
    np.save(os.path.join(root, "train_dstore", "quantized-keys.npy"), codes)
    qz = model.decoder.tgt_quantizer
    qfile = os.path.join(root, "quantizer")
    write_faiss_quantizer(qfile, qz.centroids_torch.numpy(), qz.A.numpy(), qz.b.numpy())
    ckpt_args = Namespace(arch="transformer_lm", decoder_embed_dim=cfg["d"], decoder_attention_heads=cfg["H"], graph_layer=2,
                          decoder_gcn_dim=cfg["d"], adaptive_softmax_cutoff="200,600", tie_adaptive_weights=False,
                          quantizer_path=qfile, task="language_modeling", tokens_per_sample=3072)
    ckpt = str(tmp_path / "checkpoint_best.pt")
    torch.save({"args": ckpt_args, "model": model.state_dict()}, ckpt)

    res = find_knn(root, "valid", k_nn, "l2", "pq", quantizer=qfile, write_dists=True, query_batch=100, device=dev,
                   log=lambda *_: None)
    ids = np.fromfile(res["neighbors"], np.int64).reshape(n_tok, k_nn)
    dists = np.fromfile(res["dists"], np.float32).reshape(n_tok, k_nn)
    cen = qz.centroids_torch.numpy().astype(np.float64)
    M = cen.shape[0]
    x = cen[np.arange(M)[None, :], codes].reshape(cfg["n_d"], -1) @ qz.A.numpy().astype(np.float64)
    q = torch.from_numpy(feats.astype(np.float32))
    assert _check(torch.from_numpy(dists), torch.from_numpy(ids), q, x, k_nn, "l2") == 0
    q64 = feats.astype(np.float64)
    s = q64 @ x.T - 0.5 * (x ** 2).sum(1)[None]
    o_ids = np.stack([_ranked(s[i], np.arange(x.shape[0]))[:k_nn] for i in range(n_tok)])
    o_d = ((q64[:, None, :] - x[o_ids]) ** 2).sum(-1).astype(np.float32)
    argv = [root, "--path", ckpt, "--graph", "--use-precompute-feat", "--gen-subset", "valid", "--tokens-per-sample", "64",
            "--gcn-k", str(cfg["k"]), "--neighbor-context", "1", "--math", "fp32", "--max-sentences", "2", "--knnlm", "--k",
            str(k_nn), "--lmbda", "0.25", "--knn-sim-func", "do_not_recomp_l2", "--temperature", "10"]
    got = main(argv + ["--knn-dists-file", res["dists"]], device=dev, log=lambda *_: None)
    o_ids.astype(np.int64).tofile(res["neighbors"])
    o_file = str(tmp_path / "oracle_dists")
    o_d.tofile(o_file)
    want = main(argv + ["--knn-dists-file", o_file], device=dev, log=lambda *_: None)
    assert got["count"] == want["count"] == n_tok
    assert abs(got["score_sum"] - want["score_sum"]) <= 1e-6 * abs(want["score_sum"])


@pytest.mark.parametrize("opq,metric", [(True, "l2"), (False, "ip")])
def test_searcher_pq_dsub4(dev, opq, metric):
    """dsub != 8: the keys are decoded by gnnlm_pq_gather_decode into the split format, with the OPQ bias subtracted there."""
    from gnnlm_b200.knn_search import KNNSearcher, PQKeys
    codes, codec, x = _pq_problem(9001, 32, 4, opq, opq, seed=21)
    q = torch.from_numpy(np.random.RandomState(2).randn(40, 128).astype(np.float32))
    s = KNNSearcher(PQKeys(codes, codec), metric, 16, span_keys=4096, device=dev)
    assert codec.dsub == 4 and len(s.schedule) > 1
    _check(*s.search(q), q, x, 16, metric)


def test_self_search_l2_clamps_at_zero(dev):
    """Searching the datastore's own keys (the train split): every key is its own nearest neighbour, at distance >= 0."""
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    keys = (np.random.RandomState(5).randn(5000, 64) * 4).astype(np.float16)
    d, i = KNNSearcher(RawKeys(keys), "l2", 4, device=dev).search(torch.from_numpy(keys[:700].astype(np.float32)))
    assert (i[:, 0].cpu() == torch.arange(700)).all()
    assert (d >= 0).all() and (d[:, 0] <= 1e-2).all() and (d[:, 1] > 1.0).all()


def test_searcher_on_another_current_device(dev):
    """A searcher runs on its own device whatever the current device is (the last GPU of the box against the current one; with a
    single GPU both are cuda:0)."""
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    other = torch.device(f"cuda:{torch.cuda.device_count() - 1}")
    keys = np.random.RandomState(6).randn(6000, 96).astype(np.float32)
    q = torch.from_numpy(np.random.RandomState(7).randn(50, 96).astype(np.float32))
    want = KNNSearcher(RawKeys(keys), "l2", 8, device=dev).search(q)
    with torch.cuda.device(dev):
        s = KNNSearcher(RawKeys(keys), "l2", 8, device=other)
        got = s.search(q)
    assert got[0].device == other and torch.equal(got[0].cpu(), want[0].cpu()) and torch.equal(got[1].cpu(), want[1].cpu())


def test_find_knn_ranks_as_separate_processes(dev, tmp_path):
    """`python -m gnnlm_b200.find_knn` launched as two ranks (RANK / WORLD_SIZE / LOCAL_RANK as torchrun sets them, LOCAL_RANK
    wrapped onto the GPUs present) writes the same files as one in-process run."""
    import json
    import subprocess
    import sys
    from gnnlm_b200.find_knn import find_knn
    rng = np.random.RandomState(8)
    roots = [str(tmp_path / n) for n in ("one", "two")]
    for root in roots:
        for split, n, dt in (("valid", 333, np.float16), ("train", 7000, np.float32)):
            os.makedirs(os.path.join(root, f"{split}_dstore"))
            json.dump({"dstore_size": n, "hidden_size": 64, "dstore_fp16": dt == np.float16, "vocab_size": 10, "val_size": 1},
                      open(os.path.join(root, f"{split}_dstore", "info.json"), "w"))
    for split, n, dt in (("valid", 333, np.float16), ("train", 7000, np.float32)):
        a = rng.randn(n, 64).astype(dt)
        for root in roots:
            a.tofile(os.path.join(root, f"{split}_dstore", "keys.npy"))
    ref = find_knn(roots[0], "valid", 16, "l2", "keys", write_dists=True, query_batch=100, device=dev, log=lambda *_: None)
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n_dev = torch.cuda.device_count()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", LOCAL_RANK=str(rank % n_dev),
                   PYTHONPATH=repo + os.pathsep + os.environ.get("PYTHONPATH", ""))
        procs.append(subprocess.Popen([sys.executable, "-m", "gnnlm_b200.find_knn", "--data-dir", roots[1], "--subset", "valid",
                                       "--k", "16", "--source", "keys", "--write-dists", "--query-batch", "100"],
                                      cwd=repo, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    try:
        for p in procs:
            out, _ = p.communicate(timeout=600)
            assert p.returncode == 0, out
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.wait()
    for name, dt in ((f"neighbors.mmap.16", np.int64), ("dists.16", np.float32)):
        a = np.fromfile(os.path.join(roots[0], "valid_dstore", name), dt)
        b = np.fromfile(os.path.join(roots[1], "valid_dstore", name), dt)
        assert a.shape == b.shape == (333 * 16,) and (a == b).all(), name
    assert ref["rows"] == (0, 333)
