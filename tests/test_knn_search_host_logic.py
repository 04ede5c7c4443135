"""Host logic of gnnlm_b200.knn_search / find_knn on the CPU (`-m "not gpu"`): the C-ABI calls the searcher makes
(gnnlm_knn_filter_f16x3, gnnlm_topk_merge, gnnlm_knn_key_bias, gnnlm_split_f16, gnnlm_to_split_f16, gnnlm_gather_rows) are
replaced by plain-torch stand-ins INSIDE THIS TEST ONLY (monkeypatch) that follow the header's contract -- including the
candidate overflow (writes stop at cap, the count keeps growing) and the merge leaving overflowed queries alone.  What is
exercised is the span schedule, the overflow re-run, the sharded row ranges and the file layout; the kernels themselves are
checked on the GPU (tests/test_gpu_knn_search.py)."""
import json
import os

import numpy as np
import pytest
import torch


@pytest.fixture
def torch_kernels(monkeypatch):
    from gnnlm_b200 import ops

    def split_f16(w, scale=None):
        hi = w.half()
        return hi, (w - hi.float()).half(), 1.0 if scale is None else scale

    def to_split(x, rows_dev=None, scale=1.0):
        x = x.float()
        hi = x.half()
        return ops.Split(torch.cat([hi, (x - hi.float()).half()], 1), x.shape[1])

    def knn_key_bias(x):
        return (-0.5 * (x.double() ** 2).sum(1)).float()

    def knn_filter(keys, id_base, q_hi, q_lo, key_bias, thr, cand_s, cand_id, cand_cnt):
        x = keys.float().double()
        q = q_hi.double() + q_lo.double()
        s = q @ x.T
        if key_bias is not None:
            s = s + key_bias.double()[None, :]
        s = s.float()
        cap = cand_s.shape[1]
        for i in range(q.shape[0]):
            sel = torch.nonzero(s[i] > thr[i]).flatten()
            c0 = int(cand_cnt[i])
            room = max(0, min(cap - c0, sel.numel()))
            cand_s[i, c0:c0 + room] = s[i, sel[:room]]
            cand_id[i, c0:c0 + room] = (sel[:room] + id_base).int()
            cand_cnt[i] = c0 + sel.numel()

    def topk_merge(top_s, top_id, cand_s, cand_id, cand_cnt, thr):
        k, cap = top_s.shape[1], cand_s.shape[1]
        for i in range(top_s.shape[0]):
            c = int(cand_cnt[i])
            if c == 0 or c > cap:
                continue
            held = top_id[i] >= 0
            s = torch.cat([top_s[i][held], cand_s[i, :c]]).numpy()
            ids = torch.cat([top_id[i][held], cand_id[i, :c]]).numpy()
            order = np.lexsort((ids, -s.astype(np.float64)))[:k]
            top_s[i] = -np.inf
            top_id[i] = -1
            top_s[i, :order.size] = torch.from_numpy(s[order])
            top_id[i, :order.size] = torch.from_numpy(ids[order])
            thr[i] = float(s[order[k - 1]]) if order.size == k else -np.inf
            cand_cnt[i] = 0

    def gather_rows(src, ids, n_cap=None, n_dev=None, out=None):
        return src[ids.long()]

    for name, fn in dict(split_f16=split_f16, to_split=to_split, knn_key_bias=knn_key_bias, knn_filter=knn_filter,
                         topk_merge=topk_merge, gather_rows=gather_rows).items():
        monkeypatch.setattr(ops, name, fn)


def _oracle(q, x, k, metric):
    """Top-k by (score descending, id ascending) with the stand-ins' fp32 scores; -1 / +-inf padding."""
    q64, x64 = q.double(), x.double()
    s = q64 @ x64.T
    if metric == "l2":
        s = s + (-0.5 * (x64 ** 2).sum(1))[None]
    s = s.float().numpy()
    n, n_d = s.shape
    ids = np.full((n, k), -1, np.int64)
    sc = np.full((n, k), -np.inf, np.float32)
    for i in range(n):
        o = np.lexsort((np.arange(n_d), -s[i].astype(np.float64)))[:k]
        ids[i, :o.size], sc[i, :o.size] = o, s[i, o]
    return sc, ids


def _split_round(t):
    hi = t.half()
    return hi.double() + (t - hi.float()).half().double()


def test_span_schedule_warmup_and_growth():
    from gnnlm_b200.knn_search import span_schedule
    sp = span_schedule(1_000_000, k=1024, cap=4096, span_keys=1 << 17)
    assert sp[0] == (0, 4096) and sp[-1][1] == 1_000_000
    assert all(a[1] == b[0] for a, b in zip(sp, sp[1:]))
    assert sp[1] == (4096, 4096 + int(4096 * (np.exp(2.0) - 1)))              # the warm-up is over: growth p (e^(cap/2k) - 1)
    assert max(e - s for s, e in sp) == 1 << 17
    small = span_schedule(100, k=64, cap=16, span_keys=1000)                      # cap < k: cap-sized spans until k keys are held
    assert [e - s for s, e in small[:4]] == [16] * 4 and all(e - s >= 16 for s, e in small[:-1])
    assert span_schedule(0, 8, 16, 100) == [] and span_schedule(5, 8, 16, 100) == [(0, 5)]


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_search_overflow_rerun_is_exact(torch_kernels, metric):
    """Small cap, large spans: queries overflow, their span is re-run in cap-sized pieces; the result is the exact top-k,
    ties (integer-valued keys) broken by the smaller id, identical for every cap / span length / query batch."""
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    g = torch.Generator().manual_seed(0)
    x = torch.randint(-2, 3, (700, 16), generator=g).float()
    q = torch.randint(-2, 3, (37, 16), generator=g).float()
    k = 12
    sc, ids = _oracle(q, x, k, metric)
    outs = []
    for cap, span, qb in ((16, 400, 64), (40, 1 << 20, 5), (4096, 64, 37)):
        s = KNNSearcher(RawKeys(x), metric, k, cap=cap, span_keys=span, query_batch=qb, device="cpu")
        d, i = s.search(q)
        assert (i.numpy() == ids).all()
        if cap == 16:
            assert s.reruns > 0
        outs.append(d)
    qn = (q.double() ** 2).sum(1, keepdim=True).float()
    want = torch.from_numpy(sc) if metric == "ip" else (-2.0 * (torch.from_numpy(sc) + (-0.5 * qn))).clamp_min(0.0)
    assert torch.equal(outs[0], want) and all(torch.equal(o, outs[0]) for o in outs)


def test_fewer_keys_than_k_pads(torch_kernels):
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    x, q = torch.randn(5, 8), torch.randn(3, 8)
    for metric, pad in (("l2", np.inf), ("ip", -np.inf)):
        d, i = KNNSearcher(RawKeys(x.half()), metric, 8, cap=32, device="cpu").search(q)
        assert (i[:, 5:] == -1).all() and (d[:, 5:] == pad).all()
        assert sorted(i[0, :5].tolist()) == list(range(5)) and torch.isfinite(d[:, :5]).all()


def test_out_of_range_operands_are_refused(torch_kernels):
    """Keys beyond the fp16 range of the split operands (or NaN), and queries beyond the 2^15 of the query split, raise instead of
    being clamped."""
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    x = torch.randn(50, 8)
    s = KNNSearcher(RawKeys(x), "l2", 4, device="cpu")
    with pytest.raises(ValueError, match="query"):
        s.search(torch.full((2, 8), 40000.0))
    for bad in (1e5, float("nan")):
        y = x.clone()
        y[7, 3] = bad
        with pytest.raises(ValueError, match="keys"):
            KNNSearcher(RawKeys(y), "l2", 4, device="cpu")
    assert KNNSearcher(RawKeys(x * 0 + 65504.0), "ip", 4, device="cpu").search(x[:2])[1].shape == (2, 4)


def _data_dir(root, n_q=50, n_d=300, d=16, seed=0):
    rng = np.random.RandomState(seed)
    for split, n, dt in (("valid", n_q, np.float16), ("train", n_d, np.float32)):
        os.makedirs(os.path.join(root, f"{split}_dstore"))
        rng.randn(n, d).astype(dt).tofile(os.path.join(root, f"{split}_dstore", "keys.npy"))
        json.dump({"dstore_size": n, "hidden_size": d, "dstore_fp16": dt == np.float16, "vocab_size": 10, "val_size": 1},
                  open(os.path.join(root, f"{split}_dstore", "info.json"), "w"))


def test_find_knn_file_layout_and_shards(torch_kernels, tmp_path):
    """neighbors.mmap.{k}: raw int64 [N_split, k]; dists.{k}: raw fp32 [N_split, k]; two ranks fill one file = one process."""
    from gnnlm_b200 import find_knn as fk
    one, two = str(tmp_path / "one"), str(tmp_path / "two")
    _data_dir(one), _data_dir(two)
    k = 7
    r = fk.find_knn(one, "valid", k, "l2", "keys", write_dists=True, query_batch=16, device="cpu", log=lambda *_: None, cap=8,
                    span_keys=64)
    assert r["rows"] == (0, 50)
    assert os.path.getsize(r["neighbors"]) == 50 * k * 8 and os.path.getsize(r["dists"]) == 50 * k * 4
    ids = np.fromfile(r["neighbors"], np.int64).reshape(50, k)
    dists = np.fromfile(r["dists"], np.float32).reshape(50, k)
    q = torch.from_numpy(np.fromfile(os.path.join(one, "valid_dstore", "keys.npy"), np.float16).reshape(50, 16).astype(np.float32))
    x = torch.from_numpy(np.fromfile(os.path.join(one, "train_dstore", "keys.npy"), np.float32).reshape(300, 16))
    sc, want = _oracle(_split_round(q).float(), x, k, "l2")
    assert (ids == want).all()
    np.testing.assert_allclose(dists, ((q[:, None, :].double() - x[torch.from_numpy(ids)].double()) ** 2).sum(-1).numpy(),
                               rtol=1e-5, atol=1e-4)
    assert (np.diff(dists, axis=1) >= -1e-4).all()
    r2 = fk.main(["--data-dir", two, "--subset", "valid", "--k", str(k), "--source", "keys", "--write-dists", "--query-batch", "16"],
                 device="cpu", log=lambda *_: None)
    assert r2["rows"] == (0, 50) and (np.fromfile(r2["neighbors"], np.int64).reshape(50, k) == ids).all()
    os.remove(r2["neighbors"])
    os.remove(r2["dists"])
    for rank in (1, 0):                       # the later rank's truncate never drops the rows the earlier one wrote
        fk.find_knn(two, "valid", k, "l2", "keys", write_dists=True, query_batch=16, rank=rank, world=2, device="cpu",
                    log=lambda *_: None)
    assert (np.fromfile(os.path.join(two, "valid_dstore", f"neighbors.mmap.{k}"), np.int64).reshape(50, k) == ids).all()
    assert (np.fromfile(os.path.join(two, "valid_dstore", f"dists.{k}"), np.float32).reshape(50, k) == dists).all()


def test_knn_model_searches_without_results(torch_kernels):
    from gnnlm_b200.knn_model import KNNModel
    from gnnlm_b200.knn_search import KNNSearcher, RawKeys
    x, q = torch.randn(40, 8), torch.randn(6, 8)
    s = KNNSearcher(RawKeys(x), "l2", 4, cap=8, device="cpu")
    m = KNNModel(torch.zeros(40, dtype=torch.int32), 10, "do_not_recomp_l2", k=4, searcher=s)
    d, i = m.get_knns(q)
    d2, i2 = s.search(q)
    assert torch.equal(d, d2) and torch.equal(i, i2)
    m.set_search_results(d2 + 1, i2)                # provided results still win
    assert torch.equal(m.get_knns(q)[0], d2 + 1)
    with pytest.raises(ValueError):
        KNNModel(torch.zeros(40, dtype=torch.int32), 10, "do_not_recomp_l2", k=8, searcher=s)
    with pytest.raises(RuntimeError):
        KNNModel(torch.zeros(40, dtype=torch.int32), 10, "do_not_recomp_l2", k=4).get_knns(q)
