"""Exact k-nearest-neighbour search over the datastore, without faiss: the search of knn/find_knn.py:29-71 (which writes the
neighbour-id files) and of KNNModel.get_knns (knn/knn_model.py:87-101).

For every query q, the k datastore rows x with the highest score, ties broken by the smaller id:

    metric l2   s = q.x - 1/2 ||x||^2    distance written out ||q||^2 - 2 s  (squared L2, faiss METRIC_L2)
    metric ip   s = q.x                  distance s

When the datastore holds fewer than k keys the rest is padded with id -1, distance +inf (l2) / -inf (ip).  The search is exact
over the vectors it is given (the PQ-decoded keys, or the raw keys): it does not reproduce the approximate results of an IVF
index.  A query that is itself a datastore key finds itself, as in the reference; the dataset's --invalid-neighbor-context
filter drops such neighbours.

Schedule.  The datastore is scanned in spans of increasing ids.  Per span, one 3xFP16 tcgen05 GEMM (keys = A, read from HBM
once; queries = W, resident in L2) whose epilogue keeps only the scores above each query's running k-th score, as candidates
(gnnlm_knn_filter_f16x3), and one merge of the candidates into the running top-k (gnnlm_topk_merge).  Because ids grow from
span to span, the strict `>` is exact: a later key with an equal score loses the tie.  Span lengths (span_schedule):
  - while a query can hold fewer than k results (the first k keys), spans of `cap` keys: every key is a candidate, and a
    span of cap keys cannot overflow the cap candidate slots;
  - then spans that grow with the number p of keys already scanned, p * (exp(cap / 2k) - 1): for scores in random order the
    expected number of candidates of such a span is cap / 2;  at most `span_keys`;
  - a query whose candidates overflow a span (more than cap) is searched again over that span alone, in pieces of cap keys.
A score does not depend on the tile it is computed in, so ids and distances are bit-identical across span lengths, cap, query
batches and ranks."""
import contextlib
import math
from typing import Optional

import numpy as np
import torch

from . import ops

MAX_K, MAX_CAP = 2048, 4096
METRICS = ("l2", "ip")
F16_MAX = 65504.0


def _on(device: torch.device):
    """The searcher's device as the current CUDA device: the C-ABI calls launch on the current stream, which must be that device's."""
    return torch.cuda.device(device) if device.type == "cuda" else contextlib.nullcontext()


def _check_range(x: torch.Tensor, what: str, limit: float = F16_MAX):
    """The split fp16 operands hold |x| <= 65504 (the query split, gnnlm_split_f16: |x| < 2^15 = the limit passed for queries):
    refuse, rather than clamp, what lies beyond.  NaN fails the comparison and is refused too."""
    amax = float(x.abs().amax()) if x.numel() else 0.0
    if not (amax <= limit if limit == F16_MAX else amax < limit):
        raise ValueError(f"{what} must be finite and at most {limit:g} in magnitude (fp16 range of the split operands); "
                         f"max |x| = {amax:g}")


def span_schedule(n_keys: int, k: int, cap: int, span_keys: int):
    """[(start, end)] covering [0, n_keys): cap-sized spans over the first k keys, then growing ones (module docstring)."""
    grow = math.exp(min(cap / (2.0 * k), 30.0)) - 1.0
    spans, pos = [], 0
    while pos < n_keys:
        n = cap if pos < k else max(cap, min(span_keys, int(pos * grow)))
        spans.append((pos, min(n_keys, pos + n)))
        pos = spans[-1][1]
    return spans


def _to_device(arr, device, chunk_rows: int = 1 << 20) -> torch.Tensor:
    """A (memory-mapped) [n, c] array -> device tensor, in chunks (never the whole array in host memory at once)."""
    if torch.is_tensor(arr):
        return arr.to(device).contiguous()
    out = torch.empty(arr.shape, dtype=torch.from_numpy(np.empty(0, arr.dtype)).dtype, device=device)
    for a in range(0, arr.shape[0], chunk_rows):
        out[a:a + chunk_rows].copy_(torch.from_numpy(np.array(arr[a:a + chunk_rows])))
    return out


class PQKeys:
    """Datastore keys as PQ codes [N_d, M] uint8 (train_dstore/quantized-keys.npy) + their quantizer (TorchPQCodec): the decoded
    keys x = (y - b) A, searched in the quantizer's space -- queries q' = q A^T against y - b (faiss IndexPQ exhaustive search
    behind the OPQ transform).  q'.(y - b) = q.x for any A; ||y - b|| = ||x|| only for an orthonormal A, so `l2` raises
    otherwise.  The codes are kept resident on the device (13.2 GB for Wiki103 at M = 128)."""

    def __init__(self, codes, quantizer):
        self.codes, self.quantizer = codes, quantizer
        self.n = codes.shape[0]

    def prepare(self, metric: str, device):
        qz = self.quantizer.to(device)
        if metric == "l2" and qz.pre_torch:
            A = qz.A.double()
            if not torch.allclose(A @ A.T, torch.eye(A.shape[0], dtype=A.dtype, device=A.device), atol=1e-4):
                raise NotImplementedError("l2 search against PQ-decoded keys needs an orthonormal OPQ transform")
        self.qz, self.metric = qz, metric
        self.codes_dev = _to_device(self.codes, device)
        assert self.codes_dev.dtype == torch.uint8 and self.codes_dev.shape[1] == qz.M
        self.b = qz.b if qz.pre_torch and qz.b.numel() > 0 else None
        self.norm2 = None
        if metric == "l2":                 # ||centroid - b_m||^2 per (m, c): one [M, 256] table per quantizer
            cen = qz.centroids_torch.double()
            if self.b is not None:
                cen = cen - self.b.double().view(qz.M, 1, qz.dsub)
            self.norm2 = (cen ** 2).sum(-1).float().contiguous()
        cb = qz.centroids_torch if self.b is None else qz.centroids_torch - self.b.view(qz.M, 1, qz.dsub)
        _check_range(cb, "PQ centroids (minus the OPQ bias)")

    @property
    def dim(self):
        return self.qz.A.shape[1] if self.qz.pre_torch else self.qz.M * self.qz.dsub

    def queries(self, q: torch.Tensor) -> torch.Tensor:
        return ops.linear(q, self.qz.A.contiguous(), None, math=0) if self.qz.pre_torch else q

    def spans(self, spans):
        """Yields (start, end, keys split fp16, bias or None) per span: decoded straight into the GEMM operand format."""
        for s, e in spans:
            rows = torch.arange(s, e, device=self.codes_dev.device, dtype=torch.int64)
            if self.qz.dsub == 8:
                hi, lo = self.qz._split_codebook()
                x = ops.pq_gather_decode_presplit(self.codes_dev, hi, lo, rows)
            else:
                x = ops.pq_gather_decode(self.codes_dev, self.qz.centroids_torch, rows, bias=self.b, out_dtype=ops.SPLIT)[0]
            yield s, e, x, (ops.knn_key_bias_pq(self.codes_dev[s:e], self.norm2) if self.metric == "l2" else None)


class RawKeys:
    """Datastore keys [N_d, d] fp16 / fp32 (keys.npy as a memmap, an array or a tensor).  Kept resident on the device when they fit
    in `device_bytes` (default: half the free device memory), otherwise streamed span by span from host memory through two
    pinned buffers: the host read and the H2D copy of span i+1 run while the GPU searches span i."""

    def __init__(self, keys, device_bytes: Optional[int] = None):
        self.keys, self.device_bytes = keys, device_bytes
        self.n, self.dim = keys.shape

    def prepare(self, metric: str, device):
        self.metric, self.device = metric, torch.device(device)
        dt = self.keys.dtype if torch.is_tensor(self.keys) else torch.from_numpy(np.empty(0, self.keys.dtype)).dtype
        if dt not in (torch.float16, torch.float32):
            raise ValueError(f"keys must be fp16 or fp32, not {dt}")
        self.dtype = dt
        budget = self.device_bytes
        if budget is None:
            budget = torch.cuda.mem_get_info(self.device)[0] // 2 if self.device.type == "cuda" else float("inf")
        self.resident = self.n * self.dim * dt.itemsize <= budget
        self.keys_dev = _to_device(self.keys, self.device) if self.resident else None
        if self.resident:
            _check_range(self.keys_dev, "keys")

    def queries(self, q: torch.Tensor) -> torch.Tensor:
        return q

    def _prep(self, s, e, x):
        return s, e, ops.to_split(x), (ops.knn_key_bias(x) if self.metric == "l2" else None)

    def spans(self, spans):
        if self.resident:
            for s, e in spans:
                yield self._prep(s, e, self.keys_dev[s:e])
            return
        host_keys = self.keys.cpu() if torch.is_tensor(self.keys) else self.keys
        rows = max(e - s for s, e in spans)
        bufs = [torch.empty((rows, self.dim), dtype=self.dtype).pin_memory() for _ in range(2)]
        copied = [None, None]                   # per pinned buffer: the event after which it may be overwritten
        copy_stream = torch.cuda.Stream(device=self.device)
        main = torch.cuda.current_stream(self.device)

        def stage(i):
            s, e = spans[i]
            if copied[i % 2] is not None:
                copied[i % 2].synchronize()
            host = bufs[i % 2][:e - s]
            if torch.is_tensor(host_keys):
                host.copy_(host_keys[s:e])
            else:
                np.copyto(host.numpy(), host_keys[s:e])
            with torch.cuda.stream(copy_stream):
                x = host.to(self.device, non_blocking=True)
                x.record_stream(main)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            copied[i % 2] = ev
            return x, ev

        x, ev = stage(0)
        for i, (s, e) in enumerate(spans):
            main.wait_event(ev)
            _check_range(x, "keys")             # streamed keys: checked span by span, on the device
            item = self._prep(s, e, x)
            yield item                          # the caller queues the search of span i, then asks for span i+1:
            if i + 1 < len(spans):
                x, ev = stage(i + 1)            # its host read and copy overlap that search


class KNNSearcher:
    """Exact top-k search of a datastore source (PQKeys / RawKeys); see the module docstring for the contract and the schedule.

    k <= 2048; cap (candidate slots per query and span, <= 4096, >= k is best); span_keys: largest span; query_batch: queries per
    GEMM (their split fp16 form stays in L2: 16384 queries of d = 1024 are 64 MB).  `reruns` counts overflowed spans.
    Every call runs with `device` as the current CUDA device, so searchers on several GPUs of one process are independent."""

    def __init__(self, source, metric: str = "l2", k: int = 1024, *, cap: int = MAX_CAP, span_keys: int = 1 << 19,
                 query_batch: int = 16384, device="cuda"):
        if metric not in METRICS:
            raise ValueError(f"metric must be one of {METRICS}, not {metric!r}")
        if not 1 <= k <= MAX_K:
            raise ValueError(f"k must be in [1, {MAX_K}]")
        if not 1 <= cap <= MAX_CAP:
            raise ValueError(f"cap must be in [1, {MAX_CAP}]")
        if source.n >= 2 ** 31:
            raise ValueError("datastores of 2^31 keys or more are not supported (int32 ids)")
        self.source, self.metric, self.k, self.cap = source, metric, k, cap
        self.span_keys, self.query_batch, self.device = max(span_keys, cap), query_batch, torch.device(device)
        self.reruns = 0
        with _on(self.device):
            source.prepare(metric, self.device)
        self.schedule = span_schedule(source.n, k, cap, self.span_keys)

    @torch.no_grad()
    def search(self, queries: torch.Tensor):
        """queries [n, d] (any float dtype, any device) -> (dists fp32 [n, k], ids int64 [n, k]) on the searcher's device."""
        if queries.dim() != 2 or queries.shape[1] != self.source.dim:
            raise ValueError(f"queries must be [n, {self.source.dim}], got {tuple(queries.shape)}")
        with _on(self.device):
            parts = [self._search_batch(queries[a:a + self.query_batch])
                     for a in range(0, queries.shape[0], self.query_batch)] or [self._search_batch(queries[:0])]
        return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])

    def _search_batch(self, queries):
        dev, k, cap = self.device, self.k, self.cap
        q = queries.to(dev, torch.float32).contiguous()
        n = q.shape[0]
        top_s = torch.full((n, k), -math.inf, device=dev, dtype=torch.float32)
        top_id = torch.full((n, k), -1, device=dev, dtype=torch.int32)
        if n == 0:
            return top_s, top_id.long()
        qs = self.source.queries(q)
        _check_range(qs, "query components", 32768.0)
        # Scale 1, not a per-batch scale: the split of a query, hence its scores, must not depend on the other queries.  The lo
        # half of a component below 2^-14 is subnormal: its error stays below 2^-25 per component, far under the 2^-22 relative
        # error of the split for the components that make up the score.
        q_hi, q_lo, _ = ops.split_f16(qs, scale=1.0)
        thr = torch.full((n,), -math.inf, device=dev, dtype=torch.float32)
        cnt = torch.zeros((n,), device=dev, dtype=torch.int32)
        cand_s = torch.empty((n, cap), device=dev, dtype=torch.float32)
        cand_id = torch.empty((n, cap), device=dev, dtype=torch.int32)
        spans = self.source.spans(self.schedule)
        cur = next(spans, None)
        while cur is not None:
            s, _, keys, bias = cur
            ops.knn_filter(keys, s, q_hi, q_lo, bias, thr, cand_s, cand_id, cnt)
            ops.topk_merge(top_s, top_id, cand_s, cand_id, cnt, thr)
            nxt = next(spans, None)               # the next span's preparation is queued / staged under this one
            ovf = torch.nonzero(cnt).flatten()    # the merge zeroes every count but those past cap: one small read per span
            if ovf.numel():
                self._rerun(ovf, cur, q_hi, q_lo, top_s, top_id, thr, cnt, cand_s, cand_id)
            cur = nxt
        ids = top_id.long()
        if self.metric == "ip":
            return top_s, ids
        # ||q||^2 - 2 s, clamped at 0 as faiss's exhaustive L2 does (a query that is a datastore key would otherwise come out a
        # rounding error below 0); +inf where nothing is held
        return (-2.0 * (top_s + ops.knn_key_bias(q)[:, None])).clamp_min_(0.0), ids

    def _rerun(self, ovf, span, q_hi, q_lo, top_s, top_id, thr, cnt, cand_s, cand_id):
        """The overflowed queries of one span, again over that span alone in pieces of cap keys (which cannot overflow)."""
        self.reruns += 1
        s, _, keys, bias = span
        rows = ovf.to(torch.int32)
        qh, ql = ops.gather_rows(q_hi, rows), ops.gather_rows(q_lo, rows)
        ts, ti, th = top_s[ovf], top_id[ovf], thr[ovf]
        m = ovf.numel()
        cs, ci = cand_s[:m], cand_id[:m]
        cc = torch.zeros((m,), device=cnt.device, dtype=torch.int32)
        n_span = keys.data.shape[0]
        for a in range(0, n_span, self.cap):
            b = min(n_span, a + self.cap)
            ops.knn_filter(ops.Split(keys.data[a:b], keys.d), s + a, qh, ql, None if bias is None else bias[a:b], th, cs, ci, cc)
            ops.topk_merge(ts, ti, cs, ci, cc, th)
        top_s[ovf], top_id[ovf], thr[ovf] = ts, ti, th
        cnt[ovf] = 0
