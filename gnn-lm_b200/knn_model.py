"""kNN-LM probability -- host-side mirror of knn/knn_model.py:25-217 (KNNModel) for the
precomputed-neighbour pipeline: the retrieved (dists, ids) are inputs, exactly as find_knn.py precomputes ids for the graph
(SURVEY.md Q8: the eval script's queries are the same precomputed features find_knn.py searched
with, hence precomputable).  Given a `searcher` (knn_search.KNNSearcher), get_knns searches itself when no results
were provided, as the reference's get_knns does (exact search instead of the faiss index).  Everything after the search --
similarity sign, -1 masking, softmax over sims/T, the vote on the target or the full-vocabulary scatter -- runs in
logprob_knn.cu."""
from typing import Optional

import torch

from . import ops


class KNNModel(object):
    def __init__(self, vals: torch.Tensor, vocab_size: Optional[int] = None, metric_type: str = "do_not_recomp_ip",
                 k: int = 1024, dists: Optional[torch.Tensor] = None, knns: Optional[torch.Tensor] = None,
                 keys: Optional[torch.Tensor] = None, pq_codes: Optional[torch.Tensor] = None, quantizer=None,
                 index_file: str = "", searcher=None):
        """vals: [N_d] (or [N_d,1]) int16/int32 datastore values resident in HBM (vals.npy);
        dists/knns: optional whole-split precomputed search results [N_split, k] indexed by stream position.
        metric_type `l2` / `ip` recompute the similarities (knn_model.py:159-177) from `keys` ([N_d, d] fp16/fp32 in
        HBM, the reference's keys.npy) or, when the keys only exist PQ-compressed, from `pq_codes` [N_d, M] uint8 +
        `quantizer` (TorchPQCodec) -- then against the decoded keys.  `index_file`: as in the reference, a name
        containing "cosine" switches on the query / key normalisation (:171-172,181-184), for raw and PQ-decoded keys alike.
        searcher: a knn_search.KNNSearcher with the same k, used by get_knns when neither pending nor precomputed results exist."""
        assert metric_type in ["do_not_recomp_l2", "do_not_recomp_ip", "l2", "ip"]
        self.recompute = metric_type in ("l2", "ip")
        if self.recompute and keys is None and pq_codes is None:
            raise ValueError(f"metric_type={metric_type} needs the datastore keys (keys=...) or their PQ codes "
                             "(pq_codes=..., quantizer=...)")
        self.keys, self.pq_codes, self.quantizer, self.index_file = keys, pq_codes, quantizer, index_file
        self.cosine = "cosine" in index_file
        self._key_norm2 = None
        if self.recompute and keys is None:
            if (metric_type == "l2" or self.cosine) and quantizer.pre_torch:
                A = quantizer.A.double()
                if not torch.allclose(A @ A.T, torch.eye(A.shape[0], dtype=A.dtype, device=A.device), atol=1e-4):
                    raise NotImplementedError("l2 / cosine against PQ-decoded keys needs an orthonormal OPQ transform")
        self.vals = vals.reshape(-1)
        assert self.vals.dtype in (torch.int16, torch.int32)
        self.dstore_size = self.vals.numel()
        self.vocab_size = vocab_size
        self.metric_type = metric_type
        self.k = k
        self.dists, self.knns = dists, knns
        if searcher is not None and searcher.k != k:
            raise ValueError(f"the searcher returns {searcher.k} neighbours, the model uses k = {k}")
        self.searcher = searcher
        self._pending = None

    @property
    def sim_sign(self):
        return -1.0 if self.metric_type == "do_not_recomp_l2" else 1.0      # knn_model.py:153-157 (recomputed sims carry their sign)

    def similarities(self, queries: torch.Tensor, dists: Optional[torch.Tensor], knns: torch.Tensor) -> torch.Tensor:
        """sim_func of knn_model.py:137-177 up to the sign handled by `sim_sign`: the search distances for
        do_not_recomp_*, else recomputed from the keys.  queries [num, d] fp32 on the device."""
        if not self.recompute:
            return dists
        q = queries.float()
        if q.stride(-1) != 1:
            q = q.contiguous()
        if self.keys is not None:
            return ops.knn_sims_keys(q, self.keys, knns, self.metric_type, cosine=self.cosine)
        qz = self.quantizer
        rot = ops.linear(q, qz.A.contiguous(), None, math=0) if qz.pre_torch else q        # q @ A.T, fp32
        b = qz.b if qz.pre_torch and qz.b.numel() > 0 else None
        if self.cosine and self.metric_type == "ip" and self._key_norm2 is None:
            # ||x^||^2 = ||y - b||^2 = sum_m ||centroid[m, c_m] - b_m||^2 for an orthonormal transform: one [M, 256] table per datastore
            cen = qz.centroids_torch.double()
            if b is not None:
                cen = cen - b.double().view(cen.shape[0], 1, cen.shape[2])
            self._key_norm2 = (cen ** 2).sum(-1).float().contiguous()
        return ops.knn_sims_pq(q, rot, self.pq_codes, qz.centroids_torch, b, knns, self.metric_type, key_norm2=self._key_norm2,
                               cosine=self.cosine)

    def set_search_results(self, dists: Optional[torch.Tensor], knns: torch.Tensor):
        """Provide the search output for the next get_knn_prob call: [num, k] each; dists may be None
        when the metric recomputes them."""
        self._pending = (None if dists is None else dists.contiguous().float(), knns.contiguous().long())

    def get_knns(self, queries, k: int = 0, positions: Optional[torch.Tensor] = None):
        if self._pending is not None:
            out, self._pending = self._pending, None
            return out
        if positions is not None and self.knns is not None and (self.dists is not None or self.recompute):
            positions = positions.reshape(-1)          # sample['positions'] is [B, L]: one row of search results per token
            return (None if self.dists is None else self.dists[positions].float().contiguous()), \
                self.knns[positions].long().contiguous()
        if self.searcher is not None:
            return self.searcher.search(queries)
        raise RuntimeError("no search results: pass a searcher, call set_search_results() or pass precomputed arrays")

    @torch.no_grad()
    def get_knn_prob(self, queries, k: int = 0, output_size: int = None, return_knn: bool = False, t: float = 1.0,
                     targets: torch.Tensor = None, return_recall: bool = False, positions=None):
        """knn_model.py:103-217.  `queries` [num, d] is read only by the recomputing metrics (l2 / ip)."""
        dists, knns = self.get_knns(queries, k=k, positions=positions)
        dists = self.similarities(queries, dists, knns)
        if targets is None:
            output_size = output_size or self.vocab_size
            if not output_size:
                raise ValueError("DataStore.info does not have vocab_size, please set output_size manually")
            probs = ops.knn_full_prob(dists, knns, self.vals, output_size, self.dstore_size, self.sim_sign, t)
            if return_knn:
                return probs, dists * self.sim_sign, knns
            return probs
        zero = torch.zeros(dists.shape[0], device=dists.device, dtype=torch.float32)
        # lambda = 0.5 is irrelevant here: only p_knn / recall are read back
        _, p, rec = ops.knn_mix_nll(zero, target=targets.reshape(-1).contiguous(), dists=dists, ids=knns, vals=self.vals,
                                    n_datastore=self.dstore_size, sim_sign=self.sim_sign, temperature=t, lmbda=0.5,
                                    want_knn=True)
        if not return_recall:
            return p
        return p, rec.long()
