"""The neighbour files of a split, without faiss (knn/find_knn.py:29-71): exact top-k search of the split's keys
`{subset}_dstore/keys.npy` over the train datastore (knn_search.KNNSearcher), written to `{subset}_dstore/neighbors.mmap.{k}`
(raw int64 [N_split, k], -1 = missing) -- the file the graph (--gcn-k) and the kNN-LM (--knnlm) read.  With --write-dists the
distances go to `{subset}_dstore/dists.{k}` (raw fp32 [N_split, k]; the reference drops them, :65-66), which
`eval_lm --knn-dists-file` reads as they are.

The datastore is either the PQ codes `train_dstore/quantized-keys.npy` decoded by the faiss `quantizer` file (--source pq: the
keys the graph LM sees) or the raw keys `train_dstore/keys.npy` (--source keys).  The search is exact over those vectors; it does
not reproduce the approximate results of the reference's IVF-PQ index.  Searching the train split finds every key as its own
nearest neighbour, as the reference does (--invalid-neighbor-context filters it).

Under torchrun (RANK / WORLD_SIZE) every rank searches a contiguous range of the queries and writes its rows into the shared
files; no collective is needed.

    python -m gnnlm_b200.find_knn --data-dir DATA --subset valid --k 1024 --metric l2 --source pq [--quantizer PATH] [--write-dists]
"""
import argparse
import json
import os

import numpy as np
import torch

from .dataset import dstore_path, feature_path, neighbor_path, quantized_feature_path
from .eval_lm import shard_range
from .knn_search import KNNSearcher, PQKeys, RawKeys


def dists_path(data_dir, subset, k):
    return os.path.join(dstore_path(data_dir, subset), f"dists.{k}")


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description="exact kNN search of a split's keys over the train datastore (knn/find_knn.py)")
    p.add_argument("--data-dir", type=str, required=True, help="path to binary dataset directory")
    p.add_argument("--subset", type=str, default="train", choices=["train", "valid", "test"], help="the split whose keys are the queries")
    p.add_argument("--k", type=int, default=1024, help="neighbours per query (<= 2048)")
    p.add_argument("--metric", type=str, default="l2", choices=["l2", "ip"])
    p.add_argument("--source", type=str, default="pq", choices=["pq", "keys"],
                   help="pq: the PQ-decoded keys (quantized-keys.npy + quantizer); keys: the raw keys.npy")
    p.add_argument("--quantizer", type=str, default=None, help="faiss quantizer file (default DATA/quantizer)")
    p.add_argument("--write-dists", action="store_true", help="also write {subset}_dstore/dists.{k} (raw fp32)")
    p.add_argument("--query-batch", type=int, default=16384, help="queries per search batch")
    return p


def _info(data_dir, subset):
    with open(os.path.join(dstore_path(data_dir, subset), "info.json")) as f:
        info = json.load(f)
    dt = np.float16 if info.get("dstore_fp16", False) else np.float32
    return int(info["dstore_size"]), int(info["hidden_size"]), dt


def _open_shared(path, dtype, shape):
    """The output memmap, created by whichever rank comes first; every rank sets the same size, which never drops written rows."""
    fd = os.open(path, os.O_RDWR | os.O_CREAT, 0o644)
    try:
        os.ftruncate(fd, int(np.prod(shape)) * np.dtype(dtype).itemsize)
    finally:
        os.close(fd)
    return np.memmap(path, dtype=dtype, mode="r+", shape=shape)


@torch.no_grad()
def find_knn(data_dir: str, subset: str = "train", k: int = 1024, metric: str = "l2", source: str = "pq", quantizer=None,
             write_dists: bool = False, query_batch: int = 16384, rank: int = 0, world: int = 1, device="cuda", log=print,
             **searcher_kw) -> dict:
    """Writes rows [lo, hi) = shard_range(N_split, rank, world) of the neighbour (and distance) file; returns the paths, the row
    range and the number of overflow re-runs.  `quantizer`: a file path or a TorchPQCodec (default DATA/quantizer)."""
    from .formats import read_faiss_quantizer
    from .pq_codec import TorchPQCodec
    from .quantize_features import quantizer_path
    n, d, qdt = _info(data_dir, subset)
    queries = np.memmap(feature_path(data_dir, subset), dtype=qdt, mode="r", shape=(n, d)) if n else np.zeros((0, d), qdt)
    if source == "pq":
        if quantizer is None or isinstance(quantizer, str):
            cen, A, b = read_faiss_quantizer(quantizer or quantizer_path(data_dir))
            quantizer = TorchPQCodec(centroids=cen, A=A, b=b)
        src = PQKeys(np.load(quantized_feature_path(data_dir, "train"), mmap_mode="r"), quantizer)
    elif source == "keys":
        n_d, d_d, kdt = _info(data_dir, "train")
        src = RawKeys(np.memmap(feature_path(data_dir, "train"), dtype=kdt, mode="r", shape=(n_d, d_d)))
    else:
        raise ValueError(f"unknown source {source!r}")
    searcher = KNNSearcher(src, metric, k, query_batch=query_batch, device=device, **searcher_kw)
    lo, hi = shard_range(n, rank, world)
    out = {"neighbors": neighbor_path(data_dir, subset, k), "dists": dists_path(data_dir, subset, k) if write_dists else None,
           "rows": (lo, hi)}
    ids_mm = _open_shared(out["neighbors"], np.int64, (n, k)) if n else None
    dists_mm = _open_shared(out["dists"], np.float32, (n, k)) if (n and write_dists) else None
    for a in range(lo, hi, query_batch):
        b = min(hi, a + query_batch)
        dists, ids = searcher.search(torch.from_numpy(np.asarray(queries[a:b], dtype=np.float32)))
        ids_mm[a:b] = ids.cpu().numpy()
        if dists_mm is not None:
            dists_mm[a:b] = dists.cpu().numpy()
    for mm in (ids_mm, dists_mm):
        if mm is not None:
            mm.flush()
    out["reruns"] = searcher.reruns
    log(f"{subset}: rows [{lo}, {hi}) of {n}, k = {k}, {metric} over {src.n} {source} keys -> {out['neighbors']}")
    return out


def main(argv=None, device=None, log=print):
    args = build_parser().parse_args(argv)
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if device is None:
        device = f"cuda:{int(os.environ.get('LOCAL_RANK', 0))}"
    if torch.device(device).type == "cuda":
        torch.cuda.set_device(device)           # every rank launches on its own GPU's streams
    return find_knn(args.data_dir, args.subset, args.k, args.metric, args.source, args.quantizer, args.write_dists,
                    args.query_batch, rank, world, device, log)


if __name__ == "__main__":
    main()
