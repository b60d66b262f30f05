"""Drop-in mirror of ``/root/reference/main/engine/get_knn.py`` on the B200 k-NN kernels.

``get_knn(references, queries, num_k, embeddings_come_from_same_source, with_faiss=True, distance_metric="l2")``
keeps the reference's signature and return order ``(indices, distances)``; ``with_faiss`` is accepted and ignored
(there is one implementation).  "hamming"/"cosine" rank by inner product, largest first; anything else by L2 distance,
smallest first — exactly the branches of ``get_knn_torch`` (:60-71) / ``get_knn_faiss`` (:27-57).  Ties go to the smaller
index (torch.topk / faiss leave the tie order unspecified).  -0.0 and +0.0 are the same score (reported as +0.0), and a
NaN score or distance ranks after every number for both metrics.  ±inf coordinates are supported for L2 only: the
inner-product scorer's bf16 hi/lo split turns them into NaN (inf - inf).
"""
import logging

import torch

from .. import _cabi

LOGGER = logging.getLogger("RETRIEVAL")
MAX_K = None          # no cap: lists longer than 4096 come out of the select kernel in passes of 4096 ranks


def knn_topk(references, queries, num_k, distance_metric="l2"):
    """``(distances float32 [Q, k], indices int64 [Q, k])`` on the device, like ``get_knn_torch``."""
    _cabi.require_cuda()
    refs = torch.as_tensor(references)
    qs = torch.as_tensor(queries)
    dev = refs.device if refs.is_cuda else (qs.device if qs.is_cuda else torch.device("cuda"))
    refs = refs.to(device=dev, dtype=torch.float32).contiguous()
    qs = qs.to(device=dev, dtype=torch.float32).contiguous()
    if refs.dim() != 2 or qs.dim() != 2 or refs.shape[1] != qs.shape[1]:
        raise ValueError("references [N, D] and queries [Q, D] must share D")
    n, d = int(refs.shape[0]), int(refs.shape[1])
    q = int(qs.shape[0])
    k = int(num_k)
    if k < 1 or k > n:
        # torch.topk: "selected index k out of range"
        raise RuntimeError(f"selected index k out of range (k={k}, references={n})")
    if distance_metric == "hamming" and d <= _cabi.MAX_CODE_BITS and q > 0:
        # +-1 codes: the inner-product order IS the (Hamming distance, index) order, <q, r> = B - 2 d — the counting-sort
        # evaluator ranks them exactly, for any k, without a Q x N float matrix.  Anything else (raw logits) ranks as floats.
        from . import hamming as H

        try:
            qc, rc = H.pack_codes(qs, on_nonbinary="raise"), H.pack_codes(refs, on_nonbinary="raise")
        except ValueError:
            qc = None
        if qc is not None:
            hidx, hdist = H.hamming_topk(qc, rc, k)
            return (float(d) - 2.0 * hdist.to(torch.float32)), hidx
    if d % 4:                                   # zero columns do not change inner products or distances
        pad = 4 - d % 4
        refs = torch.nn.functional.pad(refs, (0, pad))
        qs = torch.nn.functional.pad(qs, (0, pad))
        d += pad
    idx = torch.empty((q, k), dtype=torch.int64, device=dev)
    score = torch.empty((q, k), dtype=torch.float32, device=dev)
    if q == 0:
        return score, idx
    lib = _cabi.load()
    ws_bytes = lib.b200_knn_workspace_bytes(q, n, d, k)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    l2 = 0 if distance_metric in ("hamming", "cosine") else 1
    with torch.cuda.device(dev):
        rc = lib.b200_knn_topk(_cabi.ptr(refs), _cabi.ptr(qs), q, n, d, k, l2, _cabi.ptr(idx), _cabi.ptr(score), _cabi.ptr(ws),
                               ws_bytes, _cabi.stream_ptr())
    _cabi.check(rc, "b200_knn_topk")
    return score, idx


def get_knn_torch(references, queries, num_k, distance_metric="l2"):
    return knn_topk(references, queries, num_k, distance_metric)


def get_knn_faiss(references, queries, num_k, distance_metric="l2"):
    return knn_topk(references, queries, num_k, distance_metric)


def get_knn(references, queries, num_k, embeddings_come_from_same_source, with_faiss=True, distance_metric="l2"):
    num_k += embeddings_come_from_same_source
    LOGGER.info("running k-nn with k=%d" % num_k)
    LOGGER.info("embedding dimensionality is %d" % references.shape[-1])
    LOGGER.info(f"distance metric: {distance_metric}")
    with _cabi.nvtx_range("b200/get_knn"):
        distances, indices = knn_topk(references, queries, num_k, distance_metric)
    if embeddings_come_from_same_source:
        return indices[:, 1:], distances[:, 1:]
    return indices, distances


def select_topk(scores, k, largest=True):
    """Row-wise top-k of a float32 device matrix by ``b200_select_topk_f32``: ``(values [Q, k], columns int64 [Q, k])``,
    ties to the smaller column; -0.0 equals +0.0 and NaN ranks last for either ``largest``."""
    _cabi.require_cuda()
    s = torch.as_tensor(scores)
    if s.dim() != 2 or not s.is_cuda:
        raise ValueError("scores must be a 2-D CUDA tensor")
    q, n = int(s.shape[0]), int(s.shape[1])
    k = int(k)
    if k < 1 or k > n:
        raise RuntimeError(f"selected index k out of range (k={k}, columns={n})")
    ld = (n + 3) // 4 * 4
    buf = torch.zeros((q, ld), dtype=torch.float32, device=s.device)
    buf[:, :n] = s
    idx = torch.empty((q, k), dtype=torch.int64, device=s.device)
    val = torch.empty((q, k), dtype=torch.float32, device=s.device)
    with torch.cuda.device(s.device):
        rc = _cabi.load().b200_select_topk_f32(_cabi.ptr(buf), q, n, ld, k, int(bool(largest)), _cabi.ptr(idx), _cabi.ptr(val),
                                               _cabi.stream_ptr())
    _cabi.check(rc, "b200_select_topk_f32")
    return val, idx


def merge_knn_shards(shard_scores, shard_indices, num_k, distance_metric="l2"):
    """Global top-``num_k`` from per-shard lists (shards in ascending index order, each best-first with index ties
    ascending): ``shard_scores`` / ``shard_indices``: ``[n_shards, Q, k_s]``.  The concatenation shard by shard keeps equal
    scores in global index order, so one row-wise selection (ties to the smaller column) is the exact merge."""
    sc = torch.as_tensor(shard_scores)
    ix = torch.as_tensor(shard_indices)
    n_sh, q, ks = (int(v) for v in sc.shape)
    cat_s = sc.permute(1, 0, 2).reshape(q, n_sh * ks).contiguous().float()
    cat_i = ix.permute(1, 0, 2).reshape(q, n_sh * ks).contiguous()
    largest = distance_metric in ("hamming", "cosine")
    # negative index = padding of a short shard.  No score ranks after a real NaN, so the padding moves behind every real
    # entry (a stable sort keeps their order) and reads as NaN: ties go to the smaller column, so it is never chosen
    # while a real entry remains.
    order = torch.sort((cat_i < 0).to(torch.uint8), dim=1, stable=True).indices
    cat_s, cat_i = torch.gather(cat_s, 1, order), torch.gather(cat_i, 1, order)
    cat_s = cat_s.masked_fill(cat_i < 0, float("nan"))
    val, col = select_topk(cat_s, num_k, largest)
    return torch.gather(cat_i, 1, col), val


def get_knn_sharded(references_shard, queries, num_k, index_base, group=None, distance_metric="l2"):
    """``get_knn`` for a database split over the ranks of ``group`` in contiguous index ranges (the reference's faiss
    ``index_cpu_to_all_gpus(shards=True)``, get_knn.py:41-44): every rank ranks the (replicated) queries against ITS rows,
    the per-shard ``(score, global index)`` lists are all-gathered over NCCL and merged on every rank.
    Returns ``(indices, distances)`` like ``get_knn``; identical on all ranks."""
    import torch.distributed as dist

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    refs = torch.as_tensor(references_shard)
    n_local = int(refs.shape[0])
    k_local = min(int(num_k), n_local)
    q = int(torch.as_tensor(queries).shape[0])
    dev = refs.device if refs.is_cuda else torch.device("cuda", torch.cuda.current_device())
    sc = torch.zeros((q, int(num_k)), dtype=torch.float32, device=dev)
    ix = torch.full((q, int(num_k)), -1, dtype=torch.int64, device=dev)
    if k_local > 0:
        s, i = knn_topk(refs, queries, k_local, distance_metric)
        sc[:, :k_local], ix[:, :k_local] = s, i + int(index_base)
    if world == 1:
        return ix, sc
    all_s = torch.empty((world,) + tuple(sc.shape), dtype=sc.dtype, device=dev)
    all_i = torch.empty((world,) + tuple(ix.shape), dtype=ix.dtype, device=dev)
    dist.all_gather_into_tensor(all_s, sc, group=group)
    dist.all_gather_into_tensor(all_i, ix, group=group)
    return merge_knn_shards(all_s, all_i, int(num_k), distance_metric)
