"""Drop-in mirror of the reference's metric plugin, ``CustomCalculator``
(``/root/reference/main/engine/accuracy_calculator.py:16-403``), running on the B200 kernels.

Same constructor keywords, method names, argument meaning, return types (Python floats / tensors) and metric
discovery by the ``calculate_`` prefix, so ``eng.evaluate`` / ``compute_batch_map`` / ``studies/measure_random_baseline.py``
read unchanged.  pytorch-metric-learning (whose ``AccuracyCalculator`` the reference subclasses) is not a dependency:
the small part of its interface that the reference relies on is restated in :class:`AccuracyCalculator` below.

Differences a reader of the reference should know (all documented in DESIGN.md §6):

* ranking ties are broken by database index (the reference's ``torch.argsort`` leaves them implementation-defined);
* AP is accumulated in float64 from float32 quotients (the reference uses a float32 mean);
* codes must be exactly +-1 — ``sign(0) == 0`` or raw logits raise ``ValueError`` unless ``on_nonbinary='sign'``
  (binarise with ``x > 0``) or ``on_nonbinary='real'``.  ``'real'`` computes what the reference computes for any real
  codes: ``calc_hamming_dist``, ``calculate_maphashing`` and ``maphashing_details`` rank them by the float32
  ``0.5 * (B - q @ r.T)`` (summed in dimension order; ties by index, NaN last).  All-+-1 codes still take the packed
  path, so their results are byte-identical to the default; ``pr_rc_hashing`` raises ``NotImplementedError`` for
  real codes;
* everything runs on the current CUDA device whatever ``device`` says; returned tensors are moved to ``self.device``.
"""
import logging

import torch

from .. import _cabi
from . import hamming as H
from .get_knn import get_knn

LOGGER = logging.getLogger("RETRIEVAL")

EQUALITY = torch.eq


# ------------------------------------------------------------------ PML helpers the reference imports (:3-7)
def get_label_match_counts(query_labels, reference_labels, label_comparison_fn):
    """(unique query label rows, number of references each one matches)."""
    unique_query_labels = torch.unique(query_labels, dim=0)
    counts = torch.empty(len(unique_query_labels), dtype=torch.long, device=query_labels.device)
    step = 256
    for s in range(0, len(unique_query_labels), step):
        block = unique_query_labels[s:s + step]
        if label_comparison_fn is EQUALITY:
            comparison = block[:, None] == reference_labels
            while comparison.dim() > 2:
                comparison = comparison.all(dim=-1)
        else:
            comparison = label_comparison_fn(block, reference_labels)
        counts[s:s + step] = comparison.sum(dim=1)
    return unique_query_labels, counts


def get_lone_query_labels(query_labels, label_counts, ref_includes_query, label_comparison_fn):
    """Labels that cannot be retrieved at all, and the mask of queries that can."""
    unique_labels, match_counts = label_counts
    if ref_includes_query:
        # a query that is in the reference set always matches itself once
        lone_condition = match_counts - 1 <= 0
    else:
        lone_condition = match_counts == 0
    lone_query_labels = unique_labels[lone_condition]
    if len(lone_query_labels) > 0:
        comparison = query_labels[:, None] == lone_query_labels
        while comparison.dim() > 2:
            comparison = comparison.all(dim=-1)
        not_lone_query_mask = ~comparison.any(dim=1)
    else:
        not_lone_query_mask = torch.ones(query_labels.shape[0], dtype=torch.bool, device=query_labels.device)
    return lone_query_labels, not_lone_query_mask


class AccuracyCalculator:
    """The slice of pytorch-metric-learning's ``AccuracyCalculator`` interface that the reference depends on."""

    function_keyword = "calculate_"

    def __init__(self, include=(), exclude=(), avg_of_avgs=False, return_per_class=False, k=None, label_comparison_fn=None,
                 device=None, knn_func=None, kmeans_func=None):
        if not (isinstance(k, int) and k > 0) and k not in (None, "max_bin_count"):
            raise ValueError("k must be a positive integer, None, or 'max_bin_count'")
        self.k = k
        self.avg_of_avgs = avg_of_avgs
        self.return_per_class = return_per_class
        self.device = torch.device("cuda" if torch.cuda.is_available() else "cpu") if device is None else torch.device(device)
        function_names = [x for x in dir(self) if x.startswith(self.function_keyword)]
        metrics = [x.replace(self.function_keyword, "", 1) for x in function_names]
        self.original_function_dict = {x: getattr(self, y) for x, y in zip(metrics, function_names)}
        self.check_primary_metrics(include, exclude)
        self.original_function_dict = self.get_function_dict(include, exclude)
        self.curr_function_dict = self.get_function_dict()

    def get_function_dict(self, include=(), exclude=()):
        if len(include) == 0:
            include = list(self.original_function_dict.keys())
        included = [k for k in include if k not in exclude]
        return {k: v for k, v in self.original_function_dict.items() if k in included}

    def get_curr_metrics(self):
        return [k for k in self.curr_function_dict.keys()]

    def requires_clustering(self):
        return ["NMI", "AMI"]

    def requires_knn(self):
        return ["precision_at_1", "mean_average_precision", "mean_average_precision_at_r", "r_precision",
                "mean_reciprocal_rank"]

    def check_primary_metrics(self, include=(), exclude=()):
        primary = list(self.original_function_dict.keys())
        for name, seq in (("include", include), ("exclude", exclude)):
            if not isinstance(seq, (list, tuple)):
                raise TypeError(f"Arguments must be of type tuple, not {type(seq)}.")
            bad = [x for x in seq if x not in primary]
            if bad:
                raise ValueError(f"{name} argument contains names that are not in the valid metric list: {bad}. "
                                 f"Valid metrics are: {primary}")

    def description(self):
        return "avg_of_avgs" if self.avg_of_avgs else ""

    def determine_k(self, bin_counts, num_reference_embeddings, embeddings_come_from_same_source):
        self_count = int(embeddings_come_from_same_source)
        if self.k == "max_bin_count":
            return int(torch.max(bin_counts).item()) - self_count
        if self.k is None:
            return num_reference_embeddings - self_count
        return self.k

    def _get_accuracy(self, function_dict, **kwargs):
        return {k: v(**kwargs) for k, v in function_dict.items()}

    # --- PML's knn metrics, flat (no avg_of_avgs / per-class), on the knn list
    def _knn_relevance(self, knn_labels, query_labels, label_comparison_fn, **kwargs):
        return label_comparison_fn(query_labels[:, None], knn_labels)

    def calculate_precision_at_1(self, knn_labels, query_labels, not_lone_query_mask, label_comparison_fn, **kwargs):
        rel = self._knn_relevance(knn_labels[:, :1], query_labels, label_comparison_fn)[not_lone_query_mask]
        return rel.float().mean().item() if rel.numel() else 0.0

    def calculate_mean_reciprocal_rank(self, knn_labels, query_labels, not_lone_query_mask, label_comparison_fn, **kwargs):
        rel = self._knn_relevance(knn_labels, query_labels, label_comparison_fn)[not_lone_query_mask]
        if not rel.numel():
            return 0.0
        pos = torch.arange(1, rel.shape[1] + 1, device=rel.device).float()
        first = torch.where(rel, pos, torch.full_like(pos, float("inf"))).min(dim=1).values
        return (1.0 / first).mean().item()

    def calculate_mean_average_precision(self, knn_labels, query_labels, not_lone_query_mask, label_comparison_fn, **kwargs):
        rel = self._knn_relevance(knn_labels, query_labels, label_comparison_fn)[not_lone_query_mask].float()
        if not rel.numel():
            return 0.0
        pos = torch.arange(1, rel.shape[1] + 1, device=rel.device).float()
        prec = torch.cumsum(rel, dim=1) / pos * rel
        n_rel = rel.sum(dim=1)
        ap = torch.where(n_rel > 0, prec.sum(dim=1) / n_rel.clamp(min=1), torch.zeros_like(n_rel))
        return ap.mean().item()

    def _max_possible(self, query_labels, label_counts, embeddings_come_from_same_source, label_comparison_fn):
        uniq, counts = label_counts
        match = query_labels[:, None] == uniq
        while match.dim() > 2:
            match = match.all(dim=-1)
        per_query = (match.long() * counts[None, :]).sum(dim=1)
        return per_query - int(embeddings_come_from_same_source)

    def calculate_r_precision(self, knn_labels, query_labels, not_lone_query_mask, label_counts,
                              embeddings_come_from_same_source, label_comparison_fn, **kwargs):
        r = self._max_possible(query_labels, label_counts, embeddings_come_from_same_source, label_comparison_fn)
        rel = self._knn_relevance(knn_labels, query_labels, label_comparison_fn).float()
        pos = torch.arange(1, rel.shape[1] + 1, device=rel.device)
        within = (pos[None, :] <= r[:, None]).float()
        val = (rel * within).sum(dim=1) / r.clamp(min=1).float()
        val = val[not_lone_query_mask]
        return val.mean().item() if val.numel() else 0.0

    def calculate_mean_average_precision_at_r(self, knn_labels, query_labels, not_lone_query_mask, label_counts,
                                              embeddings_come_from_same_source, label_comparison_fn, **kwargs):
        r = self._max_possible(query_labels, label_counts, embeddings_come_from_same_source, label_comparison_fn)
        rel = self._knn_relevance(knn_labels, query_labels, label_comparison_fn).float()
        pos = torch.arange(1, rel.shape[1] + 1, device=rel.device)
        within = (pos[None, :] <= r[:, None]).float()
        prec = torch.cumsum(rel * within, dim=1) / pos.float() * rel * within
        val = prec.sum(dim=1) / r.clamp(min=1).float()
        val = val[not_lone_query_mask]
        return val.mean().item() if val.numel() else 0.0

    def calculate_NMI(self, **kwargs):
        raise NotImplementedError("clustering metrics (NMI/AMI) are always excluded by the reference's evaluator")

    def calculate_AMI(self, **kwargs):
        raise NotImplementedError("clustering metrics (NMI/AMI) are always excluded by the reference's evaluator")


def _numpy_to_torch(x):
    return x if isinstance(x, torch.Tensor) else torch.as_tensor(x)


class CustomCalculator(AccuracyCalculator):

    def __init__(self, *args, with_faiss=True, distance_metric="l2", on_nonbinary="raise", **kwargs):
        super().__init__(*args, **kwargs)
        LOGGER.info(f"Initializing CustomCalculator with with_faiss={with_faiss} and distance_metric={distance_metric} "
                    f"device: {self.device}")
        self.with_faiss = with_faiss
        self.distance_metric = distance_metric
        self.num_top_k = kwargs.get("k", None)
        self.on_nonbinary = on_nonbinary
        self._pack_memo = None          # active only inside get_accuracy (see _memo_pack)

    # ---------------------------------------------------------------- packing
    # Packed forms are shared between the metrics of ONE get_accuracy call only (maphashing, bit balance, pr_rc_hashing
    # ... all see the same tensors there).  The memo is keyed by the tensor OBJECT and keeps it alive, so an address or
    # id reused by a later tensor can never hit; it is dropped when get_accuracy returns, so nothing survives between
    # evaluations (a data_ptr/_version key did: the caching allocator hands the next epoch's codes the same address).
    def _memo_pack(self, kind, t, make):
        memo = self._pack_memo
        if memo is None:
            return make(t)
        key = (kind, id(t))
        hit = memo.get(key)
        if hit is None or hit[0] is not t or hit[1] != t._version:
            hit = (t, t._version, make(t))
            memo[key] = hit
        return hit[2]

    def _packed_codes(self, t):
        return self._memo_pack("c", t, lambda x: H.pack_codes(x, on_nonbinary=self.on_nonbinary))

    def _packed_labels(self, t):
        return self._memo_pack("l", t, H.pack_labels)

    def _code_pair(self, query, reference):
        """Packed codes of both sides, or None when ``on_nonbinary='real'`` and either side is not all +-1: those codes
        are then ranked by the reference's float32 distance (``H.real_hamming_*``)."""
        qc = self._packed_codes(query)
        rc = None if qc is None else self._packed_codes(reference)
        return None if rc is None else (qc, rc)

    def _label_pair(self, query_labels, reference_labels):
        ql, rl = _numpy_to_torch(query_labels), _numpy_to_torch(reference_labels)
        two_d = ql.dim() > 1 and rl.dim() > 1 and ql.shape[-1] > 1
        if not two_d:
            ql, rl = ql.reshape(-1), rl.reshape(-1)
            if ql.dtype != rl.dtype:
                # `==` in the reference promotes; bit patterns only compare within one dtype
                common = torch.promote_types(ql.dtype, rl.dtype)
                if common.is_floating_point:
                    common = torch.float64
                ql, rl = ql.to(common), rl.to(common)
        return self._packed_labels(ql), self._packed_labels(rl)

    def _knn_rowwise(self, query_labels, knn_labels):
        """Relevance of every query's OWN knn labels, ``[Q, k]`` bool: what the reference writes as
        ``label_comparison_fn(query_labels[:, None], knn_labels)`` (accuracy_calculator.py:133,146,160) — equality for 1-D
        labels (``[Q, 1]`` x ``[Q, k]``, also for k = 1), overlap for multi-hot ones (``[Q, 1, L]`` x ``[Q, k, L]``)."""
        ql, kl = _numpy_to_torch(query_labels), _numpy_to_torch(knn_labels)
        ql = ql.to(kl.device)
        if ql.dim() == 2 and ql.shape[1] == 1 and kl.dim() == 2:
            ql = ql.reshape(-1)
        return self._rowwise_labels(ql[:, None], kl)

    @staticmethod
    def _rowwise_labels(ql, rl):
        """``query_labels[:, None]`` against knn labels: [Q, 1] x [Q, k] (1-D labels) or [Q, 1, L] x [Q, k, L] (multi-hot)."""
        if ql.dim() == 3 or rl.dim() == 3:
            return (ql.float() * rl.float()).sum(dim=-1) > 0
        return ql == rl

    # ---------------------------------------------------------------- reference API
    def label_comparison_fn(self, query_labels, reference_labels):
        """accuracy_calculator.py:31-37 — bool ``[q, N]`` (2-D x 2-D multi-hot: share a tag; 1-D: equal);
        3-D ``[q, 1, L]`` against ``[q, k, L]`` knn labels: row-wise overlap."""
        ql, rl = _numpy_to_torch(query_labels), _numpy_to_torch(reference_labels)
        if ql.dim() > 1 and rl.dim() > 1:
            if ql.dim() == 2 and rl.dim() == 2:
                if ql.shape[1] == 1 and rl.shape[1] != 1 and rl.shape[0] == ql.shape[0]:
                    # 1-D labels as query_labels[:, None] against their own knn labels [Q, k] (calculate_rpr / pr / map):
                    # row-wise equality, not the all-pairs [Q, Q*k] matrix (the reference's matmul raises here)
                    return self._rowwise_labels(ql.to(rl.device), rl)
                pq, pr = self._label_pair(ql, rl)
                return H.label_relevance(pq, pr).to(self.device)
            return self._rowwise_labels(ql.to(rl.device), rl)
        if ql.dim() == 1 and rl.dim() == 1:
            pq, pr = self._label_pair(ql, rl)
            return H.label_relevance(pq, pr).to(self.device)
        return ql.unsqueeze(1) == rl

    def calc_hamming_dist(self, qB, rB):
        """accuracy_calculator.py:183-186 — float32 ``[q, N]`` holding exact integers for +-1 codes (and, with
        ``on_nonbinary='real'``, the float32 ``0.5 * (B - q @ r.T)`` of any other codes)."""
        qB, rB = _numpy_to_torch(qB), _numpy_to_torch(rB)
        packed = self._code_pair(qB, rB)
        if packed is None:
            return H.real_hamming_dist(qB, rB, qB.shape[1]).to(self.device)
        return H.hamming_dist(*packed).to(self.device)

    def per_bit_balance(self, reference):
        """accuracy_calculator.py:188-194, float32 like the reference (the counts are exact integers)."""
        packed = H.pack_codes(_numpy_to_torch(reference), on_nonbinary="sign")       # (reference > 0): any real input
        ones = H.bit_counts(packed)
        frac_positive = ones.float() / float(max(packed.rows, 1))
        return (1.0 - 2.0 * (frac_positive - 0.5).abs()).to(self.device)

    def calculate_bit_balance(self, reference, **kwargs):
        return self.per_bit_balance(reference).mean().item()

    def calculate_worst_bit_balance(self, reference, **kwargs):
        return self.per_bit_balance(reference).min().item()

    def resolve_topk(self, topk, reference_labels, ref_includes_query=False):
        """accuracy_calculator.py:204-212."""
        while isinstance(topk, (tuple, list)):
            topk = topk[0] if len(topk) else None
        if isinstance(topk, str) and topk == "max_bin_count":
            rl = _numpy_to_torch(reference_labels)
            rl = rl.cuda() if not rl.is_cuda else rl
            _, bin_counts = get_label_match_counts(rl, rl, self._device_label_comparison)
            topk = bin_counts.max().item() - int(ref_includes_query)
        if topk is not None:
            topk = int(topk)
        return topk

    def _device_label_comparison(self, a, b):
        if a.dim() > 1 and b.dim() > 1 and a.shape[-1] > 1:
            return H.label_relevance(H.pack_labels(a), H.pack_labels(b))
        return H.label_relevance(H.pack_labels(a.reshape(-1)), H.pack_labels(b.reshape(-1)))

    def maphashing_details(self, query, query_labels, reference, reference_labels, topk=None, ref_includes_query=False):
        """``(map, ap[Q], tsum[Q])`` as device tensors — no host synchronisation."""
        topk = self.resolve_topk(topk, reference_labels, ref_includes_query)
        query, reference = _numpy_to_torch(query), _numpy_to_torch(reference)
        packed = self._code_pair(query, reference)
        ql, rl = self._label_pair(query_labels, reference_labels)
        if packed is None:
            return H.real_hamming_map(query, ql, reference, rl, topk)
        qc, rc = packed
        n = rc.rows
        if topk is not None and topk < 1:
            dev = qc.words.device
            return (torch.zeros((), dtype=torch.float64, device=dev), torch.zeros(qc.rows, dtype=torch.float64, device=dev),
                    torch.zeros(qc.rows, dtype=torch.int32, device=dev))
        return H.hamming_map(qc, ql, rc, rl, n if topk is None else topk)

    def calculate_maphashing(self, query, query_labels, reference, reference_labels, topk, ref_includes_query=False, **kwargs):
        """accuracy_calculator.py:203-231 — mean over ALL queries of AP@topk under Hamming ranking; Python float."""
        with _cabi.nvtx_range("b200/calculate_maphashing"):
            m, _, _ = self.maphashing_details(query, query_labels, reference, reference_labels, topk, ref_includes_query)
            return m.item()

    def calculate_map(self, query_labels, knn_labels, knn_distances, not_lone_query_mask, knn_indices=None,
                      reference_labels=None, **kwargs):
        """accuracy_calculator.py:156-167 — RetrievalMAP over the knn list (its order), mean over not-lone queries.
        Uses the ranked-AP kernel on the index list when ``get_accuracy`` supplies it."""
        if knn_indices is not None and reference_labels is not None:
            ql, rl = self._label_pair(query_labels, reference_labels)
            m, _, _ = H.ranked_ap(knn_indices, ql, rl, query_mask=not_lone_query_mask)
            return m.item()
        rel = self._knn_rowwise(query_labels, knn_labels).float()
        mask = _numpy_to_torch(not_lone_query_mask).bool().to(rel.device)
        rel = rel[mask]
        if not rel.numel():
            return 0.0
        pos = torch.arange(1, rel.shape[1] + 1, device=rel.device).double()
        rel = rel.double()
        n_rel = rel.sum(dim=1)
        ap = torch.where(n_rel > 0, (torch.cumsum(rel, dim=1) / pos * rel).sum(dim=1) / n_rel.clamp(min=1),
                         torch.zeros_like(n_rel))
        return ap.mean().item()

    def n_relevance_at_k(self, knn_labels, query_labels, k):
        r = self.label_comparison_fn(query_labels, knn_labels[:, :k])
        return r.float().sum(1)

    def recall_at_k(self, knn_labels, query_labels, k):
        recall = self.label_comparison_fn(query_labels, knn_labels[:, :k])
        return recall.any(1).float().mean().item()

    def calculate_rpr(self, query_labels, knn_labels, knn_distances, not_lone_query_mask, **kwargs):
        """R-precision over the knn list (torchmetrics RetrievalRPrecision): hits in the first R ranks / R, R = #hits."""
        rel = self._knn_rowwise(query_labels, knn_labels)[not_lone_query_mask].float()
        if not rel.numel():
            return 0.0
        r = rel.sum(dim=1)
        pos = torch.arange(1, rel.shape[1] + 1, device=rel.device)
        top = (rel * (pos[None, :] <= r[:, None]).float()).sum(dim=1)
        return torch.where(r > 0, top / r.clamp(min=1), torch.zeros_like(r)).mean().item()

    def calculate_pr(self, query_labels, knn_labels, knn_distances, not_lone_query_mask, **kwargs):
        rel = self._knn_rowwise(query_labels, knn_labels[:, :1])[not_lone_query_mask].float()
        return rel.mean().item() if rel.numel() else 0.0

    def calculate_pr_rc(self, **kwargs):
        raise NotImplementedError("pr_rc writes a CSV of a torchmetrics curve; it is excluded by every reference caller")

    def pr_rc_hashing_curves(self, query, query_labels, reference, reference_labels, not_lone_query_mask=None, chunk=256):
        """Mean precision / recall at every rank of the full Hamming ranking (accuracy_calculator.py:235-273) over the
        queries that are not lone and have at least one relevant row: ``(precision [N], recall [N], n_queries)`` as
        float64 device tensors.  Per chunk of queries: ranking = the (distance, index) order of ``b200_hamming_topk`` with
        k = N, relevance along it as a running hit count (``b200_ranked_cumhits``: packed label words gathered by the
        ranked index, warp ballot prefix), then one pass per rank over the chunk adds the float32 quotients the
        reference forms (``b200_curve_accumulate``).  No ``[Q, N]`` float matrix is materialised; ``chunk`` bounds the
        ``[chunk, N]`` uint32 lists."""
        packed = self._code_pair(query, reference)
        if packed is None:
            raise NotImplementedError("pr_rc_hashing ranks +-1 codes only: binarise real-valued codes (torch.sign) first")
        qc, rc = packed
        ql, rl = self._label_pair(query_labels, reference_labels)
        nq, n = qc.rows, rc.rows
        dev = qc.words.device
        keep = None if not_lone_query_mask is None else \
            _numpy_to_torch(not_lone_query_mask).to(device=dev, dtype=torch.uint8).contiguous()
        prec = torch.zeros(n, dtype=torch.float64, device=dev)
        rec = torch.zeros(n, dtype=torch.float64, device=dev)
        n_used = torch.zeros(1, dtype=torch.int32, device=dev)
        for q0 in range(0, nq if n else 0, chunk):
            q1 = min(nq, q0 + chunk)
            def rows(words):                       # packed buffers hold an even number of rows (16-byte granularity)
                part = words[q0:q1]
                return (torch.cat([part, torch.zeros_like(part[:1])]) if (q1 - q0) % 2 else part).contiguous()

            sub_c = H.PackedCodes(rows(qc.words), q1 - q0, qc.bits)
            sub_l = H.PackedLabels(rows(ql.words), q1 - q0, ql.lw, ql.mode)
            cum = H.ranked_cumhits(H.hamming_topk(sub_c, rc, n, raw=True), sub_l, rl)      # [c, N] running hits
            H.curve_accumulate(cum, prec, rec, n_used, None if keep is None else keep[q0:q1])
        used = int(n_used.item())
        if used:
            prec /= used
            rec /= used
        return prec, rec, used

    def calculate_pr_rc_hashing(self, query, query_labels, reference, reference_labels, not_lone_query_mask=None, **kwargs):
        """accuracy_calculator.py:235-273: writes the mean precision / recall curve over the full ranking to ``pr_rc.csv``
        (columns ``pr``, ``rc``) and returns 0, like the reference."""
        prec, rec, used = self.pr_rc_hashing_curves(query, query_labels, reference, reference_labels, not_lone_query_mask)
        if used:
            import pandas as pd

            pd.DataFrame({"pr": prec.float().cpu().numpy(), "rc": rec.float().cpu().numpy()}).to_csv("pr_rc.csv", index=False)
        return 0

    def requires_knn(self):
        return super().requires_knn() + ["recall_classic", "rpr", "pr", "pr_rc", "map"] + \
            [f"recall_at_{k}" for k in (1, 2, 4, 8, 10, 16, 20, 30, 32, 100, 1000)]

    def get_accuracy(self, query, query_labels, reference, reference_labels, embeddings_come_from_same_source, include=(),
                     exclude=(), return_indices=False):
        """accuracy_calculator.py:279-349."""
        _cabi.require_cuda()
        self._pack_memo = {}
        try:
            return self._get_accuracy_impl(query, query_labels, reference, reference_labels, embeddings_come_from_same_source,
                                           include, exclude, return_indices)
        finally:
            self._pack_memo = None

    def _get_accuracy_impl(self, query, query_labels, reference, reference_labels, embeddings_come_from_same_source, include,
                           exclude, return_indices):
        query, reference, query_labels, reference_labels = [
            _numpy_to_torch(x).cuda() for x in (query, reference, query_labels, reference_labels)]
        if query_labels.ndim == 1 or (query_labels.ndim == 2 and query_labels.size(1) == 1):
            query_labels = query_labels.view(-1)
            reference_labels = reference_labels.view(-1)
        self.curr_function_dict = self.get_function_dict(include, exclude)
        kwargs = {
            "query": query,
            "reference": reference,
            "query_labels": query_labels,
            "reference_labels": reference_labels,
            "embeddings_come_from_same_source": embeddings_come_from_same_source,
            "label_comparison_fn": self._device_label_fn,
            "ref_includes_query": embeddings_come_from_same_source,
            "topk": self.num_top_k,
        }
        knn_indices = None
        if any(x in self.requires_knn() for x in self.get_curr_metrics()):
            label_counts = get_label_match_counts(query_labels, reference_labels, self._device_label_comparison)
            lone_query_labels, not_lone_query_mask = get_lone_query_labels(
                query_labels, label_counts, embeddings_come_from_same_source, self._device_label_comparison)
            num_k = self.determine_k(label_counts[1], len(reference), embeddings_come_from_same_source)
            knn_indices, knn_distances = get_knn(reference, query, num_k, embeddings_come_from_same_source,
                                                 with_faiss=self.with_faiss, distance_metric=self.distance_metric)
            knn_labels = reference_labels[knn_indices]
            if not any(not_lone_query_mask):
                LOGGER.warning("None of the query labels are in the reference set.")
            kwargs["label_counts"] = label_counts
            kwargs["knn_labels"] = knn_labels
            kwargs["knn_distances"] = knn_distances
            kwargs["knn_indices"] = knn_indices
            kwargs["lone_query_labels"] = lone_query_labels
            kwargs["not_lone_query_mask"] = not_lone_query_mask
        if any(x in self.requires_clustering() for x in self.get_curr_metrics()):
            raise NotImplementedError("clustering metrics (NMI/AMI) are not available")
        if return_indices:
            return knn_indices, self._get_accuracy(self.curr_function_dict, **kwargs)
        return self._get_accuracy(self.curr_function_dict, **kwargs)

    def _device_label_fn(self, query_labels, reference_labels):
        """label_comparison_fn for tensors that already live on the device (used inside get_accuracy)."""
        q, r = query_labels, reference_labels
        if q.dim() == 3 or r.dim() == 3:                       # [Q, 1, L] against knn labels [Q, k, L]
            return (q.float() * r.float()).sum(dim=-1) > 0
        if q.dim() == 2 and r.dim() == 2 and q.shape[-1] > 1:  # multi-hot [q, L] x [N, L] -> [q, N]
            return self._device_label_comparison(q, r)
        if q.dim() == 2 and r.dim() == 2:                      # 1-D labels as [Q, 1] against knn labels [Q, k]
            return q == r
        if q.dim() == 1 and r.dim() == 1:                      # [q] x [N] -> [q, N]
            return self._device_label_comparison(q, r)
        return q.unsqueeze(1) == r


for _k in (1, 2, 4, 8, 10, 16, 20, 30, 32, 100, 1000):
    def _make(k):
        def calculate_recall(self, knn_labels, query_labels, label_comparison_fn=None, **kwargs):
            """accuracy_calculator.py:50-129 — fraction of queries with a relevant item in the first k ranks."""
            fn = label_comparison_fn or self.label_comparison_fn
            rel = fn(query_labels[:, None], knn_labels[:, :k])
            return rel.any(1).float().mean().item()
        calculate_recall.__name__ = f"calculate_recall_at_{k}"
        return calculate_recall
    setattr(CustomCalculator, f"calculate_recall_at_{_k}", _make(_k))


def get_accuracy_calculator(exclude_ranks=None, k=19581, with_AP=True, **kwargs):
    """accuracy_calculator.py:352-403 — same exclude-list assembly."""
    caller_exclude = kwargs.pop("exclude", [])
    exclude = list(caller_exclude)
    if with_AP:
        exclude.extend(["NMI", "AMI"])
    else:
        exclude.extend(["NMI", "AMI", "mean_average_precision", "mean_average_precision_at_r"])
    if exclude_ranks:
        for r in exclude_ranks:
            exclude.append(f"recall_at_{r}")
    base_exclude = [
        "mean_reciprocal_rank", "precision_at_1", "recall_at_1", "recall_at_1000", "recall_at_100",
        "recall_at_10", "recall_at_16", "recall_at_20", "recall_at_30", "recall_at_32",
        "recall_at_4", "recall_at_8", "recall_at_2", "recall_at_10", "pr_rc_hashing",
    ]
    exclude = sorted(set(exclude) | set(base_exclude))
    LOGGER.info(f"Excluding metrics: {exclude}")
    return CustomCalculator(exclude=exclude, k=k, **kwargs)
