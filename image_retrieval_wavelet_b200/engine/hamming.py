"""Functional layer over the C-ABI Hamming evaluator (device tensors in, device tensors out).

What it replaces in the reference: the per-query Python loop of ``CustomCalculator.calculate_maphashing``
(``/root/reference/main/engine/accuracy_calculator.py:203-231``) together with ``calc_hamming_dist`` (:183-186),
``label_comparison_fn`` (:31-37) and ``per_bit_balance`` (:188-194).  PyTorch only provides device memory and the
stream; all arithmetic runs in ``libb200ret.so``.
"""
import ctypes
from dataclasses import dataclass

import torch

from .. import _cabi


@dataclass
class PackedCodes:
    """Bit-packed +-1 codes: ``words`` is uint64-as-int64 ``[rows_padded, CW]`` on the device."""
    words: torch.Tensor
    rows: int
    bits: int

    @property
    def cw(self):
        return _cabi.code_words(self.bits)


@dataclass
class PackedLabels:
    words: torch.Tensor
    rows: int
    lw: int
    mode: int          # _cabi.LABELS_OVERLAP / LABELS_EQUAL


def _as_cuda(x, device):
    t = torch.as_tensor(x)
    if not t.is_cuda:
        t = t.to(device if device is not None else "cuda", non_blocking=True)
    return t


def pack_codes(codes, device=None, on_nonbinary="raise"):
    """float +-1 codes ``[N, B]`` -> :class:`PackedCodes`.

    Entries that are not exactly +1/-1 (``sign(0) == 0``, raw logits, NaN) have no Hamming distance in the reference's
    sense (its ``0.5 * (B - q @ r.T)`` turns fractional); ``on_nonbinary='raise'`` (default) rejects them with
    ValueError, ``'sign'`` binarises with ``x > 0`` first, and ``'real'`` returns None for them (and for codes wider
    than the packed format), so that the caller ranks the codes as floats (:func:`real_hamming_map`).
    """
    _cabi.require_cuda()
    t = _as_cuda(codes, device)
    if t.dim() != 2:
        raise ValueError("codes must be [N, B]")
    n, b = int(t.shape[0]), int(t.shape[1])
    if b < 1:
        raise ValueError("codes need at least one bit")
    if b > _cabi.MAX_CODE_BITS:
        if on_nonbinary == "real":
            return None
        raise NotImplementedError(f"codes wider than {_cabi.MAX_CODE_BITS} bits are not supported")
    t = t.to(torch.float32).contiguous()
    cw = _cabi.code_words(b)
    padded = (n + 1) // 2 * 2
    words = torch.empty((padded, cw), dtype=torch.int64, device=t.device)
    bad = torch.zeros(1, dtype=torch.int32, device=t.device)
    if n:
        with torch.cuda.device(t.device):
            rc = _cabi.load().b200_pack_codes(_cabi.ptr(t), n, b, _cabi.ptr(words), _cabi.ptr(bad), _cabi.stream_ptr())
        _cabi.check(rc, "b200_pack_codes")
        if on_nonbinary in ("raise", "real"):
            nbad = int(bad.item())
            if nbad and on_nonbinary == "real":
                return None
            if nbad:
                raise ValueError(f"{nbad} code entries are not +-1: Hamming ranking is undefined for them "
                                 "(binarise with torch.sign and resolve zeros, or pass on_nonbinary='sign' or 'real')")
    return PackedCodes(words, n, b)


def pack_labels_unchecked(labels, device=None):
    """:func:`pack_labels` without the validity read-back (no host synchronisation): for callers that already know their
    labels are multi-hot 0/1, e.g. a benchmark loop or a second pass over the same tensors."""
    return pack_labels(labels, device, validate=False)


def pack_labels(labels, device=None, validate=True):
    """Multi-hot ``[N, L]`` (0/1) or 1-D labels -> :class:`PackedLabels` (overlap / equality relevance)."""
    _cabi.require_cuda()
    t = _as_cuda(labels, device)
    lib = _cabi.load()
    if t.dim() == 2 and t.shape[1] > 1:
        n, l = int(t.shape[0]), int(t.shape[1])
        if l > _cabi.MAX_LABEL_BITS:
            raise NotImplementedError(f"more than {_cabi.MAX_LABEL_BITS} label columns are not supported")
        t = t.to(torch.float32).contiguous()
        lw = _cabi.label_words(l)
        words = torch.empty(((n + 1) // 2 * 2, lw), dtype=torch.int64, device=t.device)
        bad = torch.zeros(1, dtype=torch.int32, device=t.device)
        if n:
            with torch.cuda.device(t.device):
                rc = lib.b200_pack_labels(_cabi.ptr(t), n, l, _cabi.ptr(words), _cabi.ptr(bad), _cabi.stream_ptr())
            _cabi.check(rc, "b200_pack_labels")
            nbad = int(bad.item()) if validate else 0
            if nbad:
                raise ValueError(f"{nbad} label entries are neither 0 nor 1: only multi-hot label matrices can be bit-packed")
        return PackedLabels(words, n, lw, _cabi.LABELS_OVERLAP)
    t = t.reshape(-1)
    n = int(t.shape[0])
    if not t.dtype.is_floating_point:
        is_int, t = 1, t.to(torch.int64).contiguous()
    elif t.dtype == torch.float64:
        is_int, t = 2, t.contiguous()                       # no float32 round trip: ids above 2^24 stay distinct
    else:
        is_int, t = 0, t.to(torch.float32).contiguous()
    words = torch.empty(((n + 1) // 2 * 2, 1), dtype=torch.int64, device=t.device)
    bad = torch.zeros(1, dtype=torch.int32, device=t.device)
    if n:
        with torch.cuda.device(t.device):
            rc = lib.b200_pack_labels_scalar(_cabi.ptr(t), int(is_int), n, _cabi.ptr(words), _cabi.ptr(bad), _cabi.stream_ptr())
        _cabi.check(rc, "b200_pack_labels_scalar")
        if validate and int(bad.item()):
            raise ValueError("NaN labels cannot be compared for equality")
    return PackedLabels(words, n, 1, _cabi.LABELS_EQUAL)


def bit_counts(packed):
    """ones[b] = number of rows with bit b set (int64 ``[B]`` on the device)."""
    ones = torch.zeros(packed.bits, dtype=torch.int32, device=packed.words.device)
    with torch.cuda.device(ones.device):
        rc = _cabi.load().b200_bit_counts(_cabi.ptr(packed.words), packed.rows, packed.bits, _cabi.ptr(ones), _cabi.stream_ptr())
    _cabi.check(rc, "b200_bit_counts")
    return ones.to(torch.int64)


def hamming_dist(qc, dc):
    """Dense Hamming distances, float32 ``[Q, N]`` (what ``calc_hamming_dist`` returns for +-1 codes)."""
    if qc.bits != dc.bits:
        raise ValueError("code widths differ")
    out = torch.empty((qc.rows, dc.rows), dtype=torch.float32, device=qc.words.device)
    with torch.cuda.device(out.device):
        rc = _cabi.load().b200_hamming_dist(_cabi.ptr(qc.words), _cabi.ptr(dc.words), qc.rows, dc.rows, qc.bits, _cabi.ptr(out),
                                            _cabi.stream_ptr())
    _cabi.check(rc, "b200_hamming_dist")
    return out


def label_relevance(ql, dl):
    """Dense relevance matrix, bool ``[Q, N]`` (``label_comparison_fn``)."""
    if ql.mode != dl.mode or ql.lw != dl.lw:
        raise ValueError("query and database labels must be packed the same way")
    out = torch.empty((ql.rows, dl.rows), dtype=torch.uint8, device=ql.words.device)
    with torch.cuda.device(out.device):
        rc = _cabi.load().b200_label_relevance(_cabi.ptr(ql.words), _cabi.ptr(dl.words), ql.rows, dl.rows, ql.lw, ql.mode,
                                               _cabi.ptr(out), _cabi.stream_ptr())
    _cabi.check(rc, "b200_label_relevance")
    return out.bool()


class MapWorkspace:
    """Plan + scratch for one (Q, N, B, labels, k) problem; reusable across calls with the same shape."""

    def __init__(self, q, n, n_total, bits, lw, mode, k, device):
        self.plan = _cabi.MapPlan()
        k_eff = n_total if k is None else int(k)
        if k_eff < 1:
            raise ValueError("topk must be >= 1")
        rc = _cabi.load().b200_map_plan_init(ctypes.byref(self.plan), q, n, n_total, bits, lw, mode, min(k_eff, max(n_total, 1)))
        _cabi.check(rc, "b200_map_plan_init")
        self.buf = torch.empty(self.plan.workspace_bytes, dtype=torch.uint8, device=device)
        self.key = (q, n, n_total, bits, lw, mode, int(self.plan.k))

    def view(self, offset, dtype, count):
        size = torch.empty((), dtype=dtype).element_size()
        return self.buf[offset:offset + count * size].view(dtype)


def select_status(ws):
    """Diagnostics of the select pipeline of the last ``hamming_map`` / ``hamming_topk`` on ``ws`` (a
    :class:`MapWorkspace`): ``None`` when the plan does not use it, else a dict (synchronises)."""
    if not ws.plan.select:
        return None
    out = (ctypes.c_uint32 * 4)()
    with torch.cuda.device(ws.buf.device):
        rc = _cabi.load().b200_map_select_status(ctypes.byref(ws.plan), _cabi.ptr(ws.buf), out, _cabi.stream_ptr())
    _cabi.check(rc, "b200_map_select_status")
    return {"pool_chunks_used": int(out[0]), "fell_back": bool(out[1]), "queries_redone": int(out[2]),
            "estimated_candidates_per_query": int(out[3]), "pool_chunks": int(ws.plan.sel_pool_chunks),
            "chunk": int(ws.plan.sel_chunk), "segments": int(ws.plan.sel_S), "sample_stride": int(ws.plan.sel_stride)}


def _check_pair(qc, ql, dc, dl):
    if qc.bits != dc.bits:
        raise ValueError(f"query codes have {qc.bits} bits, database codes {dc.bits}")
    if ql.mode != dl.mode or ql.lw != dl.lw:
        raise ValueError("query and database labels must both be multi-hot with the same width, or both 1-D")
    if ql.rows != qc.rows or dl.rows != dc.rows:
        raise ValueError("codes and labels must have the same number of rows")


def hamming_map(qc, ql, dc, dl, topk=None, workspace=None, return_workspace=False):
    """mAP@topk of packed queries against a packed database on one GPU.

    Returns ``(map, ap, tsum)``: 0-dim float64, float64 ``[Q]``, int32 ``[Q]`` device tensors (no host sync).
    """
    _check_pair(qc, ql, dc, dl)
    dev = qc.words.device
    q, n = qc.rows, dc.rows
    if q == 0:
        raise ValueError("no queries")
    ap = torch.zeros(q, dtype=torch.float64, device=dev)
    tsum = torch.zeros(q, dtype=torch.int32, device=dev)
    m = torch.zeros((), dtype=torch.float64, device=dev)
    if n == 0:
        return (m, ap, tsum, None) if return_workspace else (m, ap, tsum)
    k = n if topk is None else int(topk)
    ws = workspace
    if ws is None or ws.key[:6] != (q, n, n, qc.bits, ql.lw, ql.mode) or ws.key[6] != min(k, n):
        ws = MapWorkspace(q, n, n, qc.bits, ql.lw, ql.mode, k, dev)
    with torch.cuda.device(dev):
        rc = _cabi.load().b200_hamming_map(ctypes.byref(ws.plan), _cabi.ptr(qc.words), _cabi.ptr(ql.words), _cabi.ptr(dc.words),
                                           _cabi.ptr(dl.words), _cabi.ptr(ws.buf), _cabi.ptr(ap), _cabi.ptr(tsum), _cabi.ptr(m),
                                           _cabi.stream_ptr())
    _cabi.check(rc, "b200_hamming_map")
    return (m, ap, tsum, ws) if return_workspace else (m, ap, tsum)


def hamming_topk(qc, dc, k, raw=False, return_workspace=False):
    """Ranked list by (Hamming distance, index): ``(idx int64 [Q, k], dist int32 [Q, k])`` device tensors;
    ``raw=True``: only the uint32 index list, as the int32 tensor the kernels wrote (no widening pass)."""
    if qc.bits != dc.bits:
        raise ValueError("code widths differ")
    dev = qc.words.device
    q, n = qc.rows, dc.rows
    k = min(int(k), n)
    if k < 1 or q < 1:
        if raw:
            return torch.zeros((q, 0), dtype=torch.int32, device=dev)
        return (torch.zeros((q, 0), dtype=torch.int64, device=dev), torch.zeros((q, 0), dtype=torch.int32, device=dev))
    ws = MapWorkspace(q, n, n, qc.bits, 1, _cabi.LABELS_EQUAL, k, dev)
    idx = torch.empty((q, k), dtype=torch.int32, device=dev)
    dist = None if raw else torch.empty((q, k), dtype=torch.int16, device=dev)
    with torch.cuda.device(dev):
        rc = _cabi.load().b200_hamming_topk(ctypes.byref(ws.plan), _cabi.ptr(qc.words), _cabi.ptr(dc.words), _cabi.ptr(ws.buf),
                                            _cabi.ptr(idx), None if raw else _cabi.ptr(dist), _cabi.stream_ptr())
    _cabi.check(rc, "b200_hamming_topk")
    if raw:
        return (idx, ws) if return_workspace else idx
    out = (idx.to(torch.int64) & 0xFFFFFFFF, dist.to(torch.int32) & 0xFFFF)
    return out + (ws,) if return_workspace else out


def radius_counts(qc, ql, dc, dl):
    """Per query and Hamming radius r = 0..B: ``(#rows, #relevant rows)`` with distance <= r, int64 ``[Q, B+1, 2]``.

    Stage A of the evaluator (one pass over the packed database) followed by a running sum over distance: what DSCH's
    ``pr_curve`` and ``get_precision_recall_by_Hamming_Radius`` (``/root/reference/main/engine/DSCH/_utils.py:467-492,
    577-594``) derive from ``[Q, N]`` float matrices."""
    _check_pair(qc, ql, dc, dl)
    dev = qc.words.device
    q, n = qc.rows, dc.rows
    if q == 0:
        raise ValueError("no queries")
    bins = qc.bits + 1
    if n == 0:
        return torch.zeros((q, bins, 2), dtype=torch.int64, device=dev)
    ws = MapWorkspace(q, n, n, qc.bits, ql.lw, ql.mode, n, dev)
    cum = torch.empty((bins, q, 2), dtype=torch.int32, device=dev)
    lib = _cabi.load()
    with torch.cuda.device(dev):
        rc = lib.b200_hamming_hist(ctypes.byref(ws.plan), _cabi.ptr(qc.words), _cabi.ptr(ql.words), _cabi.ptr(dc.words),
                                   _cabi.ptr(dl.words), _cabi.ptr(ws.buf), _cabi.stream_ptr())
        _cabi.check(rc, "b200_hamming_hist")
        rc = lib.b200_hamming_radius_counts(ctypes.byref(ws.plan), _cabi.ptr(ws.buf), _cabi.ptr(cum), _cabi.stream_ptr())
    _cabi.check(rc, "b200_hamming_radius_counts")
    return (cum.to(torch.int64) & 0xFFFFFFFF).permute(1, 0, 2).contiguous()


def ranked_cumhits(idx_u32, ql, dl):
    """Running hit count along ranked lists: ``idx_u32`` int32-viewed uint32 ``[Q, k]`` (as ``hamming_topk(raw=True)``
    returns it) -> int32-viewed uint32 ``[Q, k]``, ``cum[q, p]`` = relevant rows among the first ``p + 1`` ranks."""
    if ql.mode != dl.mode or ql.lw != dl.lw:
        raise ValueError("query and database labels must be packed the same way")
    if idx_u32.dtype != torch.int32 or idx_u32.dim() != 2:
        raise ValueError("idx must be the raw uint32 list [Q, k] (int32 storage)")
    idx_u32 = idx_u32.contiguous()
    q, k = int(idx_u32.shape[0]), int(idx_u32.shape[1])
    cum = torch.empty((q, k), dtype=torch.int32, device=idx_u32.device)
    if q and k:
        with torch.cuda.device(cum.device):
            rc = _cabi.load().b200_ranked_cumhits(_cabi.ptr(idx_u32), q, k, _cabi.ptr(ql.words), _cabi.ptr(dl.words), ql.lw,
                                                  ql.mode, _cabi.ptr(cum), _cabi.stream_ptr())
        _cabi.check(rc, "b200_ranked_cumhits")
    return cum


def curve_accumulate(cum, prec_sum, rec_sum, n_used, query_mask=None):
    """``prec_sum[p] += cum[q, p] / (p + 1)``, ``rec_sum[p] += cum[q, p] / cum[q, -1]`` (float32 quotients, float64 sums)
    over the selected queries that have a relevant row; ``n_used`` (int32 ``[1]``) counts them."""
    q, k = int(cum.shape[0]), int(cum.shape[1])
    if not q or not k:
        return
    mask = None if query_mask is None else query_mask.to(device=cum.device, dtype=torch.uint8).contiguous()
    with torch.cuda.device(cum.device):
        rc = _cabi.load().b200_curve_accumulate(_cabi.ptr(cum), q, k, _cabi.ptr(mask), _cabi.ptr(prec_sum), _cabi.ptr(rec_sum),
                                                _cabi.ptr(n_used), _cabi.stream_ptr())
    _cabi.check(rc, "b200_curve_accumulate")


def ranked_ap(idx, ql, dl, query_mask=None):
    """AP over ranked index lists ``[Q, k]`` (int64, negatives = padding): ``(map, ap [Q], hits [Q])``."""
    if ql.mode != dl.mode or ql.lw != dl.lw:
        raise ValueError("query and database labels must be packed the same way")
    dev = ql.words.device
    idx = idx.to(device=dev, dtype=torch.int64).contiguous()
    q, k = int(idx.shape[0]), int(idx.shape[1])
    ap = torch.zeros(q, dtype=torch.float64, device=dev)
    hits = torch.zeros(q, dtype=torch.int32, device=dev)
    m = torch.zeros((), dtype=torch.float64, device=dev)
    mask = None if query_mask is None else query_mask.to(device=dev, dtype=torch.uint8).contiguous()
    with torch.cuda.device(dev):
        rc = _cabi.load().b200_ranked_ap(_cabi.ptr(idx), 1, q, k, _cabi.ptr(ql.words), _cabi.ptr(dl.words), ql.lw, ql.mode,
                                         _cabi.ptr(mask), _cabi.ptr(ap), _cabi.ptr(hits), _cabi.ptr(m), _cabi.stream_ptr())
    _cabi.check(rc, "b200_ranked_ap")
    return m, ap, hits


# ------------------------------------------------------------------------------------------------ real-valued codes
REAL_CHUNK_BUDGET = 1 << 30     # bytes of per-chunk scratch of real_hamming_map: distances [chunk, ldS] + top-k lists


def _real_codes(x, device=None):
    """float32 ``[rows, D]`` on the device, columns zero-padded to D % 4 == 0 (zeros add nothing to the fmaf chain)."""
    t = _as_cuda(x, device)
    if t.dim() != 2:
        raise ValueError("codes must be [N, B]")
    t = t.to(torch.float32)
    if t.shape[1] % 4:
        t = torch.nn.functional.pad(t, (0, 4 - t.shape[1] % 4))
    return t.contiguous()


def _real_dist_into(qp, rp, nbits, out):
    """``b200_real_hamming_dist`` of padded codes into ``out`` ``[Q, ldS]`` (columns ``[0, N)`` written)."""
    with torch.cuda.device(out.device):
        rc = _cabi.load().b200_real_hamming_dist(_cabi.ptr(qp), _cabi.ptr(rp), int(qp.shape[0]), int(rp.shape[0]), int(qp.shape[1]),
                                                 int(nbits), _cabi.ptr(out), int(out.shape[1]), _cabi.stream_ptr())
    _cabi.check(rc, "b200_real_hamming_dist")


def real_hamming_dist(q, r, nbits):
    """``calc_hamming_dist`` of real-valued codes: float32 ``[Q, N]`` = ``0.5 * (nbits - q @ r.T)`` as the reference
    computes it in float32, with the inner product summed in dimension order (one fmaf chain, ``b200_real_hamming_dist``).
    Raw logits, zeros, +-inf and NaN are all accepted; +-1 codes give the exact integer Hamming distances."""
    _cabi.require_cuda()
    qp = _real_codes(q)
    rp = _real_codes(r, qp.device)
    if qp.shape[1] != rp.shape[1]:
        raise ValueError("code widths differ")
    n = int(rp.shape[0])
    ld = (n + 3) // 4 * 4
    out = torch.empty((int(qp.shape[0]), ld), dtype=torch.float32, device=qp.device)
    _real_dist_into(qp, rp, nbits, out)
    return out if ld == n else out[:, :n]


def real_hamming_map(q, ql, r, rl, k, chunk=None):
    """mAP@k of real-valued codes ``q`` ``[Q, B]`` against ``r`` ``[N, B]`` ranked by :func:`real_hamming_dist` (B = the
    code width), with packed labels ``ql`` / ``rl``: ``(map, ap [Q], hits [Q])`` device tensors like :func:`hamming_map`.

    The ranking is ascending (distance, database index), NaN last.  Per chunk of queries: the distances into one
    ``[chunk, ldS]`` buffer, ``b200_select_topk_f32`` (smallest first) on it, ``b200_ranked_ap`` on the index list; then one
    ``b200_mean_f64`` over all queries, so no result depends on ``chunk``.  ``chunk`` (default: all queries) is capped so
    that the per-chunk scratch stays within ``REAL_CHUNK_BUDGET``.  ``k``: None or > N means N; < 1 gives zeros."""
    _cabi.require_cuda()
    qp = _real_codes(q)
    rp = _real_codes(r, qp.device)
    nbits = int(torch.as_tensor(q).shape[1])
    if qp.shape[1] != rp.shape[1]:
        raise ValueError(f"query codes have {nbits} bits, database codes {int(torch.as_tensor(r).shape[1])}")
    if ql.mode != rl.mode or ql.lw != rl.lw:
        raise ValueError("query and database labels must both be multi-hot with the same width, or both 1-D")
    nq, n = int(qp.shape[0]), int(rp.shape[0])
    if ql.rows != nq or rl.rows != n:
        raise ValueError("codes and labels must have the same number of rows")
    if nq == 0:
        raise ValueError("no queries")
    dev = qp.device
    ap = torch.zeros(nq, dtype=torch.float64, device=dev)
    hits = torch.zeros(nq, dtype=torch.int32, device=dev)
    m = torch.zeros((), dtype=torch.float64, device=dev)
    k = n if k is None else min(int(k), n)
    if k < 1:
        return m, ap, hits
    ld = (n + 3) // 4 * 4
    per_row = 4 * ld + 12 * k                      # distances, int64 indices, float32 scores
    c = max(1, min(nq if chunk is None else int(chunk), REAL_CHUNK_BUDGET // per_row))
    dist = torch.empty((c, ld), dtype=torch.float32, device=dev)
    idx = torch.empty((c, k), dtype=torch.int64, device=dev)
    score = torch.empty((c, k), dtype=torch.float32, device=dev)
    lib = _cabi.load()
    with torch.cuda.device(dev):
        for q0 in range(0, nq, c):
            rows = min(c, nq - q0)
            _real_dist_into(qp[q0:q0 + rows], rp, nbits, dist)
            rc = lib.b200_select_topk_f32(_cabi.ptr(dist), rows, n, ld, k, 0, _cabi.ptr(idx), _cabi.ptr(score), _cabi.stream_ptr())
            _cabi.check(rc, "b200_select_topk_f32")
            rc = lib.b200_ranked_ap(_cabi.ptr(idx), 1, rows, k, _cabi.ptr(ql.words[q0:]), _cabi.ptr(rl.words), ql.lw, ql.mode,
                                    None, _cabi.ptr(ap[q0:]), _cabi.ptr(hits[q0:]), None, _cabi.stream_ptr())
            _cabi.check(rc, "b200_ranked_ap")
        rc = lib.b200_mean_f64(_cabi.ptr(ap), None, nq, _cabi.ptr(m), _cabi.stream_ptr())
    _cabi.check(rc, "b200_mean_f64")
    return m, ap, hits
