"""Candidate lists of the select pipeline (csrc/hamming_select.cu, stage A / A') decoded from the workspace and compared
with numpy: for every query and segment, exactly the rows within the query's bound (every row for a query redone with
the bound lifted), in row order, each entry ``row_in_segment | distance << 16 | relevant << 24``.  The rank kernel, the
retry round and the fallback rely on this layout, whichever form of the select pass wrote it."""
import numpy as np
import pytest
import torch

from simlib import multi_hot, pm1

pytestmark = pytest.mark.gpu

BOUND_INACTIVE, BOUND_RETRY = 1 << 30, 1 << 31
SENTINEL = 0xA5


def _run(monkeypatch, q, ql, r, rl, k, stride=None):
    """mAP@k through the select pipeline on a workspace pre-filled with a sentinel byte; returns (plan, workspace bytes,
    status)."""
    from image_retrieval_wavelet_b200.engine import hamming as H

    monkeypatch.setenv("B200_MAP_SELECT", "1")
    if stride:
        monkeypatch.setenv("B200_SEL_STRIDE", str(stride))
    qc, rc = H.pack_codes(torch.from_numpy(q)), H.pack_codes(torch.from_numpy(r))
    qlp, rlp = H.pack_labels(torch.from_numpy(ql)), H.pack_labels(torch.from_numpy(rl))
    ws = H.MapWorkspace(qc.rows, rc.rows, rc.rows, qc.bits, qlp.lw, qlp.mode, k, qc.words.device)
    ws.buf.fill_(SENTINEL)
    H.hamming_map(qc, qlp, rc, rlp, k, workspace=ws)
    st = H.select_status(ws)
    return ws.plan, ws.buf.cpu().numpy(), ws.buf.data_ptr(), st


def _view(buf, off, count, dtype=np.uint32):
    return buf[off:off + count * np.dtype(dtype).itemsize].view(dtype)


def _check_lists(plan, buf, q, ql, r, rl):
    nq, n, bits = q.shape[0], r.shape[0], q.shape[1]
    S, seg_len, ch, maxc, qpad = plan.sel_S, plan.sel_seg_len, plan.sel_chunk, plan.sel_maxc, plan.Qpad
    bound = _view(buf, plan.off_sel_bound, qpad)
    head = _view(buf, plan.off_sel_count, qpad * S * 2).reshape(qpad, S, 2)
    table = _view(buf, plan.off_sel_table, qpad * S * maxc).reshape(qpad, S, maxc)
    pool = _view(buf, plan.off_sel_pool, plan.sel_pool_chunks * ch)
    dist = ((bits - q.astype(np.int64) @ r.astype(np.int64).T) // 2).astype(np.uint32)
    if ql.ndim == 1:
        rel = (ql[:, None] == rl[None, :]).astype(np.uint32)
    else:
        rel = ((ql.astype(np.int64) @ rl.astype(np.int64).T) > 0).astype(np.uint32)
    sentinel_word = np.uint32(int.from_bytes(bytes([SENTINEL] * 4), "little"))
    chunks_seen = []
    multi_chunk = 0
    for qi in range(qpad):
        if qi >= nq:                                   # padding queries: no list head is written
            assert bound[qi] & BOUND_INACTIVE, (qi, hex(bound[qi]))
            assert (head[qi] == sentinel_word).all(), qi
            continue
        bw = int(bound[qi])
        within = np.ones(n, bool) if bw & BOUND_RETRY else dist[qi] <= (bw & 0xFFFF)
        for s in range(S):
            lo, hi = s * seg_len, min((s + 1) * seg_len, n)
            rows = np.nonzero(within[lo:hi])[0].astype(np.uint32)
            want = rows | (dist[qi, lo:hi][rows] << 16) | (rel[qi, lo:hi][rows] << 24)
            cnt, first = int(head[qi, s, 0]), int(head[qi, s, 1])
            assert cnt == len(want), (qi, s, cnt, len(want), hex(bw))
            if cnt == 0:
                continue
            idx = np.arange(cnt)
            c = idx // ch
            ids = np.where(c == 0, first, table[qi, s, np.minimum(c, maxc - 1)]).astype(np.int64)
            assert (ids < plan.sel_pool_chunks).all(), (qi, s)
            got = pool[ids * ch + idx % ch]
            assert np.array_equal(got, want), (qi, s, np.nonzero(got != want)[0][:8])
            chunks_seen.append(np.unique(ids))
            multi_chunk += int(c[-1] > 0)
    ids = np.concatenate(chunks_seen) if chunks_seen else np.zeros(0, np.int64)
    assert len(np.unique(ids)) == len(ids), "two lists share a pool chunk"
    return multi_chunk


def _tc_plan(plan):
    return plan.off_smp_codes != plan.workspace_bytes


def _check_tc_masks(plan, buf, base, q, r):
    """The tensor-core filter's hit masks of the last round it ran, read where select_finish puts them (behind the e4m3
    copies of the codes): proof that the tensor-core form, not the SIMT kernel, wrote the lists."""
    def up(x, a):
        return (x + a - 1) // a * a

    nq, n, bits = q.shape[0], r.shape[0], q.shape[1]
    bp = up(bits, 128)
    db8 = up(base + plan.off_smp_codes, 1024) - base
    moff = db8 + up(n * bp, 1024) + up(plan.Qpad * bp, 1024)
    groups = up(n, 256) // 32
    mask = _view(buf, moff, groups * plan.Qpad).reshape(groups, plan.Qpad)
    bound = _view(buf, plan.off_sel_bound, plan.Qpad)
    dist = (bits - q.astype(np.int64) @ r.astype(np.int64).T) // 2
    retry = (bound[:nq] & BOUND_RETRY) != 0
    if retry.any():                                    # round 1 ran: every row of a redone query, nothing for the others
        within = np.broadcast_to(retry[:, None], (nq, n))
    else:
        within = dist <= (bound[:nq] & 0xFFFF).astype(np.int64)[:, None]
    bits_ = np.zeros((nq, groups * 32), np.uint64)
    bits_[:, :n] = within
    want = (bits_.reshape(nq, groups, 32) << np.arange(32, dtype=np.uint64)).sum(axis=2).astype(np.uint32).T
    assert np.array_equal(mask[:, :nq], want), np.argwhere(mask[:, :nq] != want)[:8]
    assert (mask[:, nq:] == 0).all()                   # padding queries have no hits


@pytest.mark.parametrize("nq,n,bits,nlab,k", [(300, 6001, 128, 80, 600), (130, 9000, 64, 24, 700), (256, 5000, 200, -1, 512),
                                               (40, 7001, 128, 80, 600)])
def test_lists_hold_exactly_the_rows_within_the_bound(monkeypatch, nq, n, bits, nlab, k):
    rng = np.random.default_rng(nq * 7 + n + bits)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    r[:nq] = q
    r[:nq, :3] *= -1                                                # near-duplicates: short distances exist
    if nlab > 0:
        ql, rl = multi_hot(rng, nq, nlab, 0.1), multi_hot(rng, n, nlab, 0.1)
    else:
        ql, rl = rng.integers(0, 6, nq), rng.integers(0, 6, n)
    plan, buf, base, st = _run(monkeypatch, q, ql, r, rl, k)
    assert plan.select == 1 and _tc_plan(plan) == (nq >= 128), plan.sel_T
    assert not st["fell_back"], st
    if _tc_plan(plan):
        _check_tc_masks(plan, buf, base, q, r)
    _check_lists(plan, buf, q, ql, r, rl)


def test_lists_span_several_chunks(monkeypatch):
    """Most rows are near-duplicates of two queries: those queries' lists run past one pool chunk in every segment."""
    rng = np.random.default_rng(11)
    nq, n, bits, k = 200, 7000, 128, 600
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    dup = rng.random(n) < 0.8
    r[dup] = q[np.arange(n)[dup] % 2]
    r[np.nonzero(dup)[0], rng.integers(0, bits, int(dup.sum()))] *= -1      # one flipped bit
    ql, rl = multi_hot(rng, nq, 80, 0.1), multi_hot(rng, n, 80, 0.1)
    plan, buf, base, st = _run(monkeypatch, q, ql, r, rl, k)
    assert _tc_plan(plan) and not st["fell_back"], st
    _check_tc_masks(plan, buf, base, q, r)
    assert _check_lists(plan, buf, q, ql, r, rl) > 0, (plan.sel_chunk, plan.sel_seg_len)


def test_lists_of_queries_redone_with_the_bound_lifted(monkeypatch):
    """The misleading-sample setup of test_gpu_select.py with enough queries for the tensor-core form: near neighbours of
    the first 8 queries only in the sampled 32-row groups.  Round 1 runs the filter and the append kernel for the redone
    queries, whose lists then hold every row of the database."""
    rng = np.random.default_rng(3)
    nq, n, bits, k = 200, 8192, 64, 600
    q = pm1(rng, nq, bits)
    r = pm1(rng, n, bits)
    near = q[rng.integers(0, 8, n)].copy()
    flips = rng.integers(0, bits, (n, 6))
    for c in range(6):
        near[np.arange(n), flips[:, c]] *= -1
    sampled = ((np.arange(n) // 32) % 4) == 0
    r[sampled] = near[sampled]
    ql, rl = multi_hot(rng, nq, 12, 0.2), multi_hot(rng, n, 12, 0.2)
    plan, buf, base, st = _run(monkeypatch, q, ql, r, rl, k, stride=4)
    assert _tc_plan(plan) and not st["fell_back"] and st["queries_redone"] > 0, st
    bound = _view(buf, plan.off_sel_bound, plan.Qpad)
    assert int(((bound[:nq] & BOUND_RETRY) != 0).sum()) == st["queries_redone"]
    _check_tc_masks(plan, buf, base, q, r)
    _check_lists(plan, buf, q, ql, r, rl)

