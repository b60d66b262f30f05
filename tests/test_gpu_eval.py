"""HP-EVAL parity on a B200: the CUDA path (through the C-ABI) against the CPU oracle on the same seeded inputs.

Bar (BASELINE.json north_star / SURVEY.md §8c): distances, ranked indices (index tie-break) and per-query hit counts
bit-exact; AP / mAP within 1e-6 of the float64 oracle (the kernel sums float32 quotients in float64)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import c_oracle, eval_ref
from simlib import correlated_codes, multi_hot, pack_bits, pack_labels_np, pm1, words

pytestmark = pytest.mark.gpu

AP_TOL = 1e-6


def _calc(k=None, **kw):
    from image_retrieval_wavelet_b200.engine import CustomCalculator

    return CustomCalculator(k=k, distance_metric="hamming", with_faiss=False, **kw)


def _problem(seed, nq, n, bits, nlab, dup=True):
    rng = np.random.default_rng(seed)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    if dup and n > nq:
        r[:nq] = q
        r[:nq, :3] *= -1
    if nlab > 0:
        return q, multi_hot(rng, nq, nlab, 0.1), r, multi_hot(rng, n, nlab, 0.1)
    return q, rng.integers(0, 6, nq), r, rng.integers(0, 6, n)


# ------------------------------------------------------------------------------------------------ packing
@pytest.mark.parametrize("bits", [1, 17, 32, 48, 64, 96, 128, 200, 256])
def test_pack_codes_matches_layout(bits):
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(bits)
    for n in (1, 2, 7, 1000):
        c = pm1(rng, n, bits)
        p = H.pack_codes(torch.from_numpy(c))
        assert p.rows == n and p.bits == bits
        got = p.words.cpu().numpy().view(np.uint64)
        assert np.array_equal(got, pack_bits(c, words(bits)))          # including the zeroed padding row


def test_pack_labels_and_rejections():
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(0)
    for nlab in (3, 24, 64, 80, 130, 256):
        lab = multi_hot(rng, 33, nlab, 0.2)
        p = H.pack_labels(torch.from_numpy(lab))
        assert np.array_equal(p.words.cpu().numpy().view(np.uint64), pack_labels_np(lab)[0])
    ints = rng.integers(-5, 5, 11)
    assert np.array_equal(H.pack_labels(torch.from_numpy(ints)).words.cpu().numpy().view(np.uint64), pack_labels_np(ints)[0])
    fl = np.array([0.0, -0.0, 1.5, 1.5, 3.0], np.float32)
    w = H.pack_labels(torch.from_numpy(fl)).words.cpu().numpy()[:5, 0]
    assert w[0] == w[1] and w[2] == w[3] and w[3] != w[4]              # -0.0 == 0.0, equal values <=> equal words
    with pytest.raises(ValueError):
        H.pack_codes(torch.tensor([[1.0, -1.0, 0.0]]))                 # sign(0) = 0
    with pytest.raises(ValueError):
        H.pack_codes(torch.tensor([[0.3, -2.0]]))                      # raw logits
    with pytest.raises(ValueError):
        H.pack_codes(torch.tensor([[1.0, float("nan")]]))
    assert H.pack_codes(torch.tensor([[0.3, -2.0, 0.0]]), on_nonbinary="sign").words.cpu().numpy()[0, 0] == 1
    with pytest.raises(ValueError):
        H.pack_labels(torch.tensor([[0.0, 2.0], [1.0, 0.0]]))          # not multi-hot
    with pytest.raises(NotImplementedError):
        H.pack_codes(torch.ones(2, 257))


# ------------------------------------------------------------------------------------------------ primitives
@pytest.mark.parametrize("bits", [32, 64, 96, 128])
def test_calc_hamming_dist_and_relevance_match_reference_goldens(golden, bits):
    c = _calc()
    q, r = golden[f"hamming_b{bits}/q"].astype(np.float32), golden[f"hamming_b{bits}/r"].astype(np.float32)
    d = c.calc_hamming_dist(torch.from_numpy(q), torch.from_numpy(r))
    assert d.dtype == torch.float32 and np.array_equal(d.cpu().numpy(), golden[f"hamming_b{bits}/dist"])
    rel = c.label_comparison_fn(torch.from_numpy(golden["labels2d/q"]), torch.from_numpy(golden["labels2d/r"]))
    assert rel.dtype == torch.bool and np.array_equal(rel.cpu().numpy(), golden["labels2d/rel"])
    rel1 = c.label_comparison_fn(torch.from_numpy(golden["labels1d/q"]), torch.from_numpy(golden["labels1d/r"]))
    assert np.array_equal(rel1.cpu().numpy(), golden["labels1d/rel"])


def test_bit_balance_matches_reference_golden(golden):
    c = _calc()
    codes = torch.from_numpy(golden["balance/codes"].astype(np.float32))
    assert np.allclose(c.per_bit_balance(codes).cpu().numpy(), golden["balance/per_bit"], atol=1e-7)
    assert abs(c.calculate_bit_balance(codes) - float(golden["balance/mean"])) < 1e-6
    assert abs(c.calculate_worst_bit_balance(codes) - float(golden["balance/worst"])) < 1e-6


# ------------------------------------------------------------------------------------------------ mAP
def test_maphashing_on_reference_goldens(golden):
    """Every golden case produced by the real reference code (stable tie order) through calculate_maphashing."""
    for name in golden["cases"]:
        q, r, ql, rl = (golden[f"{name}/{k}"] for k in ("q", "r", "ql", "rl"))
        tk, inc = (int(v) for v in golden[f"{name}/topk"])
        topk = None if tk == -1 else ("max_bin_count" if tk == -2 else tk)
        c = _calc(k=topk)
        got = c.calculate_maphashing(torch.from_numpy(q.astype(np.float32)), torch.from_numpy(ql),
                                     torch.from_numpy(r.astype(np.float32)), torch.from_numpy(rl), topk, ref_includes_query=bool(inc))
        assert isinstance(got, float)
        assert abs(got - float(golden[f"{name}/map_reference_stable"])) <= AP_TOL, name
        # against the literal (unstable-argsort) reference value: a tie-order effect only, large on these tiny fixtures
        assert abs(got - float(golden[f"{name}/map_reference"])) <= 0.03, name
    c = _calc(k=15)
    name = "nested_topk"
    q, r, ql, rl = (golden[f"{name}/{k}"] for k in ("q", "r", "ql", "rl"))
    got = c.calculate_maphashing(torch.from_numpy(q.astype(np.float32)), torch.from_numpy(ql), torch.from_numpy(r.astype(np.float32)),
                                 torch.from_numpy(rl), [[15]])
    assert abs(got - float(golden[f"{name}/map_reference_stable"])) <= AP_TOL


CASES = [
    (37, 500, 64, 24, 50), (37, 500, 64, 24, None), (20, 3000, 32, 20, 700), (20, 3000, 128, 80, 3000),
    (9, 2000, 96, 130, 100), (16, 70000, 64, 24, 66000), (16, 70000, 64, 24, 5000), (5, 1, 64, 8, 1), (5, 2, 64, 8, 5),
    (33, 1000, 200, 200, None), (40, 5000, 48, -1, 300), (3, 777, 17, 3, 10), (300, 4000, 64, 38, 4000),
]


@pytest.mark.parametrize("stash", [1, 0])
@pytest.mark.parametrize("nq,n,bits,nlab,k", CASES + [(7, 1029, 256, 12, 64), (6, 333, 254, 5, None)])
def test_maphashing_and_ranking_match_exact_oracle(monkeypatch, nq, n, bits, nlab, k, stash):
    """stash = 1: stage B ranks from the (distance, relevance) stash written by stage A; 0: stage B scores again."""
    from image_retrieval_wavelet_b200.engine import hamming as H

    monkeypatch.setenv("B200_MAP_STASH", str(stash))

    q, ql, r, rl = _problem(nq * 1000 + n + bits, nq, n, bits, nlab)
    m0, ap0, ts0, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    c = _calc(k=k)
    m, ap, ts = c.maphashing_details(torch.from_numpy(q), torch.from_numpy(ql), torch.from_numpy(r), torch.from_numpy(rl), k)
    assert np.array_equal(ts.cpu().numpy().astype(np.int64), ts0)
    assert np.abs(ap.cpu().numpy() - ap0).max() <= AP_TOL and abs(m.item() - m0) <= AP_TOL
    kk = n if k is None else min(k, n)
    idx, dist = H.hamming_topk(H.pack_codes(torch.from_numpy(q)), H.pack_codes(torch.from_numpy(r)), kk)
    assert np.array_equal(idx.cpu().numpy(), rank0) and np.array_equal(dist.cpu().numpy().astype(np.int64), dist0)
    # K3 on the materialised list gives the same AP
    m3, ap3, hits3 = H.ranked_ap(idx, H.pack_labels(torch.from_numpy(ql)), H.pack_labels(torch.from_numpy(rl)))
    assert np.array_equal(hits3.cpu().numpy().astype(np.int64), ts0) and np.abs(ap3.cpu().numpy() - ap0).max() <= AP_TOL


def test_c1_mirflickr_shape_full_size():
    """BASELINE config C1: 2000 x 18000, 64 bit, 24 labels, mAP@5000 — full size against the C oracle."""
    rng = np.random.default_rng(0)
    ql, rl = multi_hot(rng, 2000, 24, 0.1), multi_hot(rng, 18000, 24, 0.1)
    for q, r in (correlated_codes(rng, ql, rl, 64), (pm1(rng, 2000, 64), pm1(rng, 18000, 64))):
        m0, ap0, ts0 = c_oracle.maphashing(q, ql, r, rl, 5000)
        c = _calc(k=5000)
        m, ap, ts = c.maphashing_details(torch.from_numpy(q), torch.from_numpy(ql), torch.from_numpy(r), torch.from_numpy(rl), 5000)
        assert np.array_equal(ts.cpu().numpy().astype(np.int64), ts0)
        assert np.abs(ap.cpu().numpy() - ap0).max() <= AP_TOL and abs(m.item() - m0) <= AP_TOL


@pytest.mark.parametrize("bits,n,nlab,k,stash", [(32, 11500, 20, None, 1), (64, 11500, 20, None, 1), (128, 11500, 20, None, 0),
                                                   (128, 117000, 80, 5000, 1), (128, 117000, 80, None, 1),
                                                   (128, 117000, 80, 5000, 0)])
def test_full_size_voc_and_coco_shapes(monkeypatch, bits, n, nlab, k, stash):
    monkeypatch.setenv("B200_MAP_STASH", str(stash))
    _run_full_size(bits, n, nlab, k)


def _run_full_size(bits, n, nlab, k):
    """BASELINE configs C2 / C3 at full size (5000 queries): exact check on a query subsample + size-independent
    properties on all queries."""
    rng = np.random.default_rng(bits + n)
    ql, rl = multi_hot(rng, 5000, nlab, 0.036 if nlab == 80 else 0.1), multi_hot(rng, n, nlab, 0.036 if nlab == 80 else 0.1)
    q, r = correlated_codes(rng, ql, rl, bits)
    c = _calc(k=k)
    tq, tql, tr, trl = (torch.from_numpy(a).cuda() for a in (q, ql, r, rl))
    m, ap, ts = c.maphashing_details(tq, tql, tr, trl, k)
    sub = rng.choice(5000, 40, replace=False)
    m0, ap0, ts0 = c_oracle.maphashing(q[sub], ql[sub], r, rl, k)
    assert np.array_equal(ts.cpu().numpy()[sub].astype(np.int64), ts0)
    assert np.abs(ap.cpu().numpy()[sub] - ap0).max() <= AP_TOL
    assert abs(m.item() - ap.mean().item()) <= 1e-12 and 0.0 <= m.item() <= 1.0
    # properties: all-relevant labels => AP = 1; no relevant label => AP = 0; permuting the QUERIES permutes AP
    ones_q, ones_r = torch.ones(5000, 3, device="cuda"), torch.ones(n, 3, device="cuda")
    m1, ap1, ts1 = c.maphashing_details(tq, ones_q, tr, ones_r, k)
    kk = n if k is None else k
    assert torch.all(ap1 == 1.0) and torch.all(ts1 == kk)
    mz, apz, tsz = c.maphashing_details(tq, torch.zeros(5000, 3, device="cuda"), tr, ones_r, k)
    assert mz.item() == 0.0 and torch.all(tsz == 0)
    perm = torch.randperm(5000, device="cuda")
    mp_, app, tsp = c.maphashing_details(tq[perm].contiguous(), tql[perm].contiguous(), tr, trl, k)
    assert torch.equal(app, ap[perm]) and torch.equal(tsp, ts[perm])


def test_database_duplicates_are_ranked_by_index():
    """All ties: constant codes => the ranking is the index order (MAP-1)."""
    from image_retrieval_wavelet_b200.engine import hamming as H

    q, r = torch.ones(4, 64), torch.ones(300, 64)
    idx, dist = H.hamming_topk(H.pack_codes(q), H.pack_codes(r), 300)
    assert torch.equal(idx.cpu(), torch.arange(300).repeat(4, 1)) and int(dist.max()) == 0


# ------------------------------------------------------------------------------------------------ sharded (emulated on one GPU)
@pytest.mark.parametrize("mode", ["hist", "lists"])
@pytest.mark.parametrize("n_shards", [2, 8])
@pytest.mark.parametrize("nq,n,bits,nlab,k", [(50, 3001, 64, 24, 300), (20, 2000, 128, 80, None), (16, 70001, 64, 24, 5000)])
def test_sharded_evaluator_emulated_on_one_device(mode, n_shards, nq, n, bits, nlab, k):
    from image_retrieval_wavelet_b200.engine import hamming as H
    from image_retrieval_wavelet_b200.engine.dist import ShardedHammingEvaluator, shard_bounds

    q, ql, r, rl = _problem(n + bits, nq, n, bits, nlab)
    m0, ap0, ts0, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    qc, qlp = H.pack_codes(torch.from_numpy(q)), H.pack_labels(torch.from_numpy(ql))
    shards = []
    for b, e in shard_bounds(n, n_shards):
        shards.append((H.pack_codes(torch.from_numpy(r[b:e])), H.pack_labels(torch.from_numpy(rl[b:e]).reshape(e - b, -1)), b))
    ev = ShardedHammingEvaluator(mode=mode)
    m, ap, ts = ev.evaluate(qc, qlp, shards, n, k)
    assert np.array_equal(ts.cpu().numpy().astype(np.int64), ts0)
    assert np.abs(ap.cpu().numpy() - ap0).max() <= AP_TOL and abs(m.item() - m0) <= AP_TOL
    if mode == "lists":
        idx, dist = ev.last_ranked
        assert np.array_equal(idx.cpu().numpy().view(np.uint32).astype(np.int64), rank0)
        assert np.array_equal(dist.cpu().numpy().view(np.uint16).astype(np.int64), dist0)


# ------------------------------------------------------------------------------------------------ knn + map
@pytest.mark.parametrize("metric", ["cosine", "l2"])
@pytest.mark.parametrize("same", [False, True])
def test_get_knn_matches_reference_golden(golden, metric, same):
    from image_retrieval_wavelet_b200.engine import get_knn

    refs, qs = torch.from_numpy(golden["knn/refs"]), torch.from_numpy(golden["knn/queries"])
    src = refs[:9] if same else qs
    idx, dist = get_knn(refs, src, 10, same, with_faiss=False, distance_metric=metric)
    assert idx.dtype == torch.int64 and tuple(idx.shape) == (9, 10)
    assert np.array_equal(idx.cpu().numpy(), golden[f"knn/{metric}_same{int(same)}/idx"])
    assert np.allclose(dist.cpu().numpy(), golden[f"knn/{metric}_same{int(same)}/dist"], atol=2e-4 if metric == "l2" else 1e-5)


@pytest.mark.parametrize("nq,n,d,k", [(64, 5000, 768, 100), (7, 333, 50, 333), (130, 20000, 128, 2048)])
def test_knn_topk_against_float64_oracle(nq, n, d, k):
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk

    rng = np.random.default_rng(d)
    refs = rng.standard_normal((n, d)).astype(np.float32)
    refs /= np.linalg.norm(refs, axis=1, keepdims=True)
    qs = rng.standard_normal((nq, d)).astype(np.float32)
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    score, idx = knn_topk(torch.from_numpy(refs), torch.from_numpy(qs), k, "cosine")
    ref_idx, ref_score = eval_ref.knn_ref(refs, qs, k, False, "cosine")
    assert np.allclose(score.cpu().numpy(), ref_score, atol=1e-5)
    got = idx.cpu().numpy()
    # fp32 vs fp64 accumulation may swap near-equal neighbours: demand identical sets up to 1e-5-close scores
    same = (got == ref_idx).mean()
    assert same > 0.99
    exact = (refs.astype(np.float64) @ qs.astype(np.float64).T).T
    assert np.abs(np.take_along_axis(exact, got, 1) - ref_score).max() <= 1e-5
    assert (np.diff(score.cpu().numpy(), axis=1) <= 1e-7).all()             # best first


@pytest.mark.parametrize("nq,n,d,k", [(130, 1000, 100, 64), (5, 257, 64, 257), (300, 5000, 768, 128), (129, 513, 192, 1)])
def test_knn_tensor_core_scorer_matches_simt_scorer(monkeypatch, nq, n, d, k):
    """Inner-product k-NN: the tcgen05 scorer (bf16 hi/lo split, 3 products) against the exact float32 SIMT scorer and
    the float64 oracle; shapes with ragged Q / N / D tiles."""
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk

    rng = np.random.default_rng(n + d)
    refs = rng.standard_normal((n, d)).astype(np.float32)
    refs /= np.linalg.norm(refs, axis=1, keepdims=True)
    qs = rng.standard_normal((nq, d)).astype(np.float32)
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    monkeypatch.setenv("B200_KNN_TC", "1")
    s_tc, i_tc = knn_topk(torch.from_numpy(refs), torch.from_numpy(qs), k, "cosine")
    monkeypatch.setenv("B200_KNN_TC", "0")
    s_sm, i_sm = knn_topk(torch.from_numpy(refs), torch.from_numpy(qs), k, "cosine")
    exact = qs.astype(np.float64) @ refs.astype(np.float64).T
    # tolerance: 1e-5 for the split-bf16 tensor-core products (dropped lo.lo term ~2^-16 per product), 2e-6 for float32 FMA
    for s_, i_, tol in ((s_tc, i_tc, 1e-5), (s_sm, i_sm, 2e-6)):
        got = np.take_along_axis(exact, i_.cpu().numpy(), 1)
        assert np.abs(s_.cpu().numpy() - got).max() <= tol                        # reported score = score of that row
        assert np.abs(np.sort(exact, axis=1)[:, ::-1][:, :k] - got).max() <= tol   # and it is a true top-k
    assert (i_tc == i_sm).float().mean().item() > 0.99


def test_get_accuracy_flow_map_and_maphashing():
    """CustomCalculator.get_accuracy (accuracy_calculator.py:279-349) with the metrics the reference's CSVs read."""
    from image_retrieval_wavelet_b200.engine import get_accuracy_calculator

    q, ql, r, rl = _problem(3, 60, 2500, 64, 24)
    calc = get_accuracy_calculator(k=500, distance_metric="hamming", with_faiss=False, device=torch.device("cpu"),
                                   exclude=["mean_average_precision", "mean_average_precision_at_r", "r_precision", "rpr", "pr", "pr_rc"])
    res = calc.get_accuracy(q, ql, r, rl, False)
    assert set(res) == {"map", "maphashing", "bit_balance", "worst_bit_balance"}
    assert abs(res["maphashing"] - eval_ref.maphashing_exact(q, ql, r, rl, 500)) <= AP_TOL
    knn_idx, _ = eval_ref.knn_ref(r, q, 500, False, "hamming")
    uniq, counts = eval_ref.label_match_counts_ref(ql, rl)
    assert abs(res["map"] - eval_ref.retrieval_map_ref(ql, rl[knn_idx])) <= 1e-3      # inner-product ties are unordered in both
    _, mean_b, worst_b = eval_ref.bit_balance_ref(r)
    assert abs(res["bit_balance"] - mean_b) < 1e-6 and abs(res["worst_bit_balance"] - worst_b) < 1e-6
    idx, res2 = calc.get_accuracy(q, ql, r, rl, False, include=["map"], return_indices=True)
    assert tuple(idx.shape) == (60, 500) and set(res2) == {"map"}


def test_batch_map_mirror():
    """batch_map.py:9-36: query == reference == the batch, k = max_bin_count, raw logits binarised explicitly."""
    from image_retrieval_wavelet_b200.engine import build_batch_map_calculator, compute_batch_map

    rng = np.random.default_rng(9)
    logits = rng.standard_normal((96, 64)).astype(np.float32)
    lab = multi_hot(rng, 96, 8, 0.25)
    calc, name = build_batch_map_calculator("hamming", torch.device("cuda"))
    assert name == "maphashing"
    got = compute_batch_map(calc, name, torch.from_numpy(logits).cuda().requires_grad_(), torch.from_numpy(lab).cuda())
    codes = np.where(logits > 0, 1.0, -1.0)
    assert abs(got - eval_ref.maphashing_exact(codes, lab, codes, lab, "max_bin_count", True)) <= AP_TOL


def test_host_buffer_entry_point_directly():
    """b200_maphashing_host: float32 host buffers exactly as the reference hands them over."""
    from image_retrieval_wavelet_b200 import _cabi

    q, ql, r, rl = _problem(4, 100, 6000, 64, 24)
    ap = np.zeros(100)
    ts = np.zeros(100, np.uint32)
    m = ctypes.c_double()
    bad = ctypes.c_int()
    rc = _cabi.load().b200_maphashing_host(q.ctypes.data, ql.ctypes.data, r.ctypes.data, rl.ctypes.data, 100, 6000, 64, 24, 0, 1000,
                                           ap.ctypes.data, ts.ctypes.data, ctypes.addressof(m), ctypes.addressof(bad))
    assert rc == 0 and bad.value == 0
    m0, ap0, ts0, _, _ = eval_ref.maphashing_exact(q, ql, r, rl, 1000, return_details=True)
    assert np.array_equal(ts.astype(np.int64), ts0) and np.abs(ap - ap0).max() <= AP_TOL and abs(m.value - m0) <= AP_TOL
    q[0, 0] = 0.0
    rc = _cabi.load().b200_maphashing_host(q.ctypes.data, ql.ctypes.data, r.ctypes.data, rl.ctypes.data, 100, 6000, 64, 24, 0, 1000,
                                           None, None, ctypes.addressof(m), ctypes.addressof(bad))
    assert rc == _cabi.ERR_INVALID_ARG and bad.value == 1


@pytest.mark.parametrize("chunks", [1, 3, 8])
@pytest.mark.parametrize("n,k,nlab", [(30000, 2000, 24), (777, None, -1), (70001, 70001, 24)])
def test_host_buffer_entry_point_chunked_pipeline(monkeypatch, chunks, n, k, nlab):
    """The H2D / stage-A pipeline of b200_maphashing_host (chunks of whole segments on a copy stream) for any chunk
    count, including more chunks than segments, 1-D labels and the all-rows mode."""
    from image_retrieval_wavelet_b200 import _cabi

    monkeypatch.setenv("B200_HOST_CHUNKS", str(chunks))
    q, ql, r, rl = _problem(n + chunks, 50, n, 64, nlab)
    kk = n if k is None else k
    ap, ts = np.zeros(50), np.zeros(50, np.uint32)
    m, bad = ctypes.c_double(), ctypes.c_int()
    if nlab > 0:
        lq, lr, mode, L = ql.astype(np.float32), rl.astype(np.float32), 0, nlab
    else:
        lq, lr, mode, L = ql.astype(np.float32).reshape(-1, 1).copy(), rl.astype(np.float32).reshape(-1, 1).copy(), 1, 1
    rc = _cabi.load().b200_maphashing_host(q.ctypes.data, lq.ctypes.data, r.ctypes.data, lr.ctypes.data, 50, n, 64, L, mode, kk,
                                           ap.ctypes.data, ts.ctypes.data, ctypes.addressof(m), ctypes.addressof(bad))
    assert rc == 0 and bad.value == 0
    m0, ap0, ts0, _, _ = eval_ref.maphashing_exact(q, ql, r, rl, kk, return_details=True)
    assert np.array_equal(ts.astype(np.int64), ts0) and np.abs(ap - ap0).max() <= AP_TOL and abs(m.value - m0) <= AP_TOL


@pytest.mark.parametrize("streamed", ["1", "0"])
@pytest.mark.parametrize("chunks", [2, 3, 8])
@pytest.mark.parametrize("nq,n,k,bits,nlab,collapse", [
    pytest.param(40, 70001, 5000, 64, 24, False, id="70001-5000-64-24-False"),
    pytest.param(40, 40000, 600, 128, -1, False, id="40000-600-128--1-False"),
    pytest.param(40, 45000, 1000, 64, 24, True, id="45000-1000-64-24-True"),
    pytest.param(200, 70001, 5000, 128, 24, False, id="200q-70001-5000-128-24-False"),
])
def test_host_buffer_entry_point_streams_the_select_pipeline(monkeypatch, streamed, chunks, nq, n, k, bits, nlab, collapse):
    """Select plans in b200_maphashing_host: the sample rows cross PCIe first (strided 2-D copy), every chunk's segments are
    scored while the next chunk is in flight (B200_HOST_STREAMED=0: the whole database first).  Same integers and AP as
    the oracle either way — also when the codes collapse (every row ties: pool overflow -> the gated three stages).  With
    128 queries or more the streamed round 0 runs the SIMT select kernel on 128-query groups (the unstreamed call runs the
    tensor-core form there)."""
    from image_retrieval_wavelet_b200 import _cabi

    monkeypatch.setenv("B200_HOST_CHUNKS", str(chunks))
    monkeypatch.setenv("B200_HOST_STREAMED", streamed)
    q, ql, r, rl = _problem(n + chunks, nq, n, bits, nlab)
    if collapse:
        r[:] = r[0]
    ap, ts = np.zeros(nq), np.zeros(nq, np.uint32)
    m, bad = ctypes.c_double(), ctypes.c_int()
    if nlab > 0:
        lq, lr, mode, L = ql.astype(np.float32), rl.astype(np.float32), 0, nlab
    else:
        lq, lr, mode, L = ql.astype(np.float32).reshape(-1, 1).copy(), rl.astype(np.float32).reshape(-1, 1).copy(), 1, 1
    plan = _cabi.MapPlan()
    assert _cabi.load().b200_map_plan_init(ctypes.byref(plan), nq, n, n, bits, words(L), mode, k) == 0
    assert plan.select == 1 and (plan.sel_T == 128 or nq < 128), (plan.select, plan.sel_T)
    rc = _cabi.load().b200_maphashing_host(q.ctypes.data, lq.ctypes.data, r.ctypes.data, lr.ctypes.data, nq, n, bits, L, mode, k,
                                           ap.ctypes.data, ts.ctypes.data, ctypes.addressof(m), ctypes.addressof(bad))
    assert rc == 0 and bad.value == 0
    m0, ap0, ts0, _, _ = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    assert np.array_equal(ts.astype(np.int64), ts0) and np.abs(ap - ap0).max() <= AP_TOL and abs(m.value - m0) <= AP_TOL


@pytest.mark.parametrize("nq,n,bits,nlab", [(37, 501, 64, 24), (300, 2000, 32, 20), (9, 1000, 128, -1)])
def test_pr_rc_hashing_curves_match_oracle(tmp_path, monkeypatch, nq, n, bits, nlab):
    """calculate_pr_rc_hashing (accuracy_calculator.py:235-273): precision / recall at every rank of the full ranking."""
    q, ql, r, rl = _problem(nq + n, nq, n, bits, nlab)
    mask = np.ones(nq, bool)
    mask[::5] = False
    c = _calc(k=None)
    prec, rec, used = c.pr_rc_hashing_curves(torch.from_numpy(q), torch.from_numpy(ql), torch.from_numpy(r), torch.from_numpy(rl),
                                             torch.from_numpy(mask), chunk=64)
    p0, r0, u0 = eval_ref.pr_rc_hashing_ref(q, ql, r, rl, mask)
    assert used == u0
    # float32 quotients like the reference (accuracy_calculator.py:255-256), float64 sums: <= 2^-24 relative per term
    assert np.abs(prec.cpu().numpy() - p0).max() <= 1e-6 and np.abs(rec.cpu().numpy() - r0).max() <= 1e-6
    monkeypatch.chdir(tmp_path)
    assert c.calculate_pr_rc_hashing(torch.from_numpy(q), torch.from_numpy(ql), torch.from_numpy(r), torch.from_numpy(rl),
                                     torch.from_numpy(mask)) == 0
    import pandas as pd

    df = pd.read_csv(tmp_path / "pr_rc.csv")
    assert list(df.columns) == ["pr", "rc"] and len(df) == n and abs(df["rc"].iloc[-1] - 1.0) <= 1e-6


@pytest.mark.parametrize("tpq", ["1", "2", "3", "4"])
def test_stage_a_threads_per_query_agree(monkeypatch, tpq):
    """B200_MAP_TPQ: stage A with 1-4 threads per query sharing a counter column — identical integers, identical AP."""
    monkeypatch.setenv("B200_MAP_TPQ", tpq)
    for seed, (nq, n, bits, nlab, k) in enumerate([(130, 5000, 128, 80, 500), (33, 2100, 64, 24, None), (20, 1777, 32, -1, 100)]):
        q, ql, r, rl = _problem(40 + seed, nq, n, bits, nlab)
        m0, ap0, ts0, _, _ = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
        m, ap, ts = _calc(k=k).maphashing_details(torch.from_numpy(q), torch.from_numpy(ql), torch.from_numpy(r), torch.from_numpy(rl), k)
        assert np.array_equal(ts.cpu().numpy().astype(np.int64), ts0)
        assert np.abs(ap.cpu().numpy() - ap0).max() <= AP_TOL and abs(float(m) - m0) <= AP_TOL


def test_kernels_are_the_thing_that_ran():
    from image_retrieval_wavelet_b200 import _cabi

    before = _cabi.launch_count()
    q, ql, r, rl = _problem(5, 10, 500, 64, 8)
    _calc(k=50).calculate_maphashing(torch.from_numpy(q), torch.from_numpy(ql), torch.from_numpy(r), torch.from_numpy(rl), 50)
    assert _cabi.launch_count() - before >= 8       # 4 packs + hist + scan + ap + finalize + mean


# ------------------------------------------------------------------------------------------------ k-NN: any k, fused selection
@pytest.mark.parametrize("metric,nq,n,d,k", [("cosine", 40, 20000, 64, 5000), ("cosine", 9, 9000, 32, 9000), ("l2", 12, 12000, 48, 5717),
                                              ("cosine", 6, 4097, 16, 4097), ("l2", 5, 300, 8, 300)])
def test_knn_lists_longer_than_one_select_pass(metric, nq, n, d, k):
    """k above 4096 (the reference's own settings: 5000, 5717, 19581, the whole database): passes of 4096 ranks, each
    continuing strictly after the last (score, index) of the one before."""
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk

    rng = np.random.default_rng(n + k)
    refs = rng.standard_normal((n, d)).astype(np.float32)
    refs[::7] = refs[3]                                   # exact score ties across pass boundaries: index order decides
    qs = rng.standard_normal((nq, d)).astype(np.float32)
    if metric == "cosine":
        refs /= np.linalg.norm(refs, axis=1, keepdims=True)
        qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    score, idx = knn_topk(torch.from_numpy(refs), torch.from_numpy(qs), k, metric)
    got, sc = idx.cpu().numpy(), score.cpu().numpy()
    assert got.shape == (nq, k)
    assert all(len(set(row.tolist())) == k for row in got)                      # a permutation prefix: no row twice
    if metric == "cosine":
        exact = qs.astype(np.float64) @ refs.astype(np.float64).T
        assert (np.diff(sc, axis=1) <= 1e-7).all()
        assert np.abs(np.take_along_axis(exact, got, 1) - sc).max() <= 1e-5
        assert np.abs(np.sort(exact, axis=1)[:, ::-1][:, :k] - sc).max() <= 1e-5  # a true top-k, best first
    else:
        exact = np.sqrt(np.maximum(((qs[:, None, :].astype(np.float64) - refs[None].astype(np.float64)) ** 2).sum(-1), 0))
        assert (np.diff(sc, axis=1) >= -1e-6).all()
        assert np.abs(np.sort(exact, axis=1)[:, :k] - sc).max() <= 2e-4
    tied = sc[:, 1:] == sc[:, :-1]                                              # equal scores: smaller index first
    assert (got[:, 1:][tied] > got[:, :-1][tied]).all()


def test_get_knn_hamming_metric_any_k(golden):
    """distance_metric='hamming' on +-1 codes goes through the counting-sort evaluator: exact (distance, index) order."""
    from image_retrieval_wavelet_b200.engine import get_knn

    q, ql, r, rl = _problem(21, 30, 7000, 64, 8)
    idx, dist = get_knn(torch.from_numpy(r), torch.from_numpy(q), 5000, False, with_faiss=False, distance_metric="hamming")
    _, _, _, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, 5000, return_details=True)
    assert np.array_equal(idx.cpu().numpy(), rank0) and np.array_equal(dist.cpu().numpy(), 64.0 - 2.0 * dist0)


@pytest.mark.parametrize("k", [2048, 5000])
def test_c3_cosine_shape_fused_selection(k):
    """BASELINE configs[2] cosine rerank at full size (5000 x 117000 x 768): k = 2048 takes the fused path (threshold
    from a sampled pass, candidate filter in the tcgen05 epilogue, no score matrix), k = 5000 the matrix path (2.3 GB of
    scores, two select passes); a query sample against float64, and the first 2048 entries of the k = 5000 lists equal
    the k = 2048 lists: the same GEMM tiles score both, and both selections are exact by (key, index)."""
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk

    g = torch.Generator().manual_seed(0)
    refs = torch.nn.functional.normalize(torch.randn(117000, 768, generator=g), dim=1)
    qs = torch.nn.functional.normalize(torch.randn(5000, 768, generator=g), dim=1)
    refs_d, qs_d = refs.cuda(), qs.cuda()
    score, idx = knn_topk(refs_d, qs_d, k, "cosine")
    sub = np.random.default_rng(1).choice(5000, 24, replace=False)
    exact = qs[sub].double() @ refs.double().T
    want_s, want_i = torch.topk(exact, k, dim=1)
    got_i, got_s = idx.cpu()[sub], score.cpu()[sub]
    assert (got_s.double() - want_s).abs().max().item() <= 1e-5
    assert (torch.gather(exact, 1, got_i) - want_s).abs().max().item() <= 1e-5     # the reported rows ARE a top-k
    # random 768-d unit vectors: neighbouring scores of the top k are ~1e-6 apart, below the 1e-5 score tolerance, so
    # positions may swap against float64; the SETS must agree except at the k-th boundary
    overlap = np.mean([len(set(a.tolist()) & set(b.tolist())) / float(k) for a, b in zip(got_i.numpy(), want_i.numpy())])
    assert overlap > 0.98, overlap
    if k > 2048:
        s_f, i_f = knn_topk(refs_d, qs_d, 2048, "cosine")
        assert torch.equal(idx[:, :2048], i_f) and torch.equal(score[:, :2048].view(torch.int32), s_f.view(torch.int32))


@pytest.mark.parametrize("metric", ["cosine", "l2"])
@pytest.mark.parametrize("n_shards,n,k", [(2, 6001, 300), (8, 9000, 5000), (3, 500, 500)])
def test_sharded_knn_merge_emulated_on_one_device(metric, n_shards, n, k):
    """SURVEY 8e cosine row: per-shard top-k lists merged by (score, index) equal the unsharded top-k (ties included)."""
    from image_retrieval_wavelet_b200.engine.dist import shard_bounds
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk, merge_knn_shards

    rng = np.random.default_rng(n + k)
    refs = rng.standard_normal((n, 40)).astype(np.float32)
    refs[::5] = refs[2]                                    # ties across shards
    qs = rng.standard_normal((17, 40)).astype(np.float32)
    tr, tq = torch.from_numpy(refs).cuda(), torch.from_numpy(qs).cuda()
    want_s, want_i = knn_topk(tr, tq, k, metric)
    ss, ii = [], []
    for b, e in shard_bounds(n, n_shards):
        s = torch.zeros((17, k), device="cuda")
        i = torch.full((17, k), -1, dtype=torch.int64, device="cuda")
        kl = min(k, e - b)
        if kl > 0:
            s[:, :kl], i_ = knn_topk(tr[b:e].contiguous(), tq, kl, metric)
            i[:, :kl] = i_ + b
        ss.append(s), ii.append(i)
    got_i, got_s = merge_knn_shards(torch.stack(ss), torch.stack(ii), k, metric)
    assert torch.equal(got_i, want_i) and torch.allclose(got_s, want_s, atol=1e-6)
