"""Bit-exact continuous-embedding k-NN on integer embeddings, every scoring and selection route against an exact oracle.

Integers with |x| <= 256 are exact in bfloat16, so the tensor-core scorer's hi/lo split has lo = 0; while every partial
sum stays below 2^24, float32 accumulation is exact in any order, on the tensor cores and on the FMA path alike.  On such
inputs every route of ``b200_knn_topk`` (tcgen05 matrix, fused candidate filter and both of its fallbacks, float32 SIMT,
L2), of ``select_topk`` and of ``merge_knn_shards`` must return exactly the oracle's list: indices equal, scores
bit-equal, ordered by (score, then index), -0.0 equal to +0.0, NaN after every number.  Small value ranges give dense
exact ties, which is where the selection kernels branch (rank k, 4096-rank pass boundaries, sampled thresholds,
candidate-buffer overflow).  The tolerance tests in test_gpu_eval.py cover real float inputs."""
import math

import numpy as np
import pytest
import torch

FUSED_CAP = 8192          # knn.cu: kKnnFusedCap, candidate pairs per query of the fused path
MAX_K = 4096              # knn.cu: kKnnMaxK, ranks per select pass
SPECIAL = 100             # coordinate that makes the "special" rows of a tie pattern rank first


# ------------------------------------------------------------------------------------------------ generator + oracle
def check_exact(q, r, metric):
    """The premises of exactness on these inputs: finite entries are integers with |x| <= 256 (exact in bfloat16), and
    every partial sum the scorers form stays below 2^24 (inner product) or below 2^22 (L2: |q|^2, |r|^2, 2<q, r> and
    |q - r|^2, where float32 sqrtf of distinct integers also stays distinct)."""
    qf, rf = (np.where(np.isfinite(x), x, 0).astype(np.float64) for x in (q, r))
    for x in (qf, rf):
        assert np.array_equal(x, np.round(x)) and np.abs(x).max(initial=0) <= 256
    cross = np.abs(qf).sum(1).max(initial=0) * np.abs(rf).max(initial=0)          # >= any partial sum of |q_j r_j|
    if metric == "l2":
        assert (qf ** 2).sum(1).max(initial=0) + (rf ** 2).sum(1).max(initial=0) + 2 * cross < 2 ** 22
    else:
        assert cross < 2 ** 24


def int_embeddings(rng, rows, d, bound):
    return rng.integers(-bound, bound + 1, (rows, d)).astype(np.float32)


def make_case(seed, nq, n, d, bound, pattern, metric):
    """(queries, refs) with integer entries, |x| <= bound, and one tie pattern:
    dense        uniform integers: exact ties at every rank;
    top_tie      every 7th row is the same best row for every query (N / 7 rows tied at the top);
    stride<s>    every s-th row ranks ahead of all others (a sample of every s-th row sees only those)."""
    rng = np.random.default_rng(seed)
    q, r = int_embeddings(rng, nq, d, bound), int_embeddings(rng, n, d, bound)
    if pattern != "dense":
        step = 7 if pattern == "top_tie" else int(pattern[len("stride"):])
        special = np.zeros(n, bool)
        special[::step] = True
        if metric == "l2":          # special rows near the origin (and so near every query), the others far out
            r[:, 0] = np.where(special, 0, SPECIAL)
        else:                       # every query leans on coordinate 0, the special rows with it
            q[:, 0] = SPECIAL
            r[:, 0] = np.where(special, SPECIAL, r[:, 0])
        if pattern == "top_tie":
            r[special, 1:] = 0
    check_exact(q, r, metric)
    return q, r


def rank_order(score, k, largest):
    """Stable argsort by (score, then index): largest or smallest first; -0.0 == +0.0 and numpy sorts NaN after every
    number (-NaN is NaN), for either direction."""
    return np.argsort(-score if largest else score, axis=1, kind="stable")[:, :k]


def oracle(q, r, k, metric):
    """(scores float32 [Q, k], indices [Q, k]).  Scores in float64, exact for these integers, then rounded to float32
    (for L2, rounding sqrt from float64 equals float32 sqrtf of the same integer); rows with a NaN score NaN."""
    nan_rows = np.isnan(r).any(1)
    q64, r64 = q.astype(np.float64), np.where(nan_rows[:, None], 0, r).astype(np.float64)
    s = q64 @ r64.T
    if metric == "l2":
        s = np.sqrt((q64 * q64).sum(1)[:, None] + (r64 * r64).sum(1)[None, :] - 2 * s)
    s = s.astype(np.float32) + np.float32(0)                 # -0.0 reads as +0.0
    s[:, nan_rows] = np.nan
    idx = rank_order(s, k, metric != "l2")
    return np.take_along_axis(s, idx, 1), idx


def assert_exact(score, idx, want_s, want_i, what=""):
    """Indices equal, scores bit-equal (NaN where the oracle has NaN)."""
    s = score.cpu().numpy() if torch.is_tensor(score) else score
    i = idx.cpu().numpy() if torch.is_tensor(idx) else idx
    assert s.shape == want_s.shape and i.shape == want_i.shape, what
    nan = np.isnan(want_s)
    bad = (i != want_i) | (np.isnan(s) != nan) | (~nan & (s.view(np.int32) != want_s.view(np.int32)))
    if bad.any():
        row, col = (int(v) for v in np.argwhere(bad)[0])
        lo = max(col - 2, 0)
        raise AssertionError(f"{what}: {int(bad.sum())} mismatches, first at query {row}, rank {col}: "
                             f"got idx {i[row, lo:col + 3].tolist()} score {s[row, lo:col + 3].tolist()}, "
                             f"want idx {want_i[row, lo:col + 3].tolist()} score {want_s[row, lo:col + 3].tolist()}")


def bits_equal(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32)) if a.dtype == torch.float32 else torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ routes + probe
COSINE_ROUTES = {
    # tcgen05 scorer: where fused_rank(N, k) > 0 the sampled threshold, filtering epilogue and knn_select_cand_kernel (with
    # the score matrix as fallback), elsewhere the score matrix and knn_select_kernel
    "tc": {"B200_KNN_TC": "1"},
    "simt": {"B200_KNN_TC": "0"},                            # exact float32 FMA scorer, score matrix
}


def fused_rank(n, k):
    """knn.cu: knn_fused_rank — the sample rank of the fused path's threshold; 0: the fused path does not apply."""
    if n // 16 < 4 * 1024 or k > MAX_K:
        return 0
    ks = k / 16
    r = ks + 5.0 * math.sqrt(ks) + 2.0
    if r > MAX_K or r * 16 + 5.0 * math.sqrt(r) * 16 > 0.9 * FUSED_CAP:
        return 0
    return int(r + 0.5)


def fused_probe_offsets(lib, nq, n, d, k):
    """Byte offsets of the fused path's cand_cnt [Q] and fail word in the workspace, mirroring the carve-up in
    b200_knn_topk; None when the fused path does not apply.  The total must equal b200_knn_workspace_bytes, so a layout
    change fails here instead of reading the wrong words."""
    ru = lambda a, b: (a + b - 1) // b * b                                      # noqa: E731
    off = ru(nq * ru(n, 4) * 4, 256) + ru((nq + n) * 4, 256)                    # score matrix, norms
    off += ru(nq * FUSED_CAP * 8, 256)                                          # candidate lists
    scratch = off                                                               # sample top list (idx, score), thr, counters
    off += ru(nq * (MAX_K * 12 + 16), 256) + 256
    off += ru(2 * (nq + n) * ru(d, 64) * 2, 1024) + 1024                        # bf16 hi / lo copies (knn_tc.cu)
    assert off == lib.b200_knn_workspace_bytes(nq, n, d, k), "b200_knn_topk's workspace layout changed"
    rank = fused_rank(n, k)
    if rank == 0:
        return None
    cnt = scratch + nq * rank * 12 + nq * 4
    return cnt, cnt + nq * 4


POISON = 0xFFFFFFFF


def knn_call(monkeypatch, env, refs, qs, k, metric):
    """b200_knn_topk on a workspace filled with 0xFF: (score, idx, probe); probe = (fail word, cand_cnt [Q]) where the
    fused path applies to the shape, else None.  A fail word still 0xFFFFFFFF: the fused path did not run."""
    from image_retrieval_wavelet_b200 import _cabi

    for key, val in env.items():
        monkeypatch.setenv(key, val)
    nq, n, d = int(qs.shape[0]), int(refs.shape[0]), int(refs.shape[1])
    lib = _cabi.load()
    nbytes = lib.b200_knn_workspace_bytes(nq, n, d, k)
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device="cuda")
    idx = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    score = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    _cabi.check(lib.b200_knn_topk(_cabi.ptr(refs), _cabi.ptr(qs), nq, n, d, k, int(metric == "l2"), _cabi.ptr(idx), _cabi.ptr(score),
                                  _cabi.ptr(ws), nbytes, _cabi.stream_ptr()), "b200_knn_topk")
    torch.cuda.synchronize()
    offs = fused_probe_offsets(lib, nq, n, d, k)
    probe = None
    if offs is not None:
        cnt = ws[offs[0]:offs[0] + nq * 4].view(torch.int32).cpu().numpy().view(np.uint32)
        probe = (int(ws[offs[1]:offs[1] + 4].view(torch.int32).cpu().numpy().view(np.uint32)[0]), cnt)
    return score, idx, probe


def run_routes(monkeypatch, q, r, k, metric):
    """{route: (score, idx, probe)} for every route of the metric; the cosine routes must agree bit for bit."""
    refs, qs = torch.from_numpy(r).cuda(), torch.from_numpy(q).cuda()
    routes = COSINE_ROUTES if metric == "cosine" else {"l2": {}}
    out = {name: knn_call(monkeypatch, env, refs, qs, k, metric) for name, env in routes.items()}
    for name, (_, _, probe) in out.items():
        if probe is not None and name != "tc":
            assert probe[0] == POISON, f"{name}: the fused path ran"
    if metric == "cosine":
        assert bits_equal(out["simt"][0], out["tc"][0]) and bits_equal(out["simt"][1], out["tc"][1]), "simt != tc"
    return out


def check_fused_probe(probe, k, fail):
    """fail == 0: every list was complete and inside the cap (the fused path produced the answer); fail == 1: some
    list was too short or overflowed (the score matrix produced it)."""
    assert probe is not None and probe[0] in (0, 1), probe
    ok = (probe[1] >= k) & (probe[1] <= FUSED_CAP)
    assert probe[0] == int(not ok.all()), (probe[0], int(probe[1].min()), int(probe[1].max()))
    if fail is not None:
        assert probe[0] == fail, (probe[0], int(probe[1].min()), int(probe[1].max()))


# ------------------------------------------------------------------------------------------------ CPU: premises + oracle
def test_generator_premises_and_oracle_policy():
    rng = np.random.default_rng(0)
    x = np.arange(-256, 257, dtype=np.float32)
    assert torch.equal(torch.from_numpy(x).to(torch.bfloat16).float(), torch.from_numpy(x))        # hi = x, lo = 0
    assert not torch.equal(torch.tensor([257.0]).to(torch.bfloat16).float(), torch.tensor([257.0]))
    check_exact(int_embeddings(rng, 5, 768, 15), int_embeddings(rng, 9, 768, 15), "cosine")        # 172 800 < 2^24
    check_exact(int_embeddings(rng, 5, 64, 127), int_embeddings(rng, 9, 64, 127), "l2")
    for d, b, metric in ((768, 148, "cosine"), (64, 128, "l2"), (4, 257, "cosine")):
        q = np.full((1, d), b, np.float32)
        with pytest.raises(AssertionError):
            check_exact(q, q, metric)
    with pytest.raises(AssertionError):
        check_exact(np.full((1, 4), 0.5, np.float32), np.ones((1, 4), np.float32), "cosine")
    for metric in ("cosine", "l2"):
        for pattern in ("dense", "top_tie", "stride16"):
            make_case(1, 3, 4099, 64, 3, pattern, metric)
    # the patterns put their special rows first
    q, r = make_case(2, 4, 700, 64, 3, "top_tie", "cosine")
    assert (oracle(q, r, 100, "cosine")[1] == np.arange(0, 700, 7)).all()
    q, r = make_case(2, 4, 700, 64, 3, "stride16", "l2")
    assert (np.sort(oracle(q, r, 44, "l2")[1], axis=1) == np.arange(0, 700, 16)).all()
    # oracle: ties by index, -0.0 == +0.0 (reported +0.0), NaN after every number, +-inf in between, either direction
    s = np.array([[0.0, np.nan, -0.0, np.inf, 1.0, -np.inf, -0.0, np.nan, 0.0]], np.float32)
    assert rank_order(s, 9, True)[0].tolist() == [3, 4, 0, 2, 6, 8, 5, 1, 7]
    assert rank_order(s, 9, False)[0].tolist() == [5, 0, 2, 6, 8, 4, 3, 1, 7]
    q = np.zeros((1, 4), np.float32)
    r = np.array([[-1, -2, -3, -4], [1, 1, 1, 1], [np.nan] * 4, [-5, 0, 0, 0]], np.float32)
    want_s, want_i = oracle(q, r, 4, "cosine")
    assert want_i[0].tolist() == [0, 1, 3, 2] and (want_s[0, :3].view(np.int32) == 0).all() and np.isnan(want_s[0, 3])
    want_s, want_i = oracle(np.ones((1, 4), np.float32), r, 4, "l2")
    assert want_i[0].tolist() == [1, 3, 0, 2] and want_s[0, :3].tolist() == [0.0, np.float32(math.sqrt(39)), np.float32(math.sqrt(54))]
    assert fused_rank(65535, 2048) == 0 and fused_rank(65536, 4096) > 0 and fused_rank(70001, 4097) == 0


def test_route_probe_mirrors_the_workspace_layout():
    """The probe's copy of b200_knn_topk's workspace carve-up adds up to b200_knn_workspace_bytes (host function: no
    device needed) on every shape the GPU tests use."""
    from image_retrieval_wavelet_b200 import _cabi

    lib = _cabi.load()
    shapes = [(nq, n, d, k) for nq, n, d, k, *_ in CASES] + [(5000, 117000, 768, 2048), (9, 70001, 64, 2048), (3, 70001, 64, 2048)]
    for nq, n, d, k in shapes:
        offs = fused_probe_offsets(lib, nq, n, d, k)
        assert (offs is None) == (fused_rank(n, k) == 0) and (offs is None or offs[1] == offs[0] + 4 * nq)


# ------------------------------------------------------------------------------------------------ GPU: every route
# (Q, N, D, k, bound, pattern, fused fail word expected on the "tc" route where the fused path applies: 0, 1 or None = either)
CASES = [
    (1, 257, 4, 257, 2, "dense", None),               # k = N; scores in [-16, 16]
    (129, 4099, 12, 4097, 3, "dense", None),          # ties straddle rank k and the 4096-rank pass boundary
    (127, 16383, 60, 2048, 4, "dense", None),         # one row below the select kernel's sampled threshold
    (128, 16384, 64, 4095, 3, "dense", None),         # sampled threshold of the select kernel
    (127, 16384, 4, 8193, 7, "dense", None),          # three passes
    (300, 65535, 68, 1, 5, "dense", None),            # one row below the fused path
    (129, 65536, 64, 4096, 2, "dense", None),         # fused at its largest k, dense ties at the threshold
    (300, 70001, 768, 2048, 15, "dense", 0),          # (f) the fused path produces the answer
    (128, 70001, 64, 2048, 3, "top_tie", 1),          # (c) 10 001 rows tied at the top: fused cap and kKnnCand overflow
    (129, 65536, 64, 2048, 3, "stride16", 1),         # (d) the fused sample sees only the best rows: lists too short
    (127, 70001, 60, 2048, 3, "stride68", None),      # (e) the select kernel's sample (stride N / 1024) sees only those
    (1, 70001, 64, 4096, 3, "top_tie", 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "l2"])
@pytest.mark.parametrize("nq,n,d,k,bound,pattern,fail", CASES)
def test_every_route_returns_the_exact_list(monkeypatch, metric, nq, n, d, k, bound, pattern, fail):
    q, r = make_case(n + k + d, nq, n, d, bound, pattern, metric)
    want_s, want_i = oracle(q, r, k, metric)
    for name, (score, idx, probe) in run_routes(monkeypatch, q, r, k, metric).items():
        assert_exact(score, idx, want_s, want_i, name)
        if name == "tc" and fused_rank(n, k):
            check_fused_probe(probe, k, fail)


@pytest.mark.gpu
def test_c3_shape_every_route_exact(monkeypatch):
    """BASELINE configs[2] shape (5000 x 117000 x 768, k = 2048) on integers |x| <= 15: the fused path (which must have
    produced the answer) and the SIMT path agree bit for bit on all queries, and a 48-query sample equals the oracle."""
    q, r = make_case(3, 5000, 117000, 768, 15, "dense", "cosine")
    out = run_routes(monkeypatch, q, r, 2048, "cosine")
    check_fused_probe(out["tc"][2], 2048, 0)
    sub = np.random.default_rng(4).choice(5000, 48, replace=False)
    want_s, want_i = oracle(q[sub], r, 2048, "cosine")
    assert_exact(out["tc"][0].cpu()[sub], out["tc"][1].cpu()[sub], want_s, want_i, "c3")


# ------------------------------------------------------------------------------------------------ GPU: edges
@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "l2"])
@pytest.mark.parametrize("n,k", [(257, 257), (20000, 20000), (70001, 2048)])
def test_nan_rows_rank_after_every_number(monkeypatch, metric, n, k):
    q, r = make_case(n, 9, n, 64, 3, "dense", metric)
    r[3::41] = np.nan
    want_s, want_i = oracle(q, r, k, metric)
    for name, (score, idx, _) in run_routes(monkeypatch, q, r, k, metric).items():
        assert_exact(score, idx, want_s, want_i, name)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [257, 20000])
def test_inf_coordinates_never_outrank_a_finite_row_l2(monkeypatch, n):
    """L2 with +-inf coordinates (the inner product is out of scope: the bf16 split makes it NaN): such a row's
    distance is inf or NaN (inf - inf, 0 * inf), so it ranks after every finite row — infinite distances first, then
    NaN, each in index order — and the finite prefix equals the oracle of the finite rows."""
    q, r = make_case(n, 9, n, 64, 3, "dense", "l2")
    q[:, 5] = 0                                          # 0 * inf: NaN distances too
    bad = np.zeros(n, bool)
    bad[2::53] = True
    r[2::106, 5] = np.inf
    r[55::106, 7] = -np.inf
    score, idx, _ = run_routes(monkeypatch, q, r, n, "l2")["l2"]
    s, i = score.cpu().numpy(), idx.cpu().numpy()
    fin = np.flatnonzero(~bad)
    want_s, want_i = oracle(q, r[fin], len(fin), "l2")
    assert_exact(s[:, :len(fin)], i[:, :len(fin)], want_s, fin[want_i], "finite prefix")
    tail, tail_s = i[:, len(fin):], s[:, len(fin):]
    assert (np.isinf(tail_s) | np.isnan(tail_s)).all() and (tail_s[~np.isnan(tail_s)] > 0).all()
    for row, row_s in zip(tail, tail_s):
        assert row.tolist() == sorted(np.flatnonzero(bad).tolist(), key=lambda j: (bool(np.isnan(row_s[row == j][0])), j))


@pytest.mark.gpu
@pytest.mark.parametrize("n,k", [(257, 257), (70001, 2048)])
def test_all_zero_query_lists_rows_in_index_order(monkeypatch, n, k):
    """Every score of an all-zero query is zero, +0.0 or -0.0 by the signs of the products (all-negative rows): one
    tie, so the list is the index order and every score reads +0.0."""
    q, r = make_case(n, 3, n, 64, 3, "dense", "cosine")
    q[:] = 0
    r[1::3] = -np.abs(r[1::3]) - 1
    for name, (score, idx, _) in run_routes(monkeypatch, q, r, k, "cosine").items():
        assert_exact(score, idx, np.zeros((3, k), np.float32), np.tile(np.arange(k), (3, 1)), name)


@pytest.mark.gpu
@pytest.mark.parametrize("largest", [True, False])
@pytest.mark.parametrize("n,k", [(16383, 4097), (16384, 1), (16384, 16384), (20000, 8193)])
def test_select_topk_signed_zero_nan_and_inf(largest, n, k):
    from image_retrieval_wavelet_b200.engine.get_knn import select_topk

    rng = np.random.default_rng(n + k)
    s = rng.integers(-3, 4, (7, n)).astype(np.float32)
    u = rng.random((7, n))
    s[(s == 0) & (u < 0.5)] = -0.0
    s[u > 0.95] = np.nan
    s[(u > 0.93) & (u <= 0.94)] = np.inf
    s[(u > 0.94) & (u <= 0.95)] = -np.inf
    s[1] = np.where(u[1] < 0.5, -0.0, 0.0)                      # one row of zeros of both signs
    s[2] = np.nan
    idx = rank_order(s, k, largest)
    want_s = np.take_along_axis(s, idx, 1) + np.float32(0)
    val, col = select_topk(torch.from_numpy(s).cuda(), k, largest)
    assert_exact(val, col, want_s, idx, f"largest={largest}")


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "l2"])
@pytest.mark.parametrize("n_shards,n,k,nan_step", [(3, 700, 700, 37), (8, 9000, 5000, 2)])
def test_sharded_merge_with_short_shards_and_nan_rows(metric, n_shards, n, k, nan_step):
    """Shards shorter than k (padded with index -1) and NaN rows that reach into the list: the merge equals the
    unsharded list and never picks padding while a real entry remains."""
    from image_retrieval_wavelet_b200.engine.dist import shard_bounds
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk, merge_knn_shards

    q, r = make_case(n + k, 17, n, 16, 3, "dense", metric)
    r[1::nan_step] = np.nan
    tr, tq = torch.from_numpy(r).cuda(), torch.from_numpy(q).cuda()
    want_s, want_i = oracle(q, r, k, metric)
    s_all, i_all = knn_topk(tr, tq, k, metric)
    assert_exact(s_all, i_all, want_s, want_i, "unsharded")
    ss, ii = [], []
    for b, e in shard_bounds(n, n_shards):
        s = torch.zeros((17, k), device="cuda")
        i = torch.full((17, k), -1, dtype=torch.int64, device="cuda")
        kl = min(k, e - b)
        if kl > 0:
            s[:, :kl], i_ = knn_topk(tr[b:e].contiguous(), tq, kl, metric)
            i[:, :kl] = i_ + b
        ss.append(s), ii.append(i)
    assert any(int((i < 0).sum()) for i in ii)
    got_i, got_s = merge_knn_shards(torch.stack(ss), torch.stack(ii), k, metric)
    assert_exact(got_s, got_i, want_s, want_i, "merged")
