"""Real-valued codes on a B200: ``on_nonbinary='real'`` ranks codes that are not all +-1 by the reference's float32
``0.5 * (B - q @ r.T)``.

Bar: distances bit-identical to the C oracle (same fmaf chain; NaN where it has NaN); ranked indices (index tie-break,
NaN last) and per-query hit counts bit-exact against ``maphashing_real_exact``; AP / mAP within 1e-6 of it."""
import numpy as np
import pytest
import torch

from oracle import eval_ref, real_codes
from simlib import multi_hot, pm1

pytestmark = pytest.mark.gpu

AP_TOL = 1e-6


def _calc(mode, k=None):
    from image_retrieval_wavelet_b200.engine import CustomCalculator

    return CustomCalculator(k=k, distance_metric="hamming", with_faiss=False, on_nonbinary=mode)


def _logits(rng, n, bits, specials=True):
    x = rng.standard_normal((n, bits)).astype(np.float32)
    if specials:
        x[rng.random((n, bits)) < 0.08] = 0.0                        # sign(0) entries
    return x


def _labels(rng, nq, n, two_d):
    if two_d:
        return multi_hot(rng, nq, 12, 0.15), multi_hot(rng, n, 12, 0.15)
    return rng.integers(0, 5, nq), rng.integers(0, 5, n)


def _same_bits(got, want):
    """float32 arrays equal bit for bit, NaN matching NaN (payloads are not part of the contract)."""
    assert got.shape == want.shape and got.dtype == np.float32
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


# ------------------------------------------------------------------------------------------------ distances
@pytest.mark.parametrize("nbits", [1, 17, 48, 64, 128, 300, 768])
def test_distances_bit_identical_to_c_oracle(nbits):
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(nbits)
    q, r = _logits(rng, 37, nbits), _logits(rng, 1001, nbits)
    q[3, rng.integers(0, nbits)] = np.inf
    q[5, 0] = -np.inf
    r[10, rng.integers(0, nbits)] = np.nan
    r[11, nbits - 1] = np.inf
    r[12] = 0.0
    got = H.real_hamming_dist(_cuda(q), _cuda(r), nbits)
    assert tuple(got.shape) == (37, 1001) and got.dtype == torch.float32
    want = real_codes.real_hamming_dist(q, r)
    _same_bits(got.cpu().numpy(), want)
    assert np.isnan(want).any() and np.isinf(want).any()


def test_distance_buffer_guards_and_row_padding_stay_intact():
    """b200_real_hamming_dist writes columns [0, N) of each row and nothing else: not the ldS padding, not the guards."""
    from image_retrieval_wavelet_b200 import _cabi

    rng = np.random.default_rng(5)
    nq, n, d, ld, guard = 130, 1001, 20, 1012, 64
    q, r = _logits(rng, nq, d), _logits(rng, n, d)
    sentinel = np.int32(0x7FBADBAD)
    buf = torch.full((2 * guard + nq * ld,), int(sentinel), dtype=torch.int32, device="cuda")
    dist = buf[guard:guard + nq * ld]
    qd, rd = _cuda(q), _cuda(r)
    rc = _cabi.load().b200_real_hamming_dist(_cabi.ptr(qd), _cabi.ptr(rd), nq, n, d, d, _cabi.ptr(dist), ld, _cabi.stream_ptr())
    assert rc == _cabi.OK
    host = buf.cpu().numpy()
    assert (host[:guard] == sentinel).all() and (host[guard + nq * ld:] == sentinel).all()
    rows = host[guard:guard + nq * ld].reshape(nq, ld)
    assert (rows[:, n:] == sentinel).all()
    _same_bits(rows[:, :n].view(np.float32).copy(), real_codes.real_hamming_dist(q, r))


# ------------------------------------------------------------------------------------------------ ranking and mAP
N_RANK = 6000
K_CASES = [0, 1, 7, 4096, 4097, N_RANK, None, N_RANK + 5, "max_bin_count"]


@pytest.fixture(scope="module", params=[False, True], ids=["labels1d", "labels2d"])
def rank_problem(request):
    rng = np.random.default_rng(11 + int(request.param))
    nq, bits = 40, 48
    q, r = _logits(rng, nq, bits), _logits(rng, N_RANK, bits)
    r[3000:3100] = r[:100]                                            # exact ties: index order decides
    r[7, 5] = np.nan                                                  # a NaN distance for every query: ranks last
    ql, rl = _labels(rng, nq, N_RANK, request.param)
    return q, ql, r, rl


@pytest.mark.parametrize("k", K_CASES)
def test_map_and_ranking_match_real_exact_oracle(rank_problem, k):
    from image_retrieval_wavelet_b200.engine import hamming as H
    from image_retrieval_wavelet_b200.engine.get_knn import select_topk

    q, ql, r, rl = rank_problem
    m, ap, hits = _calc("real").maphashing_details(_cuda(q), _cuda(ql), _cuda(r), _cuda(rl), k)
    m_o, ap_o, ts_o, ranked_o, _ = real_codes.maphashing_real_exact(q, ql, r, rl, k, return_details=True)
    assert np.array_equal(hits.cpu().numpy().astype(np.int64), ts_o)
    assert np.abs(ap.cpu().numpy() - ap_o).max() <= AP_TOL and abs(m.item() - m_o) <= AP_TOL
    kk = ranked_o.shape[1]
    if kk:
        # the route's ranking: the same distances through the same selection
        _, idx = select_topk(H.real_hamming_dist(_cuda(q), _cuda(r), q.shape[1]), kk, largest=False)
        assert np.array_equal(idx.cpu().numpy(), ranked_o)
    else:
        assert m.item() == 0.0 and not ap.any() and not hits.any()


def test_small_chunks_give_the_same_bytes(rank_problem):
    from image_retrieval_wavelet_b200.engine import hamming as H

    q, ql, r, rl = rank_problem
    pq, pr = H.pack_labels(_cuda(ql)), H.pack_labels(_cuda(rl))
    one = H.real_hamming_map(_cuda(q), pq, _cuda(r), pr, 4097)
    for chunk in (1, 7, 16):
        part = H.real_hamming_map(_cuda(q), pq, _cuda(r), pr, 4097, chunk=chunk)
        assert all(torch.equal(a, b) for a, b in zip(one, part)), chunk


def test_ternary_sign_codes_are_exact():
    """torch.sign of logits keeps exact zeros: integer distances, ranked exactly."""
    rng = np.random.default_rng(3)
    q, r = np.sign(_logits(rng, 25, 64)), np.sign(_logits(rng, 3000, 64))
    ql, rl = _labels(rng, 25, 3000, True)
    c = _calc("real")
    d = c.calc_hamming_dist(_cuda(q), _cuda(r)).cpu().numpy()
    assert np.array_equal(d.astype(np.float64), 0.5 * (64 - q.astype(np.float64) @ r.astype(np.float64).T))
    m, ap, hits = c.maphashing_details(_cuda(q), _cuda(ql), _cuda(r), _cuda(rl), 500)
    m_o, ap_o, ts_o, _, _ = real_codes.maphashing_real_exact(q, ql, r, rl, 500, return_details=True)
    assert np.array_equal(hits.cpu().numpy().astype(np.int64), ts_o) and np.abs(ap.cpu().numpy() - ap_o).max() <= AP_TOL
    assert abs(c.calculate_maphashing(_cuda(q), _cuda(ql), _cuda(r), _cuda(rl), 500) - m_o) <= AP_TOL


@pytest.mark.parametrize("two_d", [False, True])
def test_pm1_codes_take_the_packed_path_and_the_float_route_agrees(two_d):
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(21)
    q, r = pm1(rng, 50, 128), pm1(rng, 4000, 128)
    r[:50] = q
    ql, rl = _labels(rng, 50, 4000, two_d)
    args = (_cuda(q), _cuda(ql), _cuda(r), _cuda(rl), 300)
    real, default = _calc("real").maphashing_details(*args), _calc("raise").maphashing_details(*args)
    assert all(torch.equal(a, b) for a, b in zip(real, default))                     # same bytes: the packed path ran
    assert torch.equal(_calc("real").calc_hamming_dist(_cuda(q), _cuda(r)), _calc("raise").calc_hamming_dist(_cuda(q), _cuda(r)))
    # the float route forced on the same +-1 codes: the packed integers, the same ranking, the same hits
    from image_retrieval_wavelet_b200.engine.get_knn import select_topk

    qc, rc = H.pack_codes(_cuda(q)), H.pack_codes(_cuda(r))
    dist = H.real_hamming_dist(_cuda(q), _cuda(r), 128)
    assert torch.equal(dist, H.hamming_dist(qc, rc))
    assert torch.equal(select_topk(dist, 300, largest=False)[1], H.hamming_topk(qc, rc, 300)[0])
    m, ap, hits = H.real_hamming_map(_cuda(q), H.pack_labels(_cuda(ql)), _cuda(r), H.pack_labels(_cuda(rl)), 300)
    assert torch.equal(hits, default[2]) and (ap - default[1]).abs().max().item() <= AP_TOL
    assert abs(m.item() - default[0].item()) <= AP_TOL


def test_codes_wider_than_the_packed_format():
    """No width limit on the float route: 300-bit +-1 codes under 'real' rank exactly like the integer oracle."""
    rng = np.random.default_rng(8)
    q, r = pm1(rng, 20, 300), pm1(rng, 2000, 300)
    ql, rl = _labels(rng, 20, 2000, True)
    got = _calc("real", k=100).calculate_maphashing(_cuda(q), _cuda(ql), _cuda(r), _cuda(rl), 100)
    assert abs(got - eval_ref.maphashing_exact(q, ql, r, rl, 100)) <= AP_TOL
    with pytest.raises(NotImplementedError):
        _calc("raise").calculate_maphashing(_cuda(q), _cuda(ql), _cuda(r), _cuda(rl), 100)     # default: unchanged


def test_edge_cases_and_unsupported_metrics():
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(2)
    q, ql = _logits(rng, 6, 20), rng.integers(0, 3, 6)
    c = _calc("real")
    m, ap, hits = c.maphashing_details(_cuda(q), _cuda(ql), _cuda(q[:0]), _cuda(ql[:0]), 5)             # N == 0
    assert m.item() == 0.0 and not ap.any() and not hits.any()
    m, ap, hits = c.maphashing_details(_cuda(q), _cuda(ql), _cuda(q), _cuda(ql), -3)                     # k < 1
    assert m.item() == 0.0 and not ap.any()
    with pytest.raises(ValueError):
        _calc("raise").calculate_maphashing(_cuda(q), _cuda(ql), _cuda(q), _cuda(ql), 5)                 # default: unchanged
    with pytest.raises(NotImplementedError):
        c.calculate_pr_rc_hashing(_cuda(q), _cuda(ql), _cuda(q), _cuda(ql))
    with pytest.raises(ValueError):
        H.real_hamming_map(_cuda(q), H.pack_labels(_cuda(ql)), _cuda(q[:, :16]), H.pack_labels(_cuda(ql)), 5)


# ------------------------------------------------------------------------------------------------ in-training proxy
@pytest.mark.parametrize("bits", [64, 128])
@pytest.mark.parametrize("batch", [96, 256, 1024])
def test_batch_map_on_raw_logits_is_the_reference_number(batch, bits):
    """batch_map.py:9-36 on raw logits, as the reference's training loop calls it."""
    from image_retrieval_wavelet_b200.engine import build_batch_map_calculator, compute_batch_map

    rng = np.random.default_rng(batch + bits)
    logits = rng.standard_normal((batch, bits)).astype(np.float32)
    lab = multi_hot(rng, batch, 10, 0.2)
    calc, name = build_batch_map_calculator("hamming", torch.device("cuda"), on_nonbinary="real")
    got = compute_batch_map(calc, name, _cuda(logits).requires_grad_(), _cuda(lab))
    assert abs(got - real_codes.maphashing_real_exact(logits, lab, logits, lab, "max_bin_count", True)) <= AP_TOL
    assert abs(got - eval_ref.maphashing_literal(logits, lab, logits, lab, "max_bin_count", True)) <= 1e-3
