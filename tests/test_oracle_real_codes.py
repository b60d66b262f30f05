"""Real-valued codes on the CPU: the oracle of the float Hamming route (C distances, ``maphashing_real_exact``) against the
exact +-1 oracle, the reference's literal op sequence and exact integer arithmetic; and the host-side argument checks of
``b200_real_hamming_dist``, which run before any CUDA call."""
import ctypes

import numpy as np
import pytest

from oracle import eval_ref, real_codes
from simlib import multi_hot, pm1


@pytest.mark.parametrize("nbits", [1, 5, 17, 64, 300])
def test_c_distances_are_exact_on_integer_codes(nbits):
    """Small integers (zeros included): every partial sum is exact, so the fmaf chain equals 0.5 * (B - q @ r.T) in float64."""
    rng = np.random.default_rng(nbits)
    q = rng.integers(-3, 4, (9, nbits)).astype(np.float32)
    r = rng.integers(-3, 4, (31, nbits)).astype(np.float32)
    got = real_codes.real_hamming_dist(q, r)
    want = 0.5 * (nbits - q.astype(np.float64) @ r.astype(np.float64).T)
    assert got.dtype == np.float32 and np.array_equal(got.astype(np.float64), want)


def test_c_distances_take_nbits_and_zero_padding():
    """Zero columns past nbits add nothing: the device route pads D to a multiple of 4 and passes the code width."""
    rng = np.random.default_rng(1)
    q, r = rng.standard_normal((5, 17)).astype(np.float32), rng.standard_normal((8, 17)).astype(np.float32)
    pad = lambda x: np.pad(x, ((0, 0), (0, 3)))                         # noqa: E731
    assert np.array_equal(real_codes.real_hamming_dist(pad(q), pad(r), nbits=17), real_codes.real_hamming_dist(q, r))


def _golden_case(g, name):
    q, r, ql, rl = (g[f"{name}/{k}"] for k in ("q", "r", "ql", "rl"))
    tk, inc = (int(v) for v in g[f"{name}/topk"])
    topk = None if tk == -1 else ("max_bin_count" if tk == -2 else tk)
    return q.astype(np.float32), ql, r.astype(np.float32), rl, topk, bool(inc)


def _same(a, b):
    m1, ap1, ts1, rk1, d1 = a
    m2, ap2, ts2, rk2, d2 = b
    assert m1 == m2 and np.array_equal(ap1, ap2) and np.array_equal(ts1, ts2) and np.array_equal(rk1, rk2)
    assert np.array_equal(d1.astype(np.int64), d2)


def test_real_exact_equals_exact_on_pm1_goldens(golden):
    """The reference's own +-1 fixtures: the float route ranks them exactly like the integer one."""
    n_cases = 0
    for name in golden["cases"]:
        q, ql, r, rl, topk, inc = _golden_case(golden, name)
        if not (np.all(np.abs(q) == 1) and np.all(np.abs(r) == 1)):
            continue
        n_cases += 1
        _same(real_codes.maphashing_real_exact(q, ql, r, rl, topk, inc, return_details=True),
              eval_ref.maphashing_exact(q, ql, r, rl, topk, inc, return_details=True))
        assert abs(real_codes.maphashing_real_exact(q, ql, r, rl, topk, inc) - float(golden[f"{name}/map_reference_stable"])) <= 1e-6
    assert n_cases >= 3


@pytest.mark.parametrize("nq,n,bits,nlab,k", [(20, 300, 64, 12, 50), (7, 1000, 17, -1, None), (12, 500, 130, 40, 1000),
                                              (5, 64, 8, 4, 0)])
def test_real_exact_equals_exact_on_pm1_codes(nq, n, bits, nlab, k):
    rng = np.random.default_rng(nq * n)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    r[:nq] = q                                                          # exact duplicates: ties at distance 0
    ql, rl = (multi_hot(rng, nq, nlab, 0.2), multi_hot(rng, n, nlab, 0.2)) if nlab > 0 else \
        (rng.integers(0, 5, nq), rng.integers(0, 5, n))
    _same(real_codes.maphashing_real_exact(q, ql, r, rl, k, return_details=True),
          eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True))


def _separated_fixture(seed, nq, n, bits, gap):
    """Continuous codes whose distances (per query) are at least `gap` apart: any summation order ranks them alike."""
    rng = np.random.default_rng(seed)
    q = rng.standard_normal((nq, bits)).astype(np.float32)
    cand = rng.standard_normal((40 * n, bits)).astype(np.float32)
    d = 0.5 * (bits - q.astype(np.float64) @ cand.astype(np.float64).T)
    keep = []
    for j in range(cand.shape[0]):
        if not keep or np.abs(d[:, keep] - d[:, j:j + 1]).min() > gap:
            keep.append(j)
            if len(keep) == n:
                break
    assert len(keep) == n
    return q, cand[keep]


@pytest.mark.parametrize("two_d", [True, False])
@pytest.mark.parametrize("k", [None, 10, "max_bin_count"])
def test_real_exact_matches_literal_reference_on_separated_codes(two_d, k):
    q, r = _separated_fixture(3, 6, 150, 32, 0.02)
    rng = np.random.default_rng(4)
    ql, rl = (multi_hot(rng, 6, 5, 0.3), multi_hot(rng, 150, 5, 0.3)) if two_d else \
        (rng.integers(0, 4, 6), rng.integers(0, 4, 150))
    got = real_codes.maphashing_real_exact(q, ql, r, rl, k)
    assert abs(got - eval_ref.maphashing_literal(q, ql, r, rl, k)) <= 1e-6
    # and the float distances order the rows as float64 arithmetic does
    _, _, _, ranked, _ = real_codes.maphashing_real_exact(q, ql, r, rl, None, return_details=True)
    d64 = 0.5 * (32 - q.astype(np.float64) @ r.astype(np.float64).T)
    assert np.array_equal(ranked, np.argsort(d64, axis=1, kind="stable"))


def test_real_exact_ranks_nan_last_and_ties_by_index():
    q = np.array([[1.0, 0.0, 0.5, -2.0]], np.float32)
    r = np.array([[np.nan, 0, 0, 0], [1, 0, 0.5, -2], [0, 0, 0, 0], [1, 0, 0.5, -2], [np.inf, 0, 0, 0], [0, 1, 0, 0]],
                 np.float32)
    _, _, _, ranked, d = real_codes.maphashing_real_exact(q, np.zeros(1), r, np.zeros(6), None, return_details=True)
    # distances: nan, -0.625, 2, -0.625, -inf, 2
    assert ranked[0].tolist() == [4, 1, 3, 2, 5, 0] and np.isnan(d[0, -1])
    assert real_codes.maphashing_real_exact(q, np.zeros(1), r, np.zeros(6), 0) == 0.0


def test_real_hamming_dist_checks_arguments_before_any_cuda_call():
    """Rejected on the host: these calls are safe without a device."""
    from image_retrieval_wavelet_b200 import _cabi

    fn = _cabi.load().b200_real_hamming_dist
    p = ctypes.c_void_p(4096)                                           # never dereferenced: every call below is rejected
    assert fn(None, p, 2, 3, 8, 8, p, 4, None) == _cabi.ERR_INVALID_ARG
    assert fn(p, p, -1, 3, 8, 8, p, 4, None) == _cabi.ERR_INVALID_ARG
    assert fn(p, p, 2, 3, 8, 0, p, 4, None) == _cabi.ERR_INVALID_ARG    # nbits < 1
    assert fn(p, p, 2, 3, 8, 9, p, 4, None) == _cabi.ERR_INVALID_ARG    # nbits > D
    assert fn(p, p, 2, 5, 8, 8, p, 4, None) == _cabi.ERR_INVALID_ARG    # ldS < N
    assert fn(p, p, 2, 3, 6, 6, p, 4, None) == _cabi.ERR_UNSUPPORTED    # D % 4
    assert fn(p, p, 2, 3, 8, 8, p, 6, None) == _cabi.ERR_ALIGNMENT      # ldS % 4
    assert fn(p, p, 2, 3, 8, 8, ctypes.c_void_p(4100), 4, None) == _cabi.ERR_ALIGNMENT
    assert fn(None, None, 0, 3, 8, 8, None, 4, None) == _cabi.OK       # empty is a no-op
