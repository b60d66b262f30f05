"""Select pipeline of the Hamming evaluator (csrc/hamming_select.cu) on a B200 against the CPU oracle: sampled bound ->
candidate lists -> one warp per query.  Same bar as test_gpu_eval.py: hit counts, ranked indices and distances
bit-exact, AP within 1e-6 — including the cases where the sample misleads (bound lifted for those queries) and where
the candidate pool overflows (the gated three-stage path takes over)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import c_oracle, eval_ref
from simlib import correlated_codes, multi_hot, pm1, words

pytestmark = pytest.mark.gpu

AP_TOL = 1e-6


def _run(q, ql, r, rl, k, want_rank=True):
    from image_retrieval_wavelet_b200.engine import hamming as H

    qc, rc = H.pack_codes(torch.from_numpy(q)), H.pack_codes(torch.from_numpy(r))
    qlp, rlp = H.pack_labels(torch.from_numpy(ql)), H.pack_labels(torch.from_numpy(rl))
    m, ap, ts, ws = H.hamming_map(qc, qlp, rc, rlp, k, return_workspace=True)
    st = H.select_status(ws)
    out = {"m": m.item(), "ap": ap.cpu().numpy(), "ts": ts.cpu().numpy().astype(np.int64), "status": st}
    if want_rank:
        idx, dist, ws2 = H.hamming_topk(qc, rc, k, return_workspace=True)
        out["idx"], out["dist"] = idx.cpu().numpy(), dist.cpu().numpy().astype(np.int64)
        out["status_topk"] = H.select_status(ws2)
    return out


def _check(out, q, ql, r, rl, k):
    m0, ap0, ts0, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    assert np.array_equal(out["ts"], ts0), out["status"]
    assert np.abs(out["ap"] - ap0).max() <= AP_TOL and abs(out["m"] - m0) <= AP_TOL, out["status"]
    if "idx" in out:
        assert np.array_equal(out["idx"], rank0) and np.array_equal(out["dist"], dist0), out["status_topk"]


SMALL = [
    (37, 2000, 64, 24, 50), (20, 3000, 32, 20, 700), (33, 4096, 128, 80, 1500), (9, 2000, 96, 130, 100),
    (40, 5000, 48, -1, 300), (3, 777, 17, 3, 10), (130, 6000, 254, 38, 600), (5, 64, 64, 8, 2), (200, 2049, 200, 200, 1024),
]


@pytest.mark.parametrize("stride", [0, 2, 5])
@pytest.mark.parametrize("nq,n,bits,nlab,k", SMALL)
def test_select_pipeline_matches_exact_oracle(monkeypatch, nq, n, bits, nlab, k, stride):
    monkeypatch.setenv("B200_MAP_SELECT", "1")
    if stride:
        monkeypatch.setenv("B200_SEL_STRIDE", str(stride))
    rng = np.random.default_rng(nq * 1000 + n + bits)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    r[:nq] = q
    r[:nq, :3] *= -1                                                # near-duplicates: short distances exist
    if nlab > 0:
        ql, rl = multi_hot(rng, nq, nlab, 0.1), multi_hot(rng, n, nlab, 0.1)
    else:
        ql, rl = rng.integers(0, 6, nq), rng.integers(0, 6, n)
    out = _run(q, ql, r, rl, k)
    assert out["status"] is not None and not out["status"]["fell_back"], out["status"]     # the pipeline under test is the one that ran
    _check(out, q, ql, r, rl, k)


def test_misleading_sample_lifts_the_bound(monkeypatch):
    """Near neighbours only in the SAMPLED 32-row groups: the sample promises 4x more rows within the bound than
    there are, the lists come out shorter than k, and those queries are redone with every row listed."""
    monkeypatch.setenv("B200_MAP_SELECT", "1")
    monkeypatch.setenv("B200_SEL_STRIDE", "4")
    rng = np.random.default_rng(3)
    nq, n, bits, k = 24, 8192, 64, 600
    q = pm1(rng, nq, bits)
    r = pm1(rng, n, bits)
    near = q[rng.integers(0, nq, n)].copy()
    flips = rng.integers(0, bits, (n, 6))
    for c in range(6):
        near[np.arange(n), flips[:, c]] *= -1
    sampled = ((np.arange(n) // 32) % 4) == 0
    r[sampled] = near[sampled]                                      # close rows exactly where the sample looks
    ql, rl = multi_hot(rng, nq, 12, 0.2), multi_hot(rng, n, 12, 0.2)
    out = _run(q, ql, r, rl, k)
    assert not out["status"]["fell_back"] and out["status"]["queries_redone"] > 0, out["status"]
    _check(out, q, ql, r, rl, k)


def test_collapsed_codes_overflow_the_pool_and_fall_back(monkeypatch):
    """One code for everybody (the collapsed-code floor, RESULTS.md:460): every row ties at distance 0, every row is a
    candidate of every query, the pool cannot hold that and the three-stage path takes over — ranking = index order."""
    monkeypatch.setenv("B200_MAP_SELECT", "1")
    rng = np.random.default_rng(4)
    nq, n, k = 300, 40000, 700
    q, r = np.ones((nq, 64), np.float32), np.ones((n, 64), np.float32)
    ql, rl = multi_hot(rng, nq, 20, 0.15), multi_hot(rng, n, 20, 0.15)
    out = _run(q, ql, r, rl, k, want_rank=True)
    assert out["status"]["fell_back"], out["status"]
    assert np.array_equal(out["idx"], np.tile(np.arange(k), (nq, 1))) and (out["dist"] == 0).all()
    for i in (0, 17, 299):
        want, hits = eval_ref.ap_from_ranked_relevance((ql[i] @ rl[:k].T) > 0)
        assert out["ts"][i] == hits and abs(out["ap"][i] - want) <= AP_TOL


def test_class_sorted_database(monkeypatch):
    """Database stored class by class: the top k of a query sit in a few segments (lists of very uneven length)."""
    monkeypatch.setenv("B200_MAP_SELECT", "1")
    rng = np.random.default_rng(5)
    nq, n, bits, k = 64, 50000, 64, 1000
    cls_r = np.sort(rng.integers(0, 25, n))
    cls_q = rng.integers(0, 25, nq)
    proto = pm1(rng, 25, bits)

    def noisy(c):
        x = proto[c].copy()
        x[rng.random(x.shape) < 0.12] *= -1
        return x

    q, r = noisy(cls_q), noisy(cls_r)
    out = _run(q, cls_q, r, cls_r, k)
    assert not out["status"]["fell_back"], out["status"]
    _check(out, q, cls_q, r, cls_r, k)


@pytest.mark.parametrize("select", ["1", "0"])
def test_c3_full_size_both_pipelines_agree(monkeypatch, select):
    """BASELINE configs[2] at full size: select pipeline (default there) and three-stage path give the same bits; a query
    sample against the C oracle."""
    from image_retrieval_wavelet_b200.engine import hamming as H

    monkeypatch.setenv("B200_MAP_SELECT", select)
    rng = np.random.default_rng(117)
    nq, n, k = 5000, 117000, 5000
    ql, rl = multi_hot(rng, nq, 80, 0.036), multi_hot(rng, n, 80, 0.036)
    q, r = correlated_codes(rng, ql, rl, 128)
    qc, rc = H.pack_codes(torch.from_numpy(q)), H.pack_codes(torch.from_numpy(r))
    qlp, rlp = H.pack_labels(torch.from_numpy(ql)), H.pack_labels(torch.from_numpy(rl))
    m, ap, ts, ws = H.hamming_map(qc, qlp, rc, rlp, k, return_workspace=True)
    st = H.select_status(ws)
    assert (st is not None and not st["fell_back"]) if select == "1" else st is None, st
    sub = rng.choice(nq, 48, replace=False)
    m0, ap0, ts0 = c_oracle.maphashing(q[sub], ql[sub], r, rl, k)
    assert np.array_equal(ts.cpu().numpy()[sub].astype(np.int64), ts0), st
    assert np.abs(ap.cpu().numpy()[sub] - ap0).max() <= AP_TOL
    # checksum over ALL queries, compared between the two parametrisations through a module-level memo
    key = (float(m.item()), int(ts.sum().item()))
    seen = _C3_MEMO.setdefault("c3", key)
    assert seen == key, (seen, key, st)


_C3_MEMO = {}


def test_c5_scale_out_shape_query_sample():
    """BASELINE configs[4] (10 000 x 1 000 000, 64 bit, mAP@5000) on one GPU: a query sample against the C oracle, and the
    ranked list of a few queries against the exact numpy oracle."""
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(1000000)
    nq, n, k = 10000, 1000000, 5000
    ql, rl = multi_hot(rng, nq, 80, 0.036), multi_hot(rng, n, 80, 0.036)
    q, r = correlated_codes(rng, ql, rl, 64)
    qc, rc = H.pack_codes(torch.from_numpy(q)), H.pack_codes(torch.from_numpy(r))
    qlp, rlp = H.pack_labels(torch.from_numpy(ql)), H.pack_labels(torch.from_numpy(rl))
    m, ap, ts, ws = H.hamming_map(qc, qlp, rc, rlp, k, return_workspace=True)
    st = H.select_status(ws)
    assert st is not None and not st["fell_back"], st
    sub = rng.choice(nq, 24, replace=False)
    m0, ap0, ts0 = c_oracle.maphashing(q[sub], ql[sub], r, rl, k)
    assert np.array_equal(ts.cpu().numpy()[sub].astype(np.int64), ts0), st
    assert np.abs(ap.cpu().numpy()[sub] - ap0).max() <= AP_TOL
    assert abs(m.item() - ap.mean().item()) <= 1e-12


@pytest.mark.parametrize("nq,n,bits,nlab,k", [(300, 6000, 128, 80, 600), (130, 9000, 64, 24, 700), (256, 5000, 200, -1, 512),
                                               (64, 6000, 128, 80, 600), (40, 9000, 64, 24, 700), (33, 5000, 200, -1, 512)])
def test_tensor_core_select_kernel_agrees(monkeypatch, nq, n, bits, nlab, k):
    """The tcgen05 form of the select pass (distances as e4m3 dot products of the +-1 codes, TMA tiles, TMEM accumulators,
    hit masks, SIMT append; DESIGN 4.2), which the plan picks for 128-query groups, and the SIMT kernel, which it picks for
    fewer queries, give the oracle's lists — hit counts bit-exact, AP within 1e-6 — and the form the plan picks is the one
    that runs (the tensor-core form's "expand" and "filter" stages show up in the stage times)."""
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.engine.map_engine import HammingMapEngine

    monkeypatch.setenv("B200_MAP_SELECT", "1")
    plan = _cabi.MapPlan()
    assert _cabi.load().b200_map_plan_init(ctypes.byref(plan), nq, n, n, bits, words(max(nlab, 1)), 0 if nlab > 0 else 1, k) == 0
    tc = plan.off_smp_codes != plan.workspace_bytes
    assert plan.select == 1 and tc == (nq >= 128), (plan.select, plan.sel_T)
    rng = np.random.default_rng(nq + n + bits)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    r[:nq] = q
    r[:nq, :3] *= -1
    if nlab > 0:
        ql, rl = multi_hot(rng, nq, nlab, 0.1), multi_hot(rng, n, nlab, 0.1)
    else:
        ql, rl = rng.integers(0, 6, nq), rng.integers(0, 6, n)
    eng = HammingMapEngine(use_graph=False)
    m, ap, ts = eng.evaluate(torch.from_numpy(q).cuda(), torch.from_numpy(ql).cuda(), torch.from_numpy(r).cuda(),
                             torch.from_numpy(rl).cuda(), k)
    stages = eng.stage_ms()
    eng.close()
    assert ("expand" in stages and "filter" in stages) == tc, stages
    m0, ap0, ts0, _, _ = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    assert np.array_equal(ts.cpu().numpy().astype(np.int64), ts0)
    assert np.abs(ap.cpu().numpy() - ap0).max() <= AP_TOL and abs(m - m0) <= AP_TOL
