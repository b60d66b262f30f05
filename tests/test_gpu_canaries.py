"""Out-of-bounds writes of the device kernels, caught with poisoned guard regions around every buffer the C-ABI writes
(compute-sanitizer is closed on this project's GPU pool: profiles/r2_sanitizer.md)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import eval_ref
from simlib import multi_hot, pm1

pytestmark = pytest.mark.gpu

GUARD = 4096


class Guarded:
    """A device buffer of `nbytes` with GUARD poisoned bytes on both sides."""

    def __init__(self, nbytes, fill=0):
        self.n = int(nbytes)
        self.raw = torch.full((self.n + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        self.raw[GUARD:GUARD + self.n] = fill
        self.ptr = self.raw.data_ptr() + GUARD

    def view(self, dtype):
        return self.raw[GUARD:GUARD + self.n].view(dtype)

    def intact(self):
        return bool((self.raw[:GUARD] == 0xA5).all()) and bool((self.raw[GUARD + self.n:] == 0xA5).all())


def _packed(seed, nq, n, bits, nlab):
    from image_retrieval_wavelet_b200.engine import hamming as H

    rng = np.random.default_rng(seed)
    q, r = pm1(rng, nq, bits), pm1(rng, n, bits)
    r[:nq] = q
    ql, rl = multi_hot(rng, nq, nlab, 0.15), multi_hot(rng, n, nlab, 0.15)
    return (q, ql, r, rl), (H.pack_codes(torch.from_numpy(q)), H.pack_labels(torch.from_numpy(ql)), H.pack_codes(torch.from_numpy(r)),
                            H.pack_labels(torch.from_numpy(rl)))


@pytest.mark.parametrize("env", [{"B200_MAP_SELECT": "1"}, {"B200_MAP_SELECT": "1", "B200_SEL_STRIDE": "4"}, {"B200_MAP_SELECT": "0"},
                                 {"B200_MAP_SELECT": "0", "B200_MAP_STASH": "0"}])
@pytest.mark.parametrize("nq,n,bits,nlab,k", [(37, 4099, 64, 24, 300), (130, 9001, 128, 80, 900), (5, 777, 200, 130, 50)])
def test_hamming_map_and_topk_stay_inside_their_buffers(monkeypatch, env, nq, n, bits, nlab, k):
    from image_retrieval_wavelet_b200 import _cabi

    for key, val in env.items():
        monkeypatch.setenv(key, val)
    (q, ql, r, rl), (qc, qlp, rc, rlp) = _packed(nq + n, nq, n, bits, nlab)
    lib = _cabi.load()
    plan = _cabi.MapPlan()
    _cabi.check(lib.b200_map_plan_init(ctypes.byref(plan), nq, n, n, bits, qlp.lw, qlp.mode, k), "plan")
    ws, ap, ts, m = Guarded(plan.workspace_bytes), Guarded(nq * 8), Guarded(nq * 4), Guarded(8)
    rc_ = lib.b200_hamming_map(ctypes.byref(plan), _cabi.ptr(qc.words), _cabi.ptr(qlp.words), _cabi.ptr(rc.words), _cabi.ptr(rlp.words),
                               ws.ptr, ap.ptr, ts.ptr, m.ptr, _cabi.stream_ptr())
    _cabi.check(rc_, "b200_hamming_map")
    torch.cuda.synchronize()
    assert ws.intact() and ap.intact() and ts.intact() and m.intact(), "b200_hamming_map wrote outside a buffer"
    m0, ap0, ts0, rank0, dist0 = eval_ref.maphashing_exact(q, ql, r, rl, k, return_details=True)
    assert np.array_equal(ts.view(torch.int32).cpu().numpy().astype(np.int64), ts0) and abs(m.view(torch.float64).item() - m0) <= 1e-6
    # the ranked list (label-free plan)
    plan2 = _cabi.MapPlan()
    _cabi.check(lib.b200_map_plan_init(ctypes.byref(plan2), nq, n, n, bits, 1, _cabi.LABELS_EQUAL, k), "plan")
    ws2, idx, dist = Guarded(plan2.workspace_bytes), Guarded(nq * k * 4), Guarded(nq * k * 2)
    _cabi.check(lib.b200_hamming_topk(ctypes.byref(plan2), _cabi.ptr(qc.words), _cabi.ptr(rc.words), ws2.ptr, idx.ptr, dist.ptr,
                                      _cabi.stream_ptr()), "b200_hamming_topk")
    torch.cuda.synchronize()
    assert ws2.intact() and idx.intact() and dist.intact(), "b200_hamming_topk wrote outside a buffer"
    assert np.array_equal(idx.view(torch.int32).cpu().numpy().reshape(nq, k).astype(np.int64), rank0)


def test_select_pool_overflow_stays_inside_the_pool(monkeypatch):
    """Collapsed codes: every row is a candidate of every query; the pool runs out and nothing may be written past it."""
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.engine import hamming as H

    monkeypatch.setenv("B200_MAP_SELECT", "1")
    rng = np.random.default_rng(1)
    nq, n, k = 200, 30000, 600
    ones_q, ones_r = torch.ones(nq, 64), torch.ones(n, 64)
    ql, rl = multi_hot(rng, nq, 12, 0.2), multi_hot(rng, n, 12, 0.2)
    qc, rc = H.pack_codes(ones_q), H.pack_codes(ones_r)
    qlp, rlp = H.pack_labels(torch.from_numpy(ql)), H.pack_labels(torch.from_numpy(rl))
    lib = _cabi.load()
    plan = _cabi.MapPlan()
    _cabi.check(lib.b200_map_plan_init(ctypes.byref(plan), nq, n, n, 64, qlp.lw, qlp.mode, k), "plan")
    assert plan.select == 1
    ws, ap, ts = Guarded(plan.workspace_bytes), Guarded(nq * 8), Guarded(nq * 4)
    _cabi.check(lib.b200_hamming_map(ctypes.byref(plan), _cabi.ptr(qc.words), _cabi.ptr(qlp.words), _cabi.ptr(rc.words),
                                     _cabi.ptr(rlp.words), ws.ptr, ap.ptr, ts.ptr, None, _cabi.stream_ptr()), "b200_hamming_map")
    torch.cuda.synchronize()
    assert ws.intact() and ap.intact() and ts.intact()
    flags = ws.view(torch.uint8)[plan.off_sel_flags:plan.off_sel_flags + 16].view(torch.int32).cpu()
    assert int(flags[1]) == 1                              # the fallback really ran
    want, hits = eval_ref.ap_from_ranked_relevance((ql[3] @ rl[:k].T) > 0)
    assert int(ts.view(torch.int32)[3]) == hits and abs(float(ap.view(torch.float64)[3]) - want) <= 1e-6


@pytest.mark.parametrize("fused,k,n,top_tie", [pytest.param("1", 1000, 70000, False, id="1-1000-70000"),
                                               pytest.param("0", 1000, 70000, False, id="0-1000-70000"),
                                               pytest.param("1", 5000, 20000, False, id="1-5000-20000"),
                                               pytest.param("1", 2048, 70001, True, id="1-2048-70001-top_tie")])
def test_knn_topk_stays_inside_its_buffers(monkeypatch, fused, k, n, top_tie):
    """top_tie: every 7th row is the best row of every query (integer inputs, 10 001 exact ties): the fused path's
    candidate lists and the select kernel's candidate buffer overflow, and the fallbacks run."""
    from image_retrieval_wavelet_b200 import _cabi

    monkeypatch.setenv("B200_KNN_FUSED", fused)
    g = torch.Generator().manual_seed(n)
    nq, d = 70, 64
    if top_tie:
        refs = torch.randint(-3, 4, (n, d), generator=g).float()
        qs = torch.randint(-3, 4, (nq, d), generator=g).float()
        qs[:, 0] = 100
        refs[::7] = 0
        refs[::7, 0] = 100
        refs, qs = refs.cuda(), qs.cuda()
    else:
        refs = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).cuda()
        qs = torch.nn.functional.normalize(torch.randn(nq, d, generator=g), dim=1).cuda()
    lib = _cabi.load()
    nbytes = lib.b200_knn_workspace_bytes(nq, n, d, k)
    ws, idx, score = Guarded(nbytes), Guarded(nq * k * 8), Guarded(nq * k * 4)
    _cabi.check(lib.b200_knn_topk(_cabi.ptr(refs), _cabi.ptr(qs), nq, n, d, k, 0, idx.ptr, score.ptr, ws.ptr, nbytes, _cabi.stream_ptr()),
                "b200_knn_topk")
    torch.cuda.synchronize()
    assert ws.intact() and idx.intact() and score.intact(), "b200_knn_topk wrote outside a buffer"
    want = torch.topk(qs.double() @ refs.double().T, k, dim=1).values
    assert (score.view(torch.float32).reshape(nq, k).double() - want).abs().max().item() <= 1e-5
    if top_tie:                                            # the tied rows in index order
        assert torch.equal(idx.view(torch.int64).reshape(nq, k).cpu(), torch.arange(0, 7 * k, 7).expand(nq, k))


# per level, a short, an 8-tap and a long filter: level 1 two-pass (uint8 in 4- or 8-pixel staging units by W), sliding
# last pass, two-pass F = 10; levels 2-3 hybrid, two-pass F = 8, two-pass F = 10; level 4 the generic program
CANARY_FILTERS = {1: ("haar", "db4", "bior4.4"), 2: ("db2", "sym4", "bior4.4"), 3: ("db2", "sym4", "bior4.4"), 4: ("haar", "db2", "db4")}


@pytest.mark.parametrize("filt", [0, 1, 2])
@pytest.mark.parametrize("shape,level,u8", [((2, 3, 70, 518), 1, True), ((1, 2, 136, 200), 2, True), ((1, 1, 256, 256), 3, False),
                                            ((1, 1, 8, 8), 3, True), ((2, 3, 64, 224), 1, True), ((1, 1, 24, 36), 1, False),
                                            ((1, 1, 64, 64), 4, False)])
def test_swt_stays_inside_its_output(filt, shape, level, u8):
    """Guard bytes around the input and the output of b200_swt2_fwd, for every planned pass form and both uint8 staging
    forms (filt: index into CANARY_FILTERS[level])."""
    from image_retrieval_wavelet_b200 import _cabi
    from oracle import c_oracle, filters

    rng = np.random.default_rng(sum(shape))
    x = rng.integers(0, 256, shape).astype(np.uint8) if u8 else rng.random(shape, dtype=np.float32)
    lo, hi = filters.filter_bank(CANARY_FILTERS[level][filt])
    b, c, h, w = shape
    xin = Guarded(x.nbytes)
    xin.view(torch.uint8).copy_(torch.from_numpy(x.view(np.uint8).reshape(-1)))
    out = Guarded(b * c * 4 * h * w * 4)
    flo, fhi = (ctypes.c_float * len(lo))(*lo), (ctypes.c_float * len(hi))(*hi)
    # the input sits 4096 bytes into an allocation: 16-byte aligned, as the entry point asks
    _cabi.check(_cabi.load().b200_swt2_fwd(xin.ptr, int(u8), out.ptr, b, c, h, w, flo, fhi, len(lo), level, _cabi.stream_ptr()),
                "b200_swt2_fwd")
    torch.cuda.synchronize()
    assert out.intact() and xin.intact()
    ref = c_oracle.swt2(x, lo, hi, level)
    got = out.view(torch.float32).cpu().numpy().reshape(b, c, 4, h, w)
    assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()
