"""Test support: loader for ``libb200ret_sim.so`` + synthetic-data and packing helpers shared by the tests."""
import ctypes
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SIM = None


def load_sim():
    global _SIM
    if _SIM is None:
        from image_retrieval_wavelet_b200 import build

        _SIM = ctypes.CDLL(os.environ.get("B200RET_SIM_LIB") or build.build_sim())      # override: a sanitizer build (tools/sim_asan.sh)
    return _SIM


def vp(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def words(n):
    return 1 if n <= 64 else (2 if n <= 128 else 4)


def pack_bits(m, nwords):
    """[n, b] (> 0 means set) -> uint64 [n rounded up to even, nwords]; the layout include/b200ret.h documents."""
    m = np.asarray(m)
    n, b = m.shape
    out = np.zeros((n + (n % 2), nwords), np.uint64)
    for j in range(b):
        out[:n, j // 64] |= (m[:, j] > 0).astype(np.uint64) << np.uint64(j % 64)
    return out


def pack_labels_np(lab):
    lab = np.asarray(lab)
    if lab.ndim == 2 and lab.shape[1] > 1:
        return pack_bits(lab, words(lab.shape[1])), words(lab.shape[1]), 0
    lab = lab.reshape(-1)
    out = np.zeros((len(lab) + len(lab) % 2, 1), np.uint64)
    if np.issubdtype(lab.dtype, np.integer):
        out[:len(lab), 0] = lab.astype(np.int64).view(np.uint64)
    else:
        out[:len(lab), 0] = (lab.astype(np.float64) + 0.0).view(np.uint64)
    return out, 1, 1


def multi_hot(rng, n, nlab, p):
    x = (rng.random((n, nlab)) < p).astype(np.float32)
    empty = x.sum(1) == 0
    x[empty, rng.integers(0, nlab, int(empty.sum()))] = 1
    return x


def pm1(rng, n, b):
    return rng.integers(0, 2, (n, b)).astype(np.float32) * 2 - 1


def correlated_codes(rng, q_labels, r_labels, bits, noise=0.8):
    """(q, r) codes = sign(labels . W + noise) with one shared projection W: rankings are non-trivial and mAP is well
    above the relevance density (SURVEY.md §8d "correlated variant")."""
    w = rng.standard_normal((q_labels.shape[1], bits)).astype(np.float32)

    def enc(lab):
        z = lab @ w + noise * rng.standard_normal((lab.shape[0], bits)).astype(np.float32)
        return np.where(z > 0, 1.0, -1.0).astype(np.float32)
    return enc(q_labels), enc(r_labels)


def sim_map(sim, q, ql, r, rl, k, n_shards=1, force_ext=0, sms=148, want_rank=False):
    """Run the Hamming-mAP stage programs on the CPU simulator.  Returns (map, ap, tsum, rank_idx, rank_dist, plan)."""
    nq, bits = q.shape
    n = r.shape[0]
    qc, dc = pack_bits(q, words(bits)), pack_bits(r, words(bits))
    qlp, lw, mode = pack_labels_np(ql)
    dlp, _, _ = pack_labels_np(rl)
    kk = n if k is None else min(int(k), n)
    ap = np.zeros(nq)
    ts = np.zeros(nq, np.uint32)
    m = ctypes.c_double()
    ri = np.zeros((nq, max(kk, 1)), np.uint32) if want_rank else None
    rd = np.zeros((nq, max(kk, 1)), np.uint16) if want_rank else None
    plan = (ctypes.c_int * 4)()
    rc = sim.sim_hamming_map(vp(qc), vp(qlp), vp(dc), vp(dlp), nq, ctypes.c_longlong(n), bits, lw, mode, ctypes.c_longlong(kk),
                             n_shards, force_ext, sms, vp(ap), vp(ts), ctypes.byref(m), vp(ri), vp(rd), plan)
    assert rc == 0, rc
    return m.value, ap, ts, ri, rd, list(plan)


def sim_swt(sim, x, lo, hi, level, sms=148):
    lo = np.ascontiguousarray(lo, np.float32)
    hi = np.ascontiguousarray(hi, np.float32)
    x = np.ascontiguousarray(x)
    b, c, h, w = x.shape
    out = np.full((b, c, 4, h, w), np.nan, np.float32)
    plan = (ctypes.c_int * 8)()            # TH, TW, rw form, threads, vs form, RH, RWp, u8_stage
    rc = sim.sim_swt2_fwd(vp(x), int(x.dtype == np.uint8), vp(out), b, c, h, w, vp(lo), vp(hi), len(lo), level, sms, plan)
    return rc, out, list(plan)
