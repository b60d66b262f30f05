"""CPU oracle of the Hamming mAP of real-valued codes (test infrastructure; see ``oracle/__init__.py``).

The reference's ``calc_hamming_dist`` (``accuracy_calculator.py:183-186``) is ``0.5 * (B - q @ r.T)`` in float32 for any
code matrix, and ``calculate_maphashing`` (:203-231) ranks rows by it with ``argsort``.  For codes that are not +-1 (raw
logits, ``sign(0) == 0``, +-inf, NaN) the float32 sum depends on its order, so this oracle fixes the order of the device
scorer:

``real_hamming_dist``      ``oracle/c/real_codes.c``: the inner product as one fmaf chain in dimension order, then
                           ``0.5f * ((float)nbits - s)`` — bit for bit what ``b200_real_hamming_dist`` computes.
``maphashing_real_exact``  ranking = stable ascending argsort of those float32 distances (ties to the smaller index,
                           NaN last), AP in float64: the parity target of ``on_nonbinary='real'``.  Equal to
                           ``eval_ref.maphashing_exact`` on +-1 codes.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from . import eval_ref

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "c", "real_codes.c")
# the flags of oracle/Makefile; plain "gcc" on purpose (an exported CC may be a wrapper without libgomp.spec)
_CFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-shared"]
_LIB = None


def _targets():
    yield os.path.join(_HERE, "libreal_codes.so")
    # a read-only checkout: build next to the other per-user temporaries instead
    yield os.path.join(tempfile.gettempdir(), f"b200_oracle_{os.getuid()}", "libreal_codes.so")


def build(force=False):
    """Compile ``oracle/c/real_codes.c`` when the library is missing or older than the source; returns its path."""
    err = None
    for so in _targets():
        if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(_SRC):
            return so
        try:
            os.makedirs(os.path.dirname(so), exist_ok=True)
            if not os.access(os.path.dirname(so), os.W_OK):
                continue
            env = dict(os.environ)
            env.pop("CC", None)
            subprocess.check_call(["gcc"] + _CFLAGS + ["-o", so, _SRC, "-lm"], env=env)
            return so
        except (OSError, subprocess.CalledProcessError) as e:
            err = e
    raise RuntimeError(f"cannot build the real-code oracle: {err}")


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
        _LIB.oracle_real_hamming_dist.restype = ctypes.c_int
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def real_hamming_dist(q, r, nbits=None, nthreads=0):
    """float32 ``0.5 * (nbits - q @ r.T)`` with the inner product as one fmaf chain in dimension order (the device
    scorer's order); nbits defaults to the code width.  -> float32 [Q, N]."""
    q = np.ascontiguousarray(q, dtype=np.float32)
    r = np.ascontiguousarray(r, dtype=np.float32)
    assert q.ndim == 2 and r.ndim == 2 and q.shape[1] == r.shape[1]
    out = np.empty((q.shape[0], r.shape[0]), dtype=np.float32)
    rc = lib().oracle_real_hamming_dist(_p(q), _p(r), q.shape[0], ctypes.c_long(r.shape[0]), q.shape[1],
                                        int(q.shape[1] if nbits is None else nbits), _p(out), int(nthreads))
    if rc:
        raise ValueError(f"oracle_real_hamming_dist failed with {rc}")
    return out


def maphashing_real_exact(query, query_labels, reference, reference_labels, topk=None, ref_includes_query=False,
                          return_details=False):
    """Parity target for real-valued codes: ranking = stable ascending argsort of :func:`real_hamming_dist` (ties go to
    the smaller index, NaN comes last); AP in float64, mean over all queries; topk as ``eval_ref.maphashing_exact``."""
    topk = eval_ref.resolve_topk_ref(topk, reference_labels, ref_includes_query)
    q = np.asarray(query, dtype=np.float32)
    r = np.asarray(reference, dtype=np.float32)
    nq, n = q.shape[0], r.shape[0]
    k = n if topk is None else max(0, min(int(topk), n))
    aps = np.zeros(nq, dtype=np.float64)
    tsums = np.zeros(nq, dtype=np.int64)
    ranked = np.zeros((nq, k), dtype=np.int64)
    dists = np.zeros((nq, k), dtype=np.float32)
    d_all = real_hamming_dist(q, r) if n else np.zeros((nq, 0), np.float32)
    ql = np.asarray(query_labels)
    rl = np.asarray(reference_labels)
    for i in range(nq):
        rel = eval_ref.label_rel_ref(ql[i:i + 1], rl).reshape(-1)
        order = np.argsort(d_all[i], kind="stable")[:k]
        aps[i], tsums[i] = eval_ref.ap_from_ranked_relevance(rel[order])
        ranked[i] = order
        dists[i] = d_all[i][order]
    m = float(aps.sum() / nq) if nq else float("nan")
    if return_details:
        return m, aps, tsums, ranked, dists
    return m
