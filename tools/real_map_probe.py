"""Hamming mAP of real-valued codes (``on_nonbinary='real'``) on the device.

    python tools/real_map_probe.py [--iters 30] [--out profiles/real_map_probe.json]

Reports, with the card's name, power limit and max SM clock read in the same run:

* the in-training proxy ``compute_batch_map`` on raw logits with ``'real'`` against ``'sign'`` at batch 96 / 256 / 1024 and
  B = 64 / 128 (multi-hot labels, k = max_bin_count): time per call from CUDA events around the whole call (it reads
  results back, so the host work between its kernels is included), median over ``--iters`` calls after warm-up, the two
  modes alternating;
* a C3-shaped real-code mAP@5000 (5000 queries x 117000 rows x 128 dims, 80 multi-hot labels): ``real_hamming_map`` end
  to end, and its three steps on the full [5000, 117000] matrix (distance kernel, top-5000 selection, ranked AP), each
  from CUDA events after warm-up; the packed ``hamming_map`` of the same codes after ``sign`` beside it.  The 2.3 GB
  distance matrix is far larger than L2, so every pass reads it from HBM.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                   # the numbers below still carry the torch device name
        q = f"nvidia-smi unavailable: {e}"
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0)}


def event_ms(fn, iters, warmup=3):
    """Median over `iters` of CUDA-event time around one call, after `warmup` calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times))


def multi_hot(rng, n, nlab, p):
    x = (rng.random((n, nlab)) < p).astype(np.float32)
    x[x.sum(1) == 0, 0] = 1
    return x


def batch_proxy(iters):
    from image_retrieval_wavelet_b200.engine import build_batch_map_calculator, compute_batch_map

    rows = []
    for bits in (64, 128):
        for batch in (96, 256, 1024):
            rng = np.random.default_rng(batch + bits)
            logits = torch.from_numpy(rng.standard_normal((batch, bits)).astype(np.float32)).cuda()
            lab = torch.from_numpy(multi_hot(rng, batch, 20, 0.1)).cuda()
            calcs = {m: build_batch_map_calculator("hamming", torch.device("cuda"), on_nonbinary=m) for m in ("real", "sign")}
            res = {m: compute_batch_map(*calcs[m], logits, lab) for m in calcs}
            times = {m: [] for m in calcs}
            for _ in range(3):
                for m in calcs:
                    compute_batch_map(*calcs[m], logits, lab)
            for _ in range(iters):                          # alternate the two modes
                for m in calcs:
                    times[m].append(event_ms(lambda: compute_batch_map(*calcs[m], logits, lab), 1, warmup=0))
            rows.append({"batch": batch, "bits": bits, "map_real": res["real"], "map_sign": res["sign"],
                         "ms_real": float(np.median(times["real"])), "ms_sign": float(np.median(times["sign"]))})
            print(rows[-1], flush=True)
    return rows


def c3_real(iters):
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.engine import hamming as H

    nq, n, bits, k = 5000, 117000, 128, 5000
    g = torch.Generator(device="cuda").manual_seed(0)
    q = torch.randn((nq, bits), device="cuda", generator=g)
    r = torch.randn((n, bits), device="cuda", generator=g)
    ql = H.pack_labels((torch.rand((nq, 80), device="cuda", generator=g) < 0.04).float())
    rl = H.pack_labels((torch.rand((n, 80), device="cuda", generator=g) < 0.04).float())
    lib = _cabi.load()
    out = {"shape": {"Q": nq, "N": n, "B": bits, "k": k, "labels": 80}}
    ld = (n + 3) // 4 * 4
    out["chunk_rows"] = min(nq, H.REAL_CHUNK_BUDGET // (4 * ld + 12 * k))
    m, _, _ = H.real_hamming_map(q, ql, r, rl, k)
    out["map"] = m.item()
    out["ms_real_hamming_map"] = event_ms(lambda: H.real_hamming_map(q, ql, r, rl, k), iters)
    # the steps on the whole matrix at once
    dist = torch.empty((nq, ld), dtype=torch.float32, device="cuda")
    idx = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    score = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    ap = torch.empty(nq, dtype=torch.float64, device="cuda")
    hits = torch.empty(nq, dtype=torch.int32, device="cuda")
    st = _cabi.stream_ptr()

    def dist_step():
        _cabi.check(lib.b200_real_hamming_dist(_cabi.ptr(q), _cabi.ptr(r), nq, n, bits, bits, _cabi.ptr(dist), ld, st))

    def select_step():
        _cabi.check(lib.b200_select_topk_f32(_cabi.ptr(dist), nq, n, ld, k, 0, _cabi.ptr(idx), _cabi.ptr(score), st))

    def ap_step():
        _cabi.check(lib.b200_ranked_ap(_cabi.ptr(idx), 1, nq, k, _cabi.ptr(ql.words), _cabi.ptr(rl.words), ql.lw, ql.mode, None,
                                       _cabi.ptr(ap), _cabi.ptr(hits), None, st))

    out["ms_distance_kernel"] = event_ms(dist_step, iters)
    out["distance_tflops"] = 2.0 * nq * n * bits / (out["ms_distance_kernel"] * 1e-3) / 1e12
    out["ms_select_top5000"] = event_ms(select_step, iters)
    out["ms_ranked_ap"] = event_ms(ap_step, iters)
    qc, rc = H.pack_codes(q, on_nonbinary="sign"), H.pack_codes(r, on_nonbinary="sign")
    out["ms_packed_hamming_map_of_sign_codes"] = event_ms(lambda: H.hamming_map(qc, ql, rc, rl, k), iters)
    out["map_sign"] = H.hamming_map(qc, ql, rc, rl, k)[0].item()
    print(out, flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("real_map_probe needs a CUDA device")
    res = {"card": card(), "batch_map": batch_proxy(a.iters), "c3_real_map_at_5000": c3_real(max(5, a.iters // 3))}
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
