#!/usr/bin/env python
"""bench.py — headline benchmark of the two hot paths (contract in the task statement; metric from BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl reference] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1)

Primary line: Hamming mAP@k queries/s on the MS-COCO shape (BASELINE.json configs[2]: 5k queries x 117k database rows,
80 labels, 128-bit codes, k = 5000 — the configuration quoted "1/2/4/8 B200" like the metric).  One step = one full
evaluation of all queries through ``HammingMapEngine.evaluate``: bit-pack the float32 +-1 codes / multi-hot labels as the
reference hands them over, evaluate (select pipeline: sampled bound, candidate lists, ranking), average, read the
result back — one CUDA graph replay.  With N > 1 GPUs every rank holds the float rows of ITS database shard, packs them
into every rank's copy of the packed database over NVLink peer memory, evaluates its slice of the (replicated) queries
and exchanges the per-query results the same way: total work is fixed, so "scaling" is "strong".

`value`   : device-resident float32 inputs, CUDA-event time per step, max over ranks (streams aligned by a device
            barrier ahead of the start event), L2 flushed between steps (memset + read pass).
`e2e`     : from PINNED HOST float32 buffers, copies inside the timed region, result read back.  N = 1: the
            reference-facing C-ABI call ``b200_maphashing_host`` (streams the database over PCIe while the select kernel
            scores the chunks that have landed), with the engine step on staging tensors (`engine_*`) and the packed host
            entry (`packed_*`) beside it; N > 1: the engine step (H2D of all queries + this rank's shard).
`roofline`: the dominant kernel of the step, its stage time measured with CUDA events in an eager re-run of the same
            kernels on the same inputs (a graph replay cannot be timed stage by stage), plus flat copies of the numbers
            the other workloads produce (`c5_*`: BASELINE configs[4] at this N; `swt_*`: configs[0] / [3]).
`extras`  : everything else (other Hamming shapes, cosine k-NN, SWT grid, DSCH metrics, DWT, fix_size) at N = 1, printed
            as a JSON line of its own on stderr.
`--impl reference` times the reference's own CPU implementation: the REAL ``CustomCalculator.calculate_maphashing`` loaded
from /root/reference when that tree is readable (kind "reference"), else the literal torch restatement of it (kind "port";
the reference's third-party stack is not installable offline, see DESIGN.md §3) — on a bounded query sample.
`--dump-outputs DIR` writes what the last timed step of the main workload computed (map.npy, and the per-query ap.npy and
hits.npy, float64); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "hamming_map_at_k_queries_per_sec"
WORKLOADS = {
    # name: (description from BASELINE.json, Q, N, bits, labels, k, label density)
    "c1": ("MIRFlickr-25K shape: 2k queries x 18k db, 24 labels, 64-bit codes, mAP@5000", 2000, 18000, 64, 24, 5000, 0.10),
    "c2": ("PASCAL VOC shape: 5k queries x 11.5k db, 20 labels, 64-bit codes, mAP@all", 5000, 11500, 64, 20, None, 0.10),
    "c2_32": ("PASCAL VOC shape, 32-bit codes", 5000, 11500, 32, 20, None, 0.10),
    "c2_128": ("PASCAL VOC shape, 128-bit codes", 5000, 11500, 128, 20, None, 0.10),
    "c3": ("MS-COCO shape: 5k queries x 117k db, 80 labels, 128-bit codes, mAP@5000", 5000, 117000, 128, 80, 5000, 0.036),
    "c3_all": ("MS-COCO shape, mAP@all (k = 117000)", 5000, 117000, 128, 80, None, 0.036),
    "c5": ("Scale-out: 1M-image db, 64-bit codes, 10k queries, mAP@5000", 10000, 1000000, 64, 80, 5000, 0.036),
}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(key):
    """DRAM bytes per launch of a kernel from the committed ncu captures (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f).get(key)
        return (int(e["bytes"]), e.get("source")) if e else (None, None)
    except Exception:
        return None, None


def make_problem(name, seed=0):
    """Synthetic evaluator inputs (SURVEY.md §8d): multi-hot labels Bernoulli(p) with >= 1 tag, codes =
    sign(labels . W + noise) so that rankings are informative.  float32, CPU, torch.Generator().manual_seed(seed)."""
    _, nq, n, bits, nlab, k, p = WORKLOADS[name]
    g = torch.Generator().manual_seed(seed)

    def labels(rows):
        lab = (torch.rand(rows, nlab, generator=g) < p).float()
        empty = lab.sum(1) == 0
        lab[empty, torch.randint(0, nlab, (int(empty.sum()),), generator=g)] = 1.0
        return lab

    ql, rl = labels(nq), labels(n)
    w = torch.randn(nlab, bits, generator=g)

    def codes(lab):
        z = lab @ w + 0.8 * torch.randn(lab.shape[0], bits, generator=g)
        return torch.where(z > 0, 1.0, -1.0).float()

    return codes(ql), ql, codes(rl), rl, (n if k is None else k)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            pass
    return local_rank


# ---------------------------------------------------------------------------------------------- reference arm (CPU)
def base_config(name):
    desc, nq, n, bits, nlab, k, _ = WORKLOADS[name]
    return {"workload": f"{name}: {desc}", "queries": nq, "database": n, "code_bits": bits, "labels": nlab, "top_k": n if k is None else k}


def reference_step_fn():
    """(callable(q, ql, r, rl, k) -> mAP, kind, description)."""
    try:
        from oracle import ref_loader

        if ref_loader.available():
            acc, _ = ref_loader.load_reference()
            calc = acc.CustomCalculator(k=None, device=torch.device("cpu"), distance_metric="hamming", with_faiss=False)
            return (lambda q, ql, r, rl, k: calc.calculate_maphashing(q, ql, r, rl, k), "reference",
                    "the reference's own CustomCalculator.calculate_maphashing (main/engine/accuracy_calculator.py:203-231), loaded "
                    "unmodified from /root/reference with its absent third-party imports stubbed (oracle/ref_loader.py)")
    except Exception:
        pass
    from oracle.eval_ref import maphashing_literal

    return (maphashing_literal, "port", "literal torch restatement of calculate_maphashing (accuracy_calculator.py:203-231; "
            "the reference tree is not on this box)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    nq = WORKLOADS[name][1]
    q, ql, r, rl, k = make_problem(name)
    step_fn, kind, how = reference_step_fn()
    cores = os.cpu_count() or 1
    # bounded sample: as many queries as take about 2 s per step with the better thread setting
    probe = min(8, nq)
    best = None
    for threads in sorted({1, cores}):
        torch.set_num_threads(threads)
        step_fn(q[:2], ql[:2], r, rl, k)
        t0 = time.perf_counter()
        step_fn(q[:probe], ql[:probe], r, rl, k)
        per_q = (time.perf_counter() - t0) / probe
        if best is None or per_q < best[1]:
            best = (threads, per_q)
    threads, per_q = best
    torch.set_num_threads(threads)
    budget = 90.0 / max(1, args.steps + args.warmup)                     # whole run well inside a few minutes
    sample = int(max(4, min(nq, min(2.0, budget) / per_q)))
    for _ in range(args.warmup):
        step_fn(q[:sample], ql[:sample], r, rl, k)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_fn(q[:sample], ql[:sample], r, rl, k)
    dt = (time.perf_counter() - t0) / args.steps
    value = sample / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": base_config(name),
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": threads, "kind": kind,
                         "sample": f"{sample} of {nq} queries per step against the full database; {how}; host has "
                                   f"{cores} logical cores, {threads} torch thread(s) was the faster setting"},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- own arm (GPU)
def l2_flusher(device):
    """Untimed between steps: a 256 MiB memset (> the 126 MB L2) evicts what the previous step left, then a 256 MiB READ of
    a second buffer evicts the memset's own dirty lines — otherwise their write-back (up to 126 MB) competes with the first
    ~20 us of the timed step for HBM bandwidth.  B200_BENCH_FLUSH=memset: the memset alone (the round-1 / early round-2 form)."""
    buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)    # > 126 MB L2
    if os.environ.get("B200_BENCH_FLUSH", "") == "memset":
        return lambda: buf.zero_()
    src = torch.zeros(64 * 1024 * 1024, dtype=torch.int32, device=device)

    def flush():
        buf.zero_()
        return src.max()                        # a pure read pass: leaves clean lines behind

    return flush


L2_NOTE = ("flushed between steps (256 MiB memset, untimed)" if os.environ.get("B200_BENCH_FLUSH", "") == "memset"
           else "flushed between steps (256 MiB memset, then a 256 MiB read so that no dirty lines are left to write back; untimed)")
POPC_PER_PAIR = {1: 2, 2: 3, 4: 4}        # select kernel: carry-save adders in front of the POPC pipe (hamming_select.cu)
XU_LANES_PER_CLK_PER_SM = 16.0              # POPC is a quarter-rate XU instruction (measured: tools/ubench_int.cu)


def dump_outputs(out_dir, engine, m):
    """Write what the last timed step computed as ``out_dir/<name>.npy``: the mAP and the per-query AP and hit counts that
    ``evaluate(details=True)`` hands a caller, read from the engine's result region after that step (float64)."""
    st = engine._last
    arrays = {"map": np.array([m], dtype=np.float64),
              "ap": engine._result(st, st.off_ap, torch.float64, st.nq).cpu().numpy(),
              "hits": engine._result(st, st.off_tsum, torch.int32, st.nq).cpu().numpy().astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for key, a in arrays.items():
        np.save(os.path.join(out_dir, f"{key}.npy"), a)


def bench_map(name, args, world, rank, device, dist, engine, with_e2e=True, with_cpu=True, check=True, dump_dir=None):
    """One Hamming-mAP workload through HammingMapEngine at this world size."""
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.engine.dist import shard_bounds

    desc, nq, n, bits, nlab, _, _ = WORKLOADS[name]
    q, ql, r, rl, k = make_problem(name)
    b0, b1 = shard_bounds(n, world)[rank]
    dq, dql = q.to(device), ql.to(device)
    dr, drl = r[b0:b1].contiguous().to(device), rl[b0:b1].contiguous().to(device)
    flush = l2_flusher(device)

    def step(details=False):
        return engine.evaluate(dq, dql, dr, drl, k, n_total=n, details=details)

    m, ap, tsum = step(details=True)
    checked = None
    if check and rank == 0:
        from oracle import c_oracle

        sub = np.random.default_rng(0).choice(nq, 16, replace=False)
        m0, ap0, ts0 = c_oracle.maphashing(q[sub].numpy(), ql[sub].numpy(), r.numpy(), rl.numpy(), k)
        ok = np.array_equal(tsum.cpu().numpy()[sub].astype(np.int64), ts0) and np.abs(ap.cpu().numpy()[sub] - ap0).max() <= 1e-6
        if not ok:
            raise SystemExit(f"bench: {name}: CUDA result differs from the oracle on the check sample")
        checked = "16-query sample bit-exact (hits) / 1e-6 (AP) against the C oracle"
    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(gpu_index(int(os.environ.get("LOCAL_RANK", "0"))))
    sampler.start()
    starts, ends = [], []
    redone = 0
    for _ in range(args.steps):
        flush()
        if dist is not None:
            dist.barrier()                       # ranks start the step together (the barriers are ahead of the start event):
            engine.align()                       # hosts first, then the streams (a barrier kernel over peer memory)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = step()
        e.record()
        starts.append(s), ends.append(e)
        torch.cuda.synchronize()
        redone += int(engine.last_info.get("redone", False))
    total_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    t = torch.tensor([total_ms], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, engine, out[0])
    # keep the GPU busy a little longer (about 0.25 s) so that the clock sampler sees the kernels under load; the count
    # comes from the all-reduced time, so every rank runs the SAME number of steps (they contain barriers)
    for _ in range(int(min(400, max(3, 250.0 / max(ms_per_step, 1e-3))))):
        step()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    value = nq / (ms_per_step * 1e-3)
    info = dict(engine.last_info)
    kernels_per_step = int(info.get("kernels_per_step") or 0)
    # per-stage device time: the same kernels launched eagerly with an event behind each, L2 flushed, on this rank's slice
    stage_runs = []
    for _ in range(5):
        flush()
        stage_runs.append(engine.stage_ms())
    # (median of the 5 runs: an eager run now and then catches a one-off stall of tens of ms in one of its 14 stages)
    stage_avg = {key: float(np.median([sr[key] for sr in stage_runs])) for key in stage_runs[0]} if stage_runs and stage_runs[0] else {}
    live = {key: v for key, v in stage_avg.items() if not key.startswith("gated") and "round1" not in key and key != "finalize"}
    cw, lw = _cabi.code_words(bits), _cabi.label_words(nlab)
    qs = info["query_slice"][1] - info["query_slice"][0]
    algo_bytes = n * (cw + lw) * 8 + qs * (cw + lw) * 8 + qs * 12              # SURVEY.md §8d compulsory traffic, per launch
    dom = max(live, key=live.get) if live else None
    dom_ms = live.get(dom, float("nan")) if dom else float("nan")
    tc_form = "filter" in live                  # tensor-core form of the select pass: tcgen05 filter -> hit masks -> SIMT append ("select")
    kernel_of = {"select": "hamming_select_kernel", "rank": "hamming_select_rank_kernel", "sample_hist": "select_sample_kernel",
                 "filter": "hamming_select_tc_kernel", "expand": "select_expand_fp8_kernel",
                 "hist": "hamming_hist_kernel", "ap": "hamming_rank_kernel" if 4 * k <= n else "hamming_walk_kernel",
                 "scan": "hamming_scan_kernel", "bound": "select_bound_kernel"}
    dom_kernel = kernel_of.get(dom, str(dom))
    peak, peak_src = measured_peaks()
    achieved = algo_bytes / (dom_ms * 1e-3) / 1e9
    sm_mhz = clocks.get("sm_mhz") or 1900.0
    score_ms = live.get("select", live.get("hist", float("nan")))           # the kernel that scores every (query, row) pair
    popc = POPC_PER_PAIR[cw] if info.get("select") else 2 * cw
    pair_rate = qs * n / (score_ms * 1e-3)
    pairs_clk_sm = pair_rate / (sm_mhz * 1e6) / 148.0
    traffic, traffic_src = measured_traffic(f"{dom_kernel}:{name}") if world == 1 else (None, None)
    roofline = {
        "bound": "hbm", "kernel": f"{dom_kernel} (stage '{dom}')", "achieved": achieved, "peak": peak,
        "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": dom_ms,
        "issue_frac": pairs_clk_sm * popc / XU_LANES_PER_CLK_PER_SM,
        "pairs_per_clk_per_sm": pairs_clk_sm, "popc32_per_pair": popc, "scoring_kernel_ms": score_ms,
        "note": "the packed database is L2-resident by design: the scoring kernel is bound by the POPC (XU) pipe, 16 lanes/clk/SM, "
                "not by HBM — issue_frac = pairs/clk/SM x POPC per pair / 16 is the fraction of that pipe's peak; frac is the "
                "mandated HBM figure on SURVEY 8d's compulsory bytes; stage times from an eager re-run with CUDA events",
    }
    if tc_form:
        # the pairs are scored on the tensor cores (e4m3 dot products of the +-1 codes, K padded to 128): the POPC figure does
        # not apply; what is reported instead is the filter kernel against the nominal dense fp8 rate and the pair rate of
        # filter + append together.  The dominant kernel is the append half (latency-bound list writes).
        kpad = (bits + 127) // 128 * 128
        flt_ms = live["filter"]
        both_ms = flt_ms + live.get("select", 0.0) + live.get("expand", 0.0)
        roofline.update({
            "issue_frac": None, "popc32_per_pair": 0, "scoring_kernel_ms": both_ms,
            "pairs_per_clk_per_sm": qs * n / (both_ms * 1e-3) / (sm_mhz * 1e6) / 148.0,
            "filter_kernel": "hamming_select_tc_kernel (tcgen05.mma kind::f8f6f4, M128 N256 K32, TMA tiles, TMEM accumulators)",
            "filter_ms": flt_ms, "filter_tflops": 2.0 * qs * n * kpad / (flt_ms * 1e-3) / 1e12,
            "filter_frac_of_fp8_peak": 2.0 * qs * n * kpad / (flt_ms * 1e-3) / 4.5e15,
            "filter_peak_source": "nominal dense fp8 4.5 PFLOP/s (B200_PROFILING.md)",
            "note": "tensor-core form of the select pass: the pairs are scored by a tcgen05 fp8 GEMM (filter), which writes one hit bit per "
                    "pair; the append kernel ('select' stage) scores only the rows within the bound again and writes the candidate lists — it "
                    "is latency-bound on those scattered 4-byte writes, not on HBM or POPC; frac is the mandated HBM figure on SURVEY 8d's "
                    "compulsory bytes; stage times from an eager re-run with CUDA events",
        })
    result = {
        "value": value, "ms_per_step": ms_per_step, "stage_ms": stage_avg, "roofline": roofline, "clocks": clocks,
        "gpu_launches": kernels_per_step * args.steps, "checked": checked, "map": float(out[0]), "top_k": k,
        "config": base_config(name), "steps_redone_with_full_sequence": redone, "plan": engine.plan_info(),
        "run": {"sharding": (f"database rows in {world} contiguous float32 shards, packed into every rank's copy over NVLink peer memory; "
                             f"queries replicated, each rank evaluates a slice of {qs}; results exchanged the same way (2 barrier kernels, no NCCL)")
                if world > 1 else "single GPU", "l2": L2_NOTE,
                "timed": f"one CUDA graph replay ({kernels_per_step} kernels: pack + select pipeline + mean) + result read-back, CUDA events, "
                         "max over ranks"},
    }
    # ---- end to end: pinned host float32 -> H2D -> the same step -> result on the host
    if with_e2e:
        hq, hql = q.pin_memory(), ql.pin_memory()
        hr, hrl = r[b0:b1].contiguous().pin_memory(), rl[b0:b1].contiguous().pin_memory()
        h2d = (hq.numel() + hql.numel() + hr.numel() + hrl.numel()) * 4
        sq, sql, sr, srl = (torch.empty_like(t_, device=device) for t_ in (hq, hql, hr, hrl))

        def e2e_step():
            sq.copy_(hq, non_blocking=True), sql.copy_(hql, non_blocking=True)
            sr.copy_(hr, non_blocking=True), srl.copy_(hrl, non_blocking=True)
            return engine.evaluate(sq, sql, sr, srl, k, n_total=n, details=False)[0]

        def timed(fn):
            for _ in range(3):
                fn()
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                last = fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=device)
            if dist is not None:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()) / args.steps, last

        dt, e2e_map = timed(e2e_step)
        result["e2e"] = {"value": nq / dt, "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 16,
                         "ms_per_step": dt * 1e3, "map": float(e2e_map),
                         "api": "HammingMapEngine.evaluate on staging tensors filled from pinned host float32 buffers "
                                "(H2D + pack + evaluation + result read-back per step)"}
        if world == 1:
            lib = _cabi.load()
            m_out, bad = ctypes.c_double(), ctypes.c_int()

            def cabi_step():
                rc = lib.b200_maphashing_host(hq.data_ptr(), hql.data_ptr(), hr.data_ptr(), hrl.data_ptr(), nq, n, bits, nlab, 0, k,
                                              None, None, ctypes.addressof(m_out), ctypes.addressof(bad))
                _cabi.check(rc, "b200_maphashing_host")
                return m_out.value

            dt, cm = timed(cabi_step)
            # the headline e2e at N = 1 is the reference-facing C-ABI call on HOST buffers (the drop-in boundary); the engine
            # figure (device staging tensors filled from the same pinned buffers, then one graph replay) is kept beside it
            eng = result["e2e"]
            result["e2e"] = {"value": nq / dt, "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 16,
                             "ms_per_step": dt * 1e3, "map": float(cm),
                             "api": "b200_maphashing_host (C-ABI, pinned float32 host buffers in, mAP out: database streamed over PCIe in "
                                    "8 row chunks, each chunk packed and scored by the select kernel while the next one is in flight)",
                             "engine_value": eng["value"], "engine_ms_per_step": eng["ms_per_step"], "engine_map": eng["map"],
                             "engine_api": eng["api"],
                             "cabi_fp32_value": nq / dt, "cabi_fp32_ms_per_step": dt * 1e3, "cabi_fp32_map": float(cm),
                             "cabi_fp32_api": "b200_maphashing_host (C-ABI, float32 host buffers, same bytes over PCIe)"}
            # packed host buffers: what crosses PCIe once the glue packs behind the model (SURVEY 8 f1)
            from image_retrieval_wavelet_b200.engine import hamming as H

            pk = [H.pack_codes(dq, on_nonbinary="sign").words[:nq], H.pack_labels_unchecked(dql).words[:nq],
                  H.pack_codes(dr, on_nonbinary="sign").words[:n], H.pack_labels_unchecked(drl).words[:n]]
            hp = [t_.cpu().contiguous().pin_memory() for t_ in pk]

            def packed_step():
                rc = lib.b200_maphashing_host_packed(hp[0].data_ptr(), hp[1].data_ptr(), hp[2].data_ptr(), hp[3].data_ptr(), nq, n, bits,
                                                     lw, 0, k, None, None, ctypes.addressof(m_out))
                _cabi.check(rc, "b200_maphashing_host_packed")
                return m_out.value

            dt, pm = timed(packed_step)
            result["e2e"].update({"packed_value": nq / dt, "packed_ms_per_step": dt * 1e3, "packed_map": float(pm),
                                  "packed_h2d_bytes_per_step": int(sum(t_.numel() * 8 for t_ in hp)),
                                  "packed_api": "b200_maphashing_host_packed (C-ABI, bit-packed host buffers)"})
    # ---- CPU baseline (rank 0, single GPU runs only): C/OpenMP port of the reference loop on a bounded query sample
    if with_cpu and rank == 0 and world == 1:
        from oracle import c_oracle

        threads = c_oracle.num_threads()
        probe = min(nq, 2 * threads)
        t0 = time.perf_counter()
        c_oracle.maphashing(q[:probe].numpy(), ql[:probe].numpy(), r.numpy(), rl.numpy(), k)
        per_q = (time.perf_counter() - t0) / probe
        sample = int(max(threads, min(nq, 12.0 / per_q)))
        t0 = time.perf_counter()
        c_oracle.maphashing(q[:sample].numpy(), ql[:sample].numpy(), r.numpy(), rl.numpy(), k)
        dt = time.perf_counter() - t0
        result["cpu_baseline"] = {"value": sample / dt, "unit": "queries/s", "cores": threads, "kind": "port",
                                  "sample": f"{sample} of {nq} queries against the full database ({dt:.1f} s); oracle/c/oracle.c "
                                            "(float dot products, comparison sort, AP) with OpenMP over queries"}
    return result


def bench_swt(shape, wavelet, level, dtype, args, device, with_cpu=False):
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms import swt2

    b, c, h, w = shape
    g = torch.Generator().manual_seed(0)
    x8 = torch.randint(0, 256, (min(b, 8), c, h, w), dtype=torch.uint8, generator=g)
    x8 = x8.repeat((b + x8.shape[0] - 1) // x8.shape[0], 1, 1, 1)[:b].contiguous()
    x = (x8.to(device) if dtype == "u8" else (x8.float() / 255.0).to(device)).contiguous()
    out = torch.empty((b, c, 4, h, w), dtype=torch.float32, device=device)
    flush = l2_flusher(device)
    for _ in range(max(args.warmup, 3)):
        swt2(x, wavelet, level, out=out)
    torch.cuda.synchronize()
    times = []
    launches0 = _cabi.launch_count()
    for _ in range(args.steps):
        flush()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        swt2(x, wavelet, level, out=out)
        e.record()
        torch.cuda.synchronize()
        times.append(s.elapsed_time(e))
    ms = float(np.mean(times))
    px = b * c * h * w
    algo = px * ((1 if dtype == "u8" else 4) + 16)                    # SURVEY.md §8d: 17 / 20 bytes per image-channel pixel
    peak, peak_src = measured_peaks()
    res = {
        "workload": f"SWT {wavelet} level {level} on {b}x{c}x{h}x{w} {dtype}", "images_per_s": b / (ms * 1e-3), "ms": ms,
        "ms_min": float(np.min(times)), "gpu_launches_per_step": (_cabi.launch_count() - launches0) // args.steps,
        "roofline": {"bound": "hbm", "kernel": "swt2_tile_kernel", "achieved": algo / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": algo / (ms * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes_per_launch": algo,
                     "peak_source": peak_src},
    }
    res["roofline"]["traffic"], res["roofline"]["traffic_source"] = measured_traffic("swt2_tile_kernel:" + res["workload"])
    if with_cpu and dtype == "u8":
        # end to end as the transform is used: uint8 batch in pinned host memory -> H2D -> kernel; the float32 sub-bands
        # stay on the device, where the model consumes them (custom_transforms.py:145-157 + base_update.py:65)
        hx = x8.pin_memory()
        sx = torch.empty_like(x)

        def e2e():
            sx.copy_(hx, non_blocking=True)
            swt2(sx, wavelet, level, out=out)

        for _ in range(3):
            e2e()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e()
            torch.cuda.synchronize()
        res["e2e_images_per_s"] = b / ((time.perf_counter() - t0) / args.steps)
        res["e2e_h2d_bytes_per_step"] = int(hx.numel())
    if with_cpu:
        from oracle import c_oracle, filters

        lo, hi = filters.filter_bank(wavelet)
        sample = x8[:min(b, 64)].numpy()
        c_oracle.swt2(sample[:2], lo, hi, level)
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 5.0:
            c_oracle.swt2(sample, lo, hi, level)
            reps += 1
        dt = (time.perf_counter() - t0) / reps
        res["cpu_baseline"] = {"value": sample.shape[0] / dt, "unit": "images/s", "cores": c_oracle.num_threads(), "kind": "port",
                               "sample": f"{sample.shape[0]} images x {reps} repetitions; oracle/c/oracle.c periodised a-trous loops "
                                         "(CPU restatement of pywt.swt2), OpenMP over image channels"}
    return res


def bench_knn(args, device, nq=5000, n=117000, d=768, k=2048):
    """BASELINE configs[2] cosine rerank: get_knn (inner product) on L2-normalised float32 embeddings, tensor-core scorer."""
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.engine.get_knn import knn_topk

    g = torch.Generator().manual_seed(0)
    refs = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).to(device)
    qs = torch.nn.functional.normalize(torch.randn(nq, d, generator=g), dim=1).to(device)
    flush = l2_flusher(device)
    res = {"workload": f"cosine k-NN: {nq} queries x {n} refs, D={d}, k={k} (get_knn, inner product)"}
    for label, env in (("tensor_core", "1"), ("simt_fp32", "0")):
        os.environ["B200_KNN_TC"] = env
        for _ in range(2):
            knn_topk(refs, qs, k, "cosine")
        torch.cuda.synchronize()
        times, l0 = [], _cabi.launch_count()
        steps = min(args.steps, 5)
        for _ in range(steps):
            flush()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            knn_topk(refs, qs, k, "cosine")
            e.record()
            torch.cuda.synchronize()
            times.append(s.elapsed_time(e))
        ms = float(np.mean(times))
        res[label] = {"ms": ms, "queries_per_s": nq / (ms * 1e-3), "gpu_launches_per_step": (_cabi.launch_count() - l0) // steps}
    os.environ.pop("B200_KNN_TC", None)
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak, src = float(json.load(f)["bf16_tflops_sustained"]), "measured sustained bf16 (MEASURED_PEAKS.json)"
    except Exception:
        peak, src = 1400.0, "fallback (B200_PROFILING.md)"
    flops = 2.0 * nq * n * d
    ms = res["tensor_core"]["ms"]
    res["roofline"] = {"bound": "tensor", "kernel": "knn_scores_tc_kernel (+ split, select)", "achieved": flops / (ms * 1e-3) / 1e12,
                       "peak": peak, "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / peak, "traffic": None, "peak_source": src,
                       "note": "achieved counts the algorithmic 2*Q*N*D flops over the whole call (split + GEMM + select); the "
                               "GEMM executes 3x that (bf16 hi/lo split for float32-grade scores)"}
    return res


def bench_fix_size(shape, level, wavelet, args, device):
    """SURVEY §8 f3: fix_size on the device (Pillow-exact bicubic, 518 -> 520) and fix_size + SWT as SWTTransform.forward runs it."""
    from image_retrieval_wavelet_b200.transforms import SWTTransform, resize_u8

    b, c, h, w = shape
    g = torch.Generator().manual_seed(0)
    x8 = torch.randint(0, 256, (min(b, 8), c, h, w), dtype=torch.uint8, generator=g)
    x = x8.repeat((b + x8.shape[0] - 1) // x8.shape[0], 1, 1, 1)[:b].contiguous().to(device)
    f = 1 << level
    ho, wo = -(-h // f) * f, -(-w // f) * f
    t = SWTTransform(level=level, wavelet=wavelet)
    flush = l2_flusher(device)
    res = {"workload": f"fix_size {h}x{w} -> {ho}x{wo} (PIL bicubic) + SWT {wavelet} level {level} on {b}x{c} uint8 planes"}
    for key, fn in (("resize_ms", lambda: resize_u8(x, (ho, wo))), ("resize_plus_swt_ms", lambda: t.forward(x))):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.steps):
            flush()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            times.append(s.elapsed_time(e))
        res[key] = float(np.mean(times))
    res["images_per_s"] = b / (res["resize_plus_swt_ms"] * 1e-3)
    res["note"] = "includes torch's allocation of the outputs; resize = horizontal + vertical pass through a uint8 intermediate"
    return res


def bench_dsch(args, device):
    """SURVEY §8 f2: DSCH's metrics on the C3 shape (5k x 117k, 128 bit, 80 labels), wall time per call incl. packing."""
    from image_retrieval_wavelet_b200.engine import DSCH

    q, ql, r, rl, _ = make_problem("c3")
    q, ql, r, rl = (t.to(device) for t in (q, ql, r, rl))
    res = {"workload": "DSCH metrics, MS-COCO shape (5000 x 117000, 128 bit, 80 labels), device-resident float inputs"}
    for key, fn in (("pr_curve_ms", lambda: DSCH.pr_curve(q, r, ql, rl)), ("p_topK_ms", lambda: DSCH.p_topK(q, r, ql, rl)),
                    ("radius2_precision_ms", lambda: DSCH.get_precision_recall_by_Hamming_Radius(r, rl, q, ql)),
                    ("mean_average_precision_at_5000_ms", lambda: DSCH.mean_average_precision(q, r, ql, rl, 5000))):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        res[key] = (time.perf_counter() - t0) / 3 * 1e3
    try:                                    # calculate_pr_rc_hashing: full ranking of every query, 500 queries of the 5000
        from image_retrieval_wavelet_b200.engine import CustomCalculator

        calc = CustomCalculator(k=None, distance_metric="hamming", with_faiss=False)
        calc.pr_rc_hashing_curves(q[:64], ql[:64], r, rl)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, _, used = calc.pr_rc_hashing_curves(q[:500], ql[:500], r, rl)
        torch.cuda.synchronize()
        res["pr_rc_hashing_500_queries_ms"] = (time.perf_counter() - t0) * 1e3
        res["pr_rc_hashing_queries_used"] = used
    except Exception as exc:
        res["pr_rc_hashing_error"] = repr(exc)
    return res


def bench_dwt(args, device):
    """SURVEY §8 f4: DWTTransform on the CIFAR shape of config/transform/cifar_dwt.yaml and on a 224 x 224 batch."""
    from image_retrieval_wavelet_b200.transforms import dwt2

    res = {}
    g = torch.Generator().manual_seed(0)
    for key, shape, wv, lv in (("cifar_haar_L2_1024x3x32x32_ms", (1024, 3, 32, 32), "haar", 2),
                               ("db4_L3_64x3x224x224_ms", (64, 3, 224, 224), "db4", 3)):
        x = torch.randint(0, 256, shape, dtype=torch.uint8, generator=g).to(device)
        for _ in range(3):
            dwt2(x, wv, lv)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(args.steps):
            dwt2(x, wv, lv)
        e.record()
        torch.cuda.synchronize()
        res[key] = s.elapsed_time(e) / args.steps
    return res


def run_own(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 hot paths have no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_mod.init_process_group("nccl", device_id=device)
        dist = dist_mod
    from image_retrieval_wavelet_b200.engine.map_engine import HammingMapEngine

    engine = HammingMapEngine()
    main = bench_map(args.workload, args, world, rank, device, dist, engine, dump_dir=args.dump_outputs)
    engine.close()
    small = argparse.Namespace(**{**vars(args), "steps": min(args.steps, 10)})
    flat = {}                     # scalar copies for the retained `roofline` object (the driver drops `extras`)
    scaleout = None
    if not args.no_extras and args.workload != "c5":
        # BASELINE configs[4] (1M-row database, 10k queries, 64 bit) at EVERY world size
        try:
            engine = HammingMapEngine()
            r_ = bench_map("c5", small, world, rank, device, dist, engine, with_e2e=False, with_cpu=False, check=(world == 1))
            engine.close()
            scaleout = {kk: r_[kk] for kk in ("value", "ms_per_step", "stage_ms", "map", "checked", "config", "plan", "run")}
            scaleout["unit"] = "queries/s"
            scaleout["issue_frac"] = r_["roofline"]["issue_frac"]
            flat.update({"c5_queries_per_s": r_["value"], "c5_ms_per_step": r_["ms_per_step"], "c5_issue_frac": r_["roofline"]["issue_frac"],
                         "c5_filter_tflops": r_["roofline"].get("filter_tflops"),
                         "c5_map": r_["map"]})
        except Exception as exc:                                       # an extra must never take the headline down
            scaleout = {"error": repr(exc)}
    extras = {}
    if not args.no_extras and world == 1:
        for name in ("c1", "c2_32", "c2", "c2_128", "c3_all"):
            if name == args.workload:
                continue
            try:
                engine = HammingMapEngine()
                r_ = bench_map(name, small, 1, 0, device, None, engine, with_e2e=name in ("c1", "c2"), with_cpu=False, check=True)
                engine.close()
                extras[name] = {kk: r_[kk] for kk in ("value", "ms_per_step", "stage_ms", "map", "checked", "plan") if kk in r_}
                extras[name]["unit"] = "queries/s"
                extras[name]["workload"] = r_["config"]["workload"]
                if "e2e" in r_:
                    extras[name]["e2e"] = r_["e2e"]
                extras[name]["issue_frac"] = r_["roofline"]["issue_frac"]
            except Exception as exc:
                extras[name] = {"error": repr(exc)}
        # C1 (both input types) and the whole C4 grid: haar/db2/db4/sym4 x levels 1-3 (518 at level 1, fix_size's 520 above)
        swt_cases = [((64, 3, 224, 224), "haar", 1, "u8", True), ((64, 3, 224, 224), "haar", 1, "f32", False)]
        for lv in (1, 2, 3):
            for wv in ("haar", "db2", "db4", "sym4"):
                swt_cases.append(((256, 3, 518, 518) if lv == 1 else (256, 3, 520, 520), wv, lv, "u8", False))
        try:
            extras["knn"] = bench_knn(small, device)
        except Exception as exc:
            extras["knn"] = {"error": repr(exc)}
        for key, fn in (("dsch", lambda: bench_dsch(small, device)), ("dwt", lambda: bench_dwt(small, device)),
                        ("fix_size", lambda: bench_fix_size((256, 3, 518, 518), 2, "haar", small, device))):
            try:
                extras[key] = fn()
            except Exception as exc:
                extras[key] = {"error": repr(exc)}
        extras["swt"] = []
        for shape, wv, lv, dt, cpu in swt_cases:
            try:
                extras["swt"].append(bench_swt(shape, wv, lv, dt, small, device, with_cpu=cpu))
            except Exception as exc:
                extras["swt"].append({"workload": f"SWT {wv} L{lv} {shape} {dt}", "error": repr(exc)})
        ok = [c for c in extras["swt"] if "roofline" in c]
        if ok:
            c1 = ok[0]
            grid = [c for c in ok if "256x3x51" in c["workload"] or "256x3x52" in c["workload"]]
            flat.update({"swt_c1_images_per_s": c1["images_per_s"], "swt_c1_frac": c1["roofline"]["frac"],
                         "swt_c1_traffic": c1["roofline"]["traffic"], "swt_c1_algorithmic_bytes": c1["roofline"]["algorithmic_bytes_per_launch"],
                         "swt_c1_note": "measured DRAM bytes per launch are BELOW the algorithmic bytes: part of the 154 MB output is "
                                        "still dirty in the 126 MB L2 when the kernel ends, so this fraction is L2-assisted; the C4 "
                                        "shapes (3.5 GB per launch) are the honest HBM figures",
                         "swt_c1_e2e_images_per_s": c1.get("e2e_images_per_s")})
            if grid:
                haar1 = next((c for c in grid if "haar level 1" in c["workload"]), grid[0])
                worst = min(grid, key=lambda c: c["roofline"]["frac"])
                flat.update({"swt_c4_haar_l1_images_per_s": haar1["images_per_s"], "swt_c4_haar_l1_frac": haar1["roofline"]["frac"],
                             "swt_c4_worst_frac": worst["roofline"]["frac"], "swt_c4_worst_case": worst["workload"],
                             "swt_c4_worst_images_per_s": worst["images_per_s"],
                             "swt_c4_cases_at_or_above_0p6": sum(1 for c in grid if c["roofline"]["frac"] >= 0.6), "swt_c4_cases": len(grid)})
        if isinstance(extras.get("knn"), dict) and "roofline" in extras["knn"]:
            flat.update({"knn_c3_ms": extras["knn"]["tensor_core"]["ms"], "knn_c3_frac_of_bf16_peak": extras["knn"]["roofline"]["frac"]})
    if rank == 0:
        roofline = dict(main["roofline"])
        roofline.update(flat)
        line = {
            "metric": METRIC, "value": main["value"], "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            # bit-packed uint64 codes / labels (XOR + POPC, integer ranks); with the tensor-core form of the select pass every
            # pair is first scored as an e4m3 dot product of the +-1 codes with float32 accumulation (exact integers)
            "dtype": "u64+e4m3" if "filter" in (main.get("stage_ms") or {}) else "u64",
            "data": "synthetic", "config": main["config"], "clocks": main["clocks"], "e2e": main.get("e2e"),
            "gpu_launches": main["gpu_launches"], "roofline": roofline, "cpu_baseline": main.get("cpu_baseline"),
            "stage_ms": main["stage_ms"], "map": main["map"], "checked": main["checked"], "run": main["run"], "plan": main["plan"],
            "steps_redone_with_full_sequence": main["steps_redone_with_full_sequence"], "scaleout": scaleout,
        }
        if extras:
            # about 14 KB: on a line of their own (stderr), so that readers with a line-length limit still parse the result
            # line; `roofline` keeps flat copies of their headline figures
            print(json.dumps({"extras": extras}), file=sys.stderr)
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the main workload as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
