"""The eval pixel step on a COCO-like ragged batch: ``resize_center_crop`` (Resize(256) -> CenterCrop(224), one launch of
``resize_crop_kernel``) against torchvision on PIL images on the CPU.

    python tools/pixel_probe.py [--images 256] [--iters 50] [--out profiles/pixel_probe.json]

Reports, with the card's name and power limit read in the same run:
  * kernel time per batch (torch.profiler, device time of ``resize_crop_kernel``) and images/s, with and without the large
    photos; the inputs (> 200 MB) exceed the 126 MB L2, so no explicit flush is done;
  * the kernel's share of HBM bandwidth from algorithmic bytes: source bytes inside each crop's support + output bytes,
    against 6552.6 GB/s (the project's measured copy bandwidth, DESIGN.md §6);
  * host time of the call (table build, one H2D copy, launch), with the stream idle;
  * end to end: pinned ragged host buffer -> H2D -> crop -> SWT (haar L1), CUDA events;
  * torchvision Compose([Resize(256), CenterCrop(224)]) on the PIL images, one core and all cores.
"""
import argparse
import json
import math
import multiprocessing as mp
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

HBM_GBPS = 6552.6
COMMON = [(480, 640), (640, 480), (427, 640), (375, 500)]
LARGE = [(3000, 4000), (4000, 3000)]


def make_batch(n, seed=0, large=4):
    rng = np.random.default_rng(seed)
    shapes = [COMMON[int(rng.integers(0, len(COMMON)))] for _ in range(n)]
    for i in range(min(large, n)):                   # a few large photos
        shapes[int(rng.integers(0, n))] = LARGE[i % 2]
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]


def _support(n_in, n_out, first, count):
    """[lo, hi) of the input samples the bilinear windows of outputs [first, first + count) read (Pillow's precompute_coeffs)."""
    if n_in == n_out:
        return first, first + count
    scale = n_in / n_out
    support = max(scale, 1.0)

    def window(xx):
        center = (xx + 0.5) * scale
        return max(int(center - support + 0.5), 0), min(int(center + support + 0.5), n_in)
    return window(first)[0], window(first + count - 1)[1]


def algorithmic_bytes(imgs, crop=224):
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin, resized_size

    total = 0
    for a in imgs:
        h, w, c = a.shape
        rh, rw = resized_size(h, w, 256)
        top, left = center_crop_origin(rh, rw, crop, crop)
        y0, y1 = _support(h, rh, top, crop)
        x0, x1 = _support(w, rw, left, crop)
        total += (y1 - y0) * (x1 - x0) * c + c * crop * crop
    return total


_PIL_IMAGES = []            # filled before the worker pool forks: workers index it instead of receiving pickled pixels


def _tv_worker(indices):
    torch.set_num_threads(1)
    from torchvision.transforms import CenterCrop, Compose, Resize

    t = Compose([Resize(256), CenterCrop(224)])
    for i in indices:
        np.asarray(t(_PIL_IMAGES[i]))
    return len(indices)


def cpu_baseline(imgs):
    try:
        import torchvision  # noqa: F401
        from PIL import Image
    except ImportError:
        return {"skipped": "torchvision is not importable"}
    _PIL_IMAGES[:] = [Image.fromarray(a) for a in imgs]
    idx = list(range(len(imgs)))
    _tv_worker(idx[:4])
    t0 = time.perf_counter()
    _tv_worker(idx)
    one = time.perf_counter() - t0
    cores = os.cpu_count() or 1
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_tv_worker, [[i] for i in range(cores)])   # start the workers
        t0 = time.perf_counter()
        pool.map(_tv_worker, [[i] for i in idx], chunksize=1)
        allc = time.perf_counter() - t0
    return {"one_core_s": one, "one_core_img_per_s": len(imgs) / one, "cores": cores, "all_cores_s": allc,
            "all_cores_img_per_s": len(imgs) / allc}


def kernel_time(dev, imgs, iters):
    """Device time of resize_crop_kernel under torch.profiler, per launch."""
    from torch.profiler import ProfilerActivity, profile

    from image_retrieval_wavelet_b200.transforms import resize_center_crop

    for _ in range(5):
        resize_center_crop(dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            resize_center_crop(dev)
        torch.cuda.synchronize()
    ks = [e for e in prof.key_averages() if "resize_crop_kernel" in e.key]
    dev_us = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) for e in ks)
    count = sum(e.count for e in ks)
    ms = dev_us / max(count, 1) / 1e3
    nbytes = algorithmic_bytes(imgs)
    return {"ms_per_batch": ms, "launches": count, "img_per_s": len(imgs) / (ms / 1e3), "input_mb": sum(x.size for x in imgs) / 1e6,
            "algorithmic_bytes": nbytes, "gbps": nbytes / (ms / 1e3) / 1e9, "hbm_fraction": nbytes / (ms / 1e3) / 1e9 / HBM_GBPS}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                   # the numbers below still carry the torch device name
        q = f"nvidia-smi unavailable: {e}"
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pixel_probe needs a CUDA device")
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms import SWTTransform, collate_ragged, resize_center_crop

    res = {"card": card(), "images": a.images, "iters": a.iters}
    imgs = make_batch(a.images)
    host = collate_ragged(imgs).pin_memory()
    dev = host.cuda()
    res["input_mb"] = host.data.numel() / 1e6
    res["l2_flushed"] = False
    out = resize_center_crop(dev)
    torch.cuda.synchronize()

    res["kernel"] = kernel_time(dev, imgs, a.iters)
    coco = make_batch(a.images, large=0)
    res["kernel_without_large_photos"] = kernel_time(collate_ragged(coco).cuda(), coco, a.iters)

    # host time of the call with the stream idle (tables + one H2D copy + launch enqueue)
    lib = _cabi.load()
    host_ms = []
    for _ in range(20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        resize_center_crop(dev)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    res["host_call_ms_median"] = float(np.median(host_ms))
    geom_only = []
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin, resized_size
    import ctypes
    geom = np.array([(h, w) + resized_size(h, w, 256) + center_crop_origin(*resized_size(h, w, 256), 224, 224)
                     for h, w in host.sizes.tolist()], dtype=np.int32)
    for _ in range(20):
        t0 = time.perf_counter()
        lib.b200_resize_crop_workspace_bytes(len(imgs), ctypes.c_void_p(geom.ctypes.data), 3, 224, 224, _cabi.RESIZE_BILINEAR)
        geom_only.append((time.perf_counter() - t0) * 1e3)
    res["host_workspace_query_ms_median"] = float(np.median(geom_only))

    # end to end: pinned ragged host buffer -> H2D -> crop -> SWT
    swt = SWTTransform(level=1, wavelet="haar")
    for _ in range(3):
        swt.forward(resize_center_crop(host.cuda(non_blocking=True)))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(a.iters):
        y = swt.forward(resize_center_crop(host.cuda(non_blocking=True)))
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / a.iters * 1e3
    ev = e0.elapsed_time(e1) / a.iters
    res["e2e_h2d_crop_swt"] = {"ms_per_batch_events": ev, "ms_per_batch_wall": wall, "img_per_s": a.images / (wall / 1e3),
                               "out_shape": list(y.shape)}
    res["cpu_torchvision"] = cpu_baseline(imgs)
    res["check"] = {"out_shape": list(out.shape), "finite": bool(math.isfinite(float(y[0, 0, 0, 0, 0])))}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
