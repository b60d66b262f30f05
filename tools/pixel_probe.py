"""The pixel step on a COCO-like ragged batch: the eval transform ``resize_center_crop`` (Resize(256) -> CenterCrop(224), one
launch of ``resize_crop_kernel``) and the training transform ``resize_random_crop_flip`` (Resize(256) ->
RandomResizedCrop(224) -> RandomHorizontalFlip, two launches) against torchvision on PIL images on the CPU.

    python tools/pixel_probe.py [--images 256] [--iters 50] [--out profiles/pixel_probe.json]

Reports, with the card's name and power limit read in the same run:
  * kernel time per batch (torch.profiler, device time of ``resize_crop_kernel``) and images/s, with and without the large
    photos; the inputs (> 200 MB) exceed the 126 MB L2, so no explicit flush is done;
  * the kernel's share of HBM bandwidth from algorithmic bytes: source bytes inside each crop's support + output bytes,
    against 6552.6 GB/s (the project's measured copy bandwidth, DESIGN.md §6);
  * host time of the call (table build, one H2D copy, launch), with the stream idle;
  * end to end: pinned ragged host buffer -> H2D -> crop -> SWT (haar L1), CUDA events;
  * torchvision Compose([Resize(256), CenterCrop(224)]) on the PIL images, one core and all cores;
  * the same for the training transform (boxes and flips drawn by ``collate_ragged_train`` under torch seed 0): device
    time of both launches, host time of the call, end to end through the SWT, and torchvision's training Compose.
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


def _tv_transform(train):
    from torchvision.transforms import CenterCrop, Compose, RandomHorizontalFlip, RandomResizedCrop, Resize

    return Compose([Resize(256), RandomResizedCrop(224), RandomHorizontalFlip()] if train else [Resize(256), CenterCrop(224)])


def _tv_worker(indices, train=False):
    torch.set_num_threads(1)
    t = _tv_transform(train)
    for i in indices:
        np.asarray(t(_PIL_IMAGES[i]))
    return len(indices)


def _tv_train_worker(indices):
    return _tv_worker(indices, True)


def cpu_baseline(imgs, train=False):
    try:
        import torchvision  # noqa: F401
        from PIL import Image
    except ImportError:
        return {"skipped": "torchvision is not importable"}
    _PIL_IMAGES[:] = [Image.fromarray(a) for a in imgs]
    work = _tv_train_worker if train else _tv_worker
    idx = list(range(len(imgs)))
    work(idx[:4])
    t0 = time.perf_counter()
    work(idx)
    one = time.perf_counter() - t0
    cores = os.cpu_count() or 1
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(work, [[i] for i in range(cores)])         # start the workers
        t0 = time.perf_counter()
        pool.map(work, [[i] for i in idx], chunksize=1)
        allc = time.perf_counter() - t0
    return {"one_core_s": one, "one_core_img_per_s": len(imgs) / one, "cores": cores, "all_cores_s": allc,
            "all_cores_img_per_s": len(imgs) / allc}


def _device_us(prof, name):
    ks = [e for e in prof.key_averages() if name in e.key]
    return sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) for e in ks), sum(e.count for e in ks)


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
    dev_us, count = _device_us(prof, "resize_crop_kernel")
    ms = dev_us / max(count, 1) / 1e3
    nbytes = algorithmic_bytes(imgs)
    return {"ms_per_batch": ms, "launches": count, "img_per_s": len(imgs) / (ms / 1e3), "input_mb": sum(x.size for x in imgs) / 1e6,
            "algorithmic_bytes": nbytes, "gbps": nbytes / (ms / 1e3) / 1e9, "hbm_fraction": nbytes / (ms / 1e3) / 1e9 / HBM_GBPS}


def train_kernel_time(dev, iters):
    """Device time of the training chain's two launches under torch.profiler, per batch: the boxes of the first resize
    (resize_crop_kernel<3, true>) and the full resize of every box plane to 224 x 224 (resize_crop_kernel<1, true>)."""
    from torch.profiler import ProfilerActivity, profile

    from image_retrieval_wavelet_b200.transforms import resize_random_crop_flip

    for _ in range(5):
        resize_random_crop_flip(dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            resize_random_crop_flip(dev)
        torch.cuda.synchronize()
    box_us, box_n = _device_us(prof, "resize_crop_kernel<3,")
    full_us, full_n = _device_us(prof, "resize_crop_kernel<1,")
    ms = (box_us + full_us) / iters / 1e3
    return {"ms_per_batch": ms, "boxes_ms": box_us / max(box_n, 1) / 1e3, "resize_ms": full_us / max(full_n, 1) / 1e3,
            "launches": box_n + full_n, "img_per_s": len(dev) / (ms / 1e3)}


def host_call_ms(fn, dev, reps=20):
    """Median host time of one call with the stream idle (tables + one H2D copy + launch enqueue)."""
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(dev)
        times.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    return float(np.median(times))


def e2e_ms(host, step, iters):
    """Pinned ragged host buffer -> H2D -> ``step`` -> SWT haar L1 per batch: CUDA events and wall clock."""
    from image_retrieval_wavelet_b200.transforms import SWTTransform

    swt = SWTTransform(level=1, wavelet="haar")
    for _ in range(3):
        swt.forward(step(host.cuda(non_blocking=True)))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(iters):
        y = swt.forward(step(host.cuda(non_blocking=True)))
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / iters * 1e3
    return {"ms_per_batch_events": e0.elapsed_time(e1) / iters, "ms_per_batch_wall": wall, "img_per_s": len(host) / (wall / 1e3),
            "out_shape": list(y.shape), "finite": bool(math.isfinite(float(y[0, 0, 0, 0, 0])))}


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
    import ctypes

    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms import collate_ragged, collate_ragged_train, resize_center_crop, resize_random_crop_flip
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin, resized_size

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
    res["host_call_ms_median"] = host_call_ms(resize_center_crop, dev)
    lib = _cabi.load()
    geom_only = []
    geom = np.array([(h, w) + resized_size(h, w, 256) + center_crop_origin(*resized_size(h, w, 256), 224, 224)
                     for h, w in host.sizes.tolist()], dtype=np.int32)
    for _ in range(20):
        t0 = time.perf_counter()
        lib.b200_resize_crop_workspace_bytes(len(imgs), ctypes.c_void_p(geom.ctypes.data), 3, 224, 224, _cabi.RESIZE_BILINEAR)
        geom_only.append((time.perf_counter() - t0) * 1e3)
    res["host_workspace_query_ms_median"] = float(np.median(geom_only))
    res["e2e_h2d_crop_swt"] = e2e_ms(host, resize_center_crop, a.iters)

    # the training chain on the same images, boxes and flips drawn once under torch seed 0
    torch.manual_seed(0)
    train_host = collate_ragged_train(imgs).pin_memory()
    train_dev = train_host.cuda()
    torch.manual_seed(0)
    train_coco = collate_ragged_train(coco).cuda()
    res["train"] = {
        "kernel": train_kernel_time(train_dev, a.iters),
        "kernel_without_large_photos": train_kernel_time(train_coco, a.iters),
        "host_call_ms_median": host_call_ms(resize_random_crop_flip, train_dev),
        "host_call_ms_median_without_large_photos": host_call_ms(resize_random_crop_flip, train_coco),
        "e2e_h2d_train_swt": e2e_ms(train_host, resize_random_crop_flip, a.iters),
        "flips": int(train_host.crop_params[:, 4].sum()),
    }
    res["cpu_torchvision"] = cpu_baseline(imgs)
    res["cpu_torchvision_train"] = cpu_baseline(imgs, train=True)
    res["check"] = {"out_shape": list(out.shape)}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
