"""The device JPEG decoder on a COCO-like batch: 256 photo-like images of the pixel_probe sizes encoded by Pillow at quality
90, 4:2:0, and the same batch with four 12 MP photos.

    python tools/jpeg_probe.py [--images 256] [--iters 30] [--out profiles/jpeg_probe.json]

Reports, with the card's name, power limit and max SM clock read in the same run: bits per pixel of the batch; device time
per kernel and per batch (torch.profiler, after warm-up); the synchronisation rounds of the parallel Huffman decode; H2D
bytes and time of the pinned compressed batch against the pinned decoded one; host time of ``decode_jpeg``; worker-side
``collate_jpeg`` time per image against Pillow's decode per image on the same host (one core); end to end, pinned
encoded batch -> H2D -> decode -> resize_center_crop -> SWT haar L1 per batch against the decoded-pixel path.
"""
import argparse
import io
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pixel_probe import COMMON, LARGE, card, e2e_ms, host_call_ms  # noqa: E402

KERNELS = ("jpeg_entropy_kernel", "jpeg_idct_kernel", "jpeg_color_kernel")


def photo(rng, h, w):
    """Smooth shapes, gradients, texture and sensor noise: entropy close to a photo's at quality 90."""
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.empty((h, w, 3), np.float32)
    for c in range(3):
        f = rng.uniform(0.004, 0.03, 4)
        img[:, :, c] = (110 + 60 * np.sin(x * f[0] + y * f[1] + c) + 40 * np.cos(x * f[2] - y * f[3])
                        + 20 * np.sin(x * 0.3 + c) * np.cos(y * 0.21))
    img += rng.normal(0, 6, (h, w, 3)).astype(np.float32)
    return np.clip(img, 0, 255).astype(np.uint8)


def make_files(n, seed=0, large=0):
    from PIL import Image

    rng = np.random.default_rng(seed)
    shapes = [COMMON[int(rng.integers(0, len(COMMON)))] for _ in range(n)]
    for i in range(min(large, n)):
        shapes[int(rng.integers(0, n))] = LARGE[i % 2]
    files = []
    for h, w in shapes:
        f = io.BytesIO()
        Image.fromarray(photo(rng, h, w)).save(f, "JPEG", quality=90, subsampling=2)
        files.append(f.getvalue())
    return files


def _dev_us(prof, name):
    ks = [e for e in prof.key_averages() if name in e.key]
    return sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) for e in ks), sum(e.count for e in ks)


def kernel_times(dev, iters):
    from torch.profiler import ProfilerActivity, profile

    from image_retrieval_wavelet_b200.transforms import decode_jpeg

    for _ in range(3):
        decode_jpeg(dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            decode_jpeg(dev)
        torch.cuda.synchronize()
    out = {}
    for k in KERNELS:
        us, n = _dev_us(prof, k)
        out[k + "_ms"] = us / max(n, 1) / 1e3
    out["ms_per_batch"] = sum(out[k + "_ms"] for k in KERNELS)
    out["img_per_s"] = len(dev) / (out["ms_per_batch"] / 1e3)
    return out


def rounds(dev):
    """Synchronisation rounds: the first uint32 of the workspace after a call."""
    import ctypes

    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms.jpeg import output_offsets

    lib = _cabi.load()
    desc, tab = np.ascontiguousarray(dev.desc.numpy()), np.ascontiguousarray(dev.tables.numpy())
    offs, total = output_offsets(dev.sizes)
    dp, tp, op = (ctypes.c_void_p(a.ctypes.data) for a in (desc, tab, offs))
    nbytes = lib.b200_jpeg_decode_workspace_bytes(dp, tp, tab.size, len(dev))
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.empty(total, dtype=torch.uint8, device="cuda")
    _cabi.check(lib.b200_jpeg_decode_u8(_cabi.ptr(dev.data), dp, tp, tab.size, len(dev), _cabi.ptr(out), op, _cabi.ptr(ws), nbytes,
                                        _cabi.stream_ptr()))
    torch.cuda.synchronize()
    return {"rounds": int(ws[:4].cpu().numpy().view(np.uint32)[0]), "workspace_mb": nbytes / 1e6}


def h2d_ms(t, iters=20):
    dst = torch.empty(t.numel(), dtype=torch.uint8, device="cuda")
    dst.copy_(t, non_blocking=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        dst.copy_(t, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def worker_side(files, reps=3):
    from PIL import Image

    from image_retrieval_wavelet_b200.transforms import collate_jpeg

    t_col, t_pil = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        collate_jpeg(files)
        t_col.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for b in files:
            np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))
        t_pil.append(time.perf_counter() - t0)
    return {"collate_jpeg_ms_per_image": min(t_col) / len(files) * 1e3, "pillow_decode_ms_per_image": min(t_pil) / len(files) * 1e3,
            "one_core": True}


def batch_report(files, iters):
    from image_retrieval_wavelet_b200.transforms import collate_jpeg, collate_ragged, decode_jpeg, resize_center_crop

    enc = collate_jpeg(files).pin_memory()
    dev = enc.cuda()
    sizes = enc.sizes.numpy()
    pixels = int((sizes[:, 0] * sizes[:, 1]).sum())
    decoded = [np.asarray(decode_jpeg(dev).image(i).cpu()) for i in range(len(dev))]
    ragged = collate_ragged(decoded).pin_memory()
    r = {"images": len(files), "host_decoded": enc.n_host_decoded, "file_mb": sum(len(b) for b in files) / 1e6,
         "bits_per_pixel": sum(len(b) for b in files) * 8 / pixels, "megapixels": pixels / 1e6}
    r["kernels"] = kernel_times(dev, iters)
    r.update(rounds(dev))
    r["h2d"] = {"compressed_mb": enc.data.numel() / 1e6, "compressed_ms": h2d_ms(enc.data),
                "decoded_mb": ragged.data.numel() / 1e6, "decoded_ms": h2d_ms(ragged.data)}
    r["decode_jpeg_host_ms_median"] = host_call_ms(decode_jpeg, dev)
    r["e2e_encoded_h2d_decode_crop_swt"] = e2e_ms(enc, lambda b: resize_center_crop(decode_jpeg(b)), iters)
    r["e2e_decoded_h2d_crop_swt"] = e2e_ms(ragged, resize_center_crop, iters)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("jpeg_probe needs a CUDA device")
    res = {"card": card(), "quality": 90, "subsampling": "4:2:0", "l2_flushed": False}
    coco = make_files(a.images)
    res["coco"] = batch_report(coco, a.iters)
    res["coco_worker_side"] = worker_side(coco[:64])
    res["with_12mp_photos"] = batch_report(make_files(a.images, large=4), a.iters)
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
