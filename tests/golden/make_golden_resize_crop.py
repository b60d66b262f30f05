#!/usr/bin/env python
"""Generate ``tests/golden/resize_crop_golden.npz``: outputs of torchvision's own eval transform
``Compose([Resize(size, interpolation), CenterCrop(crop)])`` on PIL images (config/transform/basic_swt.yaml without the SWT),
the pin of ``resize_center_crop``.  Only the cropped outputs are stored: each case's input is regenerated from its seed and
shape by ``make_image``, which uses integer arithmetic alone so that it gives the same bytes everywhere.

    python tests/golden/make_golden_resize_crop.py
"""
import os

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "resize_crop_golden.npz")

# name: (H, W, channels, size, crop, interpolation, seed); size / crop are an int or an (h, w) pair
CASES = {
    "landscape_480x640": (480, 640, 3, 256, 224, "bilinear", 1),
    "portrait_640x480": (640, 480, 3, 256, 224, "bilinear", 2),
    "landscape_375x500": (375, 500, 3, 256, 224, "bilinear", 3),
    "portrait_500x375": (500, 375, 3, 256, 224, "bilinear", 4),
    "noop_resize_256x341": (256, 341, 3, 256, 224, "bilinear", 5),      # Resize(256) keeps it; left = round(58.5) = 58
    "square_257x257": (257, 257, 3, 256, 224, "bilinear", 6),
    "half_even_480x674": (480, 674, 3, 256, 224, "bilinear", 7),        # resized 256 x 359: left = round(67.5) = 68
    "extreme_224x1000": (224, 1000, 3, 256, 224, "bilinear", 8),        # resized 256 x 1142
    "upscale_12x10": (12, 10, 3, 256, 224, "bilinear", 9),              # resized 307 x 256
    "large_1800x2400": (1800, 2400, 3, 256, 224, "bilinear", 10),       # a 7x reduction
    "bicubic_480x640": (480, 640, 3, 256, 224, "bicubic", 11),
    "bicubic_large_1800x2400": (1800, 2400, 3, 256, 224, "bicubic", 12),
    "pair_size_375x500": (375, 500, 3, (256, 300), 224, "bilinear", 13),
    "nonsquare_crop_480x640": (480, 640, 3, 256, (224, 160), "bilinear", 14),
    "gray_333x517": (333, 517, 1, 256, 224, "bilinear", 15),
}


def make_image(seed, h, w, c):
    """uint8 [h, w, c]: per-channel ramps that wrap from 255 to 0 (sharp edges, so bicubic overshoot reaches the clip) plus
    isolated spikes at one pixel in 256 (so every window sees uneven weights); smooth enough to keep the npz small."""
    rng = np.random.default_rng(seed)
    ax, ay = rng.integers(1, 12, c), rng.integers(1, 12, c)
    y, x = np.meshgrid(np.arange(h, dtype=np.int64), np.arange(w, dtype=np.int64), indexing="ij")
    spikes = (rng.integers(0, 256, (h, w, c)) == 0) * rng.integers(0, 256, (h, w, c))
    img = ((x[..., None] * ax + y[..., None] * ay) // 8 + spikes) % 256
    return img.astype(np.uint8)


def main():
    import PIL
    import torchvision
    from PIL import Image
    from torchvision.transforms import CenterCrop, Compose, InterpolationMode, Resize

    out = {"torchvision_version": np.array(torchvision.__version__), "pillow_version": np.array(PIL.__version__)}
    for name, (h, w, c, size, crop, interp, seed) in CASES.items():
        arr = make_image(seed, h, w, c)
        pil = Image.fromarray(arr[:, :, 0] if c == 1 else arr, mode="L" if c == 1 else "RGB")
        t = Compose([Resize(size, interpolation=InterpolationMode(interp)), CenterCrop(crop)])
        res = np.asarray(t(pil))
        res = res[:, :, None] if res.ndim == 2 else res
        out[name] = np.ascontiguousarray(res.transpose(2, 0, 1))                # [C, Hc, Wc], the PILToTensor layout
        print(name, out[name].shape)
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes), torchvision {torchvision.__version__}, Pillow {PIL.__version__}")


if __name__ == "__main__":
    main()
