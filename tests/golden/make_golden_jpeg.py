"""Goldens of the device JPEG decoder: JPEG files written by Pillow and Pillow's own ``Image.open(f).convert("RGB")`` of
each, plus files the device does not decode (progressive, CMYK, PNG) for the routing tests.

    python tests/golden/make_golden_jpeg.py        # writes tests/golden/jpeg_golden.npz

Content is seeded: smooth gradients with mild noise (photo-like, short Huffman codes) and uniform noise (long codes, large
coefficients at quality 100)."""
import io
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# name -> (h, w, gray, quality, subsampling (0 4:4:4, 1 4:2:2, 2 4:2:0), content, extra save options)
CASES = {}
for h, w in ((1, 1), (17, 9), (31, 17), (9, 33), (2, 3)):
    for ss in (0, 1, 2):
        CASES[f"s{ss}_{h}x{w}"] = (h, w, False, 90, ss, "smooth", {})
    CASES[f"gray_{h}x{w}"] = (h, w, True, 90, 0, "smooth", {})
for q in (1, 50, 90, 100):
    CASES[f"q{q}_420"] = (40, 56, False, q, 2, "noise", {})
    CASES[f"q{q}_gray"] = (24, 40, True, q, 0, "noise", {})
CASES["optimize_422"] = (48, 63, False, 75, 1, "smooth", {"optimize": True})
CASES["optimize_gray"] = (33, 20, True, 75, 0, "noise", {"optimize": True})
CASES["rst_blocks_420"] = (45, 70, False, 85, 2, "smooth", {"restart_marker_blocks": 3})
CASES["rst_rows_444"] = (30, 41, False, 85, 0, "noise", {"restart_marker_rows": 1})
CASES["rst_blocks_gray"] = (27, 35, True, 85, 0, "smooth", {"restart_marker_blocks": 1})
CASES["large_420"] = (240, 320, False, 92, 2, "smooth", {})             # hundreds of 1024-bit subsequences in one interval


def make_image(seed, h, w, gray, content):
    rng = np.random.default_rng(seed)
    if content == "noise":
        a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    else:
        y, x = np.mgrid[0:h, 0:w].astype(np.float64)
        base = np.stack([128 + 100 * np.sin(x / 9.0 + y / 17.0), x * 255.0 / max(w, 1), y * 255.0 / max(h, 1)], axis=2)
        a = np.clip(base + rng.normal(0, 12, (h, w, 3)), 0, 255).astype(np.uint8)
    return a[:, :, 0] if gray else a


def encode(arr, quality, subsampling, **extra):
    from PIL import Image

    f = io.BytesIO()
    Image.fromarray(arr).save(f, "JPEG", quality=quality, subsampling=subsampling, **extra)
    return f.getvalue()


def case_bytes(name):
    h, w, gray, q, ss, content, extra = CASES[name]
    return encode(make_image(sorted(CASES).index(name), h, w, gray, content), q, ss, **extra)


def unsupported_files():
    """Files the worker decodes: a progressive JPEG, a CMYK JPEG and a PNG."""
    from PIL import Image

    rgb = make_image(99, 23, 29, False, "smooth")
    out = {}
    f = io.BytesIO()
    Image.fromarray(rgb).save(f, "JPEG", quality=80, progressive=True)
    out["progressive"] = f.getvalue()
    f = io.BytesIO()
    Image.fromarray(rgb).convert("CMYK").save(f, "JPEG", quality=80)
    out["cmyk"] = f.getvalue()
    f = io.BytesIO()
    Image.fromarray(rgb).save(f, "PNG")
    out["png"] = f.getvalue()
    return out


def pil_rgb(b):
    from PIL import Image

    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


def main():
    arrays = {}
    files = {name: case_bytes(name) for name in CASES}
    files.update({f"unsupported_{k}": v for k, v in unsupported_files().items()})
    for name, b in files.items():
        arrays[f"{name}.jpg"] = np.frombuffer(b, dtype=np.uint8)
        arrays[f"{name}.rgb"] = pil_rgb(b)
    np.savez_compressed(os.path.join(HERE, "jpeg_golden.npz"), **arrays)


if __name__ == "__main__":
    main()
