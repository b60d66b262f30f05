#!/usr/bin/env python
"""Generate ``tests/golden/resize_train_golden.npz``: outputs of torchvision's own training transform
``Compose([Resize(size, interpolation), RandomResizedCrop(crop, interpolation=interpolation), RandomHorizontalFlip(p)])``
on PIL images (config/transform/basic_swt.yaml without the SWT) under ``torch.manual_seed(seed)``, the pin of
``resize_random_crop_flip``.  Only the outputs are stored: each input is regenerated from its seed and shape by
``make_image`` of ``make_golden_resize_crop.py``, and the boxes and flips are drawn again from the same torch seed.

    python tests/golden/make_golden_resize_train.py
"""
import importlib.util
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "resize_train_golden.npz")

# name: (H, W, channels, size, crop, interpolation, seed, p); size / crop are an int or an (h, w) pair
CASES = {
    "landscape_480x640": (480, 640, 3, 256, 224, "bilinear", 1, 0.5),
    "portrait_640x480": (640, 480, 3, 256, 224, "bilinear", 2, 0.5),
    "odd_width_375x501": (375, 501, 3, 256, 224, "bilinear", 3, 0.5),
    "coco_427x640_flip": (427, 640, 3, 256, 224, "bilinear", 4, 1.0),
    "coco_427x640_noflip": (427, 640, 3, 256, 224, "bilinear", 4, 0.0),
    "bicubic_480x640": (480, 640, 3, 256, 224, "bicubic", 5, 0.5),
    "bicubic_odd_333x517": (333, 517, 3, 256, 224, "bicubic", 6, 1.0),
    "gray_333x517": (333, 517, 1, 256, 224, "bilinear", 7, 1.0),
    "rgbx_300x451": (300, 451, 4, 256, 224, "bilinear", 8, 1.0),          # 4 channels as Pillow's "RGBX" (no alpha)
    "rgbx_bicubic_257x255": (257, 255, 4, 256, 224, "bicubic", 9, 0.0),
    "tiny_12x10": (12, 10, 3, 256, 224, "bilinear", 10, 0.5),            # resized 307 x 256, boxes upscaled
    "tiny_bicubic_31x17": (31, 17, 3, 256, 224, "bicubic", 11, 1.0),
    "identity_256x256": (256, 256, 3, 256, 224, "bilinear", 12, 0.5),    # Resize(256) keeps it
    "fallback_1999x37": (1999, 37, 3, 256, 224, "bilinear", 13, 1.0),    # no try fits: the central box
    "photo_3000x4000": (3000, 4000, 3, 256, 224, "bilinear", 14, 1.0),
    "pair_size_crop_375x500": (375, 500, 3, (256, 300), (224, 160), "bilinear", 15, 1.0),
}


def make_image(seed, h, w, c):
    spec = importlib.util.spec_from_file_location("make_golden_resize_crop", os.path.join(HERE, "make_golden_resize_crop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.make_image(seed, h, w, c)


def to_pil(arr):
    """uint8 [H, W, C] -> the PIL image a decoder would give: "L", "RGB", or "RGBX" for 4 channels (Pillow premultiplies
    "RGBA" by its alpha while it resizes, which a plain per-channel resize does not)."""
    from PIL import Image

    c = arr.shape[2]
    if c == 4:
        return Image.frombytes("RGBX", (arr.shape[1], arr.shape[0]), np.ascontiguousarray(arr).tobytes())
    return Image.fromarray(arr[:, :, 0] if c == 1 else arr, mode="L" if c == 1 else "RGB")


def from_pil(img, c):
    res = np.asarray(img.convert("RGBX") if c == 4 else img)
    res = res[:, :, None] if res.ndim == 2 else res
    return np.ascontiguousarray(res.transpose(2, 0, 1))                      # [C, h, w], the PILToTensor layout


def train_transform(size, crop, interp, p):
    from torchvision.transforms import Compose, InterpolationMode, RandomHorizontalFlip, RandomResizedCrop, Resize

    mode = InterpolationMode(interp)
    return Compose([Resize(size, interpolation=mode), RandomResizedCrop(crop, interpolation=mode), RandomHorizontalFlip(p)])


def chain_ref(img, rh, rw, box, out_hw, interp):
    """The chain on ``oracle/resize_ref.py``: the box ``(top, left, h, w, flip)`` of the ``rh x rw`` resize of ``img``
    ([H, W, C] uint8), rounded to uint8, resized in full to ``out_hw``, its columns mirrored when flip is set -> [C, Ho, Wo]."""
    from oracle import resize_ref

    top, left, h, w, flip = (int(v) for v in box)
    win = resize_ref.resize_ref(np.ascontiguousarray(img.transpose(2, 0, 1)), (rh, rw), interp)[:, top:top + h, left:left + w]
    out = resize_ref.resize_ref(np.ascontiguousarray(win), out_hw, interp)
    return np.ascontiguousarray(out[:, :, ::-1]) if flip else out


def main():
    import PIL
    import torch
    import torchvision

    out = {"torchvision_version": np.array(torchvision.__version__), "pillow_version": np.array(PIL.__version__)}
    for name, (h, w, c, size, crop, interp, seed, p) in CASES.items():
        torch.manual_seed(seed)
        out[name] = from_pil(train_transform(size, crop, interp, p)(to_pil(make_image(seed, h, w, c))), c)
        print(name, out[name].shape)
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes), torchvision {torchvision.__version__}, Pillow {PIL.__version__}")


if __name__ == "__main__":
    main()
