"""Ragged batches of decoded images and the eval transform ``Resize(size) -> CenterCrop(crop)`` on the device.

The reference's eval transform (``config/transform/basic_swt.yaml``: ``Resize(256) -> CenterCrop(224) -> SWTTransform``) runs
per PIL image in the DataLoader workers.  Here the workers only decode (``PIL.open(...).convert("RGB")``),
``collate_ragged`` packs the images of a batch, whatever their sizes, into one flat uint8 buffer, and
``resize_center_crop`` produces the cropped ``[B, C, Hc, Wc]`` uint8 batch on the device in one kernel launch
(``b200_resize_crop_u8``), bit-identical to torchvision's ``Compose([Resize(size), CenterCrop(crop)])`` on each PIL image.
It feeds ``SWTTransform.forward`` directly.
"""
import ctypes

import numpy as np
import torch

from .. import _cabi

__all__ = ["RaggedImages", "collate_ragged", "resize_center_crop", "resized_size", "center_crop_origin"]

ALIGN = 16          # byte alignment of every image in the packed buffer


class RaggedImages:
    """Images of different sizes in one flat buffer: image ``i`` is HWC-interleaved uint8 ``[H_i, W_i, channels]`` at byte
    ``offsets[i]`` of ``data``.  ``sizes`` (int64 ``[B, 2]`` = H, W) and ``offsets`` (int64 ``[B]``) stay on the host;
    ``pin_memory()`` and ``cuda()`` act on ``data``, so a DataLoader with ``pin_memory=True`` pins the batch."""

    def __init__(self, data, sizes, offsets, channels):
        self.data = data
        self.sizes = sizes
        self.offsets = offsets
        self.channels = int(channels)

    def __len__(self):
        return int(self.sizes.shape[0])

    def _with(self, data):
        return RaggedImages(data, self.sizes, self.offsets, self.channels)

    def pin_memory(self, device=None):
        return self._with(self.data.pin_memory())

    def cuda(self, device=None, non_blocking=False):
        return self._with(self.data.cuda(device, non_blocking=non_blocking))

    def image(self, i):
        """Image ``i`` as an ``[H, W, C]`` view of ``data``."""
        h, w = (int(v) for v in self.sizes[i])
        o = int(self.offsets[i])
        return self.data[o:o + h * w * self.channels].view(h, w, self.channels)

    def __repr__(self):
        return f"RaggedImages(n={len(self)}, channels={self.channels}, bytes={self.data.numel()}, device={self.data.device})"


def _as_hwc(img):
    if isinstance(img, np.ndarray):
        arr = img
    elif isinstance(img, torch.Tensor):
        arr = img.numpy()
    else:                                   # a PIL image: np.asarray gives [H, W] ("L") or [H, W, C]
        arr = np.asarray(img)
    if arr.dtype != np.uint8 or arr.ndim not in (2, 3):
        raise TypeError(f"collate_ragged expects uint8 HWC images (PIL images or arrays), got {arr.dtype} {arr.shape}")
    return arr[:, :, None] if arr.ndim == 2 else arr


def _pack(images):
    arrs = [_as_hwc(im) for im in images]
    channels = {a.shape[2] for a in arrs}
    if len(channels) > 1:
        raise ValueError(f"collate_ragged: images with different channel counts {sorted(channels)} in one batch")
    c = channels.pop() if channels else 3
    offsets = np.zeros(len(arrs), dtype=np.int64)
    total = 0
    for i, a in enumerate(arrs):
        offsets[i] = total
        total += -(-a.size // ALIGN) * ALIGN
    buf = np.zeros(max(total, ALIGN), dtype=np.uint8)
    for a, o in zip(arrs, offsets):
        buf[o:o + a.size] = a.reshape(-1)
    sizes = np.array([a.shape[:2] for a in arrs], dtype=np.int64).reshape(len(arrs), 2)
    return RaggedImages(torch.from_numpy(buf), torch.from_numpy(sizes), torch.from_numpy(offsets), c)


def collate_ragged(samples, key="image"):
    """``collate_fn`` for decoded images of any sizes (CPU only, safe in forked workers).

    ``samples``: PIL images / HWC uint8 arrays, or dicts holding one under ``key``.  Images are packed into a
    ``RaggedImages`` with 16-byte-aligned offsets; the other keys of dict samples go through ``default_collate``, so
    ``{"image", "label", "path"}`` samples collate as before with ``batch["image"]`` ragged."""
    from torch.utils.data import default_collate

    samples = list(samples)
    if samples and isinstance(samples[0], dict):
        rest = default_collate([{k: v for k, v in s.items() if k != key} for s in samples])
        rest[key] = _pack([s[key] for s in samples])
        return rest
    return _pack(samples)


def resized_size(h, w, size):
    """torchvision ``Resize(size)``'s output size ``(RH, RW)`` for an ``h x w`` PIL image: an int scales the shorter side
    to ``size`` keeping the aspect ratio (``int(size * long / short)``, Python float arithmetic); a pair is used as given."""
    if isinstance(size, (tuple, list)):
        if len(size) != 2:
            raise ValueError("size must be an int or an (h, w) pair")
        return int(size[0]), int(size[1])
    size = int(size)
    short, long = (w, h) if w <= h else (h, w)
    new_short, new_long = size, int(size * long / short)
    return (new_long, new_short) if w <= h else (new_short, new_long)


def center_crop_origin(rh, rw, ch, cw):
    """torchvision ``CenterCrop``'s ``(top, left)`` inside an ``rh x rw`` image: ``int(round((rh - ch) / 2.0))``, Python's
    round-half-to-even (58.5 -> 58, 67.5 -> 68)."""
    return int(round((rh - ch) / 2.0)), int(round((rw - cw) / 2.0))


def _pair(v, what):
    if isinstance(v, (tuple, list)):
        if len(v) != 2:
            raise ValueError(f"{what} must be an int or an (h, w) pair")
        return int(v[0]), int(v[1])
    return int(v), int(v)


def resize_center_crop(images, size=256, crop=224, interpolation="bilinear"):
    """``Compose([Resize(size, interpolation), CenterCrop(crop)])`` of torchvision on every image of a ragged batch, on the
    device and bit for bit as on PIL images: ``RaggedImages`` with CUDA data -> uint8 CUDA ``[B, C, Hc, Wc]``.

    ``size``: int (shorter side) or ``(h, w)``; ``crop``: int or ``(h, w)``; ``interpolation``: ``"bilinear"`` or
    ``"bicubic"`` (Pillow's antialiased filters).  Raises ``ValueError`` for a crop larger than a resized image (torchvision
    would pad with zeros) and ``NotImplementedError`` for a reduction wider than the 64-tap window (~31x bilinear,
    ~15x bicubic), like ``resize_u8``."""
    _cabi.require_cuda()
    if not isinstance(images, RaggedImages):
        raise TypeError("resize_center_crop expects a RaggedImages batch (collate_ragged)")
    data = images.data
    if not isinstance(data, torch.Tensor) or not data.is_cuda or data.dtype != torch.uint8 or data.dim() != 1:
        raise TypeError("resize_center_crop expects RaggedImages with flat uint8 CUDA data (batch.cuda())")
    filt = {"bicubic": _cabi.RESIZE_BICUBIC, "bilinear": _cabi.RESIZE_BILINEAR}.get(interpolation)
    if filt is None:
        raise ValueError("interpolation must be 'bilinear' or 'bicubic'")
    ch, cw = _pair(crop, "crop")
    if ch < 1 or cw < 1:
        raise ValueError("crop must be positive")
    c = images.channels
    if not 1 <= c <= 4:
        raise ValueError(f"images must have 1 to 4 channels, got {c}")
    n = len(images)
    sizes = images.sizes.cpu().numpy().astype(np.int64).reshape(n, 2)
    offsets = np.ascontiguousarray(images.offsets.cpu().numpy().astype(np.int64).reshape(n))
    geom = np.zeros((n, 6), dtype=np.int32)
    for i in range(n):
        h, w = int(sizes[i, 0]), int(sizes[i, 1])
        if h < 1 or w < 1:
            raise ValueError(f"image {i} is empty ({h} x {w})")
        if offsets[i] < 0 or offsets[i] + h * w * c > data.numel():
            raise ValueError(f"image {i} lies outside the data buffer")
        if offsets[i] % 4:
            raise ValueError(f"image {i}: offset {offsets[i]} is not a multiple of 4")
        rh, rw = resized_size(h, w, size)
        if rh < 1 or rw < 1:
            raise ValueError("size must be positive")
        if ch > rh or cw > rw:
            raise ValueError(f"image {i}: crop {ch}x{cw} is larger than the resized image {rh}x{rw}")
        geom[i] = (h, w, rh, rw) + center_crop_origin(rh, rw, ch, cw)
    out = torch.empty((n, c, ch, cw), dtype=torch.uint8, device=data.device)
    if n == 0:
        return out
    lib = _cabi.load()
    gp, op = ctypes.c_void_p(geom.ctypes.data), ctypes.c_void_p(offsets.ctypes.data)
    nbytes = int(lib.b200_resize_crop_workspace_bytes(n, gp, c, ch, cw, filt))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=data.device)
    with torch.cuda.device(data.device), _cabi.nvtx_range("b200/resize_crop"):
        rc = lib.b200_resize_crop_u8(_cabi.ptr(data), op, gp, n, c, ch, cw, filt, _cabi.ptr(out), _cabi.ptr(ws), ws.numel(),
                                     _cabi.stream_ptr())
    _cabi.check(rc, "b200_resize_crop_u8")
    return out
