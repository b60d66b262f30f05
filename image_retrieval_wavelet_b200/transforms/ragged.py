"""Ragged batches of decoded images, and the eval transform ``Resize(size) -> CenterCrop(crop)`` and the training transform
``Resize(size) -> RandomResizedCrop(crop) -> RandomHorizontalFlip`` on the device.

The reference's eval transform (``config/transform/basic_swt.yaml``: ``Resize(256) -> CenterCrop(224) -> SWTTransform``) runs
per PIL image in the DataLoader workers.  Here the workers only decode (``PIL.open(...).convert("RGB")``),
``collate_ragged`` packs the images of a batch, whatever their sizes, into one flat uint8 buffer, and
``resize_center_crop`` produces the cropped ``[B, C, Hc, Wc]`` uint8 batch on the device in one kernel launch
(``b200_resize_crop_u8``), bit-identical to torchvision's ``Compose([Resize(size), CenterCrop(crop)])`` on each PIL image.
It feeds ``SWTTransform.forward`` directly.

The training transform (``Resize -> RandomResizedCrop(224) -> RandomHorizontalFlip``) draws its boxes and flips in the
workers: ``collate_ragged_train`` draws them per sample with torchvision's own torch RNG calls, in sample order, so a worker
consumes the torch random stream exactly as the per-sample ``Compose`` would.  ``resize_random_crop_flip`` then resizes,
crops, resizes again and mirrors on the device (``b200_resize_random_crop_u8``), bit-identical to torchvision on each PIL
image for those draws.
"""
import ctypes
import math

import numpy as np
import torch

from .. import _cabi

__all__ = ["RaggedImages", "collate_ragged", "resize_center_crop", "resized_size", "center_crop_origin",
           "random_resized_crop_params", "collate_ragged_train", "resize_random_crop_flip"]

ALIGN = 16          # byte alignment of every image in the packed buffer


class RaggedImages:
    """Images of different sizes in one flat buffer: image ``i`` is HWC-interleaved uint8 ``[H_i, W_i, channels]`` at byte
    ``offsets[i]`` of ``data``.  ``sizes`` (int64 ``[B, 2]`` = H, W) and ``offsets`` (int64 ``[B]``) stay on the host;
    ``pin_memory()`` and ``cuda()`` act on ``data``, so a DataLoader with ``pin_memory=True`` pins the batch.
    ``crop_params`` (int64 ``[B, 7]`` = top, left, h, w, flip and the resized size RH, RW the box was drawn in, from
    ``collate_ragged_train``) also stays on the host."""

    def __init__(self, data, sizes, offsets, channels, crop_params=None):
        self.data = data
        self.sizes = sizes
        self.offsets = offsets
        self.channels = int(channels)
        self.crop_params = crop_params

    def __len__(self):
        return int(self.sizes.shape[0])

    def _with(self, data):
        return RaggedImages(data, self.sizes, self.offsets, self.channels, self.crop_params)

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
    filt, (ch, cw), sizes, offsets = _device_batch(images, crop, interpolation, "resize_center_crop", "collate_ragged")
    n = len(images)
    geom = np.zeros((n, 6), dtype=np.int32)
    for i in range(n):
        h, w = int(sizes[i, 0]), int(sizes[i, 1])
        rh, rw = resized_size(h, w, size)
        if rh < 1 or rw < 1:
            raise ValueError("size must be positive")
        if ch > rh or cw > rw:
            raise ValueError(f"image {i}: crop {ch}x{cw} is larger than the resized image {rh}x{rw}")
        geom[i] = (h, w, rh, rw) + center_crop_origin(rh, rw, ch, cw)
    return _launch(images, geom, offsets, ch, cw, filt, "b200_resize_crop", "b200/resize_crop")


def _device_batch(images, crop, interpolation, what, collate):
    """The checks both device calls share: (filter id, crop (h, w), host sizes [B, 2], host offsets [B])."""
    _cabi.require_cuda()
    if not isinstance(images, RaggedImages):
        raise TypeError(f"{what} expects a RaggedImages batch ({collate})")
    data = images.data
    if not isinstance(data, torch.Tensor) or not data.is_cuda or data.dtype != torch.uint8 or data.dim() != 1:
        raise TypeError(f"{what} expects RaggedImages with flat uint8 CUDA data (batch.cuda())")
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
    for i in range(n):
        h, w = int(sizes[i, 0]), int(sizes[i, 1])
        if h < 1 or w < 1:
            raise ValueError(f"image {i} is empty ({h} x {w})")
        if offsets[i] < 0 or offsets[i] + h * w * c > data.numel():
            raise ValueError(f"image {i} lies outside the data buffer")
        if offsets[i] % 4:
            raise ValueError(f"image {i}: offset {offsets[i]} is not a multiple of 4")
    return filt, (ch, cw), sizes, offsets


def _launch(images, geom, offsets, ch, cw, filt, entry, nvtx):
    """``<entry>_u8`` on the batch into a new uint8 CUDA ``[B, C, ch, cw]``, with a workspace of ``<entry>_workspace_bytes``."""
    data, n, c = images.data, len(images), images.channels
    out = torch.empty((n, c, ch, cw), dtype=torch.uint8, device=data.device)
    if n == 0:
        return out
    lib = _cabi.load()
    gp, op = ctypes.c_void_p(geom.ctypes.data), ctypes.c_void_p(offsets.ctypes.data)
    nbytes = int(getattr(lib, entry + "_workspace_bytes")(n, gp, c, ch, cw, filt))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=data.device)
    with torch.cuda.device(data.device), _cabi.nvtx_range(nvtx):
        rc = getattr(lib, entry + "_u8")(_cabi.ptr(data), op, gp, n, c, ch, cw, filt, _cabi.ptr(out), _cabi.ptr(ws), ws.numel(),
                                         _cabi.stream_ptr())
    _cabi.check(rc, entry + "_u8")
    return out


def random_resized_crop_params(h, w, size, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3), p=0.5):
    """What ``Compose([Resize(size), RandomResizedCrop(_, scale, ratio), RandomHorizontalFlip(p)])`` of torchvision draws for an
    ``h x w`` PIL image: ``(top, left, ch, cw, flip)``, the box inside the image after ``Resize(size)`` and the flip.

    The torch RNG calls are torchvision's, in its order (``RandomResizedCrop.get_params``: up to 10 tries of
    ``uniform_`` for the area, ``exp(uniform_)`` of the log-ratio and, for the first box that fits, ``randint`` for its
    row and column, else a central box; then ``torch.rand(1) < p``), so the same torch seed gives the same draws."""
    height, width = resized_size(h, w, size)
    area = height * width
    log_ratio = torch.log(torch.tensor(ratio))
    for _ in range(10):
        target_area = area * torch.empty(1).uniform_(scale[0], scale[1]).item()
        aspect_ratio = torch.exp(torch.empty(1).uniform_(log_ratio[0], log_ratio[1])).item()
        cw = int(round(math.sqrt(target_area * aspect_ratio)))
        ch = int(round(math.sqrt(target_area / aspect_ratio)))
        if 0 < cw <= width and 0 < ch <= height:
            top = torch.randint(0, height - ch + 1, size=(1,)).item()
            left = torch.randint(0, width - cw + 1, size=(1,)).item()
            break
    else:                                   # the central box of the ratio range
        in_ratio = float(width) / float(height)
        if in_ratio < min(ratio):
            cw, ch = width, int(round(width / min(ratio)))
        elif in_ratio > max(ratio):
            ch, cw = height, int(round(height * max(ratio)))
        else:
            ch, cw = height, width
        top, left = (height - ch) // 2, (width - cw) // 2
    flip = bool(torch.rand(1) < p)
    return int(top), int(left), ch, cw, flip


def collate_ragged_train(samples, key="image", size=256, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3), p=0.5):
    """``collate_ragged`` plus each sample's ``random_resized_crop_params`` and the resized size they were drawn in
    (``[B, 7]`` = top, left, h, w, flip, RH, RW) in ``crop_params`` of the ``RaggedImages``,
    drawn in sample order in the process that collates (the worker): the torch random stream is consumed exactly as by
    ``Compose([Resize(size), RandomResizedCrop(_, scale, ratio), RandomHorizontalFlip(p)])`` in ``__getitem__``, so an
    identically seeded DataLoader gives the same boxes and flips.  Other parameters: ``functools.partial``."""
    batch = collate_ragged(samples, key)
    images = batch[key] if isinstance(batch, dict) else batch
    images.crop_params = draw_crop_params(images.sizes, size, scale, ratio, p)
    return batch


def draw_crop_params(sizes, size=256, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3), p=0.5):
    """``random_resized_crop_params`` and the resized size of every image of a batch (``sizes``: ``[B, 2]`` = H, W), drawn
    in image order: the ``crop_params`` (int64 ``[B, 7]``) of a training batch."""
    params = [random_resized_crop_params(h, w, size, scale, ratio, p) + resized_size(h, w, size) for h, w in sizes.tolist()]
    return torch.tensor(params, dtype=torch.int64).reshape(len(params), 7)


def resize_random_crop_flip(images, size=256, crop=224, interpolation="bilinear"):
    """``Compose([Resize(size, interpolation), RandomResizedCrop(crop, interpolation=interpolation),
    RandomHorizontalFlip()])`` of torchvision on every image of a ragged batch, on the device and bit for bit as on PIL
    images, for the boxes and flips ``collate_ragged_train`` drew: ``RaggedImages`` with CUDA data -> uint8 CUDA
    ``[B, C, crop_h, crop_w]``.

    ``size`` must be the one the collate drew with.  Raises ``ValueError`` for a batch without ``crop_params``, for boxes
    drawn in another resized size than ``size`` gives, or for a box outside its resized image, and ``NotImplementedError`` for a window of either resize wider than 64 taps, like
    ``resize_center_crop``."""
    filt, (ch, cw), sizes, offsets = _device_batch(images, crop, interpolation, "resize_random_crop_flip", "collate_ragged_train")
    n = len(images)
    if images.crop_params is None:
        raise ValueError("resize_random_crop_flip expects a batch with crop_params (collate_ragged_train)")
    params = images.crop_params.cpu().numpy().astype(np.int64).reshape(n, 7)
    geom = np.zeros((n, 9), dtype=np.int32)
    for i in range(n):
        h, w = int(sizes[i, 0]), int(sizes[i, 1])
        rh, rw = resized_size(h, w, size)
        if rh < 1 or rw < 1:
            raise ValueError("size must be positive")
        top, left, bh, bw, flip, drawn_rh, drawn_rw = (int(v) for v in params[i])
        if (drawn_rh, drawn_rw) != (rh, rw):
            raise ValueError(f"image {i}: its box was drawn in a {drawn_rh}x{drawn_rw} resize, but size={size} resizes it to {rh}x{rw}")
        if bh < 1 or bw < 1 or top < 0 or left < 0 or top + bh > rh or left + bw > rw or flip not in (0, 1):
            raise ValueError(f"image {i}: box {bh}x{bw} at ({top}, {left}) (flip {flip}) does not fit the resized image {rh}x{rw}")
        geom[i] = (h, w, rh, rw, top, left, bh, bw, flip)
    return _launch(images, geom, offsets, ch, cw, filt, "b200_resize_random_crop", "b200/resize_random_crop")
