"""JPEG files -> ragged RGB batches, decoded on the device bit for bit as ``PIL.Image.open(f).convert("RGB")`` decodes them.

The DataLoader workers only read file bytes.  ``collate_jpeg`` (CPU only, safe in forked workers) parses each file's
markers, builds its Huffman decode tables (libjpeg's 8-bit lookahead table plus maxcode / valoffset) and natural-order
quantisation tables, and strips byte stuffing and restart markers from the entropy-coded segment with numpy, recording
where each restart interval starts.  ``decode_jpeg`` then decodes the whole batch on the device (``b200_jpeg_decode_u8``):
a self-synchronising parallel Huffman decode, libjpeg's integer "islow" IDCT, fancy (triangle) chroma upsampling and
libjpeg's fixed-point YCbCr -> RGB, into the ``RaggedImages`` layout ``collate_ragged`` + ``.cuda()`` produce, so
``resize_center_crop``, ``resize_random_crop_flip`` and ``SWTTransform.forward`` take it unchanged.

Device-decodable: 8-bit, Huffman-coded, single-scan sequential (SOF0 / SOF1) files with one component (grayscale,
replicated to RGB as ``convert("RGB")`` does) or three YCbCr components with luma sampling 1x1, 2x1 or 2x2 and chroma 1x1,
any restart interval.  Every other file (progressive, arithmetic-coded, 12-bit, lossless, CMYK / YCCK, Adobe RGB,
multi-scan, other sampling factors, non-JPEG data) is decoded in the worker with ``Image.open(...).convert("RGB")``, exactly
as without this module, and travels as raw HWC pixels in the same buffer; ``EncodedImages.n_host_decoded`` counts them.
"""
import ctypes
import io

import numpy as np
import torch

from .. import _cabi
from .ragged import ALIGN, RaggedImages, draw_crop_params

__all__ = ["EncodedImages", "collate_jpeg", "collate_jpeg_train", "decode_jpeg"]

KIND_HUFFMAN, KIND_RAW = 0, 1
DESC_WORDS = 19             # int64 fields of b200_jpeg_desc (include/b200ret.h)
HUFF_BYTES, QUANT_BYTES = 1024, 128

# zigzag position -> natural (row-major) position
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                   21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53,
                   60, 61, 54, 47, 55, 62, 63], dtype=np.int64)


class EncodedImages:
    """A batch of JPEG files as the device decoder takes it.

    ``data``: flat uint8 tensor; image ``i``'s bytes start at ``desc[i, 3]`` (16-byte aligned): its entropy-coded segment
    without stuffing or restart markers (kind 0), or its decoded HWC RGB pixels (kind 1, the worker path).
    ``sizes`` (int64 ``[B, 2]`` = H, W), ``desc`` (int64 ``[B, 19]``, ``b200_jpeg_desc``), ``tables`` (uint8: Huffman
    records, quantisation records and restart-interval starts the descriptors point into) and ``crop_params`` (from
    ``collate_jpeg_train``) stay on the host; ``pin_memory()`` and ``cuda()`` act on ``data`` alone, as for
    ``RaggedImages``.  ``n_host_decoded``: how many images of the batch took the worker path."""

    def __init__(self, data, sizes, desc, tables, crop_params=None, n_host_decoded=0):
        self.data = data
        self.sizes = sizes
        self.desc = desc
        self.tables = tables
        self.crop_params = crop_params
        self.n_host_decoded = int(n_host_decoded)

    def __len__(self):
        return int(self.sizes.shape[0])

    def _with(self, data):
        return EncodedImages(data, self.sizes, self.desc, self.tables, self.crop_params, self.n_host_decoded)

    def pin_memory(self, device=None):
        return self._with(self.data.pin_memory())

    def cuda(self, device=None, non_blocking=False):
        return self._with(self.data.cuda(device, non_blocking=non_blocking))

    def __repr__(self):
        return (f"EncodedImages(n={len(self)}, bytes={self.data.numel()}, host_decoded={self.n_host_decoded}, "
                f"device={self.data.device})")


class _WorkerPath(Exception):
    """A well-formed file outside the device envelope: Pillow decodes it in the worker."""


def _u16(b, i):
    return (b[i] << 8) | b[i + 1]


def huffman_record(counts, values, is_dc, name):
    """libjpeg's decode form of one DHT table (jdhuff.c jpeg_make_d_derived_tbl) as a 1024-byte record: uint16 look[256]
    ((length << 8) | symbol for codes of up to 8 bits, 0 otherwise) at 0, int32 maxcode[18] at 512, int32 valoffset[18]
    at 584, uint8 huffval[256] at 656.  Raises ValueError for the tables libjpeg rejects."""
    counts = [int(c) for c in counts]
    values = np.asarray(values, dtype=np.uint8)
    if sum(counts) > 256 or sum(counts) != len(values):
        raise ValueError(f"{name}: bad Huffman table (counts)")
    if is_dc and len(values) and int(values.max()) > 15:
        raise ValueError(f"{name}: bad DC Huffman table (symbol > 15)")
    code, p = 0, 0
    codes, sizes = [], []
    maxcode = np.full(18, -1, dtype=np.int32)
    valoff = np.zeros(18, dtype=np.int32)
    for length in range(1, 17):
        n = counts[length - 1]
        if n:
            valoff[length] = p - code
            codes += range(code, code + n)
            sizes += [length] * n
            p += n
            code += n
            maxcode[length] = code - 1
        if code >= (1 << length):
            raise ValueError(f"{name}: bad Huffman table (oversubscribed code lengths)")
        code <<= 1
    maxcode[17] = 0x7FFFFFFF
    look = np.zeros(256, dtype=np.uint16)
    for i, (c, s) in enumerate(zip(codes, sizes)):
        if s <= 8:
            lo = c << (8 - s)
            look[lo:lo + (1 << (8 - s))] = (s << 8) | int(values[i])
    rec = np.zeros(HUFF_BYTES, dtype=np.uint8)
    rec[0:512] = look.view(np.uint8)
    rec[512:584] = maxcode.view(np.uint8)
    rec[584:656] = valoff.view(np.uint8)
    rec[656:656 + len(values)] = values
    return rec


def _entropy_segment(b, start, n_intervals, name):
    """Strips the entropy-coded segment at ``b[start:]``: returns (clean bytes, interval starts, end of segment in ``b``).
    ``FF 00`` is a data byte ``FF``, ``FF FF`` fill bytes are dropped, ``FF D0``..``FF D7`` (restart markers) are dropped
    and start a new interval, and any other ``FF xx`` ends the segment."""
    seg = np.frombuffer(b, dtype=np.uint8, offset=start)
    nxt = np.empty_like(seg)
    nxt[:-1] = seg[1:]
    if len(seg):
        nxt[-1] = 0xFF                                   # a final FF has no code byte: the segment is unterminated
    is_ff = seg == 0xFF
    rst = is_ff & (nxt >= 0xD0) & (nxt <= 0xD7)
    term = np.flatnonzero(is_ff & (nxt != 0) & (nxt != 0xFF) & ~rst)
    if not len(term):
        raise ValueError(f"{name}: truncated file (the entropy-coded segment has no terminating marker)")
    end = int(term[0])
    seg, nxt, is_ff, rst = seg[:end], nxt[:end], is_ff[:end], rst[:end]
    keep = ~(is_ff & (nxt == 0xFF)) & ~rst
    keep[1:] &= ~(is_ff[:-1] & (nxt[:-1] == 0)) & ~rst[:-1]
    pos = np.flatnonzero(rst)
    if len(pos) != n_intervals - 1 or np.any((nxt[pos] - 0xD0) != np.arange(len(pos)) % 8):
        raise ValueError(f"{name}: {len(pos)} restart markers where the restart interval implies {n_intervals - 1}, or out of sequence")
    before = np.concatenate([[0], np.cumsum(keep)])
    starts = np.concatenate([[0], before[pos]]).astype(np.int64)
    return seg[keep], starts, start + end


def parse_jpeg(b, name="sample"):
    """Markers of one file -> dict of what the device decoder needs.  Raises ``_WorkerPath`` for a file outside the
    device envelope and ``ValueError`` for a malformed one."""
    n = len(b)
    if n < 4 or b[0] != 0xFF or b[1] != 0xD8:
        raise _WorkerPath("not a JPEG file")
    quant, huff = {}, {}
    frame, restart, jfif, adobe = None, 0, False, None
    pos = 2
    while True:
        if pos + 1 >= n:
            raise ValueError(f"{name}: truncated file (no scan)")
        if b[pos] != 0xFF:
            raise ValueError(f"{name}: expected a marker at byte {pos}")
        while pos + 1 < n and b[pos + 1] == 0xFF:
            pos += 1
        if pos + 1 >= n:
            raise ValueError(f"{name}: truncated file (no scan)")
        m = b[pos + 1]
        if m == 0x01 or 0xD0 <= m <= 0xD7:
            pos += 2
            continue
        if m in (0xD8, 0xD9):
            raise ValueError(f"{name}: marker FF{m:02X} before the first scan")
        if pos + 4 > n:
            raise ValueError(f"{name}: truncated marker segment")
        length = _u16(b, pos + 2)
        if length < 2 or pos + 2 + length > n:
            raise ValueError(f"{name}: bad length {length} of marker FF{m:02X}")
        seg = b[pos + 4:pos + 2 + length]
        pos += 2 + length
        if m == 0xDB:                                                    # DQT
            i = 0
            while i < len(seg):
                pq, tq = seg[i] >> 4, seg[i] & 15
                size = 64 * (2 if pq else 1)
                if pq > 1 or tq > 3 or i + 1 + size > len(seg):
                    raise ValueError(f"{name}: bad quantisation table (id {tq}, precision {pq}, length)")
                raw = np.frombuffer(seg[i + 1:i + 1 + size], dtype=">u2" if pq else np.uint8).astype(np.uint16)
                q = np.zeros(64, dtype=np.uint16)
                q[ZIGZAG] = raw
                quant[tq] = q
                i += 1 + size
        elif m == 0xC4:                                                  # DHT
            i = 0
            while i < len(seg):
                if i + 17 > len(seg):
                    raise ValueError(f"{name}: bad Huffman table length")
                tc, th = seg[i] >> 4, seg[i] & 15
                if tc > 1 or th > 3:
                    raise ValueError(f"{name}: bad Huffman table id (class {tc}, id {th})")
                counts = list(seg[i + 1:i + 17])
                total = sum(counts)
                if i + 17 + total > len(seg):
                    raise ValueError(f"{name}: bad Huffman table length")
                huff[(tc, th)] = huffman_record(counts, list(seg[i + 17:i + 17 + total]), tc == 0, name)
                i += 17 + total
        elif m in (0xC0, 0xC1):                                          # SOF0 / SOF1
            if frame is not None:
                raise ValueError(f"{name}: two frame headers")
            if len(seg) < 6 or len(seg) != 6 + 3 * seg[5]:
                raise ValueError(f"{name}: bad frame header length")
            prec, h, w, nf = seg[0], _u16(seg, 1), _u16(seg, 3), seg[5]
            comps = [(seg[6 + 3 * c], seg[7 + 3 * c] >> 4, seg[7 + 3 * c] & 15, seg[8 + 3 * c]) for c in range(nf)]
            if h == 0 or w == 0 or nf == 0:
                raise ValueError(f"{name}: bad frame size {h} x {w} x {nf}")
            if any(not (1 <= hs <= 4 and 1 <= vs <= 4) or tq > 3 for _, hs, vs, tq in comps):
                raise ValueError(f"{name}: bad sampling factors or quantisation table id")
            frame = (prec, h, w, comps)
        elif m in (0xC2, 0xC3, 0xC5, 0xC6, 0xC7, 0xC9, 0xCA, 0xCB, 0xCC, 0xCD, 0xCE, 0xCF):
            raise _WorkerPath(f"frame type FF{m:02X}")                   # progressive, lossless, arithmetic, hierarchical
        elif m == 0xDD:                                                  # DRI
            if len(seg) != 2:
                raise ValueError(f"{name}: bad restart interval length")
            restart = _u16(seg, 0)
        elif m == 0xE0:
            jfif = jfif or (len(seg) >= 12 and seg[:5] == b"JFIF\0")
        elif m == 0xEE:
            if len(seg) >= 12 and seg[:5] == b"Adobe":
                adobe = seg[11]
        elif m == 0xDA:                                                  # SOS
            break
    if frame is None:
        raise ValueError(f"{name}: scan before the frame header")
    prec, h, w, comps = frame
    if len(seg) < 1 or len(seg) != 4 + 2 * seg[0]:
        raise ValueError(f"{name}: bad scan header length")
    ns = seg[0]
    scan = [(seg[1 + 2 * j], seg[2 + 2 * j] >> 4, seg[2 + 2 * j] & 15) for j in range(ns)]
    ss, se, ahal = seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns]
    if prec != 8:
        raise _WorkerPath(f"{prec}-bit samples")
    if len(comps) not in (1, 3):
        raise _WorkerPath(f"{len(comps)} components")
    if len(comps) == 3:
        ids = tuple(c[0] for c in comps)
        rgb = (not jfif) and ((adobe == 0) if adobe is not None else ids == (82, 71, 66))   # libjpeg's colour-space guess
        if rgb:
            raise _WorkerPath("RGB colour space")
        if (comps[0][1], comps[0][2]) not in ((1, 1), (2, 1), (2, 2)) or any((c[1], c[2]) != (1, 1) for c in comps[1:]):
            raise _WorkerPath("sampling factors")
    if ns != len(comps) or [s[0] for s in scan] != [c[0] for c in comps] or (ss, se, ahal) != (0, 63, 0):
        raise _WorkerPath("multi-scan or non-sequential scan")
    for c, (_, td, ta) in zip(comps, scan):
        if td > 3 or ta > 3 or (0, td) not in huff or (1, ta) not in huff:
            raise ValueError(f"{name}: bad Huffman table id (DC {td}, AC {ta})")
        if c[3] not in quant:
            raise ValueError(f"{name}: quantisation table {c[3]} is not defined")
    hmax, vmax = (comps[0][1], comps[0][2]) if len(comps) == 3 else (1, 1)
    mcus = -(-w // (8 * hmax)) * -(-h // (8 * vmax))
    n_int = -(-mcus // restart) if restart else 1
    clean, starts, end = _entropy_segment(b, pos, n_int, name)
    tail = end
    while tail + 1 < n and b[tail] == 0xFF and b[tail + 1] == 0xFF:
        tail += 1
    if tail + 1 >= n or b[tail + 1] != 0xD9:
        raise _WorkerPath("markers after the first scan")               # a second scan, DNL, ...: Pillow's business
    return {"h": h, "w": w, "ncomp": len(comps), "hmax": hmax, "vmax": vmax, "restart": restart, "entropy": clean,
            "starts": starts, "quant": [quant[c[3]] for c in comps],
            "dc": [huff[(0, s[1])] for s in scan], "ac": [huff[(1, s[2])] for s in scan]}


def _pil_rgb(b):
    from PIL import Image

    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


def _pack(files, names):
    pieces, desc, sizes = [], np.zeros((len(files), DESC_WORDS), dtype=np.int64), np.zeros((len(files), 2), dtype=np.int64)
    tab_index, tab_blobs, tab_bytes = {}, [], [0]
    starts_blobs = []
    host = 0

    def table(rec):
        key = rec.tobytes()
        if key not in tab_index:
            tab_index[key] = tab_bytes[0]
            tab_blobs.append(rec)
            tab_bytes[0] += len(rec)
        return tab_index[key]

    for i, (b, name) in enumerate(zip(files, names)):
        if isinstance(b, (bytearray, memoryview)):
            b = bytes(b)
        if not isinstance(b, bytes):
            raise TypeError(f"collate_jpeg expects file bytes (open(path, 'rb').read()), got {type(b).__name__} for {name}")
        try:
            p = parse_jpeg(b, name)
        except _WorkerPath:
            p = None
        if p is None:
            rgb = _pil_rgb(b)
            host += 1
            pieces.append(np.ascontiguousarray(rgb).reshape(-1))
            desc[i, :3] = (KIND_RAW, rgb.shape[0], rgb.shape[1])
            desc[i, 5:8] = (3, 1, 1)
        else:
            pieces.append(p["entropy"])
            desc[i, :3] = (KIND_HUFFMAN, p["h"], p["w"])
            desc[i, 5:9] = (p["ncomp"], p["hmax"], p["vmax"], p["restart"])
            starts_blobs.append((i, p["starts"]))
            for c in range(p["ncomp"]):
                desc[i, 10 + c] = table(np.ascontiguousarray(p["quant"][c]).view(np.uint8))
                desc[i, 13 + c] = table(p["dc"][c])
                desc[i, 16 + c] = table(p["ac"][c])
        sizes[i] = desc[i, 1:3]
    for i, s in starts_blobs:
        desc[i, 9] = table(s.view(np.uint8))
    offsets, total = [], 0
    for a in pieces:
        offsets.append(total)
        total += -(-len(a) // ALIGN) * ALIGN
    buf = np.zeros(max(total, ALIGN), dtype=np.uint8)
    for i, (a, o) in enumerate(zip(pieces, offsets)):
        buf[o:o + len(a)] = a
        desc[i, 3:5] = (o, len(a))
    tables = np.concatenate(tab_blobs) if tab_blobs else np.zeros(8, dtype=np.uint8)
    return EncodedImages(torch.from_numpy(buf), torch.from_numpy(sizes), torch.from_numpy(desc), torch.from_numpy(tables),
                         n_host_decoded=host)


def collate_jpeg(samples, key="image"):
    """``collate_fn`` for JPEG file bytes (``open(path, "rb").read()``; CPU only, safe in forked workers).

    ``samples``: bytes, or dicts holding them under ``key``; the other keys go through ``default_collate``, as in
    ``collate_ragged``.  Returns an ``EncodedImages`` (or the dict with it under ``key``) for ``decode_jpeg``.  Raises
    ``ValueError`` naming the sample for a malformed JPEG file."""
    from torch.utils.data import default_collate

    samples = list(samples)
    if samples and isinstance(samples[0], dict):
        rest = default_collate([{k: v for k, v in s.items() if k != key} for s in samples])
        rest[key] = _pack([s[key] for s in samples], [f"sample {i}" for i in range(len(samples))])
        return rest
    return _pack(samples, [f"sample {i}" for i in range(len(samples))])


def collate_jpeg_train(samples, key="image", size=256, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3), p=0.5):
    """``collate_jpeg`` plus the boxes and flips of ``Resize(size) -> RandomResizedCrop -> RandomHorizontalFlip`` drawn in
    sample order from the header sizes, in ``crop_params`` (``[B, 7]``): the same draws ``collate_ragged_train`` makes for
    the decoded images under the same torch seed."""
    batch = collate_jpeg(samples, key)
    images = batch[key] if isinstance(batch, dict) else batch
    images.crop_params = draw_crop_params(images.sizes, size, scale, ratio, p)
    return batch


def output_offsets(sizes):
    """Byte offsets of the decoded images in the ragged output (HWC RGB, 16-byte aligned, as ``collate_ragged`` packs)."""
    n = np.asarray(sizes, dtype=np.int64).reshape(-1, 2)
    padded = -(-(n[:, 0] * n[:, 1] * 3) // ALIGN) * ALIGN
    offsets = np.zeros(len(n), dtype=np.int64)
    if len(n):
        offsets[1:] = np.cumsum(padded)[:-1]
    return offsets, int(max(padded.sum(), ALIGN))


def decode_jpeg(encoded):
    """``EncodedImages`` with CUDA data -> ``RaggedImages`` with CUDA data: every image as
    ``Image.open(f).convert("RGB")`` gives it, HWC uint8 at 16-byte-aligned offsets; ``crop_params`` carried over."""
    _cabi.require_cuda()
    if not isinstance(encoded, EncodedImages):
        raise TypeError("decode_jpeg expects an EncodedImages batch (collate_jpeg)")
    data = encoded.data
    if not isinstance(data, torch.Tensor) or not data.is_cuda or data.dtype != torch.uint8 or data.dim() != 1:
        raise TypeError("decode_jpeg expects EncodedImages with flat uint8 CUDA data (batch.cuda())")
    n = len(encoded)
    desc = np.ascontiguousarray(encoded.desc.numpy(), dtype=np.int64).reshape(n, DESC_WORDS)
    tables = np.ascontiguousarray(encoded.tables.numpy(), dtype=np.uint8)
    if n and np.any(desc[:, 3] + desc[:, 4] > data.numel()):
        raise ValueError("decode_jpeg: an image's bytes lie outside the data buffer")
    offsets, total = output_offsets(encoded.sizes)
    out = torch.empty(total, dtype=torch.uint8, device=data.device)
    if n:
        lib = _cabi.load()
        dp, tp, op = (ctypes.c_void_p(a.ctypes.data) for a in (desc, tables, offsets))
        nbytes = int(lib.b200_jpeg_decode_workspace_bytes(dp, tp, tables.size, n))
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=data.device)
        with torch.cuda.device(data.device), _cabi.nvtx_range("b200/jpeg_decode"):
            rc = lib.b200_jpeg_decode_u8(_cabi.ptr(data), dp, tp, tables.size, n, _cabi.ptr(out), op, _cabi.ptr(ws), ws.numel(),
                                         _cabi.stream_ptr())
        _cabi.check(rc, "b200_jpeg_decode_u8")
    return RaggedImages(out, encoded.sizes.clone(), torch.from_numpy(offsets), 3, encoded.crop_params)
