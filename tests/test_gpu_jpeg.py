"""The device JPEG decoder on a B200 (``decode_jpeg`` / ``b200_jpeg_decode_u8``): bit for bit against Pillow's
``Image.open(f).convert("RGB")`` (goldens, and the installed Pillow), against ``oracle/jpeg_ref.py`` on random files, for
mixed batches with worker-decoded images, with guard bytes around every buffer, and through both crop chains."""
import ctypes
import io
import os

import numpy as np
import pytest
import torch

from test_jpeg_host import _golden, _pil, _random_files

pytestmark = pytest.mark.gpu

GUARD = 4096


def _decode(files):
    from image_retrieval_wavelet_b200.transforms import collate_jpeg, decode_jpeg

    out = decode_jpeg(collate_jpeg(files).cuda())
    return [out.image(i).cpu().numpy() for i in range(len(out))], out


def test_matches_pillow_goldens_in_one_batch():
    gold = _golden()
    got, out = _decode([b for _, b, _ in gold])
    assert out.data.is_cuda and out.channels == 3
    for (name, _, want), g in zip(gold, got):
        assert np.array_equal(g, want), name


def test_matches_installed_pillow_and_the_oracle_on_random_files():
    pytest.importorskip("PIL")
    from image_retrieval_wavelet_b200.transforms import collate_jpeg
    from oracle import jpeg_ref

    files = _random_files(5, 200, max_side=90)
    got, _ = _decode(files)
    enc = collate_jpeg(files)
    for i, b in enumerate(files):
        assert np.array_equal(got[i], _pil(b)), i
        if i < 60:
            assert np.array_equal(got[i], jpeg_ref.decode(enc, i)), i


def test_large_photo_like_files():
    pytest.importorskip("PIL")
    from PIL import Image

    rng = np.random.default_rng(3)
    files = []
    for h, w, ss in ((1200, 1601, 2), (999, 1333, 1), (640, 480, 0)):
        y, x = np.mgrid[0:h, 0:w].astype(np.float64)
        a = np.clip(np.stack([128 + 90 * np.sin(x / 37.0) * np.cos(y / 23.0), x * 255 / w, y * 255 / h], 2) + rng.normal(0, 8, (h, w, 3)), 0, 255)
        f = io.BytesIO()
        Image.fromarray(a.astype(np.uint8)).save(f, "JPEG", quality=90, subsampling=ss)
        files.append(f.getvalue())
    got, _ = _decode(files)
    for i, b in enumerate(files):
        assert np.array_equal(got[i], _pil(b)), i


def test_one_ragged_call_equals_per_image_calls_and_mixed_batches():
    gold = _golden()
    files = [b for _, b, _ in gold]
    got, out = _decode(files)
    for i, b in enumerate(files):
        one, _ = _decode([b])
        assert np.array_equal(one[0], got[i]), gold[i][0]
    assert sum(n.startswith("unsupported") for n, _, _ in gold) == 3


class Guarded:
    def __init__(self, nbytes):
        self.n = int(nbytes)
        self.raw = torch.full((self.n + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        self.ptr = self.raw.data_ptr() + GUARD

    def view(self):
        return self.raw[GUARD:GUARD + self.n]

    def intact(self):
        return bool((self.raw[:GUARD] == 0xA5).all()) and bool((self.raw[GUARD + self.n:] == 0xA5).all())


def test_guard_bytes_around_input_output_and_workspace():
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms import collate_jpeg
    from image_retrieval_wavelet_b200.transforms.jpeg import output_offsets

    gold = _golden()
    enc = collate_jpeg([b for _, b, _ in gold] + _random_files(9, 30))
    desc, tab = np.ascontiguousarray(enc.desc.numpy()), np.ascontiguousarray(enc.tables.numpy())
    offs, total = output_offsets(enc.sizes)
    data = enc.data.numpy()
    inp = Guarded(data.size)
    inp.view().copy_(torch.from_numpy(data))
    lib = _cabi.load()
    dp, tp, op = (ctypes.c_void_p(a.ctypes.data) for a in (desc, tab, offs))
    nbytes = lib.b200_jpeg_decode_workspace_bytes(dp, tp, tab.size, len(enc))
    ws, out = Guarded(nbytes), Guarded(total)
    _cabi.check(lib.b200_jpeg_decode_u8(inp.ptr, dp, tp, tab.size, len(enc), out.ptr, op, ws.ptr, nbytes, _cabi.stream_ptr()),
                "b200_jpeg_decode_u8")
    torch.cuda.synchronize()
    assert inp.intact() and ws.intact() and out.intact()
    flat = out.view().cpu().numpy()
    rounds = int(ws.view()[:4].cpu().numpy().view(np.uint32)[0])
    assert rounds >= 1
    for i, (name, _, want) in enumerate(gold):
        h, w = want.shape[:2]
        assert np.array_equal(flat[offs[i]:offs[i] + h * w * 3].reshape(h, w, 3), want), name


@pytest.mark.parametrize("seed", [0, 5])
def test_eval_and_train_chains_equal_the_pillow_decode_chains(seed):
    from image_retrieval_wavelet_b200.transforms import (collate_jpeg, collate_jpeg_train, collate_ragged, collate_ragged_train,
                                                         decode_jpeg, resize_center_crop, resize_random_crop_flip)

    files = _random_files(20 + seed, 10, max_side=400) + [b for _, b, _ in _golden()][-8:]
    decoded = [_pil(b) for b in files]
    got = resize_center_crop(decode_jpeg(collate_jpeg(files).cuda()), 256, 224)
    want = resize_center_crop(collate_ragged(decoded).cuda(), 256, 224)
    assert torch.equal(got, want)
    torch.manual_seed(seed)
    got = resize_random_crop_flip(decode_jpeg(collate_jpeg_train(files).cuda()))
    torch.manual_seed(seed)
    want = resize_random_crop_flip(collate_ragged_train(decoded).cuda())
    assert torch.equal(got, want)


def test_empty_batch_and_bad_calls():
    from image_retrieval_wavelet_b200.transforms import collate_jpeg, decode_jpeg

    empty = decode_jpeg(collate_jpeg([]).cuda())
    assert len(empty) == 0 and empty.data.is_cuda
    with pytest.raises(TypeError):
        decode_jpeg(collate_jpeg([_golden()[0][1]]))                     # host data
