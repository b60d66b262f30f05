"""Worker side of the device JPEG decoder (``collate_jpeg``), the oracle and the CPU simulator of the kernels, against
Pillow: bit for bit on the goldens and on seeded random files, the routing of files the device does not decode, the
training draws, malformed files and the C-ABI argument checks.  No GPU needed."""
import ctypes
import io
import os

import numpy as np
import pytest
import torch

from image_retrieval_wavelet_b200 import _cabi
from image_retrieval_wavelet_b200.transforms import collate_jpeg, collate_jpeg_train, collate_ragged_train
from image_retrieval_wavelet_b200.transforms.jpeg import output_offsets
from oracle import jpeg_ref

import simlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "jpeg_golden.npz")


def _golden():
    g = np.load(GOLDEN)
    names = sorted({k.rsplit(".", 1)[0] for k in g.files})
    return [(n, g[f"{n}.jpg"].tobytes(), g[f"{n}.rgb"]) for n in names]


def _random_files(seed, count, max_side=40):
    pytest.importorskip("PIL")
    from PIL import Image

    rng = np.random.default_rng(seed)
    files = []
    for _ in range(count):
        h, w = int(rng.integers(1, max_side)), int(rng.integers(1, max_side))
        gray = rng.random() < 0.25
        if rng.random() < 0.5:
            a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        else:
            y, x = np.mgrid[0:h, 0:w]
            a = np.clip(np.stack([x * 7 % 256, y * 5 % 256, (x + y) * 3 % 256], 2) + rng.normal(0, 10, (h, w, 3)), 0, 255).astype(np.uint8)
        extra = {}
        r = rng.random()
        if r < 0.2:
            extra["optimize"] = True
        elif r < 0.35:
            extra["restart_marker_blocks"] = int(rng.integers(1, 4))
        elif r < 0.45:
            extra["restart_marker_rows"] = 1
        f = io.BytesIO()
        Image.fromarray(a[:, :, 0] if gray else a).save(f, "JPEG", quality=int(rng.choice([1, 25, 50, 75, 90, 95, 100])),
                                                      subsampling=int(rng.integers(0, 3)), **extra)
        files.append(f.getvalue())
    return files


def _pil(b):
    from PIL import Image

    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


def sim_decode(enc, sub_bits=1024):
    sim = simlib.load_sim()
    desc, tab, data = (np.ascontiguousarray(t.numpy()) for t in (enc.desc, enc.tables, enc.data))
    offs, total = output_offsets(enc.sizes)
    out = np.full(total, 0x5A, np.uint8)
    rounds, subs = ctypes.c_int(), ctypes.c_longlong()
    rc = sim.sim_jpeg_decode(simlib.vp(data), simlib.vp(desc), simlib.vp(tab), ctypes.c_size_t(tab.size), len(enc), simlib.vp(out),
                             simlib.vp(offs), ctypes.c_uint(sub_bits), ctypes.byref(rounds), ctypes.byref(subs))
    assert rc == 0, rc
    imgs = [out[o:o + h * w * 3].reshape(h, w, 3) for o, (h, w) in zip(offs, enc.sizes.tolist())]
    return imgs, rounds.value, subs.value


def test_goldens_are_device_decodable_and_the_oracle_matches_pillow():
    for name, b, want in _golden():
        enc = collate_jpeg([b])
        assert enc.n_host_decoded == (1 if name.startswith("unsupported") else 0), name
        assert np.array_equal(jpeg_ref.decode(enc, 0), want), name


def test_oracle_matches_pillow_on_random_files():
    files = _random_files(1, 300)
    enc = collate_jpeg(files)
    assert enc.n_host_decoded == 0
    for i, b in enumerate(files):
        assert np.array_equal(jpeg_ref.decode(enc, i), _pil(b)), i


def test_simulator_matches_pillow_on_the_goldens_in_one_batch():
    gold = _golden()
    enc = collate_jpeg([b for _, b, _ in gold])
    got, rounds, _ = sim_decode(enc)
    for (name, _, want), g in zip(gold, got):
        assert np.array_equal(g, want), name
    assert rounds >= 2


@pytest.mark.parametrize("sub_bits", [8, 40, 256])
def test_simulator_short_subsequences_synchronise_over_several_rounds(sub_bits):
    files = _random_files(2, 40, max_side=48) + [b for n, b, _ in _golden() if n in ("large_420", "rst_rows_444", "q100_420")]
    enc = collate_jpeg(files)
    got, rounds, subs = sim_decode(enc, sub_bits)
    assert subs > 3 * len(files) and rounds >= 3
    for i, b in enumerate(files):
        assert np.array_equal(got[i], _pil(b)), i


def test_routing_puts_unsupported_files_on_the_worker_path():
    g = {n: (b, want) for n, b, want in _golden()}
    names = ["unsupported_progressive", "s2_17x9", "unsupported_cmyk", "gray_31x17", "unsupported_png"]
    enc = collate_jpeg([{"image": g[n][0], "label": i} for i, n in enumerate(names)])
    batch = enc["image"]
    assert batch.n_host_decoded == 3 and enc["label"].tolist() == [0, 1, 2, 3, 4]
    assert batch.desc[:, 0].tolist() == [1, 0, 1, 0, 1]
    got, _, _ = sim_decode(batch)
    for n, img in zip(names, got):
        assert np.array_equal(img, g[n][1]), n
        assert np.array_equal(jpeg_ref.decode(batch, names.index(n)), g[n][1]), n


@pytest.mark.parametrize("seed", [0, 1, 7, 123])
def test_train_draws_match_collate_ragged_train(seed):
    files = _random_files(10 + seed, 12, max_side=300)
    torch.manual_seed(seed)
    enc = collate_jpeg_train(files)
    torch.manual_seed(seed)
    ragged = collate_ragged_train([_pil(b) for b in files])
    assert torch.equal(enc.crop_params, ragged.crop_params) and torch.equal(enc.sizes, ragged.sizes)


def test_malformed_files_raise_value_error_naming_the_sample():
    b = bytearray(_golden()[0][1])
    good = bytes(b)
    with pytest.raises(ValueError, match="sample 1"):
        collate_jpeg([good, good[:len(good) // 2]])                     # truncated inside the scan
    with pytest.raises(ValueError, match="sample 0"):
        collate_jpeg([good[:40]])                                       # truncated in the headers
    dht = good.index(b"\xff\xc4")
    bad = bytearray(good)
    bad[dht + 4] = 0x17                                                 # DHT class 1, id 7
    with pytest.raises(ValueError, match="sample 0"):
        collate_jpeg([bytes(bad)])
    bad = bytearray(good)
    bad[dht + 2:dht + 4] = b"\xff\xf0"                                  # DHT length past the end of the file
    with pytest.raises(ValueError, match="sample 0"):
        collate_jpeg([bytes(bad)])
    dqt = good.index(b"\xff\xdb")
    bad = bytearray(good)
    bad[dqt + 2:dqt + 4] = b"\x00\x01"                                  # length below 2
    with pytest.raises(ValueError):
        collate_jpeg([bytes(bad)])
    sos = good.index(b"\xff\xda")
    bad = bytearray(good)
    bad[sos + 6] = 0x55                                                 # scan refers to Huffman tables 5 / 5
    with pytest.raises(ValueError, match="sample 0"):
        collate_jpeg([bytes(bad)])


def _desc(enc):
    return np.ascontiguousarray(enc.desc.numpy()), np.ascontiguousarray(enc.tables.numpy())


def test_cabi_rejects_bad_arguments_before_any_cuda_call():
    lib = _cabi.load()
    enc = collate_jpeg([b for n, b, _ in _golden() if n in ("s2_17x9", "rst_blocks_420")])
    desc, tab = _desc(enc)
    vp = simlib.vp
    offs = np.zeros(2, np.int64)
    assert lib.b200_jpeg_decode_workspace_bytes(vp(desc), vp(tab), tab.size, 2) > 0
    assert lib.b200_jpeg_decode_u8(None, None, None, 0, 0, None, None, None, 0, None) == _cabi.OK            # n = 0
    assert lib.b200_jpeg_decode_u8(None, vp(desc), vp(tab), tab.size, -1, None, None, None, 0, None) == _cabi.ERR_INVALID_ARG
    assert lib.b200_jpeg_decode_u8(None, vp(desc), vp(tab), tab.size, 2, None, vp(offs), None, 0, None) == _cabi.ERR_INVALID_ARG
    fake = ctypes.c_void_p(256)                                       # never dereferenced: every check precedes the device
    for field, value, err in ((0, 5, _cabi.ERR_INVALID_ARG),          # kind
                              (1, 0, _cabi.ERR_INVALID_ARG),          # height
                              (5, 4, _cabi.ERR_UNSUPPORTED),          # four components
                              (6, 3, _cabi.ERR_UNSUPPORTED),          # 3x2 sampling
                              (9, tab.size, _cabi.ERR_INVALID_ARG),   # interval starts outside the tables
                              (13, tab.size - 8, _cabi.ERR_INVALID_ARG),   # Huffman record outside the tables
                              (4, 3, _cabi.ERR_INVALID_ARG)):         # interval starts past the segment
        d = desc.copy()
        d[0, field] = value                                           # image 0 has restart intervals
        assert lib.b200_jpeg_decode_workspace_bytes(vp(d), vp(tab), tab.size, 2) == 0, field
        assert lib.b200_jpeg_decode_u8(fake, vp(d), vp(tab), tab.size, 2, fake, vp(offs), fake, 1 << 30, None) == err, field
    d = desc.copy()
    d[0, 0], d[0, 4] = 1, 5                                           # raw pixels of the wrong size
    assert lib.b200_jpeg_decode_u8(fake, vp(d), vp(tab), tab.size, 2, fake, vp(offs), fake, 1 << 30, None) == _cabi.ERR_INVALID_ARG
    assert lib.b200_jpeg_decode_u8(fake, vp(desc), vp(tab), tab.size, 2, fake, vp(offs), fake, 16, None) == _cabi.ERR_WORKSPACE
