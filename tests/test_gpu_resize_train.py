"""The training transform of ragged batches on a B200 (``resize_random_crop_flip`` / ``b200_resize_random_crop_u8``): bit for
bit against torchvision's ``Compose([Resize, RandomResizedCrop, RandomHorizontalFlip])`` on PIL images (goldens, and the
installed torchvision when importable) and against the chain on ``oracle/resize_ref.py`` on random geometries."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 4096


def _gen():
    spec = importlib.util.spec_from_file_location("make_golden_resize_train",
                                                  os.path.join(ROOT, "tests", "golden", "make_golden_resize_train.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _train(images, seed, size=256, crop=224, interp="bilinear", p=0.5):
    from image_retrieval_wavelet_b200.transforms import collate_ragged_train, resize_random_crop_flip

    torch.manual_seed(seed)
    return resize_random_crop_flip(collate_ragged_train(images, size=size, p=p).cuda(), size, crop, interp)


def test_matches_torchvision_goldens():
    gen = _gen()
    g = np.load(os.path.join(ROOT, "tests", "golden", "resize_train_golden.npz"))
    for name, (h, w, c, size, crop, interp, seed, p) in gen.CASES.items():
        got = _train([gen.make_image(seed, h, w, c)], seed, size, crop, interp, p)
        assert got.dtype == torch.uint8 and np.array_equal(got[0].cpu().numpy(), g[name]), name


def test_matches_installed_torchvision():
    pytest.importorskip("torchvision")
    gen = _gen()
    rng = np.random.default_rng(7)
    shapes = [(480, 640), (640, 480), (427, 640), (375, 501), (333, 333), (1200, 1601), (224, 999), (31, 17), (1999, 37)]
    for interp in ("bilinear", "bicubic"):
        imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
        got = _train(imgs, 3, interp=interp).cpu().numpy()
        t = gen.train_transform(256, 224, interp, 0.5)
        torch.manual_seed(3)                                        # the same draws, in the same order
        for i, a in enumerate(imgs):
            assert np.array_equal(got[i], gen.from_pil(t(gen.to_pil(a)), 3)), (interp, shapes[i])


class Guarded:
    """A device buffer of `nbytes` with GUARD poisoned bytes on both sides (tests/test_gpu_canaries.py)."""

    def __init__(self, nbytes):
        self.n = int(nbytes)
        self.raw = torch.full((self.n + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        self.ptr = self.raw.data_ptr() + GUARD

    def view(self):
        return self.raw[GUARD:GUARD + self.n]

    def intact(self):
        return bool((self.raw[:GUARD] == 0xA5).all()) and bool((self.raw[GUARD + self.n:] == 0xA5).all())


def _run_c(imgs, geoms, ho, wo, filt):
    """b200_resize_random_crop_u8 over HWC uint8 images packed at 4-byte-aligned offsets; input, output and workspace
    guarded.  geoms: (RH, RW, top, left, h, w, flip) per image."""
    from image_retrieval_wavelet_b200 import _cabi

    c = imgs[0].shape[2]
    offs, total = [], 0
    for a in imgs:
        offs.append(total)
        total += (a.size + 3) // 4 * 4
    buf = np.zeros(max(total, 4), dtype=np.uint8)
    for a, o in zip(imgs, offs):
        buf[o:o + a.size] = a.reshape(-1)
    inp = Guarded(buf.size)
    inp.view().copy_(torch.from_numpy(buf))
    geom = np.array([(a.shape[0], a.shape[1]) + tuple(g) for a, g in zip(imgs, geoms)], dtype=np.int32).reshape(-1, 9)
    offsets = np.array(offs, dtype=np.int64)
    lib = _cabi.load()
    filt_id = {"bilinear": _cabi.RESIZE_BILINEAR, "bicubic": _cabi.RESIZE_BICUBIC}[filt]
    gp, op = ctypes.c_void_p(geom.ctypes.data), ctypes.c_void_p(offsets.ctypes.data)
    nbytes = lib.b200_resize_random_crop_workspace_bytes(len(imgs), gp, c, ho, wo, filt_id)
    ws, out = Guarded(nbytes), Guarded(len(imgs) * c * ho * wo)
    _cabi.check(lib.b200_resize_random_crop_u8(inp.ptr, op, gp, len(imgs), c, ho, wo, filt_id, out.ptr, ws.ptr, nbytes,
                                               _cabi.stream_ptr()), "b200_resize_random_crop_u8")
    torch.cuda.synchronize()
    assert out.intact() and ws.intact() and inp.intact(), "b200_resize_random_crop_u8 wrote outside a buffer"
    return out.view().cpu().numpy().reshape(len(imgs), c, ho, wo)


@pytest.mark.parametrize("c", [1, 3, 4])
@pytest.mark.parametrize("filt", ["bilinear", "bicubic"])
def test_random_geometries_match_the_oracle(c, filt):
    """Any box and flip: odd widths (rows and boxes on every byte offset), identity axes in either resize, enlargements,
    reductions, and output sizes that are not multiples of 4 (the mirrored stores fall back to bytes)."""
    gen = _gen()
    rng = np.random.default_rng(10 * c + len(filt))
    for trial in range(3):
        ho, wo = int(rng.integers(1, 70)), int(rng.integers(1, 270))
        imgs, geoms = [], []
        for k in range(5):
            h, w = int(rng.integers(1, 200)), int(rng.integers(1, 300)) | (k & 1)
            rh, rw = (h, w) if k == 0 else (int(rng.integers(1, 160)), int(rng.integers(1, 220)))
            rh, rw = max(rh, -(-h // 15)), max(rw, -(-w // 15))          # within the 64-tap window of both filters
            bh, bw = min(int(rng.integers(1, rh + 1)), 15 * ho), min(int(rng.integers(1, rw + 1)), 15 * wo)
            if k == 1:
                bh, bw = min(ho, rh), min(wo, rw)                     # the second resize keeps what fits
            top, left = int(rng.integers(0, rh - bh + 1)), int(rng.integers(0, rw - bw + 1))
            imgs.append(rng.integers(0, 256, (h, w, c), dtype=np.uint8))
            geoms.append((rh, rw, top, left, bh, bw, int(rng.integers(0, 2)) if k > 1 else k))
        got = _run_c(imgs, geoms, ho, wo, filt)
        for i, (img, g) in enumerate(zip(imgs, geoms)):
            want = gen.chain_ref(img, g[0], g[1], g[2:], (ho, wo), filt)
            assert np.array_equal(got[i], want), (trial, i, img.shape, g, ho, wo)


def test_one_ragged_call_equals_per_image_calls():
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged_train, resize_random_crop_flip

    gen = _gen()
    names = [n for n, case in gen.CASES.items() if case[2:6] == (3, 256, 224, "bilinear")]
    assert len(names) >= 8
    imgs = [gen.make_image(gen.CASES[n][6], *gen.CASES[n][:3]) for n in names]
    torch.manual_seed(0)
    batch = collate_ragged_train(imgs)
    out = resize_random_crop_flip(batch.cuda())
    assert tuple(out.shape) == (len(names), 3, 224, 224)
    for i, img in enumerate(imgs):
        one = collate_ragged_train([img])
        one = RaggedImages(one.data, one.sizes, one.offsets, 3, batch.crop_params[i:i + 1])
        assert torch.equal(out[i], resize_random_crop_flip(one.cuda())[0]), names[i]


def test_pinned_batch_and_dataloader_pinning():
    """The boxes travel with the pinned batch; the result is the unpinned batch's with the same boxes."""
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged, collate_ragged_train, resize_random_crop_flip

    rng = np.random.default_rng(3)
    samples = [{"image": rng.integers(0, 256, (240 + 7 * i, 320 - 5 * i, 3), dtype=np.uint8), "label": i} for i in range(6)]
    loader = torch.utils.data.DataLoader(samples, batch_size=3, collate_fn=collate_ragged_train, pin_memory=True)
    for j, batch in enumerate(loader):
        imgs = batch["image"]
        assert imgs.data.is_pinned() and tuple(imgs.crop_params.shape) == (3, 7)
        got = resize_random_crop_flip(imgs.cuda(non_blocking=True))
        plain = collate_ragged([s["image"] for s in samples[3 * j:3 * j + 3]])
        want = resize_random_crop_flip(RaggedImages(plain.data, plain.sizes, plain.offsets, 3, imgs.crop_params).cuda())
        assert torch.equal(got, want) and batch["label"].tolist() == [3 * j, 3 * j + 1, 3 * j + 2]


def test_empty_and_single_image_batches():
    from image_retrieval_wavelet_b200.transforms import collate_ragged_train, resize_random_crop_flip

    empty = resize_random_crop_flip(collate_ragged_train([]).cuda())
    assert tuple(empty.shape) == (0, 3, 224, 224) and empty.is_cuda
    img = np.random.default_rng(2).integers(0, 256, (300, 400, 3), dtype=np.uint8)
    torch.manual_seed(4)
    batch = collate_ragged_train([img])
    one = resize_random_crop_flip(batch.cuda())
    want = _gen().chain_ref(img, 256, 341, batch.crop_params[0].tolist()[:5], (224, 224), "bilinear")
    assert tuple(one.shape) == (1, 3, 224, 224) and np.array_equal(one[0].cpu().numpy(), want)


def test_rejects_unsupported_requests():
    from image_retrieval_wavelet_b200.transforms import (RaggedImages, collate_ragged, collate_ragged_train,
                                                         resize_random_crop_flip)
    from image_retrieval_wavelet_b200.transforms.ragged import resized_size

    def with_box(arr, box, size=256):
        b = collate_ragged([arr])
        params = torch.tensor([box + resized_size(arr.shape[0], arr.shape[1], size)], dtype=torch.int64)
        return RaggedImages(b.data, b.sizes, b.offsets, b.channels, params).cuda()

    img = np.zeros((100, 120, 3), np.uint8)                         # resized 256 x 307
    with pytest.raises(TypeError):
        resize_random_crop_flip(collate_ragged_train([img]))       # host data
    with pytest.raises(ValueError):
        resize_random_crop_flip(collate_ragged([img]).cuda())      # no boxes drawn
    with pytest.raises(ValueError):
        resize_random_crop_flip(collate_ragged_train([img], size=256).cuda(), size=300)       # drawn for another size
    with pytest.raises(ValueError):
        resize_random_crop_flip(with_box(img, (100, 0, 157, 200, 0)))          # rows past the resized image
    with pytest.raises(ValueError):
        resize_random_crop_flip(with_box(img, (0, 108, 100, 200, 0)))          # columns past it
    with pytest.raises(ValueError):
        resize_random_crop_flip(with_box(img, (0, 0, 100, 200, 2)))            # flip is 0 or 1
    with pytest.raises(ValueError):
        resize_random_crop_flip(with_box(img, (0, 0, 100, 200, 0)), interpolation="lanczos")
    with pytest.raises(ValueError):
        resize_random_crop_flip(with_box(img, (0, 0, 100, 200, 0)), crop=0)
    with pytest.raises(NotImplementedError):                       # first resize 8000 -> 256: 65 taps
        resize_random_crop_flip(with_box(np.zeros((8000, 300, 1), np.uint8), (0, 0, 200, 200, 0), (256, 256)), size=(256, 256))
    with pytest.raises(NotImplementedError):                       # second resize 7000 -> 224: 65 taps
        resize_random_crop_flip(with_box(np.zeros((7000, 300, 1), np.uint8), (0, 0, 7000, 300, 0), (7000, 300)), size=(7000, 300))
    near = resize_random_crop_flip(with_box(np.zeros((6944, 300, 1), np.uint8), (0, 0, 6944, 300, 1), (6944, 300)), size=(6944, 300))
    assert tuple(near.shape) == (1, 1, 224, 224) and int(near.max()) == 0      # 31x: the widest supported window
