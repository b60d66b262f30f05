"""Host side of the training transform (no device): ``random_resized_crop_params`` draws what torchvision draws, the chain
on ``oracle/resize_ref.py`` (window of the resize -> uint8 -> full resize -> mirror) is torchvision's ``Compose`` on PIL,
a seeded DataLoader with ``collate_ragged_train`` reproduces a seeded torchvision loader, and the C-ABI's argument checks."""
import ctypes
import functools
import importlib.util
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gen():
    spec = importlib.util.spec_from_file_location("make_golden_resize_train",
                                                  os.path.join(ROOT, "tests", "golden", "make_golden_resize_train.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# (h, w) before Resize(256); 1999 x 37 resizes to 13830 x 256, where no try fits and the central box is taken
SHAPES = [(480, 640), (640, 480), (427, 640), (375, 500), (1999, 37), (37, 1999), (60, 90), (3000, 4000), (257, 255),
          (256, 256), (12, 10)]


def test_draws_match_torchvision_get_params():
    pytest.importorskip("torchvision")
    from PIL import Image
    from torchvision.transforms import RandomResizedCrop

    from image_retrieval_wavelet_b200.transforms import random_resized_crop_params
    from image_retrieval_wavelet_b200.transforms.ragged import resized_size

    fallbacks = 0
    for h, w in SHAPES:
        rh, rw = resized_size(h, w, 256)
        resized = Image.new("L", (rw, rh))
        for scale, ratio, p in (((0.08, 1.0), (3 / 4, 4 / 3), 0.5), ((0.5, 0.9), (0.5, 2.0), 0.3)):
            for seed in range(12):
                torch.manual_seed(seed)
                top, left, bh, bw = RandomResizedCrop.get_params(resized, list(scale), list(ratio))
                want = (top, left, bh, bw, bool(torch.rand(1) < p))
                after = torch.rand(1)
                torch.manual_seed(seed)
                got = random_resized_crop_params(h, w, 256, scale, ratio, p)
                assert got == want, (h, w, scale, ratio, seed)
                assert torch.equal(torch.rand(1), after), "the torch stream was consumed differently"
                fallbacks += (bh, bw) == (341, 256) and (rh, rw) == (13830, 256)
    assert fallbacks >= 12


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("c", [1, 3])
def test_oracle_chain_matches_torchvision_compose(interp, c):
    """Small inputs (Resize(40) -> RandomResizedCrop(24)) so that the numpy restatement stays fast; the goldens cover the
    full-size cases on the device."""
    pytest.importorskip("torchvision")
    from image_retrieval_wavelet_b200.transforms import random_resized_crop_params
    from image_retrieval_wavelet_b200.transforms.ragged import resized_size

    gen = _gen()
    for k, (h, w) in enumerate([(48, 64), (64, 47), (31, 17), (40, 40), (41, 39), (300, 6), (9, 13)]):
        img = gen.make_image(k, h, w, c)
        for seed in range(3):
            torch.manual_seed(seed)
            want = gen.from_pil(gen.train_transform(40, 24, interp, 0.5)(gen.to_pil(img)), c)
            torch.manual_seed(seed)
            box = random_resized_crop_params(h, w, 40)
            got = gen.chain_ref(img, *resized_size(h, w, 40), box, (24, 24), interp)
            assert np.array_equal(got, want), (h, w, seed, box)


def test_oracle_chain_matches_the_golden():
    """The golden cases that are cheap in numpy: the draw under the case's seed and the oracle chain give torchvision's
    output."""
    from image_retrieval_wavelet_b200.transforms import random_resized_crop_params
    from image_retrieval_wavelet_b200.transforms.ragged import _pair, resized_size

    gen = _gen()
    g = np.load(os.path.join(ROOT, "tests", "golden", "resize_train_golden.npz"))
    for name in ("odd_width_375x501", "coco_427x640_flip", "coco_427x640_noflip", "gray_333x517", "rgbx_300x451",
                 "tiny_bicubic_31x17", "identity_256x256", "pair_size_crop_375x500"):
        h, w, c, size, crop, interp, seed, p = gen.CASES[name]
        torch.manual_seed(seed)
        box = random_resized_crop_params(h, w, size, p=p)
        got = gen.chain_ref(gen.make_image(seed, h, w, c), *resized_size(h, w, size), box, _pair(crop, "crop"), interp)
        assert np.array_equal(got, g[name]), name


class _Decoded(torch.utils.data.Dataset):
    """Small decoded images of many shapes; with ``transform`` the per-sample torchvision pipeline instead."""

    def __init__(self, transform=None):
        self.transform = transform
        self.shapes = [(20 + 7 * i % 23, 33 - 5 * i % 17) for i in range(14)]

    def __len__(self):
        return len(self.shapes)

    def __getitem__(self, i):
        h, w = self.shapes[i]
        arr = _gen().make_image(100 + i, h, w, 3)
        if self.transform is None:
            return {"image": arr, "label": i}
        return {"image": np.asarray(self.transform(_gen().to_pil(arr))).transpose(2, 0, 1).copy(), "label": i}


def test_seeded_dataloader_reproduces_torchvision_loader():
    """Two workers each: the training collate draws in the worker, in sample order, so the boxes and flips it hands over
    (applied with the oracle chain) give the batches of an identically seeded loader that runs torchvision per sample."""
    pytest.importorskip("torchvision")
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged_train
    from image_retrieval_wavelet_b200.transforms.ragged import resized_size

    gen = _gen()
    size, crop = 24, 16

    def loader(ds, collate):
        return torch.utils.data.DataLoader(ds, batch_size=3, shuffle=True, num_workers=2, collate_fn=collate,
                                           generator=torch.Generator().manual_seed(1234))

    ours = loader(_Decoded(), functools.partial(collate_ragged_train, size=size))
    theirs = loader(_Decoded(gen.train_transform(size, crop, "bilinear", 0.5)), None)
    flips = set()
    n = 0
    for a, b in zip(ours, theirs):
        imgs = a["image"]
        assert isinstance(imgs, RaggedImages) and torch.equal(a["label"], b["label"])
        assert imgs.crop_params.dtype == torch.int64 and tuple(imgs.crop_params.shape) == (len(imgs), 7)
        for i in range(len(imgs)):
            arr = imgs.image(i).numpy()
            box = imgs.crop_params[i].tolist()
            assert box[5:] == list(resized_size(arr.shape[0], arr.shape[1], size))
            box = box[:5]
            flips.add(box[4])
            got = gen.chain_ref(arr, *resized_size(arr.shape[0], arr.shape[1], size), box, (crop, crop), "bilinear")
            assert np.array_equal(got, b["image"][i].numpy()), (n, i, box)
        n += 1
    assert n == 5 and flips == {0, 1}


def test_crop_params_travel_with_the_batch():
    from image_retrieval_wavelet_b200.transforms import collate_ragged_train

    torch.manual_seed(0)
    batch = collate_ragged_train([np.zeros((30, 40, 3), np.uint8), np.zeros((50, 20, 3), np.uint8)], size=16, p=1.0)
    assert batch.crop_params[:, 4].tolist() == [1, 1] and batch.crop_params[:, 5:].tolist() == [[16, 21], [40, 16]]
    assert batch._with(batch.data.clone()).crop_params is batch.crop_params       # what pin_memory() and cuda() return


def test_random_crop_entry_points_reject_bad_arguments_without_a_device():
    """Rejected on the host before any CUDA call, so these are safe here."""
    from image_retrieval_wavelet_b200 import _cabi

    lib = _cabi.load()
    alive = []

    def geom(*rows):
        g = np.array(rows, dtype=np.int32).reshape(-1, 9)
        alive.append(g)
        return ctypes.c_void_p(g.ctypes.data)

    offs = np.zeros(4, dtype=np.int64)
    op = ctypes.c_void_p(offs.ctypes.data)
    fake = ctypes.c_void_p(1 << 20)                                     # never dereferenced: rejected first
    bil = _cabi.RESIZE_BILINEAR

    def call(g, n=1, c=3, ho=224, wo=224, filt=bil, offsets=op, inp=fake, ws_bytes=1 << 30):
        return lib.b200_resize_random_crop_u8(inp, offsets, g, n, c, ho, wo, filt, fake, fake, ws_bytes, None)

    gp = geom(480, 640, 256, 341, 10, 20, 200, 300, 1)
    assert lib.b200_resize_random_crop_workspace_bytes(1, gp, 3, 224, 224, bil) > 200 * 300 * 3
    assert call(gp, n=0) == _cabi.OK
    assert call(gp, c=0) == _cabi.ERR_INVALID_ARG and call(gp, c=5) == _cabi.ERR_INVALID_ARG
    assert call(gp, filt=7) == _cabi.ERR_INVALID_ARG and call(gp, ho=0) == _cabi.ERR_INVALID_ARG
    assert call(gp, n=-1) == _cabi.ERR_INVALID_ARG and call(None) == _cabi.ERR_INVALID_ARG
    assert call(gp, inp=None) == _cabi.ERR_INVALID_ARG and call(gp, offsets=None) == _cabi.ERR_INVALID_ARG
    assert call(geom(480, 640, 256, 341, 57, 20, 200, 300, 1)) == _cabi.ERR_INVALID_ARG      # box rows past the resized image
    assert call(geom(480, 640, 256, 341, 10, 42, 200, 300, 0)) == _cabi.ERR_INVALID_ARG      # box columns past it
    assert call(geom(480, 640, 256, 341, -1, 20, 200, 300, 0)) == _cabi.ERR_INVALID_ARG
    assert call(geom(480, 640, 256, 341, 10, 20, 0, 300, 0)) == _cabi.ERR_INVALID_ARG
    assert call(geom(480, 640, 256, 341, 10, 20, 200, 300, 2)) == _cabi.ERR_INVALID_ARG      # flip is 0 or 1
    assert call(geom(8000, 640, 256, 341, 10, 20, 200, 300, 0)) == _cabi.ERR_UNSUPPORTED     # first resize: 65 taps
    assert call(geom(7000, 300, 7000, 300, 0, 0, 7000, 300, 0)) == _cabi.ERR_UNSUPPORTED     # second: 7000 -> 224, 65 taps
    assert call(geom(3600, 300, 3600, 300, 0, 0, 3600, 300, 0), filt=_cabi.RESIZE_BICUBIC) == _cabi.ERR_UNSUPPORTED
    assert call(gp, inp=ctypes.c_void_p((1 << 20) + 2)) == _cabi.ERR_ALIGNMENT
    bad = np.array([6], dtype=np.int64)
    assert call(gp, offsets=ctypes.c_void_p(bad.ctypes.data)) == _cabi.ERR_ALIGNMENT
    assert call(gp, ws_bytes=16) == _cabi.ERR_WORKSPACE
    assert lib.b200_resize_random_crop_workspace_bytes(0, gp, 3, 224, 224, bil) == 0
    assert lib.b200_resize_random_crop_workspace_bytes(1, geom(7000, 300, 7000, 300, 0, 0, 7000, 300, 0), 3, 224, 224, bil) == 0


def test_resize_random_crop_flip_python_checks_need_no_kernel(monkeypatch):
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms import collate_ragged, collate_ragged_train, resize_random_crop_flip

    monkeypatch.setattr(_cabi, "require_cuda", lambda: None)
    with pytest.raises(TypeError):
        resize_random_crop_flip(collate_ragged_train([np.zeros((30, 40, 3), np.uint8)]))      # host data: .cuda() first
    with pytest.raises(TypeError):
        resize_random_crop_flip(collate_ragged([np.zeros((30, 40, 3), np.uint8)]).data)
    with pytest.raises(TypeError, match="collate_ragged_train"):
        resize_random_crop_flip(np.zeros((1, 3, 8, 8), np.uint8))
