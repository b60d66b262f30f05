"""Resize + center crop of ragged batches on a B200 (``resize_center_crop`` / ``b200_resize_crop_u8``): bit for bit against
torchvision's ``Compose([Resize, CenterCrop])`` on PIL images (goldens, and the installed torchvision when importable) and
against the Pillow restatement ``oracle/resize_ref.py`` (full resize, then the crop slice) on random geometries."""
import ctypes
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

from oracle import resize_ref

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 4096
SMEM_BUDGET = 32 * 1024          # kRcSmemBudget in csrc/resize.cu


def _gen():
    spec = importlib.util.spec_from_file_location("make_golden_resize_crop",
                                                  os.path.join(ROOT, "tests", "golden", "make_golden_resize_crop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "resize_crop_golden.npz"))


def _case(gen, name):
    h, w, c, size, crop, interp, seed = gen.CASES[name]
    img = gen.make_image(seed, h, w, c)
    return img, size, crop, interp


def _crop(images, size, crop, interp):
    from image_retrieval_wavelet_b200.transforms import collate_ragged, resize_center_crop

    return resize_center_crop(collate_ragged(images).cuda(), size, crop, interp)


def test_matches_torchvision_goldens(golden):
    gen = _gen()
    for name in gen.CASES:
        img, size, crop, interp = _case(gen, name)
        got = _crop([img], size, crop, interp)
        assert got.dtype == torch.uint8 and np.array_equal(got[0].cpu().numpy(), golden[name]), name


def test_one_ragged_call_equals_per_image_calls(golden):
    """All golden cases with the eval transform's parameters in one launch: each image's output is its own call's."""
    gen = _gen()
    names = [n for n, (_, _, c, size, crop, interp, _) in gen.CASES.items() if (c, size, crop, interp) == (3, 256, 224, "bilinear")]
    assert len(names) >= 8
    imgs = [_case(gen, n)[0] for n in names]
    batch = _crop(imgs, 256, 224, "bilinear")
    assert tuple(batch.shape) == (len(names), 3, 224, 224)
    for i, name in enumerate(names):
        assert torch.equal(batch[i], _crop([imgs[i]], 256, 224, "bilinear")[0]), name
        assert np.array_equal(batch[i].cpu().numpy(), golden[name]), name


def test_matches_installed_torchvision():
    pytest.importorskip("torchvision")
    from PIL import Image
    from torchvision.transforms import CenterCrop, Compose, InterpolationMode, Resize

    rng = np.random.default_rng(7)
    for interp in ("bilinear", "bicubic"):
        t = Compose([Resize(256, interpolation=InterpolationMode(interp)), CenterCrop(224)])
        shapes = [(480, 640), (640, 480), (427, 640), (375, 500), (333, 333), (1200, 1601), (224, 999), (31, 17)]
        imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
        got = _crop([Image.fromarray(a) for a in imgs], 256, 224, interp).cpu().numpy()
        for i, a in enumerate(imgs):
            assert np.array_equal(got[i], np.asarray(t(Image.fromarray(a))).transpose(2, 0, 1)), (interp, shapes[i])


# ---- the C entry point on arbitrary geometries (any crop origin, 4-byte offsets, guard bytes around every buffer)

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


def _run_c(imgs, geoms, hc, wc, filt):
    """b200_resize_crop_u8 over HWC uint8 images packed at 4-byte-aligned offsets; out and workspace guarded."""
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
    geom = np.array([(a.shape[0], a.shape[1]) + tuple(g) for a, g in zip(imgs, geoms)], dtype=np.int32).reshape(-1, 6)
    offsets = np.array(offs, dtype=np.int64)
    lib = _cabi.load()
    filt_id = {"bilinear": _cabi.RESIZE_BILINEAR, "bicubic": _cabi.RESIZE_BICUBIC}[filt]
    gp, op = ctypes.c_void_p(geom.ctypes.data), ctypes.c_void_p(offsets.ctypes.data)
    nbytes = lib.b200_resize_crop_workspace_bytes(len(imgs), gp, c, hc, wc, filt_id)
    ws, out = Guarded(nbytes), Guarded(len(imgs) * c * hc * wc)
    _cabi.check(lib.b200_resize_crop_u8(inp.ptr, op, gp, len(imgs), c, hc, wc, filt_id, out.ptr, ws.ptr, nbytes, _cabi.stream_ptr()),
                "b200_resize_crop_u8")
    torch.cuda.synchronize()
    assert out.intact() and ws.intact() and inp.intact(), "b200_resize_crop_u8 wrote outside a buffer"
    return out.view().cpu().numpy().reshape(len(imgs), c, hc, wc)


def _ref(img, geom, hc, wc, filt):
    rh, rw, top, left = geom
    return resize_ref.resize_ref(img.transpose(2, 0, 1), (rh, rw), filt)[:, top:top + hc, left:left + wc]


def _max_scale(filt):
    # the window limit of 64 taps: 2 * ceil(support * scale) + 1 <= 64
    return 31.0 if filt == "bilinear" else 15.5


@pytest.mark.parametrize("c", [1, 3, 4])
@pytest.mark.parametrize("filt", ["bilinear", "bicubic"])
def test_random_geometries_match_the_oracle(c, filt):
    rng = np.random.default_rng(100 * c + len(filt))
    for trial in range(4):
        hc, wc = int(rng.integers(1, 80)), int(rng.integers(1, 300))
        imgs, geoms = [], []
        for k in range(4):
            kind = (trial * 4 + k) % 4          # 0, 3: reductions up to the tap limit, 1: identity axis, 2: enlargement
            rh, rw = hc + int(rng.integers(0, 40)), wc + int(rng.integers(0, 60))
            if kind == 0:
                s = rng.uniform(1.0, _max_scale(filt)) if k % 2 else _max_scale(filt) - 0.01
                h, w = max(1, int(rh * s)), max(1, int(rw * rng.uniform(1.0, 3.0)))
                h = min(h, 2400)
                rh = max(rh if h >= rh else h, math.ceil(h / _max_scale(filt)), hc)
            elif kind == 1:
                h, w = rh, int(rng.integers(1, 3 * rw)) | 1      # odd widths: rows start on every byte offset
            elif kind == 2:
                h, w = int(rng.integers(1, rh + 1)), int(rng.integers(1, rw + 1))
            else:
                h, w = int(rng.integers(1, 3 * rh)), min(int(rw * (_max_scale(filt) - 0.01)), 4000)
                rw = max(rw, math.ceil(w / _max_scale(filt)))
            top, left = int(rng.integers(0, rh - hc + 1)), int(rng.integers(0, rw - wc + 1))
            imgs.append(rng.integers(0, 256, (h, w, c), dtype=np.uint8))
            geoms.append((rh, rw, top, left))
        got = _run_c(imgs, geoms, hc, wc, filt)
        for i, (img, g) in enumerate(zip(imgs, geoms)):
            assert np.array_equal(got[i], _ref(img, g, hc, wc, filt)), (trial, i, img.shape, g, hc, wc)


def _whole_tile_bytes(h, w, rh, rw, top, left, hc, wc, filt):
    """Shared memory a 32 x 128 tile of this geometry would stage in one piece (csrc/resize.cu crop_smem_bytes)."""
    def axis(n_in, n_out, first, count, tile):
        if n_in == n_out:
            return tile, 1
        xm, xc, kk = resize_ref.coeffs_ref(n_in, n_out, filt)
        xm, xc = xm[first:first + count], xc[first:first + count]
        span = max(int(xm[min(t + tile, count) - 1] + xc[min(t + tile, count) - 1] - xm[t]) for t in range(0, count, tile))
        return span, kk.shape[1]
    cols, ksh = axis(w, rw, left, wc, 128)
    rows, ksv = axis(h, rh, top, hc, 32)
    return (128 + 32) * 8 + (ksh * 128 + 32 * ksv) * 4 + rows * ((cols + 3) // 4 * 4 + 128)


def test_every_staging_route():
    """COCO-sized images stage a whole 32 x 128 tile at once; large photos and reductions near the tap limit walk the tile in
    smaller sub-blocks.  Both, in one batch, against the oracle."""
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin, resized_size

    rng = np.random.default_rng(5)
    shapes = [(480, 640), (1800, 2400), (2900, 3100)]
    imgs, geoms, need = [], [], []
    for h, w in shapes:
        rh, rw = resized_size(h, w, 256)
        top, left = center_crop_origin(rh, rw, 224, 224)
        imgs.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        geoms.append((rh, rw, top, left))
        need.append(_whole_tile_bytes(h, w, rh, rw, top, left, 224, 224, "bilinear"))
    assert need[0] <= SMEM_BUDGET < min(need[1:])
    got = _run_c(imgs, geoms, 224, 224, "bilinear")
    for i in range(len(imgs)):
        assert np.array_equal(got[i], _ref(imgs[i], geoms[i], 224, 224, "bilinear")), shapes[i]


def test_empty_and_single_image_batches():
    from image_retrieval_wavelet_b200.transforms import collate_ragged, resize_center_crop

    empty = resize_center_crop(collate_ragged([]).cuda())
    assert tuple(empty.shape) == (0, 3, 224, 224) and empty.is_cuda
    img = np.random.default_rng(2).integers(0, 256, (300, 400, 3), dtype=np.uint8)
    one = resize_center_crop(collate_ragged([img]).cuda())
    assert tuple(one.shape) == (1, 3, 224, 224)
    assert np.array_equal(one[0].cpu().numpy(), _ref(img, (256, 341, 16, 58), 224, 224, "bilinear"))


def test_pinned_batch_and_dataloader_pinning():
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged, resize_center_crop

    rng = np.random.default_rng(3)
    samples = [{"image": rng.integers(0, 256, (240 + 7 * i, 320 - 5 * i, 3), dtype=np.uint8), "label": i} for i in range(6)]
    loader = torch.utils.data.DataLoader(samples, batch_size=3, collate_fn=collate_ragged, pin_memory=True)
    for j, batch in enumerate(loader):
        assert isinstance(batch["image"], RaggedImages) and batch["image"].data.is_pinned()
        got = resize_center_crop(batch["image"].cuda(non_blocking=True))
        want = resize_center_crop(collate_ragged([s["image"] for s in samples[3 * j:3 * j + 3]]).cuda())
        assert torch.equal(got, want) and batch["label"].tolist() == [3 * j, 3 * j + 1, 3 * j + 2]


def test_rejects_unsupported_requests():
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged, resize_center_crop

    small = collate_ragged([np.zeros((100, 120, 3), np.uint8)]).cuda()
    with pytest.raises(ValueError):
        resize_center_crop(small, size=200, crop=224)                    # crop larger than the resized image
    with pytest.raises(ValueError):
        resize_center_crop(small, size=(256, 200), crop=(224, 201))
    with pytest.raises(ValueError):
        resize_center_crop(small, interpolation="lanczos")
    with pytest.raises(ValueError):
        resize_center_crop(small, crop=0)
    with pytest.raises(NotImplementedError):                             # 8000 / 256 = 31.25x bilinear: 65 taps
        resize_center_crop(collate_ragged([np.zeros((8000, 300, 1), np.uint8)]).cuda(), size=(256, 256), crop=224)
    with pytest.raises(NotImplementedError):                             # 16x bicubic
        resize_center_crop(collate_ragged([np.zeros((4096, 300, 1), np.uint8)]).cuda(), (256, 256), 224, "bicubic")
    near = resize_center_crop(collate_ragged([np.zeros((7936, 300, 1), np.uint8)]).cuda(), size=(256, 256), crop=224)
    assert tuple(near.shape) == (1, 1, 224, 224) and int(near.max()) == 0    # 31x: the widest window that is supported
    five = RaggedImages(torch.zeros(5 * 300 * 300, dtype=torch.uint8, device="cuda"), torch.tensor([[300, 300]]), torch.tensor([0]), 5)
    with pytest.raises(ValueError):
        resize_center_crop(five)
    shifted = RaggedImages(small.data, small.sizes, torch.tensor([2]), 3)
    with pytest.raises(ValueError):
        resize_center_crop(shifted)                                      # offset not a multiple of 4
    with pytest.raises(TypeError):
        resize_center_crop(collate_ragged([np.zeros((300, 300, 3), np.uint8)]))      # host data


@pytest.mark.parametrize("wavelet,level", [("haar", 1), ("db2", 3)])
def test_swt_of_the_crop_is_the_reference_transform(golden, wavelet, level):
    """SWTTransform(level, wavelet).forward(resize_center_crop(batch))[i] is what the reference computes per image:
    SWTTransform(level, wavelet)(CenterCrop(224)(Resize(256)(pil_i))) — with the golden crops as the PIL images, and with
    torchvision itself when it is importable."""
    from PIL import Image

    from image_retrieval_wavelet_b200.transforms import SWTTransform

    gen = _gen()
    names = ["landscape_480x640", "portrait_640x480", "half_even_480x674", "upscale_12x10", "large_1800x2400"]
    imgs = [_case(gen, n)[0] for n in names]
    t = SWTTransform(level=level, wavelet=wavelet)
    batch = t.forward(_crop(imgs, 256, 224, "bilinear"))
    assert tuple(batch.shape) == (len(names), 3, 4, 224, 224)
    for i, name in enumerate(names):
        assert torch.equal(batch[i].cpu(), t(Image.fromarray(np.ascontiguousarray(golden[name].transpose(1, 2, 0))))), name
    try:
        from torchvision.transforms import CenterCrop, Compose, Resize
    except ImportError:
        return
    eval_t = Compose([Resize(256), CenterCrop(224)])
    for i, img in enumerate(imgs):
        assert torch.equal(batch[i].cpu(), t(eval_t(Image.fromarray(img)))), names[i]
