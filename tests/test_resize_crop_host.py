"""Host side of ``resize_center_crop`` (no device): torchvision's size and crop rules, the premise that a crop of a resize is the
resize evaluated inside the crop window, the ragged packing of ``collate_ragged`` and the C-ABI's argument checks."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import resize_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _golden_module():
    spec = importlib.util.spec_from_file_location("make_golden_resize_crop",
                                                  os.path.join(ROOT, "tests", "golden", "make_golden_resize_crop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


SIZES = [(h, w) for h in (1, 2, 10, 12, 223, 224, 255, 256, 257, 333, 375, 427, 480, 500, 640, 1000, 1800, 3000)
         for w in (1, 7, 10, 224, 256, 341, 359, 375, 480, 499, 500, 640, 674, 1000, 2400, 4000)]


def test_resized_size_matches_torchvision():
    F = pytest.importorskip("torchvision.transforms.functional")
    from image_retrieval_wavelet_b200.transforms.ragged import resized_size

    for h, w in SIZES:
        for size in (256, 224, 32, (256, 300), [100, 80]):
            want = F._compute_resized_output_size((h, w), [size] if isinstance(size, int) else list(size))
            assert list(resized_size(h, w, size)) == list(want), (h, w, size)
    assert resized_size(480, 640, 256) == (256, 341) and resized_size(224, 1000, 256) == (256, 1142)


def test_center_crop_origin_matches_torchvision():
    F = pytest.importorskip("torchvision.transforms.functional")
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin

    for rh, rw in ((256, 341), (256, 359), (256, 256), (257, 257), (307, 256), (256, 1142), (225, 224), (224, 224)):
        for ch, cw in ((224, 224), (224, 160), (1, 1), (223, 7)):
            index = torch.arange(rh * rw, dtype=torch.int64).view(1, rh, rw)
            corner = int(F.center_crop(index, [ch, cw])[0, 0, 0])
            assert center_crop_origin(rh, rw, ch, cw) == divmod(corner, rw), (rh, rw, ch, cw)
    assert center_crop_origin(256, 341, 224, 224) == (16, 58)          # 58.5 -> 58
    assert center_crop_origin(256, 359, 224, 224) == (16, 68)          # 67.5 -> 68


def _windowed(img, rh, rw, top, left, ch, cw, resample):
    """The crop computed from the table rows of the crop window alone: horizontal pass over the source rows the window's
    vertical taps need, then the vertical pass — what b200_resize_crop_u8 does per tile."""
    h, w = img.shape
    if rw != w:
        xm, xc, xk = (a[left:left + cw] for a in resize_ref.coeffs_ref(w, rw, resample))
    else:
        xm, xc, xk = np.arange(left, left + cw), np.ones(cw, np.int64), np.full((cw, 1), 1 << resize_ref.PRECISION_BITS)
    if rh != h:
        ym, yc, yk = (a[top:top + ch] for a in resize_ref.coeffs_ref(h, rh, resample))
    else:
        ym, yc, yk = np.arange(top, top + ch), np.ones(ch, np.int64), np.full((ch, 1), 1 << resize_ref.PRECISION_BITS)
    y0, y1 = int(ym[0]), int(ym[-1] + yc[-1])
    x0, x1 = int(xm[0]), int(xm[-1] + xc[-1])
    src = img[y0:y1, x0:x1].astype(np.int64)                          # the source inside the crop's support
    half = 1 << (resize_ref.PRECISION_BITS - 1)
    tmp = np.empty((y1 - y0, cw), np.int64)
    for j in range(cw):
        n, s = int(xc[j]), int(xm[j]) - x0
        tmp[:, j] = np.clip((half + (src[:, s:s + n] * xk[j, :n]).sum(1)) >> resize_ref.PRECISION_BITS, 0, 255)
    out = np.empty((ch, cw), np.uint8)
    for i in range(ch):
        n, s = int(yc[i]), int(ym[i]) - y0
        out[i] = np.clip((half + (tmp[s:s + n] * yk[i, :n, None]).sum(0)) >> resize_ref.PRECISION_BITS, 0, 255)
    return out


@pytest.mark.parametrize("h,w,rh,rw,ch,cw,resample", [(480, 640, 256, 341, 224, 224, "bilinear"), (97, 131, 40, 77, 17, 30, "bicubic"),
                                                      (256, 341, 256, 341, 224, 224, "bilinear"), (12, 10, 307, 256, 224, 224, "bilinear"),
                                                      (300, 90, 256, 77, 100, 70, "bicubic"), (50, 400, 50, 128, 50, 64, "bilinear")])
def test_crop_of_resize_is_resize_inside_the_window(h, w, rh, rw, ch, cw, resample):
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin

    img = np.random.default_rng(h * w).integers(0, 256, (h, w), dtype=np.uint8)
    top, left = center_crop_origin(rh, rw, ch, cw)
    full = resize_ref.resize_ref(img, (rh, rw), resample)
    assert np.array_equal(_windowed(img, rh, rw, top, left, ch, cw, resample), full[top:top + ch, left:left + cw])


def test_oracle_slice_matches_the_golden():
    """resize_ref (Pillow restated) followed by the crop slice reproduces torchvision's outputs for the golden's cases that
    are cheap in numpy."""
    gen = _golden_module()
    from image_retrieval_wavelet_b200.transforms.ragged import center_crop_origin, resized_size

    g = np.load(os.path.join(ROOT, "tests", "golden", "resize_crop_golden.npz"))
    for name in ("landscape_480x640", "noop_resize_256x341", "half_even_480x674", "upscale_12x10", "bicubic_480x640",
                 "pair_size_375x500", "nonsquare_crop_480x640", "gray_333x517"):
        h, w, c, size, crop, interp, seed = gen.CASES[name]
        planes = gen.make_image(seed, h, w, c).transpose(2, 0, 1)
        ch, cw = (crop, crop) if isinstance(crop, int) else crop
        rh, rw = resized_size(h, w, size)
        top, left = center_crop_origin(rh, rw, ch, cw)
        want = resize_ref.resize_ref(planes, (rh, rw), interp)[:, top:top + ch, left:left + cw]
        assert np.array_equal(g[name], want), name


def test_golden_generator_reproduces_a_case():
    pytest.importorskip("torchvision")
    from PIL import Image
    from torchvision.transforms import CenterCrop, Compose, Resize

    gen = _golden_module()
    g = np.load(os.path.join(ROOT, "tests", "golden", "resize_crop_golden.npz"))
    h, w, c, size, crop, _, seed = gen.CASES["landscape_375x500"]
    got = np.asarray(Compose([Resize(size), CenterCrop(crop)])(Image.fromarray(gen.make_image(seed, h, w, c))))
    assert np.array_equal(got.transpose(2, 0, 1), g["landscape_375x500"])


def test_collate_ragged_layout():
    from PIL import Image

    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged

    rng = np.random.default_rng(0)
    arrs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ((5, 7), (1, 1), (480, 640), (3, 5))]
    batch = collate_ragged([Image.fromarray(arrs[0]), arrs[1], Image.fromarray(arrs[2]), arrs[3]])
    assert isinstance(batch, RaggedImages) and len(batch) == 4 and batch.channels == 3
    assert batch.data.dtype == torch.uint8 and batch.data.dim() == 1 and batch.data.numel() % 16 == 0
    assert batch.sizes.tolist() == [[5, 7], [1, 1], [480, 640], [3, 5]]
    offs = batch.offsets.tolist()
    assert offs[0] == 0 and all(o % 16 == 0 for o in offs)
    for i, a in enumerate(arrs):
        assert offs[i] + a.size <= (offs[i + 1] if i + 1 < len(offs) else batch.data.numel())
        assert np.array_equal(batch.image(i).numpy(), a)
    gray = collate_ragged([Image.fromarray(arrs[0][:, :, 0]), arrs[3][:, :, :1]])
    assert gray.channels == 1 and np.array_equal(gray.image(0).numpy()[:, :, 0], arrs[0][:, :, 0])
    with pytest.raises(ValueError):
        collate_ragged([arrs[0], arrs[0][:, :, 0]])                      # 3 and 1 channels in one batch
    with pytest.raises(TypeError):
        collate_ragged([arrs[0].astype(np.float32)])


def test_collate_ragged_dict_samples():
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged

    rng = np.random.default_rng(1)
    samples = [{"image": rng.integers(0, 256, (4 + i, 9 - i, 3), dtype=np.uint8), "label": torch.tensor([i, 1 - i]),
                "path": f"img{i}.jpg"} for i in range(3)]
    batch = collate_ragged(samples)
    assert set(batch) == {"image", "label", "path"}
    assert isinstance(batch["image"], RaggedImages) and batch["image"].sizes.tolist() == [[4, 9], [5, 8], [6, 7]]
    assert torch.equal(batch["label"], torch.tensor([[0, 1], [1, 0], [2, -1]])) and batch["path"] == ["img0.jpg", "img1.jpg", "img2.jpg"]
    other = collate_ragged([{"pixels": s["image"], "label": 0} for s in samples], key="pixels")
    assert isinstance(other["pixels"], RaggedImages) and other["label"].tolist() == [0, 0, 0]
    empty = collate_ragged([])
    assert len(empty) == 0 and tuple(empty.sizes.shape) == (0, 2)


def test_ragged_batch_goes_through_a_dataloader():
    from image_retrieval_wavelet_b200.transforms import RaggedImages, collate_ragged

    class Images(torch.utils.data.Dataset):
        def __len__(self):
            return 5

        def __getitem__(self, i):
            return {"image": np.full((10 + i, 20 - i, 3), i, dtype=np.uint8), "label": i}

    loader = torch.utils.data.DataLoader(Images(), batch_size=3, num_workers=2, collate_fn=collate_ragged)
    batches = list(loader)
    assert [len(b["image"]) for b in batches] == [3, 2] and isinstance(batches[1]["image"], RaggedImages)
    assert batches[1]["label"].tolist() == [3, 4] and int(batches[1]["image"].image(1)[0, 0, 0]) == 4


def test_crop_entry_points_reject_bad_arguments_without_a_device():
    """Rejected on the host before any CUDA call, so these are safe here."""
    from image_retrieval_wavelet_b200 import _cabi

    lib = _cabi.load()

    alive = []

    def geom(*rows):
        g = np.array(rows, dtype=np.int32).reshape(-1, 6)
        alive.append(g)
        return g, ctypes.c_void_p(g.ctypes.data)

    offs = np.zeros(4, dtype=np.int64)
    op = ctypes.c_void_p(offs.ctypes.data)
    fake = ctypes.c_void_p(1 << 20)                                     # never dereferenced: rejected first
    bil = _cabi.RESIZE_BILINEAR

    def call(g, n=1, c=3, hc=224, wc=224, filt=bil, offsets=op, inp=fake, ws_bytes=1 << 30):
        return lib.b200_resize_crop_u8(inp, offsets, g, n, c, hc, wc, filt, fake, fake, ws_bytes, None)

    g, gp = geom(480, 640, 256, 341, 16, 58)
    assert lib.b200_resize_crop_workspace_bytes(1, gp, 3, 224, 224, bil) > 0
    assert call(gp, n=0) == _cabi.OK                                      # empty batch: nothing to do
    assert call(gp, c=0) == _cabi.ERR_INVALID_ARG and call(gp, c=5) == _cabi.ERR_INVALID_ARG
    assert call(gp, filt=7) == _cabi.ERR_INVALID_ARG and call(gp, hc=0) == _cabi.ERR_INVALID_ARG
    assert call(gp, n=-1) == _cabi.ERR_INVALID_ARG and call(None) == _cabi.ERR_INVALID_ARG
    assert call(gp, inp=None) == _cabi.ERR_INVALID_ARG and call(gp, offsets=None) == _cabi.ERR_INVALID_ARG
    assert call(geom(480, 640, 256, 341, 33, 58)[1]) == _cabi.ERR_INVALID_ARG        # crop rows past the resized image
    assert call(geom(480, 640, 256, 341, 16, 118)[1]) == _cabi.ERR_INVALID_ARG       # crop columns past it
    assert call(geom(480, 640, 256, 341, -1, 58)[1]) == _cabi.ERR_INVALID_ARG
    assert call(geom(0, 640, 256, 341, 16, 58)[1]) == _cabi.ERR_INVALID_ARG
    assert call(geom(8000, 640, 256, 341, 16, 58)[1]) == _cabi.ERR_UNSUPPORTED        # 31.25x bilinear: 65 taps
    assert call(geom(4000, 640, 256, 341, 16, 58)[1], filt=_cabi.RESIZE_BICUBIC) == _cabi.ERR_UNSUPPORTED   # 15.6x bicubic
    assert call(gp, inp=ctypes.c_void_p((1 << 20) + 2)) == _cabi.ERR_ALIGNMENT
    bad = np.array([6], dtype=np.int64)
    assert call(gp, offsets=ctypes.c_void_p(bad.ctypes.data)) == _cabi.ERR_ALIGNMENT
    assert call(gp, ws_bytes=16) == _cabi.ERR_WORKSPACE
    assert lib.b200_resize_crop_workspace_bytes(0, gp, 3, 224, 224, bil) == 0
    assert lib.b200_resize_crop_workspace_bytes(1, geom(8000, 640, 256, 341, 16, 58)[1], 3, 224, 224, bil) == 0
    # images of one size share their tables, and so do the axes of a landscape and a portrait image of the same sizes:
    # they add a descriptor only (the descriptor block is rounded up to 256 bytes)
    two = geom(480, 640, 256, 341, 16, 58, 640, 480, 341, 256, 58, 16)[1]
    three = geom(480, 640, 256, 341, 16, 58, 640, 480, 341, 256, 58, 16, 375, 500, 256, 341, 16, 58)[1]
    one = lib.b200_resize_crop_workspace_bytes(1, gp, 3, 224, 224, bil)
    assert lib.b200_resize_crop_workspace_bytes(2, two, 3, 224, 224, bil) == one
    assert lib.b200_resize_crop_workspace_bytes(3, three, 3, 224, 224, bil) > one


def test_resize_center_crop_python_checks_need_no_kernel(monkeypatch):
    from image_retrieval_wavelet_b200 import _cabi
    from image_retrieval_wavelet_b200.transforms import collate_ragged, resize_center_crop

    monkeypatch.setattr(_cabi, "require_cuda", lambda: None)
    batch = collate_ragged([np.zeros((30, 40, 3), np.uint8)])
    with pytest.raises(TypeError):
        resize_center_crop(batch)                                         # host data: .cuda() first
    with pytest.raises(TypeError):
        resize_center_crop(np.zeros((1, 3, 8, 8), np.uint8))
