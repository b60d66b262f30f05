"""HP-SWT parity on a B200: the CUDA path (through the C-ABI) against the CPU oracle on the same seeded inputs.

Tolerance (BASELINE.json north_star / SURVEY.md §8c): per band, max |diff| <= 1e-5 * max |reference band| in float32."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import c_oracle, filters, swt_ref

pytestmark = pytest.mark.gpu


def _check(out, ref, what=""):
    out = out.cpu().numpy() if isinstance(out, torch.Tensor) else out
    assert out.shape == ref.shape and out.dtype == np.float32
    for band in range(4):
        tol = 1e-5 * max(np.abs(ref[..., band, :, :]).max(), 1e-30)
        err = np.abs(out[..., band, :, :] - ref[..., band, :, :]).max()
        assert err <= tol, f"{what} band {band}: {err} > {tol}"


CASES = [
    ((64, 3, 224, 224), "haar", 1, np.uint8),       # BASELINE config C1
    ((64, 3, 224, 224), "haar", 1, np.float32),
    ((4, 3, 518, 518), "haar", 1, np.uint8),        # C4, level 1 (W % 4 != 0)
    ((4, 3, 518, 518), "db2", 1, np.uint8),
    ((4, 3, 518, 518), "db4", 1, np.uint8),
    ((4, 3, 518, 518), "sym4", 1, np.float32),
    ((4, 3, 520, 520), "haar", 2, np.uint8),        # C4, levels 2-3 at fix_size's 520
    ((4, 3, 520, 520), "db2", 2, np.uint8),
    ((4, 3, 520, 520), "db4", 2, np.uint8),
    ((4, 3, 520, 520), "sym4", 2, np.uint8),
    ((4, 3, 520, 520), "haar", 3, np.uint8),
    ((4, 3, 520, 520), "db2", 3, np.uint8),
    ((4, 3, 520, 520), "db4", 3, np.uint8),
    ((4, 3, 520, 520), "sym4", 3, np.float32),
    ((2, 3, 224, 224), "bior4.4", 1, np.uint8),     # studies/mflickr_wavelet_type_ablation.yaml
    ((2, 3, 224, 224), "bior4.4", 3, np.uint8),
    ((1, 1, 32, 32), "db7", 2, np.float32),         # generic program (F = 14)
    ((1, 2, 64, 64), "haar", 4, np.float32),        # generic program (level 4)
    ((1, 1, 8, 8), "db4", 3, np.float32),           # image smaller than the dilated filter
    ((1, 1, 2, 2), "haar", 1, np.uint8),
    ((3, 1, 136, 200), "coif1", 3, np.uint8),
    ((1, 3, 30, 34), "db3", 1, np.float32),
    ((2, 3, 256, 256), "db2", 2, np.float32),       # float32, 16-byte aligned rows: interior tiles staged by cp.async.bulk
    ((2, 2, 520, 520), "haar", 1, np.float32),
    ((1, 1, 24, 36), "sym4", 1, np.float32),        # sliding last pass: float32, smaller than one tile
    ((1, 1, 256, 256), "db2", 3, np.float32),       # hybrid, bulk-staged float32
    ((1, 1, 8, 8), "db2", 3, np.uint8),             # hybrid: smaller than one tile
]


@pytest.mark.parametrize("shape,name,level,dtype", CASES)
def test_swt2_matches_oracle(shape, name, level, dtype):
    from image_retrieval_wavelet_b200.transforms import swt2

    rng = np.random.default_rng(sum(shape) + level)
    x = rng.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else rng.random(shape, dtype=np.float32)
    lo, hi = filters.filter_bank(name)
    ref = c_oracle.swt2(x, lo, hi, level)
    from image_retrieval_wavelet_b200.transforms import wavelets
    bank = name if name in wavelets.wavelist() else (list(lo), list(hi))      # e.g. db7: explicit (dec_lo, dec_hi)
    out = swt2(torch.from_numpy(x).cuda(), bank, level)
    _check(out, ref, f"{shape} {name} L{level}")


def _swt_rolled(x, name, level, dy, dx):
    """x rolled by (dy, dx) through its planned pass form: parity with the rolled oracle and, for a non-zero roll, the
    rolled sub-bands of x bit for bit (the periodic SWT commutes with circular shifts, and every pixel is computed in the
    same order wherever tiles, staging units and register windows cut the image)."""
    from image_retrieval_wavelet_b200.transforms import swt2

    lo, hi = filters.filter_bank(name)
    xt = torch.from_numpy(x).cuda()
    out = swt2(torch.roll(xt, (dy, dx), dims=(2, 3)), name, level)
    _check(out, np.roll(c_oracle.swt2(x, lo, hi, level), (dy, dx), axis=(3, 4)), f"{x.shape} {name} L{level} rolled by {(dy, dx)}")
    if dy or dx:
        assert torch.equal(out, torch.roll(swt2(xt, name, level), (dy, dx), dims=(3, 4)))
    return out


@pytest.mark.parametrize("shift", [0, 1, 2])
@pytest.mark.parametrize("shape,name,level,dtype", [((2, 3, 70, 518), "haar", 1, np.uint8), ((1, 2, 130, 518), "db4", 1, np.uint8),
                                                     ((2, 1, 136, 200), "db2", 2, np.uint8), ((1, 2, 256, 256), "db2", 2, np.float32),
                                                     ((1, 1, 520, 520), "sym4", 3, np.uint8), ((1, 3, 104, 96), "haar", 3, np.float32),
                                                     ((1, 1, 48, 40), "bior4.4", 2, np.uint8), ((1, 1, 8, 8), "db4", 3, np.float32)])
def test_swt_pass_forms_agree_on_device(shift, shape, name, level, dtype):
    """Every pass form the planner picks (two-pass, sliding last pass, hybrid) on the image rolled by (shift, shift)."""
    rng = np.random.default_rng(sum(shape) + level)
    x = rng.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else rng.random(shape, dtype=np.float32)
    _swt_rolled(x, name, level, shift, shift)


@pytest.mark.parametrize("dx", [0, 1])
@pytest.mark.parametrize("shape,name,level,dtype", [((2, 3, 70, 518), "haar", 1, np.uint8), ((1, 2, 130, 518), "db4", 1, np.uint8),
                                                     ((2, 3, 518, 518), "sym4", 1, np.uint8), ((2, 1, 136, 200), "db2", 2, np.uint8),
                                                     ((1, 1, 520, 520), "sym4", 3, np.uint8), ((1, 1, 48, 40), "bior4.4", 2, np.uint8),
                                                     ((1, 1, 8, 8), "db4", 3, np.float32), ((1, 2, 224, 224), "db4", 1, np.float32)])
def test_swt_sliding_last_pass_agrees_on_device(dx, shape, name, level, dtype):
    """The last vertical pass (sliding for 8-tap filters at level 1, blocked otherwise) on the image rolled by (0, dx)."""
    rng = np.random.default_rng(sum(shape) + level)
    x = rng.integers(0, 256, shape).astype(np.uint8) if dtype == np.uint8 else rng.random(shape, dtype=np.float32)
    _swt_rolled(x, name, level, 0, dx)


@pytest.mark.parametrize("dx", [0, 1])
@pytest.mark.parametrize("shape,name,level", [((3, 2, 70, 518), "haar", 1), ((2, 3, 130, 518), "db4", 1), ((2, 1, 66, 94), "bior4.4", 1),
                                              ((2, 1, 40, 36), "db2", 2), ((1, 1, 24, 10), "haar", 1), ((2, 3, 224, 224), "db2", 1),
                                              ((2, 3, 130, 518), "db2", 1), ((2, 1, 40, 10), "db2", 1), ((2, 3, 224, 222), "haar", 1)])
def test_uint8_staging_units_agree(dx, shape, name, level):
    """uint8 staging on rows that start on every byte alignment (the image rolled by dx), with wrap in x and y.  Where
    both staging forms apply (level 1, F <= 4) they give identical bits: x (W % 4 = 2) is staged in 8-pixel units of three
    aligned words, [x, x] side by side (W % 4 = 0) in 4-pixel units, and the periodic transform of [x, x] is
    [swt(x), swt(x)]."""
    from image_retrieval_wavelet_b200.transforms import swt2

    x = np.random.default_rng(len(name) + shape[3]).integers(0, 256, shape).astype(np.uint8)
    out = _swt_rolled(x, name, level, 0, dx)
    if level == 1 and len(filters.filter_bank(name)[0]) <= 4 and shape[3] % 4 == 2:
        xr = torch.roll(torch.from_numpy(x).cuda(), dx, dims=3)
        assert torch.equal(swt2(torch.cat([xr, xr], dim=-1), name, 1), torch.cat([out, out], dim=-1))


def test_full_size_c4_properties():
    """256 x 3 x 518 x 518 (BASELINE config C4): size-independent properties at the full batch."""
    from image_retrieval_wavelet_b200.transforms import swt2

    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randint(0, 256, (256, 3, 518, 518), dtype=torch.uint8, device="cuda", generator=g)
    out = swt2(x, "haar", 1)
    assert out.shape == (256, 3, 4, 518, 518) and torch.isfinite(out).all()
    xf = x.float() / 255.0
    energy = (out.double() ** 2).sum(dim=(2, 3, 4)) / (xf.double() ** 2).sum(dim=(2, 3))
    assert (energy - 4.0).abs().max() < 1e-4                              # SWT-5
    assert out[:, :, 1:].sum(dim=(3, 4)).abs().max() < 0.5                # SWT-4: detail bands sum to ~0 (fp32 sums of 268k terms)
    assert out[:, :, 0].min() >= 0 and out[:, :, 0].max() <= 2.0 + 1e-5
    # a slice against the oracle
    lo, hi = filters.filter_bank("haar")
    ref = c_oracle.swt2(x[17:19].cpu().numpy(), lo, hi, 1)
    _check(out[17:19], ref, "slice of the full batch")
    # circular shift equivariance on the device (SWT-6)
    shifted = swt2(torch.roll(x[:8], shifts=(7, -5), dims=(2, 3)), "haar", 1)
    assert torch.equal(shifted, torch.roll(out[:8], shifts=(7, -5), dims=(3, 4)))


def test_constant_and_linearity():
    from image_retrieval_wavelet_b200.transforms import swt2

    c = torch.full((2, 3, 64, 64), 0.37, device="cuda")
    for name, level in (("haar", 1), ("db4", 2), ("sym4", 3)):
        out = swt2(c, name, level)
        assert (out[:, :, 0] - 0.37 * 2 ** level).abs().max() < 1e-5 and out[:, :, 1:].abs().max() < 1e-5
    a, b = torch.rand(1, 3, 64, 64, device="cuda"), torch.rand(1, 3, 64, 64, device="cuda")
    assert (swt2(a + b, "db2", 2) - swt2(a, "db2", 2) - swt2(b, "db2", 2)).abs().max() < 1e-5


def test_swt_transform_call_on_pil_image_matches_reference_contract():
    """SWTTransform.__call__: PIL RGB in, CPU float32 [3, 4, H', W'] out (custom_transforms.py:145-166)."""
    from PIL import Image

    from image_retrieval_wavelet_b200.transforms import RawStackTransform, SWTTransform

    rng = np.random.default_rng(0)
    arr = rng.integers(0, 256, (224, 224, 3), dtype=np.uint8)
    img = Image.fromarray(arr)
    for name, level in (("haar", 1), ("db4", 2), ("bior4.4", 1)):
        out = SWTTransform(level=level, wavelet=name)(img)
        assert isinstance(out, torch.Tensor) and out.device.type == "cpu" and out.dtype == torch.float32
        assert tuple(out.shape) == (3, 4, 224, 224)
        _check(out.numpy(), swt_ref.swt_transform_ref(arr, name, level), f"PIL {name} L{level}")
    # fix_size path: 30 x 26 -> 32 x 32 at level 3 (PIL bicubic on the host, like the reference)
    small = Image.fromarray(rng.integers(0, 256, (26, 30, 3), dtype=np.uint8))
    t = SWTTransform(level=3, wavelet="haar")
    out = t(small)
    assert tuple(out.shape) == (3, 4, 32, 32)
    _check(out.numpy(), swt_ref.swt_transform_ref(np.array(t.fix_size(small)), "haar", 3), "fix_size")
    raw = RawStackTransform(level=1)(img)
    assert tuple(raw.shape) == (3, 4, 224, 224)
    assert np.array_equal(raw.numpy(), swt_ref.raw_stack_ref(arr))
    # the slicing the models do: x[:, :, i] on a batch (verify_swt_transform.py:88-91)
    assert tuple(out.unsqueeze(0)[:, :, 0].shape) == (1, 3, 32, 32)


def test_errors_are_python_exceptions():
    from image_retrieval_wavelet_b200.transforms import swt2

    with pytest.raises(ValueError):
        swt2(torch.zeros(1, 1, 6, 8, device="cuda"), "haar", 2)           # pywt.swt2 raises ValueError too
    with pytest.raises(ValueError):
        swt2(torch.zeros(1, 1, 8, 8, device="cuda"), "nope", 1)
    with pytest.raises(TypeError):
        swt2(torch.zeros(1, 1, 8, 8), "haar", 1)                          # CPU tensor: no fallback
    with pytest.raises(TypeError):
        swt2(torch.zeros(1, 1, 8, 8, device="cuda", dtype=torch.float16), "haar", 1)
    with pytest.raises(NotImplementedError):
        swt2(torch.zeros(1, 1, 64, 64, device="cuda"), "haar", 5)
    assert swt2(torch.zeros(0, 3, 8, 8, device="cuda"), "haar", 1).shape == (0, 3, 4, 8, 8)


def test_host_buffer_entry_point_directly():
    """b200_swt2_fwd_host with plain numpy buffers (what a non-torch caller binds)."""
    from image_retrieval_wavelet_b200 import _cabi

    rng = np.random.default_rng(3)
    x = rng.integers(0, 256, (2, 3, 32, 40), dtype=np.uint8)
    lo, hi = filters.filter_bank("db2")
    out = np.zeros((2, 3, 4, 32, 40), np.float32)
    lo32, hi32 = lo.astype(np.float32), hi.astype(np.float32)
    rc = _cabi.load().b200_swt2_fwd_host(x.ctypes.data, 1, 0, out.ctypes.data, 2, 3, 32, 40, lo32.ctypes.data, hi32.ctypes.data, 4, 2)
    assert rc == 0
    _check(out, c_oracle.swt2(x, lo, hi, 2), "host entry")


def test_u8_conversion_is_bit_identical_to_division_on_device():
    """RawStackTransform on all 256 byte values: the device's FMA form of x / 255 equals numpy's float32 division."""
    import ctypes

    from image_retrieval_wavelet_b200 import _cabi

    x = torch.arange(256, dtype=torch.uint8).reshape(1, 1, 16, 16).cuda()
    out = torch.empty((1, 1, 2, 16, 16), dtype=torch.float32, device="cuda")
    rc = _cabi.load().b200_raw_stack(_cabi.ptr(x), 1, _cabi.ptr(out), 1, 1, 16, 16, 2, _cabi.stream_ptr())
    _cabi.check(rc, "b200_raw_stack")
    want = (np.arange(256, dtype=np.float32) / np.float32(255.0)).reshape(16, 16)
    got = out.cpu().numpy()
    assert np.array_equal(got[0, 0, 0].view(np.uint32), want.view(np.uint32))
    assert np.array_equal(got[0, 0, 1].view(np.uint32), want.view(np.uint32))
