"""The stage-1 -> stage-2 hand-off without a GPU: the host tables of b200sr_resample_u8 plus an integer restatement of the
kernel's arithmetic against PIL.Image.resize byte for byte; planted defects the sweep rejects; PIL2Tensor's size rule on
hand-worked cases; the fp32 values of the uint8 -> [-1, 1] conversion; and, when a checkout of the reference is present,
the reference's own tensor2img / PIL2Tensor."""
import importlib.util
import os

import numpy as np
import pytest
import torch
from PIL import Image

import imageio_ref as R
from imageio_ref import SWEEP, image
from b200sr import colorfix, ops
from oracle import reference_import

@pytest.fixture(scope="module")
def sweep():
    return [(image(w, h, i), (w, h), (W, H), R.pil_resize(image(w, h, i), H, W)) for i, ((w, h), (W, H)) in
            enumerate(SWEEP)]


def test_tables_and_kernel_arithmetic_match_pillow(sweep):
    for u8, (w, h), (W, H), ref in sweep:
        got = R.resize(u8, H, W, ops.pillow_bicubic_tables)
        assert got.shape == ref.shape and np.array_equal(got, ref), ((w, h), (W, H))


def test_tables_shape_and_normalisation():
    for n_in, n_out in ((400, 1024), (1100, 1088), (300, 13), (1, 7), (9, 1)):
        bounds, coeffs, ksize = ops.pillow_bicubic_tables(n_in, n_out)
        assert bounds.dtype == np.int32 and coeffs.dtype == np.int32
        assert bounds.shape == (n_out, 2) and coeffs.shape == (n_out, ksize)
        assert (bounds[:, 0] >= 0).all() and (bounds[:, 1] >= 1).all() and (bounds.sum(1) <= n_in).all()
        assert (bounds[:, 1] <= ksize).all()
        # normalised weights: each row sums to 2^22 up to one rounding per tap
        assert (np.abs(coeffs.astype(np.int64).sum(1) - (1 << 22)) <= ksize).all()
        # coefficients past a row's tap count are zero
        assert all((coeffs[o, bounds[o, 1]:] == 0).all() for o in range(n_out))
    with pytest.raises(ValueError):
        ops.pillow_bicubic_tables(0, 4)


@pytest.mark.parametrize("variant", ["a=-0.75", "no antialias", "vertical first", "truncation"])
def test_sweep_rejects_planted_variants(sweep, variant):
    tables = {"a=-0.75": R.variant_tables(a=-0.75), "no antialias": R.variant_tables(antialias=False),
              "vertical first": ops.pillow_bicubic_tables, "truncation": R.variant_tables(truncate=True)}[variant]
    differ = [not np.array_equal(R.resize(u8, H, W, tables, vertical_first=(variant == "vertical first")), ref)
              for u8, _, (W, H), ref in sweep]
    assert any(differ), variant
    # the restatement itself is the one the sweep accepts
    assert all(np.array_equal(R.resize(u8, H, W, R.variant_tables()), ref) for u8, _, (W, H), ref in sweep[:4])


@pytest.mark.parametrize("w, h, kw, expect", [
    (400, 400, {}, (1024, 1024, 400, 400)),              # RSSCN7: x2.56
    (600, 600, {}, (1024, 1024, 600, 600)),              # WHU-RS19: 600 * (1024 / 600) is 1024 + 1 ulp
    (512, 512, {}, (1024, 1024, 512, 512)),
    (1100, 1100, {}, (1088, 1088, 1100, 1100)),          # no upscale; 17.1875 -> 17
    (200, 120, {"min_size": 256}, (448, 256, 200, 120)),  # 426.67 / 64 = 6.67 -> 7
    (1056, 1120, {"min_size": 1}, (1024, 1152, 1056, 1120)),  # 16.5 -> 16, 17.5 -> 18: numpy rounds ties to even
    (176, 112, {"min_size": 256}, (384, 256, 176, 112)),
    (1024, 1536, {}, (1024, 1536, 1024, 1536)),
    (300, 200, {"upscale": 2}, (1536, 1024, 600, 400)),
    (400, 300, {"fix_resize": 512}, (704, 512, 683, 512)),  # fix_resize also sets (w0, h0)
])
def test_pil2tensor_size_hand_worked(w, h, kw, expect):
    assert colorfix.pil2tensor_size(w, h, **kw) == expect


def test_pil2tensor_size_matches_the_pillow_reference():
    for (w, h), kw in (((37, 53), {"min_size": 100}), ((96, 96), {"min_size": 256}), ((150, 70), {"min_size": 64}),
                       ((130, 66), {"min_size": 1, "upscale": 2})):
        x, h0, w0 = R.pil2tensor(Image.fromarray(image(w, h, 0)), **kw)
        W, H, w0_, h0_ = colorfix.pil2tensor_size(w, h, **kw)
        assert (x.shape[1], x.shape[2], h0, w0) == (H, W, h0_, w0_)


def test_u8_to_unit_range_values_are_the_float64_path():
    """x / 255 * 2 - 1 is evaluated in float64 and then cast: the fp32 value the kernel must produce for every byte
    (it computes in double).  PIL2Tensor of an image already at its target size is exactly this table."""
    v = np.arange(256)
    table = np.float32(v / 255 * 2 - 1)
    u8 = np.tile(v.astype(np.uint8), (64, 1))[..., None].repeat(3, 2)          # 256 x 64, no resize at min_size 64
    x, _, _ = R.pil2tensor(Image.fromarray(u8), min_size=64)
    assert x.dtype == torch.float32 and x.shape == (3, 64, 256)
    assert np.array_equal(x[0, 0].numpy(), table) and np.array_equal(x[2, 63].numpy(), table)
    assert table[0] == -1.0 and table[255] == 1.0
    # the same formula in fp32 differs in the last bit for some bytes: fp32 arithmetic would not do
    f32 = (v.astype(np.float32) / np.float32(255) * np.float32(2) - np.float32(1)).astype(np.float32)
    assert (f32 != table).any()


def test_tensor2img_rounding():
    """Round half to even after the fp32 scaling, clamp outside [-1, 1]."""
    x = torch.tensor([-2.0, -1.0, 0.0, 1.0, 3.0, 1 / 255 - 1, 2 * (0.5 / 255) - 1, 2 * (1.5 / 255) - 1], dtype=torch.float32)
    u8 = R.tensor2img(x.view(1, 1, 8).repeat(3, 2, 1))
    t = (x.clamp(-1, 1) + 1) / 2
    expect = np.rint(t.numpy() * np.float32(255.0)).astype(np.uint8)
    assert np.array_equal(u8[0, :, 0], expect)
    assert u8[0, :5, 0].tolist() == [0, 0, 128, 255, 255]


needs_reference = pytest.mark.skipif(not reference_import.available(),
                                     reason="no reference checkout (oracle/_ref/ or B200SR_REFERENCE_ROOT)")


def _ref_module(rel):
    reference_import.install_stubs()
    spec = importlib.util.spec_from_file_location("_ref_" + rel.replace("/", "_")[:-3],
                                                  os.path.join(reference_import.REFERENCE_ROOT, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@needs_reference
def test_hand_off_against_the_reference_functions():
    util = _ref_module("models/util.py")
    t2i = _ref_module("utils/tensor2img.py")
    g = torch.Generator().manual_seed(0)
    x = torch.rand(3, 40, 56, generator=g) * 2.4 - 1.2
    assert np.array_equal(t2i.tensor2img(x), R.tensor2img(x))
    for (w, h), kw in (((56, 40), {"min_size": 128}), ((400, 400), {}), ((176, 112), {"min_size": 256}),
                       ((300, 200), {"upscale": 2}), ((400, 300), {"fix_resize": 512})):
        img = Image.fromarray(image(w, h, 1))
        ref_x, ref_h0, ref_w0 = util.PIL2Tensor(img, **kw)
        x, h0, w0 = R.pil2tensor(img, **kw)
        assert (h0, w0) == (ref_h0, ref_w0) and torch.equal(x, ref_x)
        W, H, w0_, h0_ = colorfix.pil2tensor_size(w, h, **kw)
        assert (tuple(ref_x.shape[-2:]), ref_h0, ref_w0) == ((H, W), h0_, w0_)
