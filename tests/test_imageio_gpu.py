"""GPU kernels of the stage-1 -> stage-2 hand-off, byte for byte: b200sr_resample_u8 (through resize_bicubic_u8) against
PIL.Image.resize, b200sr_tensor2img_u8 against SR3's tensor2img, b200sr_img_u8_to_tensor against numpy's float64 path,
pil_to_tensor against PIL2Tensor.  Every output is also written as a window of a sentinel-filled guard buffer, twice with
different sentinels: every byte inside the window is written, nothing outside it.  Bad arguments return EINVAL."""
import ctypes

import numpy as np
import pytest
import torch
from PIL import Image

import imageio_ref as R
from imageio_ref import SWEEP, image

pytestmark = pytest.mark.gpu

SIZES = SWEEP + [((600, 600), (1024, 1024)), ((1100, 1100), (1088, 1088)), ((1024, 1536), (1024, 1536))]


def _windows(nbytes, pad):
    """Two guard buffers (sentinels 0x5A / 0xA5 in every byte) and a contiguous window of nbytes at byte offset pad."""
    out = []
    for s in (0x5A, 0xA5):
        buf = torch.full((nbytes + pad + 37,), s, dtype=torch.uint8, device="cuda")
        out.append((buf, buf[pad:pad + nbytes]))
    return out


def _check_guards(buf, pad, nbytes, sentinel):
    host = buf.cpu().numpy()
    assert (host[:pad] == sentinel).all() and (host[pad + nbytes:] == sentinel).all()


def test_resize_matches_pillow():
    from b200sr import ops

    for i, ((w, h), (W, H)) in enumerate(SIZES):
        u8 = image(w, h, i)
        out = ops.resize_bicubic_u8(torch.from_numpy(u8).cuda(), H, W)
        assert tuple(out.shape) == (H, W, 3)
        assert np.array_equal(out.cpu().numpy(), R.pil_resize(u8, H, W)), ((w, h), (W, H))


@pytest.mark.parametrize("pad", [0, 16, 7])     # 16-byte stores, and the byte path of an unaligned destination
def test_resample_pass_writes_exactly_its_window(pad):
    from b200sr import ops

    for i, ((w, h), (W, H)) in enumerate(SIZES[:12]):
        u8 = image(w, h, i)
        src = torch.from_numpy(u8).cuda()
        for axis, n_in, n_out in ((1, w, W), (0, h, H)):
            bounds, coeffs, _ = ops.pillow_bicubic_tables(n_in, n_out)
            ref = R.resample_axis(u8, axis, bounds, coeffs)
            for s, (buf, win) in zip((0x5A, 0xA5), _windows(ref.size, pad)):
                ops.resample_u8_axis(src, n_out, axis, out=win.view(ref.shape))
                assert np.array_equal(win.view(ref.shape).cpu().numpy(), ref), ((w, h), axis)
                _check_guards(buf, pad, ref.size, s)


@pytest.mark.parametrize("hw", [(40, 56), (7, 9), (256, 384), (2, 3)])
def test_tensor2img_u8(hw):
    from b200sr import colorfix

    h, w = hw
    g = torch.Generator(device="cuda").manual_seed(h * 1000 + w)
    x = torch.rand(3, h, w, generator=g, device="cuda") * 2.6 - 1.3
    # exact ties of the * 255 rounding and the clamp edges
    ties = (torch.arange(h * w, device="cuda") % 256).float().add(0.5).div(255).mul(2).sub(1).view(h, w)
    x[1] = torch.where(torch.arange(h * w, device="cuda").view(h, w) % 2 == 0, ties, x[1])
    x[2, 0, 0] = -1.0
    x[2, -1, -1] = 1.0
    ref = R.tensor2img(x.cpu())
    assert np.array_equal(colorfix.tensor2img_u8(x.unsqueeze(0)).cpu().numpy(), ref)
    # window of a guard buffer; the input as an unaligned view takes the scalar load path
    xs = torch.empty(3 * h * w + 1, device="cuda")
    xs[1:] = x.flatten()
    for pad in (0, 5):
        for s, (buf, win) in zip((0x5A, 0xA5), _windows(3 * h * w, pad)):
            rc = _lib().b200sr_tensor2img_u8(xs[1:].data_ptr(), win.data_ptr(), 3, h, w, _stream())
            assert rc == 0
            assert np.array_equal(win.view(h, w, 3).cpu().numpy(), ref)
            _check_guards(buf, pad, 3 * h * w, s)


@pytest.mark.parametrize("hw", [(64, 256), (7, 9), (1024, 1024)])
def test_img_u8_to_tensor_is_the_float64_path(hw):
    from b200sr import ops

    h, w = hw
    rng = np.random.default_rng(h + w)
    u8 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    u8.reshape(-1)[:256] = np.arange(min(256, u8.size), dtype=np.uint8)
    ref = torch.tensor(u8 / 255 * 2 - 1, dtype=torch.float32).permute(2, 0, 1).contiguous()
    src = torch.from_numpy(u8).cuda()
    assert torch.equal(ops.img_u8_to_tensor(src).cpu(), ref)
    n = 3 * h * w * 4
    for pad in (0, 4):          # a 4-byte offset takes the scalar store path
        for s, (buf, win) in zip((0x5A, 0xA5), _windows(n, pad)):
            assert _lib().b200sr_img_u8_to_tensor(src.data_ptr(), win.data_ptr(), 3, h, w, _stream()) == 0
            torch.cuda.synchronize()
            got = win.cpu().numpy().view(np.float32).reshape(3, h, w)
            assert np.array_equal(got, ref.numpy())
            _check_guards(buf, pad, n, s)


@pytest.mark.parametrize("wh, kw", [((400, 400), {}), ((600, 600), {}), ((176, 112), {"min_size": 256}),
                                    ((1100, 1100), {}), ((37, 53), {"min_size": 100}), ((300, 200), {"upscale": 2})])
def test_pil_to_tensor_matches_pil2tensor(wh, kw):
    from b200sr import colorfix

    w, h = wh
    u8 = image(w, h, 5)
    ref, h0, w0 = R.pil2tensor(Image.fromarray(u8), **kw)
    x, h0_, w0_ = colorfix.pil_to_tensor(torch.from_numpy(u8).cuda(), **kw)
    assert (h0_, w0_) == (h0, w0) and x.shape == (1,) + tuple(ref.shape)
    assert torch.equal(x[0].cpu(), ref)


def test_bad_arguments_return_einval():
    lib, st = _lib(), _stream()
    a = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    b = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    f = torch.zeros(1024, device="cuda")
    t = torch.zeros(64, dtype=torch.int32, device="cuda")
    E = -22
    for args in ((f, b, 0, 4, 4), (f, b, 5, 4, 4), (f, b, 3, 0, 4), (f, b, 3, 4, -1), (None, b, 3, 4, 4), (f, None, 3, 4, 4)):
        assert lib.b200sr_tensor2img_u8(*(_p(v) for v in args[:2]), *args[2:], st) == E, args
        assert lib.b200sr_img_u8_to_tensor(*(_p(v) for v in args[:2][::-1]), *args[2:], st) == E, args
    ok = (a, b, 2, 8, 4, 3, t, t, 5)
    for i, bad in ((0, None), (1, None), (2, 0), (3, 0), (4, 0), (5, -3), (6, None), (7, None), (8, 0), (1, a)):
        args = list(ok)
        args[i] = bad
        assert lib.b200sr_resample_u8(*(_p(v) if isinstance(v, torch.Tensor) or v is None else v for v in args), st) == E, i
    torch.cuda.synchronize()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _lib():
    from b200sr import _lib

    return _lib.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream
