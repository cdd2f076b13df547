"""References for the stage-1 -> stage-2 hand-off (tensor2img, PIL2Tensor), written with numpy and Pillow itself: Pillow is
the third-party arithmetic the reference calls, so it is the checker for the bicubic resample.

  tensor2img   SR3's utils/tensor2img.py:4-21 (min_max = (-1, 1), out_type uint8), as infer.py:133-138 uses it.  No checkout
               of the reference was at hand when this was written: the convention is SR3 upstream's.
               test_imageio_cpu.py pins it against the reference's own function when a checkout is present.
  pil2tensor   models/util.py:132-156 (PIL2Tensor).
  resample_axis / resize
               an integer restatement of what b200sr_resample_u8 computes from the host tables
               (b200sr.ops.pillow_bicubic_tables), in numpy: the tests check it against PIL.Image.resize.
  variant_tables
               the table builder with one deliberate defect each, which a byte-for-byte sweep must reject.
"""
from __future__ import annotations

import math

import numpy as np
import torch
from PIL import Image

PB = 22


# (w, h) -> (W, H): up, down, mixed, non-square, 1-pixel inputs, ratios > 4 both ways, and the PIL2Tensor sizes of the
# reference's datasets (RSSCN7 400^2, WHU-RS19 600^2) and of an image larger than 1024.
SWEEP = [
    ((400, 400), (1024, 1024)), ((600, 600), (1024, 1024)), ((37, 53), (1024, 1472)), ((1100, 1100), (1088, 1088)),
    ((200, 120), (448, 256)), ((5, 7), (64, 3)), ((1, 9), (4, 2)), ((333, 257), (128, 448)),
    ((64, 48), (40, 96)), ((96, 80), (160, 24)), ((1, 1), (7, 5)), ((1, 30), (3, 1)), ((17, 1), (1, 9)),
    ((10, 12), (53, 61)), ((300, 260), (13, 11)), ((250, 9), (31, 50)), ((176, 112), (384, 256)),
]


def image(w, h, seed):
    """Noise plus a ramp and hard edges: every tap weight, overshoot and clamp is exercised."""
    rng = np.random.default_rng(seed)
    u8 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    u8[:, : max(w // 3, 1), 0] = 255
    u8[: max(h // 4, 1), :, 1] = 0
    u8[..., 2] = np.minimum(u8[..., 2], (np.arange(w) * 255 // max(w - 1, 1)).astype(np.uint8)[None, :])
    return u8


def tensor2img(x: torch.Tensor) -> np.ndarray:
    """[C, H, W] (or [1, C, H, W]) tensor in [-1, 1] -> uint8 HWC, as SR3's tensor2img."""
    t = x.squeeze().float().cpu().clamp_(-1, 1)
    t = (t - (-1)) / (1 - (-1))
    img = np.transpose(t.numpy(), (1, 2, 0))
    return (img * 255.0).round().astype(np.uint8)


def pil2tensor(img: Image.Image, upscale=1, min_size=1024, fix_resize=None):
    """models/util.py:132-156: returns (x [C, H, W] fp32, h0, w0)."""
    w, h = img.size
    w *= upscale
    h *= upscale
    w0, h0 = round(w), round(h)
    if min(w, h) < min_size:
        _upscale = min_size / min(w, h)
        w *= _upscale
        h *= _upscale
    if fix_resize is not None:
        _upscale = fix_resize / min(w, h)
        w *= _upscale
        h *= _upscale
        w0, h0 = round(w), round(h)
    w = int(np.round(w / 64.0)) * 64
    h = int(np.round(h / 64.0)) * 64
    x = img.resize((w, h), Image.BICUBIC)
    x = np.array(x).round().clip(0, 255).astype(np.uint8)
    x = x / 255 * 2 - 1
    x = torch.tensor(x, dtype=torch.float32).permute(2, 0, 1)
    return x, h0, w0


def pil_resize(u8: np.ndarray, oh: int, ow: int) -> np.ndarray:
    return np.asarray(Image.fromarray(u8).resize((ow, oh), Image.BICUBIC))


def resample_axis(src: np.ndarray, axis: int, bounds: np.ndarray, coeffs: np.ndarray) -> np.ndarray:
    """The kernel's arithmetic along `axis` of a uint8 [H, W, C] array: int32 accumulator from 2^21, clamp(acc >> 22)."""
    s = np.moveaxis(src, axis, 0).astype(np.int64)
    out = np.empty((bounds.shape[0],) + s.shape[1:], dtype=np.uint8)
    for o in range(bounds.shape[0]):
        xmin, n = int(bounds[o, 0]), int(bounds[o, 1])
        acc = np.full(s.shape[1:], 1 << (PB - 1), dtype=np.int64)
        for t in range(n):
            acc += s[xmin + t] * int(coeffs[o, t])
        assert np.abs(acc).max() < 2 ** 31                      # the kernel's int32 accumulator cannot overflow
        out[o] = np.clip(acc >> PB, 0, 255)
    return np.moveaxis(out, 0, axis)


def resize(u8: np.ndarray, oh: int, ow: int, tables, vertical_first: bool = False) -> np.ndarray:
    """Two passes as Image.resize: width first, each pass only when its size changes."""
    h, w = u8.shape[:2]
    passes = [(1, w, ow), (0, h, oh)]
    if vertical_first:
        passes.reverse()
    x = u8
    for axis, n_in, n_out in passes:
        if n_in != n_out:
            bounds, coeffs, _ = tables(n_in, n_out)
            x = resample_axis(x, axis, bounds, coeffs)
    return x.copy()


def variant_tables(a: float = -0.5, antialias: bool = True, truncate: bool = False):
    """A restatement of pillow_bicubic_tables with one knob changed (defaults = Pillow's rule)."""

    def filt(x):
        x = np.abs(x)
        return np.where(x < 1.0, ((a + 2.0) * x - (a + 3.0)) * x * x + 1,
                        np.where(x < 2.0, (((x - 5) * x + 8) * x - 4) * a, 0.0))

    def tables(in_len, out_len):
        scale = float(in_len) / out_len
        fs = max(scale, 1.0) if antialias else 1.0
        support = 2.0 * fs
        ksize = int(math.ceil(support)) * 2 + 1
        bounds = np.zeros((out_len, 2), np.int32)
        coeffs = np.zeros((out_len, ksize), np.int32)
        for o in range(out_len):
            center = (o + 0.5) * scale
            xmin = max(int(center - support + 0.5), 0)
            n = min(int(center + support + 0.5), in_len) - xmin
            w = [float(filt((k + xmin - center + 0.5) * (1.0 / fs))) for k in range(n)]
            ww = 0.0
            for v in w:
                ww += v
            if ww != 0.0:
                w = [v / ww for v in w]
            for k, v in enumerate(w):
                if truncate:
                    coeffs[o, k] = int(v * (1 << PB))
                else:
                    coeffs[o, k] = int(-0.5 + v * (1 << PB)) if v < 0 else int(0.5 + v * (1 << PB))
            bounds[o] = (xmin, n)
        return bounds, coeffs, ksize

    return tables
