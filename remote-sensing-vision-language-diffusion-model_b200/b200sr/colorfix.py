"""Image side of the pipeline on the sm_100a kernels (SURVEY.md section 8(f) row f3): the stage-1 -> stage-2 hand-off,
the wavelet colour fix and the tensor -> uint8 image conversion.

Mirrored reference code (relative to the reference root), same function names and argument meaning:
  tensor2img (stage-1 output -> uint8)                                infer.py:133-138, utils/tensor2img.py:4-21
  PIL2Tensor (bicubic resize to the stage-2 size, uint8 -> [-1, 1])   models/util.py:132-156
  wavelet_blur / wavelet_decomposition / wavelet_reconstruction      utils/colorfix.py:73-119
  Tensor2PIL                                                          models/util.py:159-166
The hand-off never leaves the device: ``tensor2img_u8`` and ``pil_to_tensor`` reproduce the bytes and the fp32 values
the reference gets from its PIL round trip (Pillow's own bicubic resample, not torch's).
(color_fix_type defaults to "Wavelet" in infer.py / infer_dir.py; the AdaIN variant, colorfix.py:44-71, is not selected
by the shipped drivers and is not built.)
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import ops


def wavelet_blur(image: torch.Tensor, radius: int) -> torch.Tensor:
    """colorfix.py:73-91: depthwise 3x3 binomial blur with dilation `radius`, replicate padding."""
    return ops.wavelet_level(image.float().contiguous(), radius)


def wavelet_decomposition(image: torch.Tensor, levels: int = 5):
    """colorfix.py:93-106: returns (high_freq, low_freq)."""
    image = image.float().contiguous()
    high = torch.empty_like(image)
    for i in range(levels):
        image = ops.wavelet_level(image, 2 ** i, high=high, first=(i == 0))
    return high, image


def wavelet_reconstruction(content_feat: torch.Tensor, style_feat: torch.Tensor) -> torch.Tensor:
    """colorfix.py:108-119: the content's high frequencies on the style's low frequencies."""
    content_high, _ = wavelet_decomposition(content_feat)
    style = style_feat.float().contiguous()
    for i in range(5):
        style = ops.wavelet_level(style, 2 ** i)
    return ops.add_f32(content_high, style)


def tensor_to_uint8(x: torch.Tensor, h0: int, w0: int) -> torch.Tensor:
    """Tensor2PIL without the PIL object (models/util.py:159-166): [C, H, W] in [-1, 1] -> uint8 [h0, w0, C] on the
    device (bicubic resize, * 127.5 + 127.5, clip, truncate); ``PIL.Image.fromarray(result.cpu().numpy())`` is the image."""
    return ops.image_to_u8(x.float().contiguous(), h0, w0)


def tensor2img_u8(x: torch.Tensor) -> torch.Tensor:
    """tensor2img (utils/tensor2img.py:4-21, min_max = (-1, 1)) without the host copy: [C, H, W] (or [1, C, H, W]) in
    [-1, 1] -> uint8 [H, W, C] on the device, t = (clamp(x, -1, 1) + 1) / 2, rint(t * 255) in fp32 (round half to even,
    as numpy's .round()).  This is SR3 upstream's convention; it was written without a checkout of the reference at
    hand and is pinned against the reference's own function by tests/test_imageio_cpu.py when a checkout is present."""
    if x.dim() == 4:
        if x.shape[0] != 1:
            raise ValueError("tensor2img_u8 converts one image")
        x = x[0]
    return ops.tensor2img_u8(x.float().contiguous())


def pil2tensor_size(w: int, h: int, upscale: float = 1, min_size: int = 1024,
                    fix_resize: Optional[int] = None) -> Tuple[int, int, int, int]:
    """The sizes PIL2Tensor (models/util.py:132-156) computes for a w x h image: returns (W, H, w0, h0), the resize
    target (multiples of 64, short side scaled up to at least about min_size) and the size Tensor2PIL restores."""
    w, h = w * upscale, h * upscale
    w0, h0 = round(w), round(h)
    if min(w, h) < min_size:
        s = min_size / min(w, h)
        w, h = w * s, h * s
    if fix_resize is not None:
        s = fix_resize / min(w, h)
        w, h = w * s, h * s
        w0, h0 = round(w), round(h)
    return int(np.round(w / 64.0)) * 64, int(np.round(h / 64.0)) * 64, w0, h0


def pil_to_tensor(u8_hwc: torch.Tensor, upscale: float = 1, min_size: int = 1024,
                  fix_resize: Optional[int] = None) -> Tuple[torch.Tensor, int, int]:
    """PIL2Tensor (models/util.py:132-156) on the device: uint8 [h, w, 3] -> (x [1, 3, H, W] fp32 in [-1, 1], h0, w0).
    The resize is Image.resize((W, H), Image.BICUBIC) byte for byte (Pillow's a = -0.5 filter, antialiased when it
    reduces, 22-bit fixed point), and x = float32(u8 / 255 * 2 - 1) with the arithmetic in double, as the reference's
    numpy."""
    h, w = u8_hwc.shape[:2]
    W, H, w0, h0 = pil2tensor_size(w, h, upscale, min_size, fix_resize)
    if W <= 0 or H <= 0:
        raise ValueError(f"PIL2Tensor size of a {w}x{h} image rounds to {W}x{H}")
    x = ops.img_u8_to_tensor(ops.resize_bicubic_u8(u8_hwc.contiguous(), H, W))
    return x.unsqueeze(0), h0, w0
