"""infer_dir-style driver of the two-stage restoration for a list of images, sharded over the GPUs.

Mirrored reference code (relative to the reference root):
  BatchSRPipeline.run / _process_single_image        infer_dir.py:108-206   (sequential loop over the directory)
  SR_backbone.just_sampling                          models/SR_model.py:200-298 (stage-2 loop, :265-291)
  GaussianDiffusion.super_resolution                 models/sr3_model/sr3_modules/diffusion.py:178-201
  tensor2img -> PIL2Tensor ... Tensor2PIL            infer.py:133-138, models/util.py:132-166 (with stage2_min_size)

What it runs per image (the denoiser hot path and its closest callers):
  LR image --bicubic x S--> SR3 stage 1 (T ancestral steps, CUDA-graphed) --> (hand-off) --> [first stage encode] -->
  50 RestoreEDMSampler steps with the first-block cache (img_threshold, dec_img) --> [first stage decode]
  --> [wavelet colour fix] --> [uint8 pack].

The hand-off is the reference's: with ``stage2_min_size`` set, the stage-1 image is quantised to uint8 (tensor2img) and
resized with Pillow's bicubic filter so that its short side is at least about ``stage2_min_size`` and both sides are
multiples of 64 (PIL2Tensor; the reference's drivers use 1024), and the result is resized back to the stage-1 size
(Tensor2PIL).  This is what lets stage 2 run on any SR3 output size (a 400^2 or 600^2 image would otherwise reach the
UNet as a latent whose side is not a multiple of 8).  ``stage2_min_size=None`` feeds the SR3 output to stage 2 as
is, which equals the reference only for square multiples of 64 of at least 1024 (the benchmark configurations).

The bracketed stages are the rows SURVEY.md section 8(f) ranks after the step path (VAE f2, colour fix f3).  They are
pluggable: ``first_stage`` is any object with ``encode(img) -> latent`` / ``decode(latent) -> img``
(``b200sr.vae.FirstStage`` over ``b200sr.vae.AutoencoderKL``); without one the driver stops at the latent and uses
``LatentStandIn`` — a fixed linear 8x8 pooling of the stage-1 image into 4 channels — to derive the
LQ control latent, which keeps shapes, data flow and work per image identical for throughput
purposes and is labelled as such in every result.  Captions are the fixed synthetic text embeddings
BASELINE.json prescribes (the LLaVA captioner and CLIP conditioner are not on the path).

Sharding: image i is processed by rank i mod world (``shard_images``); no communication while
sampling; ``run`` returns this rank's results and the caller gathers what it needs.
"""
from __future__ import annotations

import time
from typing import Callable, Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

from .parallel import shard_images
from .sampling import Stage2Engine


class LatentStandIn:
    """Placeholder for the SDXL VAE when none is supplied: 8x8 average pooling of the RGB image to three latent
    channels plus their mean as the fourth.  NOT a model of the VAE — it only produces a [B, 4, H/8, W/8]
    control latent with image-dependent content so the stage-2 loop runs on realistic shapes."""

    name = "stand-in (8x8 average pooling; no VAE)"

    def encode(self, img: torch.Tensor) -> torch.Tensor:
        z = F.avg_pool2d(img.float(), 8)
        return torch.cat((z, z.mean(1, keepdim=True)), 1).contiguous()

    def decode(self, z: torch.Tensor) -> Optional[torch.Tensor]:
        return None


class RestorationPipeline:
    """One GPU's worker: owns the stage-1 diffusion, the stage-2 engine and the optional first stage."""

    def __init__(self, stage2_wrapper, sr3_diffusion=None, first_stage=None, device="cuda", num_steps: int = 50,
                 s_churn: float = 5.0, s_noise: float = 1.003, cfg_scale: float = 7.5, cfg_scale_start: float = 4.0,
                 control_scale: float = 1.0, img_threshold: float = 0.3, dec_img: float = 1.0, upscale: int = 8,
                 color_fix: Optional[Callable] = None, stage2_min_size: Optional[int] = None):
        self.device = torch.device(device)
        self.sr3 = sr3_diffusion
        self.first_stage = first_stage if first_stage is not None else LatentStandIn()
        self.img_threshold, self.dec_img, self.upscale = img_threshold, dec_img, upscale
        self.color_fix = color_fix
        self.stage2_min_size = stage2_min_size
        # use_linear_CFG: guider scale = cfg_scale_start, scale_min = cfg_scale (SR_model.py:243-248)
        self.engine = Stage2Engine(stage2_wrapper, num_steps=num_steps, s_churn=s_churn, s_noise=s_noise,
                                   cfg_scale=cfg_scale_start, cfg_scale_min=cfg_scale, control_scale=control_scale,
                                   device=self.device)
        self.timings: Dict[str, float] = {}

    def _tic(self):
        torch.cuda.synchronize(self.device) if self.device.type == "cuda" else None
        return time.perf_counter()

    @torch.no_grad()
    def restore(self, lr: torch.Tensor, c: Dict[str, torch.Tensor], uc: Dict[str, torch.Tensor], seed: int = 0) -> dict:
        """lr: [1, 3, h, w] in [-1, 1].  c / uc: {"crossattn": [1, 77, 2048], "vector": [1, 2816]} (synthetic caption).
        Returns {"stage1": image, "latent": final latent, "image": decoded image or None, "uint8": [h0, w0, 3] or None,
        "trace": hit/miss list, "stage2_size": (H, W) of the stage-2 input}; with stage2_min_size also "stage2_input",
        PIL2Tensor's [1, 3, H, W] fp32 image, and (h0, w0) is the stage-1 size."""
        dev = self.device
        g = torch.Generator(device=dev).manual_seed(seed)
        t0 = self._tic()
        # ---- stage 1: bicubic xS then SR3 (infer_dir.py:118-133; diffusion.py:178-201) -----------------------------
        cond = F.interpolate(lr.to(dev).float(), scale_factor=self.upscale, mode="bicubic", align_corners=False).clamp(-1, 1)
        if self.sr3 is not None:
            steps = self.sr3.num_timesteps
            noises = [torch.randn(cond.shape, generator=g, device=dev) for _ in range(steps + 1)]
            stage1 = self.sr3.p_sample_loop(cond, continous=False, noises=noises)
            stage1 = stage1.reshape(cond.shape).clamp(-1, 1)
        else:
            stage1 = cond
        t1 = self._tic()
        x2, h0, w0 = stage1, None, None
        if self.stage2_min_size is not None:
            # ---- hand-off on the device: tensor2img + PIL2Tensor (infer.py:133-138, models/util.py:132-156) --------
            from .colorfix import pil_to_tensor, tensor2img_u8

            x2, h0, w0 = pil_to_tensor(tensor2img_u8(stage1), upscale=1, min_size=self.stage2_min_size)
        # ---- first stage encode -> LQ control latent (SR_model.py:259-263) -----------------------------------------
        lq = self.first_stage.encode(x2)                     # _z = encode_first_stage_with_denoise(x, use_sample=False)
        x_stage1 = self.first_stage.decode(lq)               # x_stage1 = decode_first_stage(_z): the colour-fix reference
        # (z_stage1 = encode_first_stage(x_stage1), SR_model.py:256, only feeds the restore_cfg > 0 branch of the
        #  sampler, which the shipped drivers switch off with restoration_scale = -1; it is not computed here.)
        t2 = self._tic()
        # ---- stage 2: num_steps RestoreEDMSampler steps with the first-block cache (SR_model.py:265-291) -------
        cc = {"crossattn": c["crossattn"].to(dev), "vector": c["vector"].to(dev), "control": lq}
        ucc = {"crossattn": uc["crossattn"].to(dev), "vector": uc["vector"].to(dev), "control": lq}
        self.engine.set_condition(cc, ucc)
        z0 = torch.randn(lq.shape, generator=g, device=dev)                       # noised_z = randn_like(_z)
        noises2 = [torch.randn(lq.shape, generator=g, device=dev) for _ in range(self.engine.sched.num_steps)]
        z = self.engine.sample(z0, noises2, threshold=self.img_threshold, dec=self.dec_img)
        trace = [t[0] for t in self.engine.trace]
        t3 = self._tic()
        # ---- decode, colour fix (SR_model.py:293-298) -------------------------------------------------------------
        img = self.first_stage.decode(z)
        u8 = None
        if img is not None:
            if self.color_fix is not None:
                img = self.color_fix(img, x_stage1)                               # wavelet_reconstruction(samples, x_stage1)
            from .colorfix import tensor_to_uint8

            oh, ow = (h0, w0) if h0 is not None else img.shape[-2:]
            u8 = tensor_to_uint8(img[0], oh, ow)                                  # Tensor2PIL(sample, h0, w0)
        t4 = self._tic()
        for k, v in (("stage1_s", t1 - t0), ("encode_s", t2 - t1), ("stage2_s", t3 - t2), ("decode_s", t4 - t3)):
            self.timings[k] = self.timings.get(k, 0.0) + v
        out = {"stage1": stage1, "latent": z, "image": img, "uint8": u8, "trace": trace,
               "stage2_size": tuple(x2.shape[-2:])}
        if self.stage2_min_size is not None:
            out["stage2_input"] = x2
        return out


def run_sharded(pipeline: RestorationPipeline, images: Sequence[torch.Tensor], captions: Sequence, rank: int = 0,
                world: int = 1, seed: int = 0, keep: bool = False) -> dict:
    """infer_dir.py:187-206 over `images` with image i on rank i mod world.  captions[i] = (c, uc).
    Returns {"indices": this rank's image indices, "seconds": wall time of this rank's share,
    "misses": cache misses per image, "results": per-image outputs when keep}."""
    mine = shard_images(len(images), rank, world)
    results, misses = [], []
    t0 = pipeline._tic()
    for i in mine:
        c, uc = captions[i]
        r = pipeline.restore(images[i], c, uc, seed=seed + i)
        misses.append(r["trace"].count("miss"))
        if keep:
            results.append(r)
    dt = pipeline._tic() - t0
    return {"indices": mine, "seconds": dt, "misses": misses, "results": results}
