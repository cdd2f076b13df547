"""ORACLE tooling — import the *real* reference modules from a checkout of the reference project
(B200SR_REFERENCE_ROOT, default oracle/_ref/, which git ignores) to pin the restatement and to generate
tests/golden/.  Without such a checkout, available() is False and the tests that need it skip.

Three third-party packages the reference imports at module scope are absent from this image and
are not executed on the denoiser path; they are replaced by empty stubs (SURVEY.md Appendix B):
omegaconf (ListConfig/OmegaConf names), pytorch_lightning (LightningModule), k_diffusion.sampling
(two names), plus kornia / open_clip placeholders.
"""
import os
import sys
import types

import torch

REFERENCE_ROOT = os.environ.get("B200SR_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "sgm"))


def install_stubs() -> None:
    if "omegaconf" not in sys.modules:
        oc = types.ModuleType("omegaconf")

        class ListConfig(list):
            pass

        class OmegaConf(dict):
            pass

        oc.ListConfig, oc.OmegaConf = ListConfig, OmegaConf
        lc = types.ModuleType("omegaconf.listconfig")
        lc.ListConfig = ListConfig
        sys.modules.update({"omegaconf": oc, "omegaconf.listconfig": lc})
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")
        pl.LightningModule = torch.nn.Module
        sys.modules["pytorch_lightning"] = pl
    if "k_diffusion" not in sys.modules:
        kd, kds = types.ModuleType("k_diffusion"), types.ModuleType("k_diffusion.sampling")
        kds.BrownianTreeNoiseSampler = object
        kds.get_sigmas_karras = lambda *a, **k: None
        kd.sampling = kds
        sys.modules.update({"k_diffusion": kd, "k_diffusion.sampling": kds})
    for name in ("kornia", "open_clip"):
        sys.modules.setdefault(name, types.ModuleType(name))
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def stage2_modules(unet_cfg: dict, control_cfg: dict):
    """Returns the reference ControlWrapper(LightGLVUNet) with GLVControl loaded, eval mode, fp32."""
    install_stubs()
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        from models.modules.SR_modules import GLVControl, LightGLVUNet
        from sgm.modules.diffusionmodules.wrappers import ControlWrapper

        unet = LightGLVUNet(**unet_cfg)
        control = GLVControl(**control_cfg)
    wrapper = ControlWrapper(unet)
    wrapper.load_control_model(control)
    return wrapper.eval()


def stage2_sampler(num_steps=50, s_churn=5.0, s_noise=1.003, scale=4.0, scale_min=7.5, device="cpu"):
    install_stubs()
    from sgm.modules.diffusionmodules.denoiser import DiscreteDenoiserWithControl
    from sgm.modules.diffusionmodules.sampling import RestoreEDMSampler

    disc = {"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"}
    denoiser = DiscreteDenoiserWithControl(
        weighting_config={"target": "sgm.modules.diffusionmodules.denoiser_weighting.EpsWeighting"},
        scaling_config={"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
        num_idx=1000, discretization_config=disc)
    sampler = RestoreEDMSampler(
        num_steps=num_steps, restore_cfg=-1.0, s_churn=s_churn, s_noise=s_noise, discretization_config=disc,
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearCFG",
                       "params": {"scale": scale, "scale_min": scale_min}},
        device=device)
    return denoiser, sampler


def sr3_modules(unet_cfg: dict, schedule: dict):
    install_stubs()
    from models.sr3_model.sr3_modules.diffusion import GaussianDiffusion
    from models.sr3_model.sr3_modules.unet import UNet

    net = UNet(in_channel=unet_cfg["in_channel"], out_channel=unet_cfg["out_channel"],
               norm_groups=unet_cfg["norm_groups"], inner_channel=unet_cfg["inner_channel"],
               channel_mults=unet_cfg["channel_mults"], attn_res=unet_cfg["attn_res"],
               res_blocks=unet_cfg["res_blocks"], dropout=unet_cfg["dropout"], image_size=unet_cfg["image_size"])
    diff = GaussianDiffusion(net, image_size=unet_cfg["image_size"], channels=3, loss_type="l1", conditional=True)
    diff.set_new_noise_schedule(dict(schedule, schedule="linear"), device="cpu")
    return diff.eval()


def vae_modules(ddconfig: dict, embed_dim: int):
    """The reference AutoencoderKLInferenceWrapper (sgm/models/autoencoder.py:282-321) with the SR_backbone's
    denoise_encoder copy (models/SR_model.py:22), eval mode, fp32."""
    install_stubs()
    import contextlib
    import copy
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        from sgm.models.autoencoder import AutoencoderKLInferenceWrapper

        vae = AutoencoderKLInferenceWrapper(embed_dim=embed_dim, ddconfig=dict(ddconfig),
                                            lossconfig={"target": "torch.nn.Identity"}, monitor="val/rec_loss")
    vae.denoise_encoder = copy.deepcopy(vae.encoder)
    return vae.eval()
