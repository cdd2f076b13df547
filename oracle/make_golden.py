"""ORACLE tooling — needs a checkout of the reference project at oracle/_ref/ (or B200SR_REFERENCE_ROOT):

    python -m oracle.make_golden

1. instantiates the real reference modules (oracle/reference_import.py), fills them with the
   name-keyed weights of oracle/weights.py and runs them in fp32 on seeded synthetic inputs;
2. runs the restatement (oracle/stage2.py, sampler.py, sr3.py) on the same state_dict / inputs and
   asserts agreement (this is what pins the oracle);
3. writes the reference outputs as small fixtures to tests/golden/*.pt (inputs and weights are
   regenerated from seeds at test time; checksums of both are stored to detect RNG drift).
"""
from __future__ import annotations

import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import configs, inputs, reference_import, sampler as osampler, sr3 as osr3, stage2 as ostage2, weights  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def maxdiff(a, b):
    return (a.float() - b.float()).abs().max().item()


def checksum(t: torch.Tensor):
    t = t.double()
    return [t.sum().item(), t.abs().sum().item()]


def stage2(latent=16, seed=0, steps=6, threshold=0.3):
    t0 = time.time()
    wrapper = reference_import.stage2_modules(configs.STAGE2_UNET_TEST, configs.STAGE2_CONTROL_TEST)
    sd = wrapper.state_dict()
    weights.fill_(sd, seed)
    sd = {k: v.clone() for k, v in wrapper.state_dict().items()}
    print(f"[stage2] reference built + filled: {len(sd)} tensors, "
          f"{sum(v.numel() for v in sd.values()) / 1e6:.0f} M params, {time.time() - t0:.1f}s")
    x, c, uc = inputs.stage2_inputs(latent=latent, seed=1234)
    den, smp = reference_import.stage2_sampler(device="cpu")
    out = {"latent": latent, "seed": seed, "threshold": threshold,
           "weight_checksum": checksum(sd["diffusion_model.input_blocks.4.1.transformer_blocks.0.attn1.to_q.weight"]),
           "input_checksum": checksum(c["crossattn"])}

    # --- single network call, CFG batch 2, fbcache_mode none / stage1+2 ---------------------------------
    import sgm.modules.diffusionmodules.guiders as guiders
    guider = guiders.LinearCFG(scale=4.0, scale_min=7.5)
    sig = torch.full((1,), 14.6146)
    xin, sin, cin = guider.prepare_inputs(x, sig, c, uc)
    idx = den.sigma_to_idx(sin)
    c_in = 1 / (den.sigmas[idx] ** 2 + 1) ** 0.5
    net_x = xin * c_in.view(-1, 1, 1, 1)
    with torch.no_grad():
        eps_ref = wrapper(net_x, idx, cin, 1.0, "none", None)
        info = wrapper(net_x, idx, cin, 1.0, "input_stage1", None)
        eps_ref2 = wrapper(net_x, idx, cin, 1.0, "input_stage2", info)
        ctrl_ref = wrapper.control_model(x=cin["control"], timesteps=idx, xt=net_x, context=cin["crossattn"],
                                         y=cin["vector"])
        eps_or = ostage2.control_wrapper(sd, net_x, idx, cin, 1.0)
        ctrl_or = ostage2.glv_control(sd, "control_model.", cin["control"], idx, net_x, cin["crossattn"], cin["vector"])
    d = maxdiff(eps_ref, eps_or)
    print(f"[stage2] eps: |ref|max={eps_ref.abs().max():.4f} std={eps_ref.std():.4f}  oracle-vs-ref max diff {d:.3e};"
          f" two-stage-vs-none {maxdiff(eps_ref, eps_ref2):.3e}")
    assert d < 2e-4 * max(1.0, eps_ref.abs().max().item()), "oracle restatement disagrees with the reference"
    for a, b in zip(ctrl_ref, ctrl_or):
        assert maxdiff(a, b) < 2e-4 * max(1.0, a.abs().max().item())
    out.update(net_x=net_x, idx=idx, eps=eps_ref, h_stage1=info["h"],
               control_stats=[[t.mean().item(), t.std().item()] for t in ctrl_ref])

    # --- sampler: `steps` RestoreEDMSampler steps with the first-block cache ------------------------------
    from models.modules.DFBCache import MyCacheContext, cache_context

    def ref_denoiser(inp, sigma, cc, control_scale=1.0, fbcache_mode="none", partial_info=None):
        return den(wrapper, inp, sigma, cc, control_scale, fbcache_mode, partial_info)

    oden = osampler.Denoiser()

    def or_net(xx, tt, cc, cs, mode, pinfo):
        with torch.no_grad():
            if mode == "none":
                return ostage2.control_wrapper(sd, xx, tt, cc, cs)
            if mode == "input_stage1":
                control = ostage2.glv_control(sd, "control_model.", cc["control"], tt, xx, cc["crossattn"], cc["vector"])
                h, hs, emb = ostage2.unet_input_stage(sd, "diffusion_model.", xx, tt, cc["crossattn"], cc["vector"])
                return {"h": h, "hs": hs, "emb": emb, "context": cc["crossattn"], "control": control}
            return ostage2.unet_output_stage(sd, "diffusion_model.", pinfo["h"], pinfo["hs"], pinfo["emb"],
                                             pinfo["context"], pinfo["control"], cs).float()

    def or_denoiser(inp, sigma, cc, control_scale, mode, pinfo):
        return oden(or_net, inp, sigma, cc, control_scale, mode, pinfo)

    z0 = torch.randn(1, 4, latent, latent, generator=torch.Generator().manual_seed(77))
    zr, s_in, sigmas, _, _, _ = smp.init_loop(z0.clone(), c, uc, num_steps=50)
    osmp = osampler.RestoreSampler(device="cpu")
    zo, os_in, osig = osmp.init_loop(z0.clone())
    assert maxdiff(sigmas, osig) == 0.0
    thr_r, thr_o, cache = threshold, threshold, osampler.CacheState()
    ref_trace = []
    with torch.no_grad(), cache_context(MyCacheContext()):
        for i in range(steps):
            torch.manual_seed(1000 + i)
            zr, new_thr = smp.step(zr, i, s_in, sigmas, ref_denoiser, c, uc, x_center=None, control_scale=1.0,
                                   threshold=thr_r)
            ref_trace.append(("hit" if new_thr == thr_r and i > 0 else "miss", float(new_thr)))
            thr_r = new_thr
            torch.manual_seed(1000 + i)
            noise = torch.randn_like(zo)
            zo, thr_o = osmp.step(zo, i, os_in, osig, or_denoiser, c, uc, 1.0, thr_o, cache, noise)
            print(f"[stage2] step {i}: ref thr {thr_r:.5f} oracle {osmp.trace[-1]} z diff {maxdiff(zr, zo):.3e}")
            assert maxdiff(zr, zo) < 5e-3 and abs(thr_r - thr_o) < 1e-4
    out.update(z0=z0, z_final=zr, trace=[list(t) for t in osmp.trace], sigmas=sigmas, steps=steps)
    torch.save(out, os.path.join(GOLDEN, f"stage2_test_{latent}.pt"))
    print(f"[stage2] wrote golden, total {time.time() - t0:.1f}s")


def sr3(size=32, seed=0):
    diff = reference_import.sr3_modules(configs.SR3_UNET, configs.SR3_SCHEDULE)
    sd = diff.denoise_fn.state_dict()
    weights.fill_(sd, seed)
    sd = {k: v.clone() for k, v in diff.denoise_fn.state_dict().items()}
    cond, noises = inputs.sr3_inputs(size=size, seed=0, steps=50)
    level = torch.tensor([[0.73]])
    xin = torch.cat([cond, noises[0]], dim=1)
    with torch.no_grad():
        e_ref = diff.denoise_fn(xin, level)
        e_or = osr3.unet(sd, "", xin, level)
    d = maxdiff(e_ref, e_or)
    print(f"[sr3] unet |ref|max {e_ref.abs().max():.4f}; oracle-vs-ref {d:.3e}")
    assert d < 1e-4 * max(1.0, e_ref.abs().max().item())
    # full 50-step loop: the reference draws torch.randn(shape) then randn_like per step (t>0) from the global RNG
    torch.manual_seed(5)
    with torch.no_grad():
        sr_ref = diff.p_sample_loop(cond, continous=False)
    torch.manual_seed(5)
    seq = [torch.randn(cond.shape) for _ in range(50)] + [torch.zeros_like(cond)]
    sched = osr3.Schedule(**configs.SR3_SCHEDULE)
    with torch.no_grad():
        sr_or = osr3.p_sample_loop(lambda x, l: osr3.unet(sd, "", x, l), sched, cond, seq)
    d2 = maxdiff(sr_ref, sr_or)
    print(f"[sr3] 50-step loop oracle-vs-ref {d2:.3e}")
    assert d2 < 1e-3
    torch.save({"size": size, "level": level, "eps": e_ref, "sr": sr_ref, "loop_seed": 5,
                "weight_checksum": checksum(sd["downs.1.res_block.block1.block.3.weight"])},
               os.path.join(GOLDEN, f"sr3_{size}.pt"))
    print("[sr3] wrote golden")


def vae(size=64, seed=0):
    """First stage: real AutoencoderKLInferenceWrapper vs oracle/vae.py; golden = the reference's outputs."""
    from oracle import vae as ovae

    ref = reference_import.vae_modules(configs.VAE_DDCONFIG, configs.VAE_EMBED_DIM)
    weights.fill_(ref.state_dict(), seed)
    sd = {k: v.clone() for k, v in ref.state_dict().items()}
    g = torch.Generator().manual_seed(31)
    img = torch.rand(1, 3, size, size, generator=g) * 2 - 1
    noise = torch.randn(1, 4, size // 8, size // 8, generator=g)
    with torch.no_grad():
        m_ref = ref.quant_conv(ref.denoise_encoder(img))                      # SR_model.py:66-71
        m_plain = ref.quant_conv(ref.encoder(img))
        z = ovae.SCALE_FACTOR * m_ref.chunk(2, dim=1)[0]                      # posterior.mode() * scale_factor
        x_ref = ref.decode(1.0 / ovae.SCALE_FACTOR * z)                       # SR_model.py:81-85
        m_or = ovae.moments(sd, img, "denoise_encoder.")
        x_or = ovae.decode_first_stage(sd, ovae.encode_with_denoise(sd, img))
    print(f"[vae] moments |ref|max {m_ref.abs().max():.4f} oracle-vs-ref {maxdiff(m_ref, m_or):.3e}; "
          f"decode |ref|max {x_ref.abs().max():.4f} oracle-vs-ref {maxdiff(x_ref, x_or):.3e}")
    assert maxdiff(m_ref, m_or) < 1e-4 * max(1.0, m_ref.abs().max().item())
    assert maxdiff(x_ref, x_or) < 1e-4 * max(1.0, x_ref.abs().max().item())
    assert maxdiff(ovae.posterior(m_plain, noise), m_plain.chunk(2, 1)[0] + torch.exp(0.5 * m_plain.chunk(2, 1)[1].clamp(-30, 20)) * noise) == 0
    torch.save({"size": size, "img": img, "moments": m_ref, "z": z, "decoded": x_ref,
                "weight_checksum": checksum(sd["decoder.mid.block_1.conv1.weight"])},
               os.path.join(GOLDEN, f"vae_{size}.pt"))
    import json

    with open(os.path.join(GOLDEN, "vae_keys.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in sd.items()}, f, indent=0, sort_keys=True)
    print("[vae] wrote golden")


def colorfix(size=48):
    """Output side: the reference's utils/colorfix.py functions vs oracle/colorfix.py; golden = the reference's outputs."""
    reference_import.install_stubs()
    from oracle import colorfix as ocf
    from utils import colorfix as rcf

    g = torch.Generator().manual_seed(17)
    content = torch.rand(1, 3, size, size + 16, generator=g) * 2.4 - 1.2
    style = torch.rand(1, 3, size, size + 16, generator=g) * 2 - 1
    ref = rcf.wavelet_reconstruction(content, style)
    assert maxdiff(ref, ocf.wavelet_reconstruction(content, style)) == 0.0
    hi, lo = rcf.wavelet_decomposition(content)
    u8_same = ocf.tensor_to_uint8(ref[0], size, size + 16)
    u8_up = ocf.tensor_to_uint8(ref[0], 70, 100)
    u8_down = ocf.tensor_to_uint8(ref[0], 31, 40)
    torch.save({"content": content, "style": style, "reconstruction": ref, "high": hi, "low": lo,
                "u8_same": u8_same, "u8_up": u8_up, "u8_down": u8_down}, os.path.join(GOLDEN, f"colorfix_{size}.pt"))
    print("[colorfix] wrote golden")


def conditioner(clip_layers=3, clip_idx=2, bigg_layers=3):
    """Text towers at reduced depth (full widths): the installed transformers implementation vs oracle/conditioner.py."""
    import transformers
    from oracle import conditioner as ocond

    sys.path.insert(0, os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200"))
    from b200sr import conditioner as pcond   # parameter containers only (names / shapes of the reference's modules)

    m = pcond.GeneralConditionerWithControl(_clip_layers=clip_layers, _clip_layer_idx=clip_idx, _bigg_layers=bigg_layers)
    sd = weights.fill_(m.state_dict(), 0)
    g = torch.Generator().manual_seed(23)
    ids = torch.randint(1, 49000, (2, 77), generator=g)
    ids[0, 20], ids[1, 33] = 49407, 49407           # eot = highest id
    ids[0, 21:], ids[1, 34:] = 0, 0
    # CLIP-L: transformers.CLIPTextModel
    cfg = transformers.CLIPTextConfig(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=clip_layers,
                                      num_attention_heads=12, max_position_embeddings=77, hidden_act="quick_gelu",
                                      eos_token_id=2, bos_token_id=0, pad_token_id=1)
    hf = transformers.CLIPTextModel(cfg).eval()
    pre = "embedders.0.transformer."
    missing = hf.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys), missing
    with torch.no_grad():
        ref_l = hf(input_ids=ids, output_hidden_states=True).hidden_states[clip_idx]
        or_l = ocond.clip_l_hidden_states(sd, pre + "text_model.", ids)[clip_idx]
    print(f"[conditioner] CLIP-L hidden[{clip_idx}] |ref|max {ref_l.abs().max():.3f} oracle-vs-transformers {maxdiff(ref_l, or_l):.3e}")
    assert maxdiff(ref_l, or_l) < 1e-4 * max(1.0, ref_l.abs().max().item())
    # bigG text tower: transformers.CLIPTextModelWithProjection with the open_clip weights re-laid-out
    cfg2 = transformers.CLIPTextConfig(vocab_size=49408, hidden_size=1280, intermediate_size=5120, num_hidden_layers=bigg_layers,
                                       num_attention_heads=20, max_position_embeddings=77, hidden_act="gelu",
                                       projection_dim=1280, eos_token_id=2, bos_token_id=0, pad_token_id=1)
    hf2 = transformers.CLIPTextModelWithProjection(cfg2).eval()
    q = "embedders.1.model."
    m2 = {"text_model.embeddings.token_embedding.weight": sd[q + "token_embedding.weight"],
          "text_model.embeddings.position_embedding.weight": sd[q + "positional_embedding"],
          "text_model.final_layer_norm.weight": sd[q + "ln_final.weight"], "text_model.final_layer_norm.bias": sd[q + "ln_final.bias"],
          "text_projection.weight": sd[q + "text_projection"].t().contiguous()}
    for i in range(bigg_layers):
        r, t = f"{q}transformer.resblocks.{i}.", f"text_model.encoder.layers.{i}."
        wq, wk, wv = sd[r + "attn.in_proj_weight"].chunk(3, 0)
        bq, bk, bv = sd[r + "attn.in_proj_bias"].chunk(3, 0)
        m2.update({t + "self_attn.q_proj.weight": wq, t + "self_attn.k_proj.weight": wk, t + "self_attn.v_proj.weight": wv,
                   t + "self_attn.q_proj.bias": bq, t + "self_attn.k_proj.bias": bk, t + "self_attn.v_proj.bias": bv,
                   t + "self_attn.out_proj.weight": sd[r + "attn.out_proj.weight"], t + "self_attn.out_proj.bias": sd[r + "attn.out_proj.bias"],
                   t + "layer_norm1.weight": sd[r + "ln_1.weight"], t + "layer_norm1.bias": sd[r + "ln_1.bias"],
                   t + "layer_norm2.weight": sd[r + "ln_2.weight"], t + "layer_norm2.bias": sd[r + "ln_2.bias"],
                   t + "mlp.fc1.weight": sd[r + "mlp.c_fc.weight"], t + "mlp.fc1.bias": sd[r + "mlp.c_fc.bias"],
                   t + "mlp.fc2.weight": sd[r + "mlp.c_proj.weight"], t + "mlp.fc2.bias": sd[r + "mlp.c_proj.bias"]})
    missing = hf2.load_state_dict(m2, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys), missing
    with torch.no_grad():
        o2 = hf2(input_ids=ids, output_hidden_states=True)
        ref_pen, ref_pool = o2.hidden_states[-2], o2.text_embeds
        or_pen, or_pool = ocond.openclip_text(sd, q, ids)
    print(f"[conditioner] bigG penultimate oracle-vs-transformers {maxdiff(ref_pen, or_pen):.3e}; pooled {maxdiff(ref_pool, or_pool):.3e}")
    assert maxdiff(ref_pen, or_pen) < 1e-4 * max(1.0, ref_pen.abs().max().item())
    assert maxdiff(ref_pool, or_pool) < 1e-4 * max(1.0, ref_pool.abs().max().item())
    batch = {"txt": (ids, ids.flip(0)), "original_size_as_tuple": torch.tensor([[1024., 1024.]] * 2),
             "crop_coords_top_left": torch.zeros(2, 2), "target_size_as_tuple": torch.tensor([[1024., 1024.]] * 2)}
    with torch.no_grad():
        out = ocond.conditioner(sd, batch, clip_idx)
    # the size embedders against sgm's own Timestep module
    reference_import.install_stubs()
    from sgm.modules.diffusionmodules.openaimodel import Timestep
    ts = Timestep(256)(torch.tensor([1024., 1024., 0., 0.]))
    assert maxdiff(ts.reshape(2, 512), torch.stack([ocond.concat_timestep(torch.tensor([[1024., 1024.]]))[0],
                                                    ocond.concat_timestep(torch.zeros(1, 2))[0]])) < 1e-6
    torch.save({"clip_layers": clip_layers, "clip_idx": clip_idx, "bigg_layers": bigg_layers, "ids": ids,
                "clip_hidden": ref_l, "bigg_penultimate": ref_pen, "bigg_pooled": ref_pool,
                "crossattn": out["crossattn"], "vector": out["vector"]}, os.path.join(GOLDEN, "conditioner_small.pt"))
    print("[conditioner] wrote golden")


def tables():
    reference_import.install_stubs()
    from sgm.modules.diffusionmodules.sampling import _sliding_windows
    import numpy as np

    den, smp = reference_import.stage2_sampler(device="cpu")
    sig50 = smp.discretization(50, device="cpu")
    assert maxdiff(sig50, osampler.ddpm_sigmas(50)) == 0.0
    assert maxdiff(den.sigmas, osampler.Denoiser().sigmas) == 0.0
    wins = _sliding_windows(256, 256, 128, 96)
    assert wins == osampler.sliding_windows(256, 256, 128, 96)
    # gaussian_weights in the reference allocates on 'cuda'; restate its numpy body for the fixture
    torch.save({"sigmas50": sig50, "sigmas1000_head": den.sigmas[:8], "sigmas1000_tail": den.sigmas[-8:],
                "windows_256_128_96": wins, "gauss_128_row64": osampler.gaussian_weights(128, 128)[64].float(),
                "gauss_128_col64": osampler.gaussian_weights(128, 128)[:, 64].float()},
               os.path.join(GOLDEN, "tables.pt"))
    print("[tables] wrote golden")


def keys():
    """state_dict key -> shape of the FULL reference configuration (meta device, no memory)."""
    import json

    with torch.device("meta"):
        wrapper = reference_import.stage2_modules(configs.STAGE2_UNET, configs.STAGE2_CONTROL)
        diff = reference_import.sr3_modules(configs.SR3_UNET, configs.SR3_SCHEDULE) if False else None
    with open(os.path.join(GOLDEN, "stage2_keys.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in wrapper.state_dict().items()}, f, indent=0, sort_keys=True)
    reference_import.install_stubs()
    from models.sr3_model.sr3_modules.unet import UNet

    cfg = configs.SR3_UNET
    with torch.device("meta"):
        net = UNet(in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=cfg["norm_groups"],
                   inner_channel=cfg["inner_channel"], channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"],
                   res_blocks=cfg["res_blocks"], dropout=cfg["dropout"], image_size=cfg["image_size"])
    with open(os.path.join(GOLDEN, "sr3_keys.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in net.state_dict().items()}, f, indent=0, sort_keys=True)
    print("[keys] wrote golden")


if __name__ == "__main__":
    assert reference_import.available(), "needs a reference checkout at oracle/_ref/ or B200SR_REFERENCE_ROOT"
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_grad_enabled(False)
    keys()
    if "--keys-only" in sys.argv:
        sys.exit(0)
    if "--vae-only" in sys.argv:
        vae()
        sys.exit(0)
    if "--conditioner-only" in sys.argv:
        conditioner()
        sys.exit(0)
    if "--colorfix-only" in sys.argv:
        colorfix()
        sys.exit(0)
    tables()
    sr3()
    vae()
    colorfix()
    conditioner()
    stage2()
