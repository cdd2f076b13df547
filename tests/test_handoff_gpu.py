"""Stage 2 at the non-square latents PIL2Tensor produces, and the driver's reference hand-off (stage2_min_size):
  - the test-config engine at a 32 x 56 latent against the fp32 oracle (same gates as the square tests), CUDA-graph
    replay of a cached trajectory equal to eager bit for bit;
  - one full-depth network call at 128 x 192 against the oracle (eps rel-L2 < 1e-2);
  - the test-config pipeline on stage-1 images of 176 x 112 and 96^2 with stage2_min_size = 256, and 400^2 with 1024:
    stage-2 input == PIL2Tensor(tensor2img(stage 1)) bit for bit, shapes from pil2tensor_size, a mixed-size
    run_sharded list == fresh pipelines per image, and stage2_min_size=None == the pipeline built without it."""
import pytest
import torch
from PIL import Image

import imageio_ref as R

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def psnr(a, b):
    import math

    a, b = a.float(), b.float()
    peak = (b.max() - b.min()).item()
    return 10 * math.log10(peak * peak / ((a - b) ** 2).mean().item())


def _build(unet_cfg, control_cfg):
    from b200sr import modules
    from oracle import weights

    w = modules.build_stage2(unet_cfg, control_cfg).eval()
    weights.fill_(w.state_dict(), 0)
    return w.cuda()


def _inputs(h, w, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(1, 4, h, w, generator=g) * (1.0 + 14.6146**2) ** 0.5
    control = torch.randn(1, 4, h, w, generator=g)
    cap = lambda: {"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}  # noqa
    c, uc = cap(), cap()
    to = lambda d: {k: v.cuda() for k, v in d.items()}  # noqa: E731
    return x.cuda(), to(dict(c, control=control)), to(dict(uc, control=control))


def test_engine_non_square_latent_vs_oracle():
    from b200sr.sampling import Stage2Engine
    from oracle import configs, sampler as osampler, stage2 as ostage2

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    small = _build(configs.STAGE2_UNET_TEST, configs.STAGE2_CONTROL_TEST)
    x, c, uc = _inputs(32, 56, 7)
    sd = {k: v.detach() for k, v in small.state_dict().items()}
    oden = osampler.Denoiser(device="cuda")
    net = lambda xx, tt, cc, cs, mode, pi: ostage2.control_wrapper(sd, xx, tt, cc, cs)  # noqa: E731
    smp = osampler.RestoreSampler(device="cuda")
    _, s_in, sig = smp.init_loop(x.clone())
    g = torch.Generator(device="cuda").manual_seed(3)
    noise = torch.randn(x.shape, generator=g, device="cuda")
    with torch.no_grad():
        ref, _ = smp.step(x, 3, s_in, sig, lambda *a: oden(net, *a), c, uc, 1.0, 0.0, None, noise)
    eng = Stage2Engine(small)
    eng.set_condition(c, uc)
    out, _ = eng.step(x, 3, noise, 0.0)
    assert out.shape == (1, 4, 32, 56)
    print(f"32x56 step: update rel-L2 {rel_l2(out - x, ref - x):.3e}, PSNR {psnr(out, ref):.1f} dB")
    assert rel_l2(out - x, ref - x) < 1e-2 and psnr(out, ref) >= 40.0
    # cached trajectory (first-block cache on): CUDA-graph replay == eager, bit for bit
    z0 = torch.randn(x.shape, generator=g, device="cuda")
    noises = [torch.randn(x.shape, generator=g, device="cuda") for _ in range(8)]
    outs, traces = [], []
    for graphs in (False, True):
        e = Stage2Engine(small, num_steps=8, use_graphs=graphs)
        e.set_condition(c, uc)
        outs.append(e.sample(z0, noises, threshold=0.3, dec=1.0))
        traces.append([t[0] for t in e.trace])
        e.close()
    print("32x56 trace", traces[0])
    assert traces[0] == traces[1] and "hit" in traces[0]
    assert torch.equal(outs[0], outs[1])
    eng.close()


def test_full_model_eps_128x192():
    from oracle import configs, sampler as osampler, stage2 as ostage2

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    full = _build(configs.STAGE2_UNET, configs.STAGE2_CONTROL)
    x, c, uc = _inputs(128, 192, 11)
    _, _, cin = osampler.cfg_prepare(x, torch.ones(1, device="cuda"), c, uc)
    oden = osampler.Denoiser(device="cuda")
    sig = torch.full((1,), 14.6146, device="cuda")
    idx = oden.sigma_to_idx(torch.cat([sig] * 2))
    net_x = torch.cat([x] * 2) / (oden.sigmas[idx] ** 2 + 1).sqrt().view(-1, 1, 1, 1)
    sd = {k: v.detach() for k, v in full.state_dict().items()}
    with torch.no_grad():
        ref = ostage2.control_wrapper(sd, net_x, idx, cin, 1.0)
        eps = full(net_x, idx, cin, 1.0, "none", None)
    err = rel_l2(eps, ref)
    print(f"full-model eps rel-L2 at 128x192 vs fp32 oracle: {err:.4e}")
    assert eps.shape == (2, 4, 128, 192) and err < 1e-2


@pytest.fixture(scope="module")
def parts():
    from b200sr import modules, sr3, vae
    from oracle import configs, weights

    wrapper = modules.build_stage2(configs.STAGE2_UNET_TEST, configs.STAGE2_CONTROL_TEST).eval()
    weights.fill_(wrapper.state_dict(), 0)
    ae = vae.AutoencoderKLInferenceWrapper(configs.VAE_EMBED_DIM, dict(configs.VAE_DDCONFIG)).add_denoise_encoder().eval()
    weights.fill_(ae.state_dict(), 0)
    net = sr3.UNet(**configs.SR3_UNET).eval()
    weights.fill_(net.state_dict(), 0)
    diff = sr3.GaussianDiffusion(net.cuda(), image_size=224, channels=3, conditional=True)
    diff.set_new_noise_schedule(dict(configs.SR3_SCHEDULE, schedule="linear", n_timestep=8), device="cuda")
    return wrapper.cuda(), ae.cuda(), diff


def _pipeline(parts, **kw):
    from b200sr import colorfix, vae
    from b200sr.driver import RestorationPipeline

    wrapper, ae, diff = parts
    return RestorationPipeline(wrapper, diff, first_stage=vae.FirstStage(ae), device="cuda", num_steps=6,
                               color_fix=colorfix.wavelet_reconstruction, **kw)


def _check_hand_off(r, min_size):
    from b200sr import colorfix

    stage1 = r["stage1"]
    h, w = stage1.shape[-2:]
    W, H, w0, h0 = colorfix.pil2tensor_size(w, h, 1, min_size)
    ref, rh0, rw0 = R.pil2tensor(Image.fromarray(R.tensor2img(stage1.cpu())), min_size=min_size)
    assert (rh0, rw0) == (h0, w0) == (h, w)
    assert torch.equal(r["stage2_input"][0].cpu(), ref)
    assert r["stage2_size"] == (H, W)
    assert r["latent"].shape == (1, 4, H // 8, W // 8)
    assert r["image"].shape == (1, 3, H, W) and torch.isfinite(r["image"]).all()
    assert r["uint8"].shape == (h0, w0, 3) and r["uint8"].dtype == torch.uint8


def test_pipeline_hand_off_mixed_sizes(parts):
    from b200sr.driver import run_sharded

    g = torch.Generator().manual_seed(5)
    # x8 -> stage 1 at 176 x 112 (-> 384 x 256 at stage 2, a 32 x 48 latent) and 96^2 (-> 256^2)
    images = [torch.rand(1, 3, 14, 22, generator=g) * 2 - 1, torch.rand(1, 3, 12, 12, generator=g) * 2 - 1,
              torch.rand(1, 3, 14, 22, generator=g) * 2 - 1]
    cap = ({"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)},
           {"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)})
    caps = [cap] * 3                            # the same caption objects at every control shape
    pipe = _pipeline(parts, stage2_min_size=256)
    whole = run_sharded(pipe, images, caps, 0, 1, seed=21, keep=True)
    for r in whole["results"]:
        _check_hand_off(r, 256)
    assert [r["stage2_size"] for r in whole["results"]] == [(256, 384), (256, 256), (256, 384)]
    pipe.engine.close()
    for i in range(3):
        fresh = _pipeline(parts, stage2_min_size=256)
        one = run_sharded(fresh, images[i:i + 1], caps[i:i + 1], 0, 1, seed=21 + i, keep=True)["results"][0]
        assert torch.equal(one["latent"], whole["results"][i]["latent"]), i
        assert torch.equal(one["uint8"], whole["results"][i]["uint8"]), i
        fresh.engine.close()


def test_pipeline_hand_off_400(parts):
    """RSSCN7's image size: 400^2 at stage 1 -> 1024^2 (a 128^2 latent) at stage 2 -> 400^2 uint8."""
    g = torch.Generator().manual_seed(6)
    lr = torch.rand(1, 3, 50, 50, generator=g) * 2 - 1
    c = {"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}
    uc = {"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}
    pipe = _pipeline(parts, stage2_min_size=1024)
    r = pipe.restore(lr, c, uc, seed=1)
    _check_hand_off(r, 1024)
    assert r["stage2_size"] == (1024, 1024) and r["uint8"].shape == (400, 400, 3)
    pipe.engine.close()


def test_stage2_min_size_none_is_the_default(parts):
    g = torch.Generator().manual_seed(8)
    lr = torch.rand(1, 3, 32, 32, generator=g) * 2 - 1
    c = {"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}
    uc = {"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}
    outs = []
    for kw in ({}, {"stage2_min_size": None}):
        pipe = _pipeline(parts, **kw)
        outs.append(pipe.restore(lr, c, uc, seed=4))
        pipe.engine.close()
    a, b = outs
    assert "stage2_input" not in a and a["stage2_size"] == (256, 256) and a["uint8"].shape == (256, 256, 3)
    for k in ("stage1", "latent", "image", "uint8"):
        assert torch.equal(a[k], b[k]), k
    assert a["trace"] == b["trace"]
