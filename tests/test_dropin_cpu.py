"""The drop-in claim, shown: the reference's OWN sampler stack — DiscreteDenoiserWithControl.__call__
(sgm/modules/diffusionmodules/denoiser.py:66-78), RestoreEDMSampler.step / denoise (sampling.py:548-694), LinearCFG
(guiders.py:44-74) and the first-block cache context (models/modules/DFBCache.py) — imported unmodified from
the reference checkout, drives ``b200sr.modules.ControlWrapper`` exactly as it drives its own ``ControlWrapper``:
positional ``network(input * c_in, c_noise, cond, control_scale, fbcache_mode, partial_info)``, the ``"h"`` entry of
the returned partial_info read by the sampler, fp32 eps back.  The kernels are replaced by the CPU test double
(tests/ops_double.py); the module wiring, signatures and return conventions are the product's.

The tests marked ``needs_reference`` import the reference checkout (oracle/_ref/ or B200SR_REFERENCE_ROOT) and skip
without one.  test_sampler_protocol_drives_b200sr_wrapper needs nothing outside the repository: the oracle's
restatement of the same sampler stack drives the wrapper, checked against the reference's stored trajectory."""
import math
import os

import pytest
import torch

from oracle import configs, inputs, reference_import, sampler as osampler, weights

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
needs_reference = pytest.mark.skipif(not reference_import.available(),
                                     reason="needs a reference checkout (oracle/_ref/ or B200SR_REFERENCE_ROOT)")


def _psnr(z, ref):
    mse = ((z - ref) ** 2).mean().item()
    peak = (ref.max() - ref.min()).item()
    return 10 * math.log10(peak * peak / mse)


def test_sampler_protocol_drives_b200sr_wrapper(monkeypatch):
    """The oracle's restatement of RestoreEDMSampler + DiscreteDenoiserWithControl + LinearCFG + the first-block
    cache (oracle/sampler.py; oracle/make_golden.py pinned it to the reference's sampler when it wrote the golden
    file) calls ``b200sr.modules.ControlWrapper`` itself, positionally, as the reference's denoiser does.  Every
    call's arguments and return convention are checked; the hit/miss trace and the final latent must match the
    reference sampler's own 6-step run stored in tests/golden/stage2_test_16.pt."""
    import ops_double
    from b200sr import modules, ops

    ops_double.install(monkeypatch, ops)
    golden = torch.load(os.path.join(GOLDEN, "stage2_test_16.pt"), weights_only=False)
    wrapper = modules.build_stage2(configs.STAGE2_UNET_TEST, configs.STAGE2_CONTROL_TEST).eval()
    weights.fill_(wrapper.state_dict(), 0)
    calls, stage1 = [], {}

    def network(*args, **kwargs):
        assert not kwargs and len(args) == 6                     # denoiser.py:66-78 passes all six positionally
        x, c_noise, cond, control_scale, mode, partial_info = args
        assert x.dtype == torch.float32 and x.shape[0] == 2 and c_noise.dtype == torch.int64 and control_scale == 1.0
        assert set(cond) >= {"crossattn", "vector", "control"}
        calls.append(mode)
        if mode == "input_stage2":
            assert partial_info is stage1["info"]                 # the stage-1 result is handed back unchanged
        else:
            assert partial_info is None
        out = wrapper(*args)
        if mode == "input_stage1":
            assert torch.is_tensor(out["h"]) and out["h"].shape[0] == 2   # the sampler reads "h" (DFBCache.py:112)
            stage1["info"] = out
        else:
            assert out.dtype == torch.float32 and out.shape == x.shape
        return out

    den = osampler.Denoiser()
    smp = osampler.RestoreSampler()
    _, c, uc = inputs.stage2_inputs(latent=golden["latent"], seed=1234)
    z, s_in, sigmas = smp.init_loop(golden["z0"].clone())
    assert torch.equal(sigmas, golden["sigmas"])
    thr, cache = golden["threshold"], osampler.CacheState()
    with torch.no_grad():
        for i in range(golden["steps"]):
            torch.manual_seed(1000 + i)                          # the reference draws randn_like(x) from the global RNG
            noise = torch.randn_like(z)
            z, thr = smp.step(z, i, s_in, sigmas, lambda *a: den(network, *a), c, uc, 1.0, thr, cache, noise)
    trace = [t[0] for t in smp.trace]
    assert trace == [t[0] for t in golden["trace"]]
    assert calls.count("input_stage1") == golden["steps"] and calls.count("input_stage2") == trace.count("miss")
    assert len(calls) == golden["steps"] + trace.count("miss")
    assert z.dtype == torch.float32
    assert _psnr(z, golden["z_final"]) >= 40.0


@needs_reference
def test_reference_sampler_drives_b200sr_wrapper(monkeypatch):
    import ops_double
    from b200sr import modules, ops

    ops_double.install(monkeypatch, ops)
    golden = torch.load(os.path.join(GOLDEN, "stage2_test_16.pt"), weights_only=False)
    wrapper = modules.build_stage2(configs.STAGE2_UNET_TEST, configs.STAGE2_CONTROL_TEST).eval()
    weights.fill_(wrapper.state_dict(), 0)
    den, smp = reference_import.stage2_sampler(device="cpu")
    from models.modules.DFBCache import MyCacheContext, cache_context

    calls = []

    def denoiser(inp, sigma, cc, control_scale=1.0, fbcache_mode="none", partial_info=None):
        calls.append(fbcache_mode)
        return den(wrapper, inp, sigma, cc, control_scale, fbcache_mode, partial_info)   # denoiser.py:66-78

    _, c, uc = inputs.stage2_inputs(latent=golden["latent"], seed=1234)
    z, s_in, sigmas, _, c, uc = smp.init_loop(golden["z0"].clone(), c, uc, num_steps=50)
    assert torch.equal(sigmas, golden["sigmas"])
    thr, trace = golden["threshold"], []
    with torch.no_grad(), cache_context(MyCacheContext()):
        for i in range(golden["steps"]):
            torch.manual_seed(1000 + i)                      # the reference draws randn_like(x) from the global RNG
            z, new_thr = smp.step(z, i, s_in, sigmas, denoiser, c, uc, x_center=None, control_scale=1.0, threshold=thr)
            trace.append("hit" if (new_thr == thr and i > 0) else "miss")
            thr = new_thr
    assert trace == [t[0] for t in golden["trace"]]
    # every step asked for stage 1; only the misses went on to stage 2 (SR_modules.py:660-730 protocol)
    assert calls.count("input_stage1") == golden["steps"] and calls.count("input_stage2") == trace.count("miss")
    assert z.dtype == torch.float32
    assert _psnr(z, golden["z_final"]) >= 40.0


@needs_reference
def test_reference_yaml_targets_resolve_to_b200sr_classes():
    """INTEGRATION.md section 2: the swap is a change of `target:` strings; the constructors take the YAML's params."""
    import yaml
    from b200sr import modules

    with open(os.path.join(reference_import.REFERENCE_ROOT, "model_configs", "juggernautXL.yaml")) as f:
        params = yaml.safe_load(f)["model"]["params"]
    for key, cls in (("control_stage_config", modules.GLVControl), ("network_config", modules.LightGLVUNet)):
        with torch.device("meta"):
            m = cls(**params[key]["params"])
        assert isinstance(m, modules.UNetModel)
