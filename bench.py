#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native stage-2 denoiser path.

Workload (BASELINE.json configs[1], SURVEY.md section 8(d) config 2): ONE RestoreEDMSampler step of the full
SDXL UNet + GLV ControlNet at 1024^2 (4x128x128 latent), CFG batch 2 ([uncond; cond]), fbcache off
(threshold <= 0), bf16 operands / fp32 accumulation, random-init weights (oracle/weights.py, seed 0),
synthetic conditioning (oracle/inputs.py).  Algorithmic work = 20.28 TFLOP per step.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this framework
  python bench.py --impl reference [--gpus N] ...                # the reference algorithm on the host cores
  python bench.py ... --dump-outputs DIR                         # also write the last timed step's output as DIR/*.npy

--dump-outputs writes what the timed step returns to its caller, float32, after the timed loop: Stage2Engine.step's
x_next (rank 0's latent) as x_next.npy, or with --impl reference the network's eps as eps.npy.  The inputs are
seeded, so two builds run with the same arguments can be compared array for array.

The JSON line's `value` is the BASELINE metric (steps/s, one independent latent per GPU: image sharding, weak
scaling).  Beside it, in the same line:
  roofline            dominant kernel (tcgen05 GEMM / conv) against the measured bf16 peak, per-launch CUDA events;
                      share_of_step_time against a whole eager step; HBM GB/s of the normalisation kernels
  cpu_baseline        ONE full step of the reference algorithm on the host cores (N = 1 only; no extrapolation)
  gpu_eager_baseline  the same step through stock torch ops on this GPU (oracle under bf16 autocast = the reference's
                      own policy, and with pre-cast bf16 weights) — what the hand-written kernels have to beat
  tiled_x8            BASELINE config 4: a pool of 256^2 latents (2048^2 images), 9 windows each, the (image, window)
                      list sharded over the N ranks with the NVLink halo exchange; tiled steps/s, bytes exchanged,
                      speed-up over the same list on rank 0 alone; single-image scaling beside it
  batched             the same step with 2 / 4 latents per network call (per-latent step time)
  images_per_s        BASELINE config 5 sample (x8, 128^2 -> 1024^2) and config 3 (x4, 256^2 -> 1024^2): infer_dir-style
                      images sharded i mod N; SR3, VAE encode, 50 cached stage-2 steps, VAE decode, colour fix, uint8
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200"))

import torch  # noqa: E402

STEP_TFLOP = 20.28071518208      # FlopCounterMode over the oracle, B=2, 128^2 latent (tools: see DESIGN.md)
METRIC = "stage2_denoise_steps_per_s_1024sq_cfg2"
UNIT = "steps/s"
LATENT = 128
WORKLOAD = "stage-2 SDXL UNet + GLV ControlNet denoise step, 4x128x128 latent (1024^2), CFG batch 2"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference algorithm on the host cores, one FULL step per timing
# ------------------------------------------------------------------------------------------------
def cpu_reference(steps: int, warmup: int, sd_cpu=None, dump_dir=None):
    """Times complete stage-2 network steps (control net + UNet, CFG batch 2, 128^2 latent, fp32, every host thread)
    of the reference algorithm on the CPU: through the reference's own modules imported from a reference checkout
    (oracle/_ref/ or B200SR_REFERENCE_ROOT) when there is one (kind "reference"), else through the oracle port of
    the same functions (kind "port").  Shapes are never scaled down.  With `dump_dir`, the last timed step's output
    (the network's eps, 2x4x128x128) is written there as eps.npy."""
    from oracle import configs, inputs, reference_import, sampler as osampler, stage2 as ostage2, weights

    torch.set_num_threads(os.cpu_count() or 1)
    x, c, uc = inputs.stage2_inputs(latent=LATENT, seed=1234)
    xin, _, cin = osampler.cfg_prepare(x, torch.ones(1), c, uc)
    t = torch.full((2,), 999.0)
    net_x = xin / (14.6146**2 + 1) ** 0.5
    kind = "port"
    if reference_import.available() and sd_cpu is None:
        kind = "reference"
        wrapper = reference_import.stage2_modules(configs.STAGE2_UNET, configs.STAGE2_CONTROL)
        weights.fill_(wrapper.state_dict(), 0)
        idx = t.long()

        def step():
            with torch.no_grad():
                return wrapper(net_x, idx, cin, 1.0, "none", None)
    else:
        if sd_cpu is None:
            from b200sr import modules

            w = modules.build_stage2(configs.STAGE2_UNET, configs.STAGE2_CONTROL).eval()
            sd_cpu = weights.fill_(w.state_dict(), 0)

        def step():
            with torch.no_grad():
                return ostage2.control_wrapper(sd_cpu, net_x, t, cin, 1.0)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = step()
    dt = (time.perf_counter() - t0) / steps
    if dump_dir:
        dump_outputs(dump_dir, {"eps": out})
    return {"value": 1.0 / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{steps} full step(s) of the workload (20.28 TFLOP each, fp32) after {warmup} warm-up step(s); "
                      f"{dt:.2f} s per step; no extrapolation",
            "seconds_per_step": dt, "cpu_tflops": STEP_TFLOP / dt}


def run_reference(args, rank: int):
    if rank != 0:
        return
    k, w = args.steps, args.warmup
    base = cpu_reference(k, w, dump_dir=args.dump_outputs)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": k, "warmup": w, "ms_per_step": 1000.0 / base["value"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD}, "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# the same step through stock torch ops on this GPU (the reference's algorithm, eager)
# ------------------------------------------------------------------------------------------------
def gpu_eager_baseline(wrapper, dev, iters: int = 5):
    from oracle import inputs, sampler as osampler, stage2 as ostage2

    x, c, uc = inputs.stage2_inputs(latent=LATENT, seed=1234)
    xin, _, cin = osampler.cfg_prepare(x, torch.ones(1), c, uc)
    t = torch.full((2,), 999.0, device=dev)
    net_x = (xin / (14.6146**2 + 1) ** 0.5).to(dev)
    cin = {k: v.to(dev) for k, v in cin.items()}
    sd = {k: v.detach() for k, v in wrapper.state_dict().items()}
    out = {}
    ostage2.ATTENTION = "sdpa"   # the reference's own attention call (attention.py:275-277), fused kernel

    def timed(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def autocast_step():
        with torch.no_grad(), torch.autocast("cuda", torch.bfloat16):
            return ostage2.control_wrapper(sd, net_x, t, cin, 1.0)

    ms = timed(autocast_step)
    out["autocast_bf16"] = {"ms_per_step": ms, "steps_per_s": 1000.0 / ms, "tflops": STEP_TFLOP / ms * 1e3,
                            "what": "oracle restatement of the reference modules (F.linear / F.conv2d / F.group_norm / SDPA) "
                                    "under torch.autocast(cuda, bf16) with fp32 master weights = the reference's policy "
                                    "(wrappers.py:84-110); weights are re-cast every step, as in the reference"}
    sd16 = {k: v.to(torch.bfloat16) for k, v in sd.items()}
    x16, c16 = net_x.to(torch.bfloat16), {k: v.to(torch.bfloat16) for k, v in cin.items()}

    def bf16_step():
        with torch.no_grad(), torch.autocast("cuda", torch.bfloat16):
            return ostage2.control_wrapper(sd16, x16, t, c16, 1.0)

    try:
        ms16 = timed(bf16_step)
        out["bf16_weights"] = {"ms_per_step": ms16, "steps_per_s": 1000.0 / ms16, "tflops": STEP_TFLOP / ms16 * 1e3,
                               "what": "same functions under the same autocast policy, but on weights pre-cast to bf16 once "
                                       "(no per-step weight casts): the fastest stock-torch form of the reference's "
                                       "numerics — cuBLASLt + cuDNN + fused SDPA, fp32 GroupNorm / LayerNorm / softmax"}
    except Exception as e:  # pragma: no cover
        out["bf16_weights"] = {"error": repr(e)[:200]}
    ostage2.ATTENTION = "manual"
    del sd16
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# BASELINE config 4: pooled tiled x8 sampler steps, (image, window) list sharded over the ranks
# ------------------------------------------------------------------------------------------------
def tiled_block(wrapper, dev, rank: int, world: int, pool: int, steps: int, tile_batch: int):
    import torch.distributed as dist
    from b200sr import ops
    from b200sr.parallel import EngineTileRunner, PooledTileStepper
    from b200sr.sampling import Stage2Engine

    L, TILE, STRIDE = 256, 128, 96

    def data(n_images, seed):
        g = torch.Generator().manual_seed(seed)     # identical on every rank
        xs, lqs, caps, noises = {}, {}, {}, {}
        for m in range(n_images):
            xs[m] = (torch.randn(1, 4, L, L, generator=g) * (1 + 14.6146**2) ** 0.5)
            lqs[m] = torch.randn(1, 4, L, L, generator=g)
            caps[m] = tuple({"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}
                            for _ in range(2))
            noises[m] = [torch.randn(1, 4, L, L, generator=g) for _ in range(steps + 1)]
        return xs, lqs, caps, noises

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(n_images, solo: bool, n_steps: int):
        xs, lqs, caps, noises = data(n_images, 4321)
        st = PooledTileStepper(n_images, L, L, TILE, STRIDE, device=dev, tile_batch=tile_batch, blend=ops)
        if solo:   # the whole list on this rank alone (no exchange): the N = 1 run of the same list
            st.world, st.rank, st.mine, st.my_images, st.strips = 1, 0, list(st.units), list(range(n_images)), {}
        mine = st.my_images
        caps_d = {m: tuple({k: v.to(dev) for k, v in d.items()} for d in caps[m]) for m in mine}
        lqs_d = {m: lqs[m].to(dev) for m in mine}
        runner = EngineTileRunner(lambda: Stage2Engine(wrapper, device=dev), caps_d, lqs_d)
        cur = {m: xs[m].to(dev) for m in mine}
        nz = {m: [n.to(dev) for n in noises[m]] for m in mine}
        cur = st.step(cur, 0, {m: nz[m][0] for m in mine}, runner)          # warm-up: packing, graph capture, snapshots
        if not solo:
            barrier()
        else:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(1, n_steps + 1):
            cur = st.step(cur, i, {m: nz[m][i] for m in mine}, runner)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if not solo:
            tt = torch.tensor([dt], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = tt.item()
        runner.close()
        del runner
        torch.cuda.empty_cache()
        return st, dt / n_steps

    res = {"latent": f"{L}x{L} (2048^2 image)", "tile": TILE, "stride": STRIDE, "windows_per_image": 9,
           "tile_batch": tile_batch, "timed_steps": steps, "tflop_per_tiled_step_per_image": 9 * STEP_TFLOP}
    st, dt = run(pool, False, steps)
    halo = torch.tensor([float(st.halo_bytes_per_step)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(halo, op=dist.ReduceOp.SUM)
    res["pooled"] = {"images": pool, "units": len(st.units), "units_per_rank": [len(p) for p in st.parts],
                     "s_per_tiled_step": dt, "tiled_steps_per_s": 1.0 / dt, "image_steps_per_s": pool / dt,
                     "window_steps_per_s": len(st.units) / dt, "halo_bytes_per_step_all_ranks": int(halo.item()),
                     "rank_pairs_exchanging": len(st.strips)}
    st1, dt1 = run(1, False, steps)
    res["single_image"] = {"units_per_rank": [len(p) for p in st1.parts], "s_per_tiled_step": dt1,
                           "tiled_steps_per_s": 1.0 / dt1,
                           "halo_bytes_per_step_rank0": int(st1.halo_bytes_per_step)}
    if world > 1:
        # the same lists on rank 0 alone (one timed step each), for the speed-up of the sharded run
        if rank == 0:
            _, solo_pool = run(pool, True, 1)
            _, solo_one = run(1, True, 1)
            res["pooled"]["s_per_tiled_step_rank0_alone"] = solo_pool
            res["pooled"]["speedup_vs_rank0_alone"] = solo_pool / dt
            res["single_image"]["s_per_tiled_step_rank0_alone"] = solo_one
            res["single_image"]["speedup_vs_rank0_alone"] = solo_one / dt1
        barrier()
    return res


# ------------------------------------------------------------------------------------------------
# BASELINE config 5 sample: infer_dir-style images sharded i mod N
# ------------------------------------------------------------------------------------------------
def images_block(wrapper, dev, rank: int, world: int, per_rank: int, upscale: int = 8):
    import torch.distributed as dist
    from b200sr import colorfix, sr3, vae
    from b200sr.driver import RestorationPipeline, run_sharded
    from oracle import configs, weights

    net = sr3.UNet(**configs.SR3_UNET).eval()
    weights.fill_(net.state_dict(), 0)
    diff = sr3.GaussianDiffusion(net.to(dev), image_size=configs.SR3_UNET["image_size"], channels=3, conditional=True)
    diff.set_new_noise_schedule(dict(configs.SR3_SCHEDULE, schedule="linear"), device=dev)
    ae = vae.AutoencoderKLInferenceWrapper(configs.VAE_EMBED_DIM, dict(configs.VAE_DDCONFIG)).add_denoise_encoder().eval()
    weights.fill_(ae.state_dict(), 0)
    pipe = RestorationPipeline(wrapper, diff, first_stage=vae.FirstStage(ae.to(dev)), device=dev,
                               color_fix=colorfix.wavelet_reconstruction, upscale=upscale)
    lr = 1024 // upscale
    n = per_rank * world
    g = torch.Generator().manual_seed(555)
    images = [torch.rand(1, 3, lr, lr, generator=g) * 2 - 1 for _ in range(n)]
    caps = [tuple({"crossattn": torch.randn(1, 77, 2048, generator=g), "vector": torch.randn(1, 2816, generator=g)}
                  for _ in range(2)) for _ in range(n)]
    run_sharded(pipe, images[:world], caps[:world], rank, world)       # warm-up: one image per rank (graph capture)
    pipe.timings.clear()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    r = run_sharded(pipe, images, caps, rank, world)
    t = torch.tensor([r["seconds"]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = t.item()
    k = max(1, len(r["indices"]))
    pipe.engine.close()
    return {"images": n, "images_per_rank": per_rank, "seconds": sec, "images_per_s": n / sec,
            "what": f"{lr}^2 -> 1024^2: bicubic x{upscale}, SR3 stage 1 (50 ancestral steps at 1024^2), VAE encode, 50 stage-2 steps "
                    "with the first-block cache (img_threshold 0.3), VAE decode, wavelet colour fix, uint8 pack; image i "
                    "on rank i mod N",
            "first_stage": pipe.first_stage.name if hasattr(pipe.first_stage, "name") else type(pipe.first_stage).__name__,
            "rank0_seconds_per_image": {kk: v / k for kk, v in pipe.timings.items()},
            "rank0_cache_misses_per_image": r["misses"]}


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each tensor whole as out_dir/<name>.npy in float32 (the step's latent is 1x4x128x128: 256 KB)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().to("cpu", torch.float32).numpy())


# ------------------------------------------------------------------------------------------------
# this framework
# ------------------------------------------------------------------------------------------------
def run_b200(args, rank: int, world: int, local_rank: int):
    import torch.distributed as dist
    from b200sr import modules, ops
    from b200sr.sampling import Stage2Engine
    from oracle import configs, inputs, weights  # weights/inputs only: seeded random init + synthetic conditioning

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    wrapper = modules.build_stage2(configs.STAGE2_UNET, configs.STAGE2_CONTROL).eval()
    weights.fill_(wrapper.state_dict(), 0)
    want_cpu = world == 1 and not args.no_cpu_baseline
    sd_cpu = {k: v.detach().clone() for k, v in wrapper.state_dict().items()} if want_cpu else None
    wrapper = wrapper.to(dev)
    x0, c, uc = inputs.stage2_inputs(latent=LATENT, seed=1234 + rank)
    eng = Stage2Engine(wrapper, use_graphs=not args.no_graphs, device=dev)
    c_dev, uc_dev = {k: v.to(dev) for k, v in c.items()}, {k: v.to(dev) for k, v in uc.items()}
    eng.set_condition(c_dev, uc_dev)
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    noise_host = torch.randn(x0.shape, generator=g).pin_memory()
    x_host = x0.clone().pin_memory()
    out_host = torch.empty_like(x_host).pin_memory()
    x, noise = x_host.to(dev), noise_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_i = 3  # a mid-schedule step (sigma ~ 9.6); every step does identical work
    for _ in range(max(args.warmup, 3)):
        eng.step(x, step_i, noise, 0.0, copy_out=False)
    launches = eng.launches.get("full", 0) + 1   # + the step loader kernel outside the graph

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # ---- device-resident timing --------------------------------------------------------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out, _ = eng.step(x, step_i, noise, 0.0, copy_out=False)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs and rank == 0:
        # `out` is the engine's output buffer, which the next step overwrites: copy it out now
        dump_outputs(args.dump_outputs, {"x_next": out})
    # ---- end-to-end timing: host buffers, H2D + D2H inside the timed region ----------------------
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        xd = x_host.to(dev, non_blocking=True)
        nd = noise_host.to(dev, non_blocking=True)
        out, _ = eng.step(xd, step_i, nd, 0.0, copy_out=False)
        out_host.copy_(out, non_blocking=True)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1) / args.steps
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    # ---- several latents per network call (SURVEY f1: batching > 1 image per step) ----------------------------
    batched = None
    if not args.no_batched:
        batched = {}
        for nb in (2, 4):
            xs, cs, ucs = zip(*(inputs.stage2_inputs(latent=LATENT, seed=1234 + 17 * j + rank) for j in range(nb)))
            cat = lambda ds: {k: torch.cat([d[k] for d in ds], 0).to(dev) for k in ds[0]}  # noqa: E731
            engb = Stage2Engine(wrapper, use_graphs=not args.no_graphs, device=dev)
            engb.set_condition(cat(cs), cat(ucs))
            xb = torch.cat(xs, 0).to(dev)
            nzb = torch.randn(xb.shape, device=dev)
            for _ in range(3):
                engb.step(xb, step_i, nzb, 0.0, copy_out=False)
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(max(4, args.steps // 2)):
                engb.step(xb, step_i, nzb, 0.0, copy_out=False)
            b1.record()
            barrier()
            msb = b0.elapsed_time(b1) / max(4, args.steps // 2)
            batched[f"latents_{nb}"] = {"ms_per_step": msb, "ms_per_latent_step": msb / nb,
                                        "latent_steps_per_s_per_gpu": 1000.0 * nb / msb,
                                        "tflops": nb * STEP_TFLOP / (msb * 1e-3)}
            engb.close()
            del engb
            torch.cuda.empty_cache()

    # ---- multi-GPU blocks (every rank takes part) ----------------------------------------------------
    tiled = images = None
    if not args.no_tiled:
        tiled = tiled_block(wrapper, dev, rank, world, args.tiled_pool, args.tiled_steps, args.tile_batch)
    if not args.no_images:
        images = {"x8": images_block(wrapper, dev, rank, world, args.images_per_rank, 8),
                  "x4": images_block(wrapper, dev, rank, world, 1, 4)}
    if rank != 0:
        return

    # ---- dominant-kernel roofline: per-launch CUDA-event timing of every instrumented kernel family -----
    # single-stream eager passes so that per-launch event pairs do not overlap
    eager = Stage2Engine(wrapper, use_graphs=False, device=dev, dual_stream=False, split_cfg=False)
    eager.set_condition(c_dev, uc_dev)
    eager.step(x, step_i, noise, 0.0)
    spin = int(0.10 * 1.9e9)
    # (1) whole eager step, no per-launch events: the denominator of share_of_step_time.  The GPU is kept busy
    #     (~100 ms spin) while the host enqueues the step, so kernels run back to back as they do inside the graph.
    torch.cuda.synchronize()
    torch.cuda._sleep(spin)
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    eager.step(x, step_i, noise, 0.0)
    w1.record()
    torch.cuda.synchronize()
    eager_ms = w0.elapsed_time(w1)
    # (2) the same step with an event pair around every gemm / conv / attention / GroupNorm / LayerNorm launch
    recs = []
    torch.cuda._sleep(spin)
    ops.set_profile(recs)
    eager.step(x, step_i, noise, 0.0)
    ops.set_profile(None)
    torch.cuda.synchronize()
    agg = {}
    for kind, work, a, b, _desc in recs:
        d = agg.setdefault(kind, [0.0, 0.0, 0])
        d[0] += work
        d[1] += a.elapsed_time(b)
        d[2] += 1
    pk, pk_src = peaks()
    dense = [agg.get("gemm", [0, 0, 0]), agg.get("conv3x3", [0, 0, 0])]
    dense_fl, dense_ms, dense_n = (sum(d[i] for d in dense) for i in range(3))
    achieved = dense_fl / (dense_ms * 1e-3) / 1e12 if dense_ms else 0.0
    peak = pk["bf16_tflops_sustained"]
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(tp):
        tp = os.path.join(ROOT, "profiles", "r01_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")

    def entry(k, v):
        e = {"ms": v[1], "launches": v[2]}
        if k in ("group_norm", "layer_norm"):   # work = algorithmic bytes (read + write of the activation once, bf16)
            e.update(gbytes=v[0] / 1e9, gb_per_s=v[0] / (v[1] * 1e-3) / 1e9 if v[1] else None,
                     frac_of_hbm_peak=(v[0] / (v[1] * 1e-3) / 1e9) / pk["hbm_gbs"] if v[1] else None)
        else:
            e.update(tflop=v[0] / 1e12, tflops=v[0] / (v[1] * 1e-3) / 1e12 if v[1] else None)
        return e

    timed_ms = sum(v[1] for v in agg.values())
    roofline = {"bound": "tensor", "kernel": "gemm_conv_kernel (tcgen05 GEMM + implicit-GEMM conv3x3)",
                "achieved": achieved, "peak": peak, "peak_source": f"{pk_src} bf16_tflops_sustained", "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": traffic, "launches_per_step": dense_n,
                "avg_launch_us": 1e3 * dense_ms / max(dense_n, 1),
                "share_of_step_time": dense_ms / eager_ms if eager_ms else None,
                "eager_step_ms": eager_ms, "event_timed_ms": timed_ms,
                "share_note": "dense kernel time / one whole single-stream eager step (all kernels, back to back)",
                "hbm_peak_gbs": pk["hbm_gbs"],
                "by_kind": {k: entry(k, v) for k, v in agg.items()},
                "step": {"tflop": STEP_TFLOP, "tflops": STEP_TFLOP / (ms * 1e-3), "frac_of_peak": STEP_TFLOP / (ms * 1e-3) / peak}}

    gpu_eager = None
    if world == 1 and not args.no_gpu_eager:
        eager.close()
        eng.close()
        del eager
        torch.cuda.empty_cache()
        gpu_eager = gpu_eager_baseline(wrapper, dev)

    cpu = None
    if want_cpu:
        cpu = cpu_reference(1, 0, sd_cpu)

    nbytes = x_host.numel() * 4
    line = {"metric": METRIC, "value": world * 1000.0 / ms, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD + ", fbcache off, one independent latent per GPU",
                       "l2": "no explicit flush: 7.7 GB of bf16 weights + 1.5 GB of folded cross-attention operands stream through the 126 MB L2 every step",
                       "cuda_graphs": not args.no_graphs, "tflop_per_step": STEP_TFLOP},
            "e2e": {"value": world * 1000.0 / ms_e2e, "unit": UNIT, "h2d_bytes_per_step": 2 * nbytes,
                    "d2h_bytes_per_step": nbytes, "ms_per_step": ms_e2e},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches, "clocks": clocks,
            "roofline": roofline}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if gpu_eager is not None:
        line["gpu_eager_baseline"] = gpu_eager
    if batched is not None:
        line["batched"] = dict(batched, what="the same step with 2 / 4 independent latents per network call (CFG batch 4 / 8): "
                                             "M = 4096 / 8192-row GEMMs, weights streamed once per call; rank 0's timing")
    if tiled is not None:
        line["tiled_x8"] = tiled
    if images is not None:
        line["images_per_s"] = images
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--no-tiled", action="store_true")
    ap.add_argument("--no-batched", action="store_true")
    ap.add_argument("--no-images", action="store_true")
    ap.add_argument("--tiled-pool", type=int, default=10, help="images in the pooled tiled x8 work list (9 windows each)")
    ap.add_argument("--tiled-steps", type=int, default=2, help="timed tiled sampler steps")
    ap.add_argument("--tile-batch", type=int, default=1, help="windows per network call")
    ap.add_argument("--images-per-rank", type=int, default=2, help="config-5 sample: images per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's output (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
