"""Times the stage-1 -> stage-2 hand-off (tensor2img + PIL2Tensor) at a 600^2 stage-1 image (WHU-RS19) -> 1024^2: the
device path (b200sr.colorfix.tensor2img_u8 + pil_to_tensor, CUDA events over many calls) against the reference's host path
(device -> host copy, numpy tensor2img, PIL.Image.resize, float64 conversion, host -> device copy).  Prints one JSON line
with the GPU's name and power limit beside the numbers.

    python tools/handoff_bench.py [--size 600] [--min-size 1024] [--iters 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200"), os.path.join(ROOT, "tests")]

import torch  # noqa: E402
from PIL import Image  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=600)
    ap.add_argument("--min-size", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("handoff_bench.py needs a CUDA device")
    import imageio_ref as R
    from b200sr import colorfix

    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(1, 3, a.size, a.size, generator=g, device="cuda") * 2 - 1

    def device_path():
        return colorfix.pil_to_tensor(colorfix.tensor2img_u8(x), min_size=a.min_size)[0]

    def host_path():
        y, _, _ = R.pil2tensor(Image.fromarray(R.tensor2img(x)), min_size=a.min_size)
        return y.unsqueeze(0).cuda()

    out_d, out_h = device_path(), host_path()
    torch.cuda.synchronize()
    assert torch.equal(out_d, out_h), "device and host hand-off differ"
    for _ in range(10):
        device_path()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(a.iters):
        device_path()
    t1.record()
    torch.cuda.synchronize()
    dev_ms = t0.elapsed_time(t1) / a.iters
    n_host = max(a.iters // 20, 3)
    host_path()
    torch.cuda.synchronize()
    s = time.perf_counter()
    for _ in range(n_host):
        host_path()
    torch.cuda.synchronize()
    host_ms = (time.perf_counter() - s) * 1e3 / n_host
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"stage1": a.size, "stage2": list(out_d.shape[-2:]), "device_ms": round(dev_ms, 4),
                      "host_pillow_ms": round(host_ms, 3), "iters": a.iters, "host_iters": n_host, "gpu": smi}))


if __name__ == "__main__":
    main()
