import os, sys, time
ROOT = "/root/repo" if os.path.isdir("/root/repo/oracle") else os.getcwd()
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "remote-sensing-vision-language-diffusion-model_b200"))
import torch
from b200sr import vae
from oracle import configs, weights
ae = vae.AutoencoderKLInferenceWrapper(configs.VAE_EMBED_DIM, dict(configs.VAE_DDCONFIG)).add_denoise_encoder().eval()
weights.fill_(ae.state_dict(), 0); ae = ae.cuda(); fs = vae.FirstStage(ae)
img = torch.rand(1, 3, 1024, 1024, device="cuda") * 2 - 1
z = fs.encode(img); x = fs.decode(z); torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(3): z = fs.encode(img)
torch.cuda.synchronize(); t1 = time.perf_counter()
for _ in range(3): x = fs.decode(z)
torch.cuda.synchronize(); t2 = time.perf_counter()
print(f"VAE encode {1e3*(t1-t0)/3:.2f} ms, decode {1e3*(t2-t1)/3:.2f} ms at 1024^2 (eager)")
