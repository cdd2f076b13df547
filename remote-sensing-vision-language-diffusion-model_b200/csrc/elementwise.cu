// b200sr — memory-bound helper kernels of the denoiser path: layout conversion at the drop-in
// boundary (NCHW fp32 <-> NHWC bf16), nearest 2x upsample, channel concat (+ControlNet add),
// SiLU, sinusoidal timestep embeddings, tiny-channel 3x3 convolutions (4->320, 320->4, 6->64,
// 64->3), the per-step sampler update and tile blend, and the first-block-cache similarity test.
//
// Reference semantics:
//   Upsample (nearest x2)                   sgm/modules/diffusionmodules/openaimodel.py:125-145
//   ZeroSFT concat / zero_conv add          models/modules/SR_modules.py:88-100
//   timestep_embedding (cos | sin)          sgm/modules/diffusionmodules/util.py:206-230
//   SR3 PositionalEncoding (sin | cos)      models/sr3_model/sr3_modules/unet.py:19-32
//   EpsScaling / DiscreteDenoiser           sgm/modules/diffusionmodules/denoiser_scaling.py:16-22, denoiser.py:67-78
//   LinearCFG / to_d / euler step           guiders.py:44-74, sampling_utils.py:39-40, sampling.py:598-621
//   tile blend                              sampling.py:753-756
//   first-block-cache similarity            models/modules/DFBCache.py:98-112
//   SR3 ancestral update                    models/sr3_model/sr3_modules/diffusion.py:142-176
#include "common.cuh"

namespace b200sr {

// ------------------------------------------------------------------------------------------
// NCHW fp32 -> NHWC bf16 (optionally scaled), and back.  32x32 smem transpose tiles over
// (C, HW) so both sides are coalesced.
// ------------------------------------------------------------------------------------------
__global__ void nchw_f32_to_nhwc_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int HW,
                                             float scale) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const float* src = x + static_cast<size_t>(n) * C * HW;
  __nv_bfloat16* dst = y + static_cast<size_t>(n) * C * HW;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pix = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && pix < HW) ? src[static_cast<size_t>(c) * HW + pix] * scale : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pix = p0 + i, c = c0 + threadIdx.x;
    if (c < C && pix < HW) dst[static_cast<size_t>(pix) * C + c] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}

// Cs = channels per pixel in the source (>= C: the first C of them are converted; convolutions to <= 4 channels run
// with their output padded to 8 channels on the tensor cores)
__global__ void nhwc_bf16_to_nchw_f32_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, int C, int Cs,
                                             int HW) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const __nv_bfloat16* src = x + static_cast<size_t>(n) * Cs * HW;
  float* dst = y + static_cast<size_t>(n) * C * HW;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pix = p0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && pix < HW) ? __bfloat162float(src[static_cast<size_t>(pix) * Cs + c]) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pix = p0 + threadIdx.x;
    if (c < C && pix < HW) dst[static_cast<size_t>(c) * HW + pix] = tile[threadIdx.x][i];
  }
}

}  // namespace b200sr

using namespace b200sr;

extern "C" int b200sr_nchw_f32_to_nhwc_bf16(const float* x, void* y, int32_t N, int32_t C, int32_t HW, float scale,
                                            void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || C <= 0 || HW <= 0) return B200SR_EINVAL;
  dim3 grid((HW + 31) / 32, (C + 31) / 32, N), block(32, 8);
  launch_k(nchw_f32_to_nhwc_bf16_kernel, dim3(grid), dim3(block), 0, stream, 1, x, reinterpret_cast<__nv_bfloat16*>(y), C, HW, scale);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}
extern "C" int b200sr_nhwc_bf16_to_nchw_f32_strided(const void* x, float* y, int32_t N, int32_t C, int32_t Cs,
                                                    int32_t HW, void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || C <= 0 || HW <= 0 || Cs < C) return B200SR_EINVAL;
  dim3 grid((HW + 31) / 32, (C + 31) / 32, N), block(32, 8);
  launch_k(nhwc_bf16_to_nchw_f32_kernel, dim3(grid), dim3(block), 0, stream, 1, reinterpret_cast<const __nv_bfloat16*>(x), y, C, Cs, HW);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}
extern "C" int b200sr_nhwc_bf16_to_nchw_f32(const void* x, float* y, int32_t N, int32_t C, int32_t HW, void* stream) {
  return b200sr_nhwc_bf16_to_nchw_f32_strided(x, y, N, C, C, HW, stream);
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// nearest 2x upsample, NHWC bf16, 16-byte vectors
// ------------------------------------------------------------------------------------------
__global__ void upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int H, int W, int C8,
                                  size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(i % C8);
    size_t t = i / C8;
    const int ow = static_cast<int>(t % (2 * W));
    t /= (2 * W);
    const int oh = static_cast<int>(t % (2 * H));
    const size_t n = t / (2 * H);
    y[i] = __ldg(x + ((n * H + (oh >> 1)) * W + (ow >> 1)) * C8 + cv);
  }
}

}  // namespace b200sr

extern "C" int b200sr_upsample2x_nhwc(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C,
                                      void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || (C % 8)) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(N) * 4 * H * W * (C / 8);
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(upsample2x_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), H, W,
                                              C / 8, total);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// out[:, :Ca] = a ; out[:, Ca:] = b (+ c)       rows of Ca / Cb channels, bf16, 16-byte vectors
// ------------------------------------------------------------------------------------------
__global__ void concat_add_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, const uint4* __restrict__ c,
                                  uint4* __restrict__ out, int Ca8, int Cb8, size_t rows) {
  pdl_launch_dependents();
  pdl_wait();
  const int Ct8 = Ca8 + Cb8;
  const size_t total = rows * Ct8;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t row = i / Ct8;
    const int cv = static_cast<int>(i - row * Ct8);
    uint4 v;
    if (cv < Ca8) {
      v = __ldg(a + row * Ca8 + cv);
    } else {
      v = __ldg(b + row * Cb8 + (cv - Ca8));
      if (c != nullptr) {
        const uint4 w = __ldg(c + row * Cb8 + (cv - Ca8));
        const uint32_t vv[4] = {v.x, v.y, v.z, v.w}, ww[4] = {w.x, w.y, w.z, w.w};
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = unpack_bf16x2(vv[j]), g = unpack_bf16x2(ww[j]);
          o[j] = pack_bf16x2(f.x + g.x, f.y + g.y);
        }
        v = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
    out[i] = v;
  }
}

}  // namespace b200sr

extern "C" int b200sr_concat_add(const void* a, int32_t Ca, const void* b, int32_t Cb, const void* c, void* out,
                                 int64_t rows, void* stream_ptr) {
  if ((a == nullptr && Ca > 0) || b == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (rows <= 0 || Ca < 0 || Cb <= 0 || (Ca % 8) || (Cb % 8)) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(rows) * ((Ca + Cb) / 8);
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(concat_add_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b),
                                              reinterpret_cast<const uint4*>(c), reinterpret_cast<uint4*>(out), Ca / 8,
                                              Cb / 8, static_cast<size_t>(rows));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// y = a + alpha * b (bf16), used for residual adds that could not be fused
// ------------------------------------------------------------------------------------------
__global__ void axpy_bf16_kernel(const __nv_bfloat162* __restrict__ a, const __nv_bfloat162* __restrict__ b,
                                 __nv_bfloat162* __restrict__ y, float alpha, size_t n2) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n2;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float2 f = __bfloat1622float2(a[i]), g = __bfloat1622float2(b[i]);
    y[i] = __floats2bfloat162_rn(f.x + alpha * g.x, f.y + alpha * g.y);
  }
}

}  // namespace b200sr

extern "C" int b200sr_axpy_bf16(const void* a, const void* b, void* y, float alpha, int64_t n, void* stream_ptr) {
  if (a == nullptr || b == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0 || (n & 1)) return B200SR_EINVAL;
  const size_t n2 = static_cast<size_t>(n) / 2;
  int grid = static_cast<int>((n2 + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(axpy_bf16_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const __nv_bfloat162*>(a),
                                             reinterpret_cast<const __nv_bfloat162*>(b),
                                             reinterpret_cast<__nv_bfloat162*>(y), alpha, n2);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// y[rows, Cpad] = [x[rows, C] | 0]: pads the latent's 4 channels to one 64-channel K chunk so the
// stem convolutions run on the tensor-core implicit-GEMM path.
// ------------------------------------------------------------------------------------------
__global__ void pad_channels_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int Cpad,
                                    size_t rows) {
  pdl_launch_dependents();
  pdl_wait();
  const int V = Cpad / 8;
  const size_t total = rows * V;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t row = i / V;
    const int c0 = static_cast<int>(i - row * V) * 8;
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (c0 + j < C) ? x[row * C + c0 + j] : __float2bfloat16(0.f);
    reinterpret_cast<uint4*>(y)[i] = *reinterpret_cast<const uint4*>(v);
  }
}

}  // namespace b200sr

extern "C" int b200sr_pad_channels(const void* x, void* y, int32_t C, int32_t Cpad, int64_t rows, void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (C <= 0 || Cpad < C || (Cpad % 8) || rows <= 0) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(rows) * (Cpad / 8);
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(pad_channels_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const __nv_bfloat16*>(x),
                                                reinterpret_cast<__nv_bfloat16*>(y), C, Cpad, static_cast<size_t>(rows));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// SiLU on a small fp32/bf16 vector (embedding path), bf16 out
// ------------------------------------------------------------------------------------------
__global__ void silu_bf16_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, size_t n) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    y[i] = __float2bfloat16(silu_f(__bfloat162float(x[i])));
}

}  // namespace b200sr

extern "C" int b200sr_silu_bf16(const void* x, void* y, int64_t n, void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0) return B200SR_EINVAL;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(silu_bf16_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const __nv_bfloat16*>(x),
                                             reinterpret_cast<__nv_bfloat16*>(y), static_cast<size_t>(n));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// sinusoidal embeddings: out[b, :] = cat(f(t*freq), g(t*freq)), freq_k = exp(-ln(max_period) k / half)
//   sin_first = 0: (cos | sin)  sgm timestep_embedding;  sin_first = 1: (sin | cos)  SR3 PositionalEncoding
// ------------------------------------------------------------------------------------------
__global__ void sinusoid_kernel(const float* __restrict__ t, __nv_bfloat16* __restrict__ out, int B, int dim,
                                float max_period, int sin_first) {
  pdl_launch_dependents();
  pdl_wait();
  const int half = dim / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half) return;
  const int b = i / half, k = i - b * half;
  const float freq = expf(-logf(max_period) * static_cast<float>(k) / static_cast<float>(half));
  const float arg = t[b] * freq;
  const float cs = cosf(arg), sn = sinf(arg);
  __nv_bfloat16* o = out + static_cast<size_t>(b) * dim;
  o[k] = __float2bfloat16(sin_first ? sn : cs);
  o[half + k] = __float2bfloat16(sin_first ? cs : sn);
  if ((dim & 1) && k == 0) o[dim - 1] = __float2bfloat16(0.f);
}

}  // namespace b200sr

extern "C" int b200sr_sinusoid_embedding(const float* t, void* out, int32_t B, int32_t dim, float max_period,
                                         int32_t sin_first, void* stream_ptr) {
  if (t == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (B <= 0 || dim < 2) return B200SR_EINVAL;
  const int total = B * (dim / 2);
  launch_k(sinusoid_kernel, dim3((total + 127) / 128), dim3(128), 0, stream, 1, t, reinterpret_cast<__nv_bfloat16*>(out), B, dim, max_period,
                                                           sin_first);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Direct 3x3 convolution (pad 1, stride 1) for tiny channel counts where an MMA tile would be
// >90 % padding: Cin <= 8 (latent / image -> features) or Cout <= 8 (features -> latent / image).
// NHWC bf16 in, weights [Cout, 3, 3, Cin] bf16, bias fp32.  Output bf16 NHWC, or fp32 NCHW when
// out_nchw_f32 (the UNet `out` conv feeds the fp32 sampler directly).
// ------------------------------------------------------------------------------------------
__global__ void conv3x3_few_in_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                      const float* __restrict__ bias, const __nv_bfloat16* __restrict__ addend,
                                      __nv_bfloat16* __restrict__ y, int N, int H, int W, int Cin, int Cout) {
  pdl_launch_dependents();
  pdl_wait();
  // one thread = one output pixel x 8 output channels; weights staged in smem as fp32
  extern __shared__ float s_w[];  // [Cout][9*Cin]
  const int K = 9 * Cin;
  for (int i = threadIdx.x; i < Cout * K; i += blockDim.x) s_w[i] = __bfloat162float(w[i]);
  __syncthreads();
  const int Co8 = Cout / 8;
  const size_t total = static_cast<size_t>(N) * H * W * Co8;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int cg = static_cast<int>(i % Co8);
    size_t t = i / Co8;
    const int ow = static_cast<int>(t % W);
    t /= W;
    const int oh = static_cast<int>(t % H);
    const size_t n = t / H;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = bias ? bias[cg * 8 + j] : 0.f;
    for (int kh = 0; kh < 3; ++kh) {
      const int ih = oh + kh - 1;
      if (ih < 0 || ih >= H) continue;
      for (int kw = 0; kw < 3; ++kw) {
        const int iw = ow + kw - 1;
        if (iw < 0 || iw >= W) continue;
        const __nv_bfloat16* px = x + ((n * H + ih) * W + iw) * Cin;
        for (int c = 0; c < Cin; ++c) {
          const float xv = __bfloat162float(px[c]);
          const int kidx = (kh * 3 + kw) * Cin + c;
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] += xv * s_w[(cg * 8 + j) * K + kidx];
        }
      }
    }
    const size_t o = (((n * H + oh) * W + ow) * Cout) + cg * 8;
    if (addend != nullptr) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(addend + o));
      const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(uu[j]);
        acc[2 * j] += f.x;
        acc[2 * j + 1] += f.y;
      }
    }
    uint4 v;
    v.x = pack_bf16x2(acc[0], acc[1]);
    v.y = pack_bf16x2(acc[2], acc[3]);
    v.z = pack_bf16x2(acc[4], acc[5]);
    v.w = pack_bf16x2(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(y + o) = v;
  }
}

template <int COUT>
__global__ void conv3x3_few_out_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                       const float* __restrict__ bias, void* __restrict__ y, int N, int H, int W,
                                       int Cin, int out_nchw_f32) {
  pdl_launch_dependents();
  pdl_wait();
  // one warp = one output pixel; lanes stride over (tap, channel-vector); warp-shuffle reduction
  const int warps_per_cta = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C8 = Cin / 8;
  const size_t total = static_cast<size_t>(N) * H * W;
  for (size_t pix = blockIdx.x * static_cast<size_t>(warps_per_cta) + warp; pix < total;
       pix += static_cast<size_t>(gridDim.x) * warps_per_cta) {
    const int ow = static_cast<int>(pix % W);
    const int oh = static_cast<int>((pix / W) % H);
    const size_t n = pix / (static_cast<size_t>(W) * H);
    float acc[COUT];
#pragma unroll
    for (int j = 0; j < COUT; ++j) acc[j] = 0.f;
    for (int idx = lane; idx < 9 * C8; idx += 32) {
      const int tap = idx / C8, cv = idx - tap * C8;
      const int kh = tap / 3, kw = tap - kh * 3;
      const int ih = oh + kh - 1, iw = ow + kw - 1;
      if (ih < 0 || ih >= H || iw < 0 || iw >= W) continue;
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + ((n * H + ih) * W + iw) * Cin) + cv);
      const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
      float xv[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(uu[j]);
        xv[2 * j] = f.x;
        xv[2 * j + 1] = f.y;
      }
#pragma unroll
      for (int co = 0; co < COUT; ++co) {
        const uint4 wv = __ldg(reinterpret_cast<const uint4*>(w + (static_cast<size_t>(co) * 9 + tap) * Cin) + cv);
        const uint32_t ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = unpack_bf16x2(ww[j]);
          acc[co] += xv[2 * j] * f.x + xv[2 * j + 1] * f.y;
        }
      }
    }
#pragma unroll
    for (int co = 0; co < COUT; ++co) acc[co] = warp_sum(acc[co]);
    if (lane == 0) {
#pragma unroll
      for (int co = 0; co < COUT; ++co) {
        const float v = acc[co] + (bias ? bias[co] : 0.f);
        if (out_nchw_f32)
          reinterpret_cast<float*>(y)[((n * COUT + co) * H + oh) * W + ow] = v;
        else
          reinterpret_cast<__nv_bfloat16*>(y)[pix * COUT + co] = __float2bfloat16(v);
      }
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_conv3x3_small(const void* x, const void* w, const float* bias, const void* addend, void* y,
                                    int32_t N, int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t out_nchw_f32,
                                    void* stream_ptr) {
  if (x == nullptr || w == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0) return B200SR_EINVAL;
  const __nv_bfloat16* xi = reinterpret_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* wi = reinterpret_cast<const __nv_bfloat16*>(w);
  if (Cin <= 8 && (Cout % 8) == 0) {
    if (out_nchw_f32) return B200SR_EINVAL;
    const size_t smem = static_cast<size_t>(Cout) * 9 * Cin * sizeof(float);
    if (smem > 96 * 1024) return B200SR_EINVAL;
    static bool attr_set[64] = {false};  // the attribute is per device
    if (first_use_on_device(attr_set))
      cudaFuncSetAttribute(conv3x3_few_in_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    const size_t total = static_cast<size_t>(N) * H * W * (Cout / 8);
    int grid = static_cast<int>((total + 255) / 256);
    if (grid > num_sms() * 4) grid = num_sms() * 4;
    launch_k(conv3x3_few_in_kernel, dim3(grid), dim3(256), smem, stream, 1, xi, wi, bias, reinterpret_cast<const __nv_bfloat16*>(addend),
                                                       reinterpret_cast<__nv_bfloat16*>(y), N, H, W, Cin, Cout);
  } else if (Cout <= 4 && (Cin % 8) == 0) {
    if (addend != nullptr) return B200SR_EINVAL;
    const size_t total = static_cast<size_t>(N) * H * W;
    int grid = static_cast<int>((total + 7) / 8);
    if (grid > num_sms() * 32) grid = num_sms() * 32;
    switch (Cout) {
      case 1: launch_k(conv3x3_few_out_kernel<1>, dim3(grid), dim3(256), 0, stream, 1, xi, wi, bias, y, N, H, W, Cin, out_nchw_f32); break;
      case 2: launch_k(conv3x3_few_out_kernel<2>, dim3(grid), dim3(256), 0, stream, 1, xi, wi, bias, y, N, H, W, Cin, out_nchw_f32); break;
      case 3: launch_k(conv3x3_few_out_kernel<3>, dim3(grid), dim3(256), 0, stream, 1, xi, wi, bias, y, N, H, W, Cin, out_nchw_f32); break;
      default: launch_k(conv3x3_few_out_kernel<4>, dim3(grid), dim3(256), 0, stream, 1, xi, wi, bias, y, N, H, W, Cin, out_nchw_f32); break;
    }
  } else {
    return B200SR_EINVAL;
  }
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Sampler step, part 1 (before the network):   sampling.py:598-606, denoiser.py:70-76, guiders.py:65-74
//   x_hat = x + noise * s_noise * sqrt(sigma_hat^2 - sigma^2)          (fp32 NCHW, kept for part 2)
//   net_in[0] = net_in[1] = x_hat * c_in,  c_in = 1/sqrt(sigma_q^2 + 1)  (bf16 NHWC, CFG batch 2)
// All per-step scalars arrive in a small device array so the launch is CUDA-graph friendly:
//   sc[0]=sigma  sc[1]=sigma_hat  sc[2]=sigma_next  sc[3]=sigma_q (quantised)  sc[4]=cfg_scale  sc[5]=s_noise
// ------------------------------------------------------------------------------------------
__global__ void sampler_pre_kernel(const float* __restrict__ x, const float* __restrict__ noise,
                                   const float* __restrict__ sc, float* __restrict__ x_hat,
                                   __nv_bfloat16* __restrict__ net_in, int B, int C, int HW, int cfg_copies) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = static_cast<size_t>(B) * C * HW;
  const float sigma = sc[0], sigma_hat = sc[1], sigma_q = sc[3], s_noise = sc[5];
  const float churn = sqrtf(fmaxf(sigma_hat * sigma_hat - sigma * sigma, 0.f)) * s_noise;
  const float c_in = rsqrtf(sigma_q * sigma_q + 1.f);
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float v = x[i];
    if (noise != nullptr) v += noise[i] * churn;
    x_hat[i] = v;
    const int pix = static_cast<int>(i % HW);
    const int c = static_cast<int>((i / HW) % C);
    const size_t b = i / (static_cast<size_t>(HW) * C);
    const __nv_bfloat16 o = __float2bfloat16(v * c_in);
    for (int k = 0; k < cfg_copies; ++k)
      net_in[((static_cast<size_t>(k) * B + b) * HW + pix) * C + c] = o;
  }
}

}  // namespace b200sr

extern "C" int b200sr_sampler_pre(const float* x, const float* noise, const float* scalars, float* x_hat, void* net_in,
                                  int32_t B, int32_t C, int32_t HW, int32_t cfg_copies, void* stream_ptr) {
  if (x == nullptr || scalars == nullptr || x_hat == nullptr || net_in == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (B <= 0 || C <= 0 || HW <= 0 || cfg_copies < 1) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(B) * C * HW;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(sampler_pre_kernel, dim3(grid), dim3(256), 0, stream, 1, x, noise, scalars, x_hat, reinterpret_cast<__nv_bfloat16*>(net_in), B, C,
                                               HW, cfg_copies);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Sampler step, part 2 (after the network):  denoiser.py:76-78, guiders.py:59-63, sampling.py:618-620
//   den_k    = eps_k * (-sigma_q) + x_hat                 k = uncond, cond   (eps: fp32 NCHW [2B,...])
//   denoised = den_u + cfg * (den_c - den_u)
//   d        = (x_hat - denoised) / sigma_hat ;  x_next = x_hat + d * (sigma_next - sigma_hat)
// Optionally accumulates the tile blend  acc[win] += x_next * w ; cnt[win] += w  (sampling.py:753-755).
// ------------------------------------------------------------------------------------------
__global__ void sampler_post_kernel(const float* __restrict__ eps, const float* __restrict__ x_hat,
                                    const float* __restrict__ sc, float* __restrict__ denoised_out,
                                    float* __restrict__ x_next, int B, int C, int HW, int use_cfg) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = static_cast<size_t>(B) * C * HW;
  const float sigma_hat = sc[1], sigma_next = sc[2], sigma_q = sc[3], cfg = sc[4];
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float xh = x_hat[i];
    float den;
    if (use_cfg) {
      const float du = eps[i] * (-sigma_q) + xh;
      const float dc = eps[total + i] * (-sigma_q) + xh;
      den = du + cfg * (dc - du);
    } else {
      den = eps[i] * (-sigma_q) + xh;
    }
    if (denoised_out != nullptr) denoised_out[i] = den;
    const float d = (xh - den) / sigma_hat;
    x_next[i] = xh + d * (sigma_next - sigma_hat);
  }
}

}  // namespace b200sr

extern "C" int b200sr_sampler_post(const float* eps, const float* x_hat, const float* scalars, float* denoised_out,
                                   float* x_next, int32_t B, int32_t C, int32_t HW, int32_t use_cfg, void* stream_ptr) {
  if (eps == nullptr || x_hat == nullptr || scalars == nullptr || x_next == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (B <= 0 || C <= 0 || HW <= 0) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(B) * C * HW;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(sampler_post_kernel, dim3(grid), dim3(256), 0, stream, 1, eps, x_hat, scalars, denoised_out, x_next, B, C, HW, use_cfg);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// Euler update from an already guided `denoised` (cache-hit path reuses the previous one).
__global__ void euler_from_denoised_kernel(const float* __restrict__ den, const float* __restrict__ x_hat,
                                           const float* __restrict__ sc, float* __restrict__ x_next, size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  const float sigma_hat = sc[1], sigma_next = sc[2];
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float xh = x_hat[i];
    const float d = (xh - den[i]) / sigma_hat;
    x_next[i] = xh + d * (sigma_next - sigma_hat);
  }
}

}  // namespace b200sr

extern "C" int b200sr_euler_from_denoised(const float* denoised, const float* x_hat, const float* scalars, float* x_next,
                                          int64_t n, void* stream_ptr) {
  if (denoised == nullptr || x_hat == nullptr || scalars == nullptr || x_next == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0) return B200SR_EINVAL;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(euler_from_denoised_kernel, dim3(grid), dim3(256), 0, stream, 1, denoised, x_hat, scalars, x_next, static_cast<size_t>(n));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Tile blend (sampling.py:753-756): acc[:, :, h0:h0+th, w0:w0+tw] += tile * weight ; cnt += weight
// and the final acc / cnt.  fp32 NCHW.  `weight` is [th, tw].
// ------------------------------------------------------------------------------------------
__global__ void tile_accumulate_kernel(const float* __restrict__ tile, const float* __restrict__ weight,
                                       float* __restrict__ acc, float* __restrict__ cnt, int BC, int th, int tw, int H,
                                       int W, int h0, int w0) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = static_cast<size_t>(BC) * th * tw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % tw);
    const int y = static_cast<int>((i / tw) % th);
    const size_t bc = i / (static_cast<size_t>(tw) * th);
    const float wgt = weight[y * tw + x];
    const size_t o = (bc * H + (h0 + y)) * W + (w0 + x);
    // explicit round-to-nearest multiply then add (no FMA contraction): a rank that ships the weighted strip
    // tile * w to the window's owner, which adds it, must produce the same bits as this local accumulation
    acc[o] = __fadd_rn(acc[o], __fmul_rn(tile[i], wgt));
    if (cnt != nullptr) cnt[o] += wgt;
  }
}
__global__ void tile_normalize_kernel(const float* __restrict__ acc, const float* __restrict__ cnt,
                                      float* __restrict__ out, size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    out[i] = acc[i] / cnt[i];
}

}  // namespace b200sr

extern "C" int b200sr_tile_accumulate(const float* tile, const float* weight, float* acc, float* cnt, int32_t BC,
                                      int32_t th, int32_t tw, int32_t H, int32_t W, int32_t h0, int32_t w0,
                                      void* stream_ptr) {
  if (tile == nullptr || weight == nullptr || acc == nullptr) return B200SR_EINVAL;  // cnt may be NULL
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (BC <= 0 || th <= 0 || tw <= 0 || h0 < 0 || w0 < 0 || h0 + th > H || w0 + tw > W) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(BC) * th * tw;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(tile_accumulate_kernel, dim3(grid), dim3(256), 0, stream, 1, tile, weight, acc, cnt, BC, th, tw, H, W, h0, w0);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}
extern "C" int b200sr_tile_normalize(const float* acc, const float* cnt, float* out, int64_t n, void* stream_ptr) {
  if (acc == nullptr || cnt == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0) return B200SR_EINVAL;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(tile_normalize_kernel, dim3(grid), dim3(256), 0, stream, 1, acc, cnt, out, static_cast<size_t>(n));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// First-block-cache similarity (DFBCache.py:98-112):
//   out[0] = sum|prev - cur|, out[1] = sum|prev|  (fp32 block partials, fp64 final atomics)
//   finalize: diff = (s0/n) / (s1/n + 1e-6);  result[0] = diff, result[1] = (diff < thr)
// ------------------------------------------------------------------------------------------
__global__ void rel_l1_partial_kernel(const __nv_bfloat16* __restrict__ prev, const __nv_bfloat16* __restrict__ cur,
                                      double* __restrict__ sums, size_t n8) {
  pdl_launch_dependents();
  pdl_wait();
  float a = 0.f, b = 0.f;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(prev) + i);
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(cur) + i);
    const uint32_t uu[4] = {u.x, u.y, u.z, u.w}, vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_bf16x2(uu[j]), g = unpack_bf16x2(vv[j]);
      a += fabsf(f.x - g.x) + fabsf(f.y - g.y);
      b += fabsf(f.x) + fabsf(f.y);
    }
  }
  a = warp_sum(a);
  b = warp_sum(b);
  __shared__ float sa[32], sb[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sa[warp] = a;
    sb[warp] = b;
  }
  __syncthreads();
  if (warp == 0) {
    a = lane < (blockDim.x >> 5) ? sa[lane] : 0.f;
    b = lane < (blockDim.x >> 5) ? sb[lane] : 0.f;
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) {
      atomicAdd(&sums[0], static_cast<double>(a));
      atomicAdd(&sums[1], static_cast<double>(b));
    }
  }
}
__global__ void rel_l1_finalize_kernel(double* __restrict__ sums, const float* __restrict__ threshold,
                                       float* __restrict__ result, double n) {
  pdl_launch_dependents();
  pdl_wait();
  const double mean_diff = sums[0] / n, mean_prev = sums[1] / n;
  const float diff = static_cast<float>(mean_diff / (mean_prev + 1e-6));
  result[0] = diff;
  result[1] = diff < threshold[0] ? 1.f : 0.f;
  sums[0] = 0.0;
  sums[1] = 0.0;
}

}  // namespace b200sr

// workspace: 2 doubles, zero on first use (re-zeroed by the finalize kernel)
extern "C" int b200sr_rel_l1_similarity(const void* prev, const void* cur, int64_t n, const float* threshold,
                                        void* workspace_ptr, float* result, void* stream_ptr) {
  if (prev == nullptr || cur == nullptr || threshold == nullptr || workspace_ptr == nullptr || result == nullptr)
    return B200SR_EINVAL;
  double* workspace = static_cast<double*>(workspace_ptr);
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0 || (n % 8)) return B200SR_EINVAL;
  const size_t n8 = static_cast<size_t>(n) / 8;
  int grid = static_cast<int>((n8 + 255) / 256);
  if (grid > num_sms() * 4) grid = num_sms() * 4;
  launch_k(rel_l1_partial_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const __nv_bfloat16*>(prev),
                                                  reinterpret_cast<const __nv_bfloat16*>(cur), workspace, n8);
  launch_k(rel_l1_finalize_kernel, dim3(1), dim3(1), 0, stream, 1, workspace, threshold, result, static_cast<double>(n));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// SR3 ancestral DDPM update (diffusion.py:142-176), fp32 NCHW:
//   x0 = clamp(c_recip * x - c_recipm1 * eps, -1, 1);  mean = coef1 * x0 + coef2 * x
//   x  = mean + noise * exp(0.5 * logvar)            (noise == nullptr on the last step)
//   sc = {sqrt_recip_ac, sqrt_recipm1_ac, coef1, coef2, logvar}
// ------------------------------------------------------------------------------------------
__global__ void sr3_update_kernel(const float* __restrict__ x, const float* __restrict__ eps,
                                  const float* __restrict__ noise, const float* __restrict__ sc, float* __restrict__ out,
                                  size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  const float cr = sc[0], crm1 = sc[1], c1 = sc[2], c2 = sc[3], std = expf(0.5f * sc[4]);
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float xv = x[i];
    float x0 = cr * xv - crm1 * eps[i];
    x0 = fminf(fmaxf(x0, -1.f), 1.f);
    float v = c1 * x0 + c2 * xv;
    if (noise != nullptr) v += noise[i] * std;
    out[i] = v;
  }
}

}  // namespace b200sr

extern "C" int b200sr_sr3_update(const float* x, const float* eps, const float* noise, const float* scalars, float* out,
                                 int64_t n, void* stream_ptr) {
  if (x == nullptr || eps == nullptr || scalars == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0) return B200SR_EINVAL;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(sr3_update_kernel, dim3(grid), dim3(256), 0, stream, 1, x, eps, noise, scalars, out, static_cast<size_t>(n));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Batched small device-to-device copies in ONE launch (per-step loader of the sampler engine: latent, noise,
// the step's row of the scalar table and of the precomputed embedding projections -> the static buffers a
// captured CUDA graph reads).  Each copy is 4-byte granular; 16-byte vectors when both ends allow it.
// ------------------------------------------------------------------------------------------
struct CopyBatchArgs {
  const void* src[B200SR_MAX_COPIES];
  void* dst[B200SR_MAX_COPIES];
  long long bytes[B200SR_MAX_COPIES];
};
__global__ void copy_batch_kernel(const CopyBatchArgs a) {
  pdl_launch_dependents();
  pdl_wait();
  const int k = blockIdx.y;
  const long long nbytes = a.bytes[k];
  const uintptr_t s = reinterpret_cast<uintptr_t>(a.src[k]), d = reinterpret_cast<uintptr_t>(a.dst[k]);
  const size_t tid = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  const size_t nth = static_cast<size_t>(gridDim.x) * blockDim.x;
  if (((s | d | static_cast<uintptr_t>(nbytes)) & 15) == 0) {
    const uint4* sp = reinterpret_cast<const uint4*>(s);
    uint4* dp = reinterpret_cast<uint4*>(d);
    for (size_t i = tid; i < static_cast<size_t>(nbytes >> 4); i += nth) dp[i] = sp[i];
  } else {
    const uint32_t* sp = reinterpret_cast<const uint32_t*>(s);
    uint32_t* dp = reinterpret_cast<uint32_t*>(d);
    for (size_t i = tid; i < static_cast<size_t>(nbytes >> 2); i += nth) dp[i] = sp[i];
  }
}

}  // namespace b200sr

extern "C" int b200sr_copy_batch(const b200sr_copy* copies, int32_t n, void* stream_ptr) {
  if (copies == nullptr || n <= 0 || n > B200SR_MAX_COPIES) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  CopyBatchArgs a;
  long long mx = 0;
  for (int i = 0; i < n; ++i) {
    const b200sr_copy& c = copies[i];
    if (c.src == nullptr || c.dst == nullptr || c.bytes <= 0 || (c.bytes & 3) || (reinterpret_cast<uintptr_t>(c.src) & 3) ||
        (reinterpret_cast<uintptr_t>(c.dst) & 3))
      return B200SR_EINVAL;
    a.src[i] = c.src;
    a.dst[i] = c.dst;
    a.bytes[i] = c.bytes;
    if (c.bytes > mx) mx = c.bytes;
  }
  int gx = static_cast<int>((mx / 16 + 255) / 256);
  if (gx < 1) gx = 1;
  if (gx > num_sms() * 4) gx = num_sms() * 4;
  launch_k(copy_batch_kernel, dim3(gx, n), dim3(256), 0, stream, 1, a);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Tile-sharded blend, halo side (sampling.py:753-756 across GPUs): strip = tile[:, y0:y0+sh, x0:x0+sw] * weight
// (the same round-to-nearest product tile_accumulate forms), packed contiguously for the peer that owns an
// overlapping window; and acc[:, h0:h0+sh, w0:w0+sw] += strip on the receiving side.
// ------------------------------------------------------------------------------------------
__global__ void tile_weighted_strip_kernel(const float* __restrict__ tile, const float* __restrict__ weight,
                                           float* __restrict__ strip, int BC, int th, int tw, int y0, int x0, int sh,
                                           int sw) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = static_cast<size_t>(BC) * sh * sw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % sw);
    const int y = static_cast<int>((i / sw) % sh);
    const size_t bc = i / (static_cast<size_t>(sw) * sh);
    strip[i] = __fmul_rn(tile[(bc * th + (y0 + y)) * tw + (x0 + x)], weight[(y0 + y) * tw + (x0 + x)]);
  }
}
__global__ void strip_add_kernel(const float* __restrict__ strip, float* __restrict__ acc, int BC, int sh, int sw, int H,
                                 int W, int h0, int w0) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = static_cast<size_t>(BC) * sh * sw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % sw);
    const int y = static_cast<int>((i / sw) % sh);
    const size_t bc = i / (static_cast<size_t>(sw) * sh);
    const size_t o = (bc * H + (h0 + y)) * W + (w0 + x);
    acc[o] = __fadd_rn(acc[o], strip[i]);
  }
}

}  // namespace b200sr

extern "C" int b200sr_tile_weighted_strip(const float* tile, const float* weight, float* strip, int32_t BC, int32_t th,
                                          int32_t tw, int32_t y0, int32_t x0, int32_t sh, int32_t sw, void* stream_ptr) {
  if (tile == nullptr || weight == nullptr || strip == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (BC <= 0 || sh <= 0 || sw <= 0 || y0 < 0 || x0 < 0 || y0 + sh > th || x0 + sw > tw) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(BC) * sh * sw;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(tile_weighted_strip_kernel, dim3(grid), dim3(256), 0, stream, 1, tile, weight, strip, BC, th, tw, y0, x0, sh, sw);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}
extern "C" int b200sr_strip_add(const float* strip, float* acc, int32_t BC, int32_t sh, int32_t sw, int32_t H, int32_t W,
                                int32_t h0, int32_t w0, void* stream_ptr) {
  if (strip == nullptr || acc == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (BC <= 0 || sh <= 0 || sw <= 0 || h0 < 0 || w0 < 0 || h0 + sh > H || w0 + sw > W) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(BC) * sh * sw;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(strip_add_kernel, dim3(grid), dim3(256), 0, stream, 1, strip, acc, BC, sh, sw, H, W, h0, w0);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// First-stage (SDXL VAE) glue around the latent: 1x1 convolutions between <= 8 channels
//   quant_conv 8 -> 8 and post_quant_conv 4 -> 4            sgm/models/autoencoder.py:298-299, :305-318
// one thread per pixel, weights in shared memory, fp32 math; bf16 NHWC in, bf16 NHWC or fp32 NCHW (x scale) out;
// and DiagonalGaussianDistribution.sample / .mode        sgm/modules/distributions/distributions.py (mean | logvar
// halves of the moments, logvar clamped to [-30, 20], z = mean + exp(0.5 logvar) * noise), times scale_factor
// (models/SR_model.py:58-78).
// ------------------------------------------------------------------------------------------
__global__ void pointwise_small_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                                       const float* __restrict__ bias, void* __restrict__ y, int Cin, int Cout,
                                       long long rows, int HW, int out_nchw_f32, float scale) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_w[64], s_b[8];
  if (threadIdx.x < Cin * Cout) s_w[threadIdx.x] = w[threadIdx.x];
  if (threadIdx.x < Cout) s_b[threadIdx.x] = bias != nullptr ? bias[threadIdx.x] : 0.f;
  __syncthreads();
  for (long long r = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; r < rows;
       r += static_cast<long long>(gridDim.x) * blockDim.x) {
    float xv[8], acc[8];
    for (int c = 0; c < Cin; ++c) xv[c] = __bfloat162float(x[r * Cin + c]);
    for (int o = 0; o < Cout; ++o) {
      float a = s_b[o];
      for (int c = 0; c < Cin; ++c) a = fmaf(xv[c], s_w[o * Cin + c], a);
      acc[o] = a * scale;
    }
    if (out_nchw_f32) {
      const long long n = r / HW, pix = r - n * HW;
      for (int o = 0; o < Cout; ++o) reinterpret_cast<float*>(y)[(n * Cout + o) * HW + pix] = acc[o];
    } else {
      for (int o = 0; o < Cout; ++o) reinterpret_cast<__nv_bfloat16*>(y)[r * Cout + o] = __float2bfloat16(acc[o]);
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_pointwise_small(const void* x, const float* w, const float* bias, void* y, int32_t Cin, int32_t Cout,
                                      int64_t rows, int32_t HW, int32_t out_nchw_f32, float scale, void* stream_ptr) {
  if (x == nullptr || w == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (Cin <= 0 || Cin > 8 || Cout <= 0 || Cout > 8 || rows <= 0 || HW <= 0 || (rows % HW) != 0) return B200SR_EINVAL;
  int grid = static_cast<int>((rows + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(pointwise_small_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const __nv_bfloat16*>(x), w, bias, y, Cin,
           Cout, rows, HW, out_nchw_f32, scale);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

__global__ void diag_gaussian_kernel(const float* __restrict__ moments, const float* __restrict__ noise,
                                     float* __restrict__ z, int C, int HW, long long total, float scale) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = i / (static_cast<long long>(C) * HW), rem = i - n * C * HW;
    const float mean = moments[n * 2 * C * HW + rem];
    float v = mean;
    if (noise != nullptr) {
      const float logvar = fminf(fmaxf(moments[n * 2 * C * HW + static_cast<long long>(C) * HW + rem], -30.f), 20.f);
      v = mean + expf(0.5f * logvar) * noise[i];
    }
    z[i] = v * scale;
  }
}

}  // namespace b200sr

extern "C" int b200sr_diag_gaussian(const float* moments, const float* noise, float* z, int32_t N, int32_t C, int32_t HW,
                                    float scale, void* stream_ptr) {
  if (moments == nullptr || z == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || C <= 0 || HW <= 0) return B200SR_EINVAL;
  const long long total = static_cast<long long>(N) * C * HW;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(diag_gaussian_kernel, dim3(grid), dim3(256), 0, stream, 1, moments, noise, z, C, HW, total, scale);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Token + position embedding of the text towers (transformers CLIPTextEmbeddings; open_clip
// model.token_embedding(text) + model.positional_embedding, sgm/modules/encoders/modules.py:569-571):
//   out[b, t, :] = tok[ids[b, t], :] + pos[t, :]      fp32 tables -> bf16 tokens
// ------------------------------------------------------------------------------------------
__global__ void embed_tokens_kernel(const long long* __restrict__ ids, const float* __restrict__ tok,
                                    const float* __restrict__ pos, __nv_bfloat16* __restrict__ out, int T, int C,
                                    int vocab, size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const size_t bt = i / C;
    const int t = static_cast<int>(bt % T);
    long long id = ids[bt];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    out[i] = __float2bfloat16(tok[static_cast<size_t>(id) * C + c] + pos[static_cast<size_t>(t) * C + c]);
  }
}

}  // namespace b200sr

extern "C" int b200sr_embed_tokens(const int64_t* ids, const float* tok, const float* pos, void* out, int32_t B, int32_t T,
                                   int32_t C, int32_t vocab, void* stream_ptr) {
  if (ids == nullptr || tok == nullptr || pos == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (B <= 0 || T <= 0 || C <= 0 || vocab <= 0) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(B) * T * C;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  launch_k(embed_tokens_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const long long*>(ids), tok, pos, reinterpret_cast<__nv_bfloat16*>(out), T, C,
           vocab, total);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}
