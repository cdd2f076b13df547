// b200sr — output side of the restoration pipeline (SURVEY.md section 8(f) row f3): wavelet colour fix and the
// bicubic resize + uint8 pack of Tensor2PIL.  fp32 NCHW images, memory-bound elementwise / stencil kernels.
//
// Reference semantics:
//   wavelet_blur / wavelet_decomposition / wavelet_reconstruction     utils/colorfix.py:73-119
//     blur = depthwise 3x3 [1 2 1; 2 4 2; 1 2 1] / 16 with dilation r = 2^level, replicate padding r;
//     high += image - low; image = low (5 levels); result = content_high + style_low
//   Tensor2PIL                                                         models/util.py:159-166
//     F.interpolate(size = (h0, w0), mode = "bicubic") (align_corners False, A = -0.75, clamped taps),
//     x * 127.5 + 127.5, clip to [0, 255], truncate to uint8, HWC
//   tensor2img (stage-1 output -> uint8)                              infer.py:133-138, utils/tensor2img.py:4-21
//     (clamp(x, -1, 1) + 1) / 2, * 255, round half to even, uint8 HWC
//   PIL2Tensor                                                         models/util.py:132-156
//     Image.resize((w, h), Image.BICUBIC): Pillow's two-pass 8-bit resample (a = -0.5, antialiased when reducing,
//     22-bit fixed point); then x / 255 * 2 - 1 in float64, cast to fp32, CHW
#include "common.cuh"

namespace b200sr {

__global__ void wavelet_level_kernel(const float* __restrict__ img, float* __restrict__ low, float* __restrict__ high,
                                     int first, int H, int W, int r, size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % W);
    const int y = static_cast<int>((i / W) % H);
    const float* plane = img + (i / (static_cast<size_t>(W) * H)) * static_cast<size_t>(W) * H;
    const int ym = max(y - r, 0), yp = min(y + r, H - 1), xm = max(x - r, 0), xp = min(x + r, W - 1);
    const float* r0 = plane + static_cast<size_t>(ym) * W;
    const float* r1 = plane + static_cast<size_t>(y) * W;
    const float* r2 = plane + static_cast<size_t>(yp) * W;
    // same tap order as a row-major 3x3 kernel
    float l = 0.0625f * r0[xm];
    l = fmaf(0.125f, r0[x], l);
    l = fmaf(0.0625f, r0[xp], l);
    l = fmaf(0.125f, r1[xm], l);
    l = fmaf(0.25f, r1[x], l);
    l = fmaf(0.125f, r1[xp], l);
    l = fmaf(0.0625f, r2[xm], l);
    l = fmaf(0.125f, r2[x], l);
    l = fmaf(0.0625f, r2[xp], l);
    low[i] = l;
    if (high != nullptr) high[i] = (first ? 0.f : high[i]) + (r1[x] - l);
  }
}

}  // namespace b200sr

using namespace b200sr;

extern "C" int b200sr_wavelet_level(const float* img, float* low, float* high, int32_t first, int32_t BC, int32_t H,
                                    int32_t W, int32_t radius, void* stream_ptr) {
  if (img == nullptr || low == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (BC <= 0 || H <= 0 || W <= 0 || radius <= 0 || img == low) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(BC) * H * W;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(wavelet_level_kernel, dim3(grid), dim3(256), 0, stream, 1, img, low, high, first, H, W, radius, total);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

__global__ void add_f32_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                               size_t n) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    out[i] = a[i] + b[i];
}

}  // namespace b200sr

extern "C" int b200sr_add_f32(const float* a, const float* b, float* out, int64_t n, void* stream_ptr) {
  if (a == nullptr || b == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (n <= 0) return B200SR_EINVAL;
  int grid = static_cast<int>((n + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(add_f32_kernel, dim3(grid), dim3(256), 0, stream, 1, a, b, out, static_cast<size_t>(n));
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// cubic convolution coefficients of torch's upsample_bicubic2d (A = -0.75)
__device__ __forceinline__ void cubic_coeffs(float t, float (&c)[4]) {
  const float A = -0.75f;
  const float x0 = t + 1.f, x1 = t, x2 = 1.f - t, x3 = 2.f - t;
  c[0] = ((A * x0 - 5.f * A) * x0 + 8.f * A) * x0 - 4.f * A;
  c[1] = ((A + 2.f) * x1 - (A + 3.f)) * x1 * x1 + 1.f;
  c[2] = ((A + 2.f) * x2 - (A + 3.f)) * x2 * x2 + 1.f;
  c[3] = ((A * x3 - 5.f * A) * x3 + 8.f * A) * x3 - 4.f * A;
}

__global__ void image_to_u8_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, int C, int H, int W, int OH,
                                   int OW, float sh, float sw) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = static_cast<size_t>(OH) * OW;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(i % OW), oy = static_cast<int>(i / OW);
    const float ry = sh * (oy + 0.5f) - 0.5f, rx = sw * (ox + 0.5f) - 0.5f;
    const int iy = static_cast<int>(floorf(ry)), ix = static_cast<int>(floorf(rx));
    float cy[4], cx[4];
    cubic_coeffs(ry - iy, cy);
    cubic_coeffs(rx - ix, cx);
    for (int c = 0; c < C; ++c) {
      const float* plane = x + static_cast<size_t>(c) * H * W;
      float v = 0.f;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float* row = plane + static_cast<size_t>(min(max(iy - 1 + a, 0), H - 1)) * W;
        float rv = 0.f;
#pragma unroll
        for (int b = 0; b < 4; ++b) rv += cx[b] * row[min(max(ix - 1 + b, 0), W - 1)];
        v += cy[a] * rv;
      }
      v = fminf(fmaxf(v * 127.5f + 127.5f, 0.f), 255.f);
      out[i * C + c] = static_cast<uint8_t>(v);   // truncation, as numpy's astype(uint8) on a clipped float
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_image_to_u8(const float* x, void* out, int32_t C, int32_t H, int32_t W, int32_t OH, int32_t OW,
                                  void* stream_ptr) {
  if (x == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (C <= 0 || C > 4 || H <= 0 || W <= 0 || OH <= 0 || OW <= 0) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(OH) * OW;
  int grid = static_cast<int>((total + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  launch_k(image_to_u8_kernel, dim3(grid), dim3(256), 0, stream, 1, x, reinterpret_cast<uint8_t*>(out), C, H, W, OH, OW,
           static_cast<float>(H) / OH, static_cast<float>(W) / OW);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ---- stage-1 -> stage-2 hand-off (infer.py:133-138, models/util.py:132-156) -------------------------------------------
static int grid_for(size_t work) {
  int grid = static_cast<int>((work + 255) / 256);
  if (grid > num_sms() * 16) grid = num_sms() * 16;
  return grid < 1 ? 1 : grid;
}

// tensor2img (utils/tensor2img.py:4-21): t = (clamp(x, -1, 1) + 1) / 2 in fp32, rint(t * 255) in fp32 (numpy .round()
// is round-half-to-even), uint8 HWC.  Each thread converts 4 pixels: one 16-byte load per plane.
__global__ void tensor2img_u8_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, int C, size_t HW,
                                     bool vec) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t quads = (HW + 3) / 4;
  for (size_t q = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; q < quads;
       q += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p0 = q * 4;
    for (int c = 0; c < C; ++c) {
      const float* plane = x + static_cast<size_t>(c) * HW;
      float v[4];
      if (vec) {
        const float4 f = *reinterpret_cast<const float4*>(plane + p0);
        v[0] = f.x, v[1] = f.y, v[2] = f.z, v[3] = f.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = p0 + j < HW ? plane[p0 + j] : 0.f;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (p0 + j >= HW) break;
        const float t = __fmul_rn(__fadd_rn(fminf(fmaxf(v[j], -1.f), 1.f), 1.f), 0.5f);  // exact halving = / 2
        out[(p0 + j) * C + c] = static_cast<uint8_t>(rintf(__fmul_rn(t, 255.f)));
      }
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_tensor2img_u8(const float* x, void* out, int32_t C, int32_t H, int32_t W, void* stream_ptr) {
  if (x == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (C <= 0 || C > 4 || H <= 0 || W <= 0) return B200SR_EINVAL;
  const size_t HW = static_cast<size_t>(H) * W;
  const bool vec = HW % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  launch_k(tensor2img_u8_kernel, dim3(grid_for((HW + 3) / 4)), dim3(256), 0, stream, 1, x,
           reinterpret_cast<uint8_t*>(out), C, HW, vec);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// One axis of Pillow's 8-bit resample (libImaging/Resample.c ImagingResampleHorizontal_8bpc / ..Vertical_8bpc) over
// src viewed as [outer, in_len, inner] bytes -> dst [outer, out_len, inner]: the horizontal pass of an HWC image is
// (outer, inner) = (H, C), the vertical pass (1, W * C).  Output o reads taps bounds[2o] .. bounds[2o] + bounds[2o+1] - 1
// with the int32 fixed-point coefficients coeffs[o * ksize + k] (22 fractional bits):
//   acc = 2^21 + sum_k src * coeff, out = clamp(acc >> 22, 0, 255).
// Each thread produces 16 consecutive output bytes and stores them with one 16-byte store when they are aligned.
constexpr int kResamplePB = 22;
__global__ void resample_u8_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int in_len, int out_len,
                                   int inner, const int* __restrict__ bounds, const int* __restrict__ coeffs, int ksize,
                                   size_t total, bool aligned) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t per_outer = static_cast<size_t>(out_len) * inner;
  const size_t chunks = (total + 15) / 16;
  for (size_t q = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; q < chunks;
       q += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t i0 = q * 16;
    alignas(16) uint8_t r[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const size_t i = i0 + j;
      r[j] = 0;
      if (i < total) {
        const size_t b = i / per_outer, rem = i - b * per_outer;
        const int o = static_cast<int>(rem / inner), e = static_cast<int>(rem - static_cast<size_t>(o) * inner);
        const int xmin = __ldg(bounds + 2 * o), n = __ldg(bounds + 2 * o + 1);
        const uint8_t* s = src + (b * in_len + xmin) * static_cast<size_t>(inner) + e;
        const int* k = coeffs + static_cast<size_t>(o) * ksize;
        int acc = 1 << (kResamplePB - 1);
        for (int t = 0; t < n; ++t) acc += static_cast<int>(s[static_cast<size_t>(t) * inner]) * __ldg(k + t);
        r[j] = static_cast<uint8_t>(min(max(acc >> kResamplePB, 0), 255));
      }
    }
    if (aligned && i0 + 16 <= total) {
      *reinterpret_cast<uint4*>(dst + i0) = *reinterpret_cast<const uint4*>(r);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (i0 + j < total) dst[i0 + j] = r[j];
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_resample_u8(const void* src, void* dst, int32_t outer, int32_t in_len, int32_t out_len, int32_t inner,
                                  const int32_t* bounds, const int32_t* coeffs, int32_t ksize, void* stream_ptr) {
  if (src == nullptr || dst == nullptr || bounds == nullptr || coeffs == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (outer <= 0 || in_len <= 0 || out_len <= 0 || inner <= 0 || ksize <= 0 || src == dst) return B200SR_EINVAL;
  const size_t total = static_cast<size_t>(outer) * out_len * inner;
  const bool aligned = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  launch_k(resample_u8_kernel, dim3(grid_for((total + 15) / 16)), dim3(256), 0, stream, 1,
           reinterpret_cast<const uint8_t*>(src), reinterpret_cast<uint8_t*>(dst), in_len, out_len, inner, bounds, coeffs,
           ksize, total, aligned);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// PIL2Tensor's conversion (models/util.py:152-154): x / 255 * 2 - 1 in float64, cast to fp32; uint8 HWC -> fp32 CHW.
// Each thread converts 4 pixels and writes one 16-byte store per plane.
__global__ void img_u8_to_tensor_kernel(const uint8_t* __restrict__ in, float* __restrict__ out, int C, size_t HW,
                                        bool vec) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t quads = (HW + 3) / 4;
  for (size_t q = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; q < quads;
       q += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p0 = q * 4;
    for (int c = 0; c < C; ++c) {
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double u = p0 + j < HW ? static_cast<double>(in[(p0 + j) * C + c]) : 0.0;
        v[j] = static_cast<float>(__dadd_rn(__dmul_rn(__ddiv_rn(u, 255.0), 2.0), -1.0));
      }
      float* plane = out + static_cast<size_t>(c) * HW;
      if (vec) {
        *reinterpret_cast<float4*>(plane + p0) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
        for (int j = 0; j < 4 && p0 + j < HW; ++j) plane[p0 + j] = v[j];
      }
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_img_u8_to_tensor(const void* in, float* out, int32_t C, int32_t H, int32_t W, void* stream_ptr) {
  if (in == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (C <= 0 || C > 4 || H <= 0 || W <= 0) return B200SR_EINVAL;
  const size_t HW = static_cast<size_t>(H) * W;
  const bool vec = HW % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  launch_k(img_u8_to_tensor_kernel, dim3(grid_for((HW + 3) / 4)), dim3(256), 0, stream, 1,
           reinterpret_cast<const uint8_t*>(in), out, C, HW, vec);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}
