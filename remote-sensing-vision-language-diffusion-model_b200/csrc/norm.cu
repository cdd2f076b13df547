// b200sr — fused GroupNorm(32)(+SiLU)(+SFT modulate) and LayerNorm for NHWC / token-major bf16
// activations.  Memory-bound kernels: 128-bit coalesced accesses, fp32 statistics, warp-shuffle +
// shared-memory reductions.
//
// Reference semantics:
//   GroupNorm32 = nn.GroupNorm(32, C, eps=1e-5)       sgm/modules/diffusionmodules/util.py:258-276
//   Normalize   = nn.GroupNorm(32, C, eps=1e-6)       sgm/modules/attention.py:122-125
//   followed by nn.SiLU in ResBlock / UNet.out        openaimodel.py:254-258, :289-292, :942-944
//   ZeroSFT modulate  GN(h) * (1 + gamma) + beta, lerp with control_scale   SR_modules.py:101-110
//   nn.LayerNorm(C) eps 1e-5                          sgm/modules/attention.py:437-439
//   SR3 nn.GroupNorm(32, C) + Swish                   models/sr3_model/sr3_modules/unet.py:81-92
#include "common.cuh"
#include <cstdlib>

namespace b200sr {

static constexpr int GN_WS_COUNTER_FLOATS = 256;

// (sum, sum of squares) of a group -> (mean, 1/sqrt(var + eps)).  The sums arrive as fp64 folds of fp32 partials: each
// thread sums its pixels in fp32 and each CTA its threads' sums in fp32, so those partials carry fp32 rounding error;
// only the fold across chunks and E[x^2] - mean^2 are fp64 (rounding negligible next to the partials'), and the final reciprocal square
// root is fp32 (correctly rounded sqrt and divide).
__device__ __forceinline__ float2 gn_mean_rstd(double sum, double sumsq, double inv_cnt, float eps) {
  const double mean = sum * inv_cnt;
  double var = sumsq * inv_cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  return make_float2(static_cast<float>(mean), 1.0f / sqrtf(static_cast<float>(var) + eps));
}  // 1 KiB of per-image arrival counters at the start of the workspace

// ------------------------------------------------------------------------------------------
// GroupNorm pass 1: per-(image, pixel-chunk, group) partial sum / sum-of-squares.
// Thread t owns channel vector (t % C8) (8 channels, one 16-byte load per pixel) and walks
// pixels t / C8, t / C8 + P, ... of its chunk, so consecutive threads read consecutive 16 B.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
gn_stats_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ workspace, float2* __restrict__ stats_out,
                int HW, int C, int groups, int pix_per_cta, int chunks, int N, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float s_red[];  // [P][C] sums, then [P][C] sums of squares (no atomics: deterministic)
  const int C8 = C >> 3;
  const int P = blockDim.x / C8;
  const int cv = threadIdx.x % C8;
  const int pl = threadIdx.x / C8;
  const int n = blockIdx.y;
  const int chunk = blockIdx.x;
  const int p_begin = chunk * pix_per_cta;
  const int p_end = min(HW, p_begin + pix_per_cta);
  float* s_sum = s_red;
  float* s_sq = s_red + P * C;
  // workspace: [N] arrival counters (zero between launches) | [N][groups] (mean, rstd) | partial sums
  unsigned int* counters = reinterpret_cast<unsigned int*>(workspace);
  float2* stats = stats_out != nullptr ? stats_out : reinterpret_cast<float2*>(workspace + GN_WS_COUNTER_FLOATS);
  float* partial = workspace + GN_WS_COUNTER_FLOATS + 2 * static_cast<size_t>(N) * groups;

  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  if (pl < P) {
    const uint4* base = reinterpret_cast<const uint4*>(x + (static_cast<size_t>(n) * HW) * C) + cv;
    int pix = p_begin + pl;
    // 4 independent 16-byte loads in flight per thread
    for (; pix + 3 * P < p_end; pix += 4 * P) {
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) u[k] = __ldg(base + static_cast<size_t>(pix + k * P) * C8);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = unpack_bf16x2(w[j]);
          s[2 * j] += f.x;
          q[2 * j] += f.x * f.x;
          s[2 * j + 1] += f.y;
          q[2 * j + 1] += f.y * f.y;
        }
      }
    }
    for (; pix < p_end; pix += P) {
      const uint4 u = __ldg(base + static_cast<size_t>(pix) * C8);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(w[j]);
        s[2 * j] += f.x;
        q[2 * j] += f.x * f.x;
        s[2 * j + 1] += f.y;
        q[2 * j + 1] += f.y * f.y;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s_sum[pl * C + cv * 8 + j] = s[j];
      s_sq[pl * C + cv * 8 + j] = q[j];
    }
  }
  __syncthreads();
  const int cpg = C / groups;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int pp = 0; pp < P; ++pp) {
      for (int c = g * cpg; c < (g + 1) * cpg; ++c) {
        a += s_sum[pp * C + c];
        b += s_sq[pp * C + c];
      }
    }
    float* dst = partial + ((static_cast<size_t>(n) * chunks + chunk) * groups + g) * 2;
    dst[0] = a;
    dst[1] = b;
  }

  // The last CTA of image n to get here folds the image's `chunks` partials into (mean, rstd) once,
  // so the apply pass reads 2 * groups floats instead of every CTA re-reading all partials
  // (that re-read was half of the apply kernel's time).  Summation order is fixed -> deterministic.
  __shared__ bool s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();  // cumulative: orders the CTA's partial-sum stores (observed through the barrier) before the arrival
    const unsigned int prev = atomicAdd(&counters[n], 1u);
    s_last = (prev == static_cast<unsigned int>(chunks) - 1u);
    __threadfence();  // ... and the other CTAs' arrivals before this CTA's reads of their partial sums
  }
  __syncthreads();
  if (!s_last) return;
  const float2* src = reinterpret_cast<const float2*>(partial) + static_cast<size_t>(n) * chunks * groups;
  const double inv_cnt = 1.0 / (static_cast<double>(HW) * cpg);
  const int T = blockDim.x;
  if (T % groups == 0 && 2 * T * sizeof(double) <= 2 * static_cast<size_t>(P) * C * sizeof(float)) {
    // thread t: group t % groups, chunk rows t / groups, + T / groups, ... (coalesced rows of float2)
    const int g = threadIdx.x % groups, r0 = threadIdx.x / groups, rstep = T / groups;
    double a = 0.0, b = 0.0;
    // every load of a batch is issued before the first add: one L2 round trip per 40 rows
    for (int k0 = r0; k0 < chunks; k0 += 40 * rstep) {
      float2 v[40];
#pragma unroll
      for (int i = 0; i < 40; ++i) {
        const int k = k0 + i * rstep;
        v[i] = k < chunks ? __ldcg(src + static_cast<size_t>(k) * groups + g) : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int i = 0; i < 40; ++i) {
        a += v[i].x;
        b += v[i].y;
      }
    }
    double* s_d = reinterpret_cast<double*>(s_red);  // the [P][C] buffers are dead by now
    __syncthreads();
    s_d[threadIdx.x] = a;
    s_d[T + threadIdx.x] = b;
    __syncthreads();
    if (threadIdx.x < groups) {
      a = 0.0;
      b = 0.0;
      for (int r = 0; r < rstep; ++r) {
        a += s_d[r * groups + threadIdx.x];
        b += s_d[T + r * groups + threadIdx.x];
      }
      stats[static_cast<size_t>(n) * groups + threadIdx.x] = gn_mean_rstd(a, b, inv_cnt, eps);
    }
  } else {
    // generic shapes: warp per group, lanes over chunks, fixed xor-shuffle tree
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = T >> 5;
    for (int g = warp; g < groups; g += nwarps) {
      double a = 0.0, b = 0.0;
      for (int k = lane; k < chunks; k += 32) {
        const float2 v = __ldcg(src + static_cast<size_t>(k) * groups + g);
        a += v.x;
        b += v.y;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
      }
      if (lane == 0) {
        stats[static_cast<size_t>(n) * groups + g] = gn_mean_rstd(a, b, inv_cnt, eps);
      }
    }
  }
  if (threadIdx.x == 0) counters[n] = 0u;  // ready for the next launch (and for graph replays)
}

// ------------------------------------------------------------------------------------------
// GroupNorm pass 2: y = (x - mean) * rstd * w + b  [-> SiLU]  [-> SFT: y * (1 + gamma) + beta,
// lerp with the un-normalised input by control_scale].  Same thread->channel mapping as pass 1
// so the per-channel scale/shift live in registers.
// ------------------------------------------------------------------------------------------
struct GnApplyArgs {
  const __nv_bfloat16* x;
  const float* stats;  // [N][groups] (mean, rstd) written by the statistics pass
  const float* weight;
  const float* bias;
  __nv_bfloat16* y;
  const __nv_bfloat16* sft_gamma;  // optional [N, HW, C]
  const __nv_bfloat16* sft_beta;   // optional [N, HW, C]
  const __nv_bfloat16* raw;        // optional un-modulated tensor for the control_scale lerp
  float control_scale;
  int HW, C, groups, pix_per_cta, silu;
};

__global__ void __launch_bounds__(1024) gn_apply_kernel(const GnApplyArgs a) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float s_ab[];  // [groups] mean, [groups] rstd
  const int C = a.C, HW = a.HW;
  const int C8 = C >> 3;
  const int P = blockDim.x / C8;
  const int cv = threadIdx.x % C8;
  const int pl = threadIdx.x / C8;
  const int n = blockIdx.y;
  const int cpg = C / a.groups;

  {
    const float2* stats = reinterpret_cast<const float2*>(a.stats) + static_cast<size_t>(n) * a.groups;
    for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
      const float2 m = __ldcg(stats + g);
      s_ab[g] = m.x;
      s_ab[a.groups + g] = m.y;
    }
  }
  __syncthreads();
  if (pl >= P) return;

  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cv * 8 + j;
    const int g = c / cpg;
    const float w = a.weight ? a.weight[c] : 1.f;
    const float b = a.bias ? a.bias[c] : 0.f;
    sc[j] = s_ab[a.groups + g] * w;
    sh[j] = b - s_ab[g] * sc[j];
  }
  const int p_begin = blockIdx.x * a.pix_per_cta;
  const int p_end = min(HW, p_begin + a.pix_per_cta);
  const size_t img = static_cast<size_t>(n) * HW;
  const bool sft = a.sft_gamma != nullptr;
  const float cs = a.control_scale;
  // one pixel-vector: normalise, activate, modulate, store
  auto emit = [&](const size_t off, const uint4 u) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float v[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_bf16x2(w[j]);
      v[2 * j] = f.x * sc[2 * j] + sh[2 * j];
      v[2 * j + 1] = f.y * sc[2 * j + 1] + sh[2 * j + 1];
    }
    if (a.silu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = silu_f(v[j]);
    }
    if (sft) {
      const uint4 ug = __ldg(reinterpret_cast<const uint4*>(a.sft_gamma) + off);
      const uint4 ub = __ldg(reinterpret_cast<const uint4*>(a.sft_beta) + off);
      const uint32_t wg[4] = {ug.x, ug.y, ug.z, ug.w};
      const uint32_t wb[4] = {ub.x, ub.y, ub.z, ub.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 g = unpack_bf16x2(wg[j]);
        const float2 b = unpack_bf16x2(wb[j]);
        v[2 * j] = v[2 * j] * (1.f + g.x) + b.x;
        v[2 * j + 1] = v[2 * j + 1] * (1.f + g.y) + b.y;
      }
      if (a.raw != nullptr && cs != 1.f) {
        const uint4 ur = __ldg(reinterpret_cast<const uint4*>(a.raw) + off);
        const uint32_t wr[4] = {ur.x, ur.y, ur.z, ur.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 r = unpack_bf16x2(wr[j]);
          v[2 * j] = v[2 * j] * cs + r.x * (1.f - cs);
          v[2 * j + 1] = v[2 * j + 1] * cs + r.y * (1.f - cs);
        }
      }
    }
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]);
    o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]);
    o.w = pack_bf16x2(v[6], v[7]);
    reinterpret_cast<uint4*>(a.y)[off] = o;
  };
  int pix = p_begin + pl;
  // 4 independent 16-byte loads in flight per thread (a one-load-at-a-time loop ran at 1/3 of the
  // statistics pass's speed on the same tensor)
  for (; pix + 3 * P < p_end; pix += 4 * P) {
    uint4 u[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = __ldg(reinterpret_cast<const uint4*>(a.x) + (img + pix + k * P) * C8 + cv);
#pragma unroll
    for (int k = 0; k < 4; ++k) emit((img + pix + k * P) * C8 + cv, u[k]);
  }
  for (; pix < p_end; pix += P) {
    const size_t off = (img + pix) * C8 + cv;
    emit(off, __ldg(reinterpret_cast<const uint4*>(a.x) + off));
  }
}

// ------------------------------------------------------------------------------------------
// GroupNorm in ONE kernel for tensors that fit the SMs' shared memory (<= ~12 MB: every GroupNorm of the 32^2 and most
// of the 64^2 levels of the stage-2 networks).  Each CTA keeps its pixel chunk in shared memory between the two phases:
//   phase 1  load the chunk (one 16-byte vector per thread and pixel), per-channel sums, per-(chunk, group) partials
//   barrier  per-image arrival counter; CTAs spin until all `chunks` CTAs of their image have published
//   fold     every CTA folds the image's partials itself, in a fixed order (deterministic), fp64
//   phase 2  normalise / activate / modulate from shared memory, write y
// x is read from L2 / HBM once, and the statistics -> apply dependency costs a spin on an L2 counter instead of a
// kernel boundary.  The launcher only takes this path when the whole grid is resident at once (chunks * N <= SMs, one
// CTA of <= 100 KB per SM, so two such kernels on two streams still fit side by side); the spin traps instead of
// hanging if that assumption is ever violated.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
gn_fused_kernel(const GnApplyArgs a, float* __restrict__ workspace, int chunks, int N, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ __align__(16) uint8_t s_raw[];
  const int C = a.C, HW = a.HW, groups = a.groups;
  const int C8 = C >> 3;
  const int P = blockDim.x / C8;
  const int cv = threadIdx.x % C8;
  const int pl = threadIdx.x / C8;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p_begin = chunk * a.pix_per_cta;
  const int p_end = min(HW, p_begin + a.pix_per_cta);
  const int cpg = C / groups;
  uint4* s_x = reinterpret_cast<uint4*>(s_raw);                                     // [pix_per_cta][C8]
  float* s_sum = reinterpret_cast<float*>(s_raw + static_cast<size_t>(a.pix_per_cta) * C * 2);   // [P][C]
  float* s_sq = s_sum + P * C;                                                      // [P][C]
  float* s_ab = s_sq + P * C;                                                       // [groups] mean | [groups] rstd
  unsigned int* arrive = reinterpret_cast<unsigned int*>(workspace);                // [N]
  unsigned int* depart = arrive + 128;                                              // [N]
  float* partial = workspace + GN_WS_COUNTER_FLOATS + 2 * static_cast<size_t>(N) * groups;
  const size_t img = static_cast<size_t>(n) * HW;

  // ---- phase 1 ----
  if (pl < P) {
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
    const uint4* base = reinterpret_cast<const uint4*>(a.x) + img * C8 + cv;
    for (int pix = p_begin + pl; pix < p_end; pix += P) {
      const uint4 u = __ldg(base + static_cast<size_t>(pix) * C8);
      s_x[(pix - p_begin) * C8 + cv] = u;
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(w[j]);
        s[2 * j] += f.x;
        q[2 * j] += f.x * f.x;
        s[2 * j + 1] += f.y;
        q[2 * j + 1] += f.y * f.y;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s_sum[pl * C + cv * 8 + j] = s[j];
      s_sq[pl * C + cv * 8 + j] = q[j];
    }
  }
  __syncthreads();
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    float sa = 0.f, sb = 0.f;
    for (int pp = 0; pp < P; ++pp)
      for (int c = g * cpg; c < (g + 1) * cpg; ++c) {
        sa += s_sum[pp * C + c];
        sb += s_sq[pp * C + c];
      }
    float* dst = partial + ((static_cast<size_t>(n) * chunks + chunk) * groups + g) * 2;
    dst[0] = sa;
    dst[1] = sb;
  }
  __syncthreads();
  // ---- per-image barrier ----
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(&arrive[n], 1u);
    long long t0 = 0;
    unsigned int spins = 0;
    while (true) {
      unsigned int v;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(arrive + n) : "memory");
      if (v >= static_cast<unsigned int>(chunks)) break;
      if (++spins == 64u) t0 = clock64();
      if (spins > 64u) {
        __nanosleep(64);
        if (clock64() - t0 > 4000000000LL) __trap();   // the grid was not resident at once: fail loudly, never hang
      }
    }
  }
  __syncthreads();
  // ---- fold (same order in every CTA and on every replay) ----
  {
    const float2* src = reinterpret_cast<const float2*>(partial) + static_cast<size_t>(n) * chunks * groups;
    const int T = blockDim.x;
    const int R = T / groups > 0 ? T / groups : 1;       // partial rows handled in parallel per group
    double* s_d = reinterpret_cast<double*>(s_sum);       // the [P][C] buffers are dead; 2 * R * groups doubles fit (R * groups <= T)
    const int g = threadIdx.x % groups, r0 = threadIdx.x / groups;
    double da = 0.0, db = 0.0;
    if (r0 < R)
      for (int k = r0; k < chunks; k += R) {
        const float2 v = __ldcg(src + static_cast<size_t>(k) * groups + g);
        da += v.x;
        db += v.y;
      }
    if (r0 < R) {
      s_d[r0 * groups + g] = da;
      s_d[(R + r0) * groups + g] = db;
    }
    __syncthreads();
    if (threadIdx.x < groups) {
      da = 0.0;
      db = 0.0;
      for (int r = 0; r < R; ++r) {
        da += s_d[r * groups + threadIdx.x];
        db += s_d[(R + r) * groups + threadIdx.x];
      }
      const float2 m = gn_mean_rstd(da, db, 1.0 / (static_cast<double>(HW) * cpg), eps);
      s_ab[threadIdx.x] = m.x;
      s_ab[groups + threadIdx.x] = m.y;
    }
    __syncthreads();
  }
  // the last CTA of the image to get here re-arms both counters (every CTA has passed the spin by then)
  if (threadIdx.x == 0) {
    const unsigned int prev = atomicAdd(&depart[n], 1u);
    if (prev == static_cast<unsigned int>(chunks) - 1u) {
      depart[n] = 0u;
      __threadfence();
      arrive[n] = 0u;
    }
  }
  if (pl >= P) return;
  // ---- phase 2: apply from shared memory ----
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cv * 8 + j;
    const int g = c / cpg;
    const float w = a.weight ? a.weight[c] : 1.f;
    const float b = a.bias ? a.bias[c] : 0.f;
    sc[j] = s_ab[groups + g] * w;
    sh[j] = b - s_ab[g] * sc[j];
  }
  const bool sft = a.sft_gamma != nullptr;
  const float cs = a.control_scale;
  for (int pix = p_begin + pl; pix < p_end; pix += P) {
    const size_t off = (img + pix) * C8 + cv;
    const uint4 u = s_x[(pix - p_begin) * C8 + cv];
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float v[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_bf16x2(w[j]);
      v[2 * j] = f.x * sc[2 * j] + sh[2 * j];
      v[2 * j + 1] = f.y * sc[2 * j + 1] + sh[2 * j + 1];
    }
    if (a.silu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = silu_f(v[j]);
    }
    if (sft) {
      const uint4 ug = __ldg(reinterpret_cast<const uint4*>(a.sft_gamma) + off);
      const uint4 ub = __ldg(reinterpret_cast<const uint4*>(a.sft_beta) + off);
      const uint32_t wg[4] = {ug.x, ug.y, ug.z, ug.w};
      const uint32_t wb[4] = {ub.x, ub.y, ub.z, ub.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 g2 = unpack_bf16x2(wg[j]);
        const float2 b2 = unpack_bf16x2(wb[j]);
        v[2 * j] = v[2 * j] * (1.f + g2.x) + b2.x;
        v[2 * j + 1] = v[2 * j + 1] * (1.f + g2.y) + b2.y;
      }
      if (a.raw != nullptr && cs != 1.f) {
        const uint4 ur = __ldg(reinterpret_cast<const uint4*>(a.raw) + off);
        const uint32_t wr[4] = {ur.x, ur.y, ur.z, ur.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 r2 = unpack_bf16x2(wr[j]);
          v[2 * j] = v[2 * j] * cs + r2.x * (1.f - cs);
          v[2 * j + 1] = v[2 * j + 1] * cs + r2.y * (1.f - cs);
        }
      }
    }
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]);
    o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]);
    o.w = pack_bf16x2(v[6], v[7]);
    reinterpret_cast<uint4*>(a.y)[off] = o;
  }
}

static void gn_geometry(int N, int HW, int C, int* threads, int* P, int* pix_per_cta, int* chunks) {
  const int C8 = C / 8;
  int p = 256 / C8;
  if (p < 1) p = 1;
  *P = p;
  *threads = ((C8 * p + 31) / 32) * 32;
  // aim for ~4 CTAs per SM across the grid, at least 4 pixels per thread row
  // One CTA per SM (two for tensors of 16 MB and more): measured best in-graph (12.9 / 15.3 / 19.4 us for the
  // 2x1024x1280 / 2x4096x640 / 2x16384x320 GroupNorms against 19.6 / 18.9 / 24.3 us with four per SM) — fewer
  // partial sums for the last-arriving CTA to fold and fewer arrival atomics outweigh the shorter per-CTA loop.
  const int ctas_per_sm = static_cast<long long>(N) * HW * C * 2 >= (16ll << 20) ? 2 : 1;
  int want = (ctas_per_sm * num_sms() + N - 1) / N;
  if (want < 1) want = 1;
  int ppc = (HW + want - 1) / want;
  const int min_ppc = p * 8;
  if (ppc < min_ppc) ppc = min_ppc;
  if (ppc > HW) ppc = HW;
  *pix_per_cta = ppc;
  *chunks = (HW + ppc - 1) / ppc;
}

static bool gn_fused_enabled() {
  static const bool v = [] {
    const char* e = getenv("B200SR_GN_FUSED");
    return e == nullptr || e[0] != '0';
  }();
  return v;
}
// one-kernel path: the whole grid resident at once (<= one CTA per SM), the chunk and the reduction scratch within
// 100 KB of shared memory, the fold's per-group parallelism covered by the thread count
static bool gn_fused_eligible(int N, int C, int groups, int threads, int P, int ppc, int chunks, size_t* smem_out) {
  const size_t smem = static_cast<size_t>(ppc) * C * 2 + 2 * static_cast<size_t>(P) * C * sizeof(float) + 2 * groups * sizeof(float);
  const bool fold_fits = groups <= threads && 2 * static_cast<size_t>(threads) * sizeof(double) <= 2 * static_cast<size_t>(P) * C * sizeof(float);
  if (smem_out) *smem_out = smem;
  return gn_fused_enabled() && chunks * N <= num_sms() && N <= 128 && smem <= 100 * 1024 && fold_fits;
}

}  // namespace b200sr

using namespace b200sr;

extern "C" int b200sr_group_norm_launches(int32_t N, int32_t HW, int32_t C, int32_t groups) {
  if (N <= 0 || HW <= 0 || C <= 0 || groups <= 0 || (C % 8) != 0 || (C % groups) != 0) return 0;
  int threads, P, ppc, chunks;
  gn_geometry(N, HW, C, &threads, &P, &ppc, &chunks);
  return gn_fused_eligible(N, C, groups, threads, P, ppc, chunks, nullptr) ? 1 : 2;
}

extern "C" size_t b200sr_group_norm_workspace_bytes(int32_t N, int32_t HW, int32_t C, int32_t groups) {
  if (N <= 0 || HW <= 0 || C < 8 || groups <= 0) return 0;
  int threads, P, ppc, chunks;
  gn_geometry(N, HW, C, &threads, &P, &ppc, &chunks);
  return (GN_WS_COUNTER_FLOATS + 2 * static_cast<size_t>(N) * groups + static_cast<size_t>(N) * chunks * groups * 2) * sizeof(float);
}

extern "C" int b200sr_group_norm_nhwc(const void* x, void* y, const float* weight, const float* bias, int32_t N,
                                      int32_t HW, int32_t C, int32_t groups, float eps, int32_t silu,
                                      const void* sft_gamma, const void* sft_beta, const void* raw,
                                      float control_scale, void* workspace_ptr, void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  float* workspace = static_cast<float*>(workspace_ptr);
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || HW <= 0 || C <= 0 || groups <= 0 || (C % 8) != 0 || (C % groups) != 0 || C / 8 > 1024)
    return B200SR_EINVAL;
  if ((sft_gamma == nullptr) != (sft_beta == nullptr)) return B200SR_EINVAL;
  if (workspace == nullptr || N > GN_WS_COUNTER_FLOATS) return B200SR_EINVAL;
  int threads, P, ppc, chunks;
  gn_geometry(N, HW, C, &threads, &P, &ppc, &chunks);
  dim3 grid(chunks, N);
  {
    size_t smem = 0;
    if (gn_fused_eligible(N, C, groups, threads, P, ppc, chunks, &smem)) {
      static bool attr_set[64] = {false};
      if (first_use_on_device(attr_set))
        cudaFuncSetAttribute(gn_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
      GnApplyArgs a;
      a.x = reinterpret_cast<const __nv_bfloat16*>(x);
      a.stats = nullptr;
      a.weight = weight;
      a.bias = bias;
      a.y = reinterpret_cast<__nv_bfloat16*>(y);
      a.sft_gamma = reinterpret_cast<const __nv_bfloat16*>(sft_gamma);
      a.sft_beta = reinterpret_cast<const __nv_bfloat16*>(sft_beta);
      a.raw = reinterpret_cast<const __nv_bfloat16*>(raw);
      a.control_scale = control_scale;
      a.HW = HW;
      a.C = C;
      a.groups = groups;
      a.pix_per_cta = ppc;
      a.silu = silu;
      launch_k(gn_fused_kernel, dim3(grid), dim3(threads), smem, stream, 1, a, workspace, chunks, N, eps);
      return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
    }
  }
  launch_k(gn_stats_kernel, dim3(grid), dim3(threads), 2 * static_cast<size_t>(P) * C * sizeof(float), stream, 1, reinterpret_cast<const __nv_bfloat16*>(x),
                                                                    workspace, static_cast<float2*>(nullptr), HW, C, groups, ppc, chunks, N, eps);
  GnApplyArgs a;
  a.x = reinterpret_cast<const __nv_bfloat16*>(x);
  a.stats = workspace + GN_WS_COUNTER_FLOATS;
  a.weight = weight;
  a.bias = bias;
  a.y = reinterpret_cast<__nv_bfloat16*>(y);
  a.sft_gamma = reinterpret_cast<const __nv_bfloat16*>(sft_gamma);
  a.sft_beta = reinterpret_cast<const __nv_bfloat16*>(sft_beta);
  a.raw = reinterpret_cast<const __nv_bfloat16*>(raw);
  a.control_scale = control_scale;
  a.HW = HW;
  a.C = C;
  a.groups = groups;
  a.pix_per_cta = ppc;
  a.silu = silu;
  launch_k(gn_apply_kernel, dim3(grid), dim3(threads), 2 * groups * sizeof(float), stream, 1, a);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

// Statistics pass alone: (mean, rstd) per (image, group) into `stats_out` [N][groups][2] for a consumer that applies
// the normalisation itself (the halo convolution's fused input GroupNorm, gemm_conv.cu).
extern "C" int b200sr_group_norm_stats(const void* x, int32_t N, int32_t HW, int32_t C, int32_t groups, float eps,
                                       float* stats_out, void* workspace_ptr, void* stream_ptr) {
  if (x == nullptr) return B200SR_EINVAL;
  float* workspace = static_cast<float*>(workspace_ptr);
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (N <= 0 || HW <= 0 || C <= 0 || groups <= 0 || (C % 8) != 0 || (C % groups) != 0 || C / 8 > 1024)
    return B200SR_EINVAL;
  if (workspace == nullptr || stats_out == nullptr || N > GN_WS_COUNTER_FLOATS) return B200SR_EINVAL;
  int threads, P, ppc, chunks;
  gn_geometry(N, HW, C, &threads, &P, &ppc, &chunks);
  launch_k(gn_stats_kernel, dim3(chunks, N), dim3(threads), 2 * static_cast<size_t>(P) * C * sizeof(float), stream, 1,
           reinterpret_cast<const __nv_bfloat16*>(x), workspace, reinterpret_cast<float2*>(stats_out), HW, C, groups, ppc,
           chunks, N, eps);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// LayerNorm over the channel dim of a token-major [M, C] bf16 matrix: one warp per row, the row
// is held in registers (C <= 2560), two-pass mean / variance in fp32.
// ------------------------------------------------------------------------------------------
template <int VEC_PER_LANE>
__global__ void __launch_bounds__(256)
layer_norm_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y,
                  const float* __restrict__ weight, const float* __restrict__ bias, int M, int C, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= M) return;
  const int C8 = C >> 3;
  const uint4* src = reinterpret_cast<const uint4*>(x + static_cast<size_t>(row) * C);
  float v[VEC_PER_LANE][8];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < VEC_PER_LANE; ++i) {
    const int vi = lane + i * 32;
    if (vi < C8) {
      const uint4 u = __ldg(src + vi);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(w[j]);
        v[i][2 * j] = f.x;
        v[i][2 * j + 1] = f.y;
        sum += f.x + f.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[i][j] = 0.f;
    }
  }
  const float mean = warp_sum(sum) / C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < VEC_PER_LANE; ++i) {
    const int vi = lane + i * 32;
    if (vi < C8) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[i][j] - mean;
        sq += d * d;
      }
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / C + eps);
  uint4* dst = reinterpret_cast<uint4*>(y + static_cast<size_t>(row) * C);
#pragma unroll
  for (int i = 0; i < VEC_PER_LANE; ++i) {
    const int vi = lane + i * 32;
    if (vi < C8) {
      float o[8];
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(weight) + vi * 2);
      const float4 w1 = __ldg(reinterpret_cast<const float4*>(weight) + vi * 2 + 1);
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias) + vi * 2);
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias) + vi * 2 + 1);
      const float ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * ww[j] + bb[j];
      uint4 u;
      u.x = pack_bf16x2(o[0], o[1]);
      u.y = pack_bf16x2(o[2], o[3]);
      u.z = pack_bf16x2(o[4], o[5]);
      u.w = pack_bf16x2(o[6], o[7]);
      dst[vi] = u;
    }
  }
}

}  // namespace b200sr

extern "C" int b200sr_layer_norm(const void* x, void* y, const float* weight, const float* bias, int32_t M, int32_t C,
                                 float eps, void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (M <= 0 || C <= 0 || (C % 8) != 0 || C > 2560 * 2 || weight == nullptr || bias == nullptr) return B200SR_EINVAL;
  const int rows_per_cta = 8;
  const int grid = (M + rows_per_cta - 1) / rows_per_cta;
  const __nv_bfloat16* xi = reinterpret_cast<const __nv_bfloat16*>(x);
  __nv_bfloat16* yo = reinterpret_cast<__nv_bfloat16*>(y);
  const int vpl = (C / 8 + 31) / 32;
  if (vpl <= 1)
    launch_k(layer_norm_kernel<1>, dim3(grid), dim3(256), 0, stream, 1, xi, yo, weight, bias, M, C, eps);
  else if (vpl <= 3)
    launch_k(layer_norm_kernel<3>, dim3(grid), dim3(256), 0, stream, 1, xi, yo, weight, bias, M, C, eps);
  else if (vpl <= 5)
    launch_k(layer_norm_kernel<5>, dim3(grid), dim3(256), 0, stream, 1, xi, yo, weight, bias, M, C, eps);
  else if (vpl <= 10)
    launch_k(layer_norm_kernel<10>, dim3(grid), dim3(256), 0, stream, 1, xi, yo, weight, bias, M, C, eps);
  else
    launch_k(layer_norm_kernel<20>, dim3(grid), dim3(256), 0, stream, 1, xi, yo, weight, bias, M, C, eps);
  return cudaGetLastError() == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

namespace b200sr {

// ------------------------------------------------------------------------------------------
// Row softmax of an fp32 [rows, cols] score matrix -> bf16 probabilities (SR3 single-head
// attention, models/sr3_model/sr3_modules/unet.py:133-138).  One warp per row, three passes
// over an L2-resident row.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
softmax_rows_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int rows, int cols, int valid,
                    float scale) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= rows) return;
  const float* src = x + static_cast<size_t>(row) * cols;
  float mx = -INFINITY;
  for (int c = lane; c < valid; c += 32) mx = fmaxf(mx, src[c]);
  mx = warp_max(mx) * scale;
  float sum = 0.f;
  for (int c = lane; c < valid; c += 32) sum += __expf(src[c] * scale - mx);
  const float inv = 1.0f / warp_sum(sum);
  __nv_bfloat16* dst = y + static_cast<size_t>(row) * cols;
  for (int c = lane; c < cols; c += 32)
    dst[c] = __float2bfloat16(c < valid ? __expf(src[c] * scale - mx) * inv : 0.f);  // padded keys get weight 0
}

// Long rows (1024 < cols <= 32768, cols % 4 == 0): one CTA per row, the row is read ONCE into registers (64 floats per
// thread), maximum and sum are block reductions, the probabilities are written once: 4 + 2 bytes per element instead
// of three passes over a row that no longer fits L1 (T = 16384 keys: 64 KB per row, 1 GB per score matrix).
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
softmax_rows_block_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int cols, int valid, float scale) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_red[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const size_t row = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(x + row * cols);
  const int c4 = cols >> 2;
  float4 v[16];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int idx = threadIdx.x + i * blockDim.x;
    v[i] = idx < c4 ? __ldcs(src + idx) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    const int c = idx * 4;
    if (c + 0 >= valid) v[i].x = -INFINITY;
    if (c + 1 >= valid) v[i].y = -INFINITY;
    if (c + 2 >= valid) v[i].z = -INFINITY;
    if (c + 3 >= valid) v[i].w = -INFINITY;
    mx = fmaxf(mx, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
  }
  mx = warp_max(mx);
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = lane < nwarps ? s_red[lane] : -INFINITY;
  mx = warp_max(mx) * scale;
  __syncthreads();
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    v[i].x = __expf(v[i].x * scale - mx);
    v[i].y = __expf(v[i].y * scale - mx);
    v[i].z = __expf(v[i].z * scale - mx);
    v[i].w = __expf(v[i].w * scale - mx);
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  sum = warp_sum(sum);
  if (lane == 0) s_red[warp] = sum;
  __syncthreads();
  sum = lane < nwarps ? s_red[lane] : 0.f;
  const float inv = 1.0f / warp_sum(sum);
  uint2* dst = reinterpret_cast<uint2*>(y + row * cols);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int idx = threadIdx.x + i * blockDim.x;
    if (idx < c4) dst[idx] = make_uint2(pack_bf16x2(v[i].x * inv, v[i].y * inv), pack_bf16x2(v[i].z * inv, v[i].w * inv));
  }
}

// Two-pass row softmax (b200sr_gemm_bf16 with row_softmax = 1 / 2): fold the per-N-tile (max, sum of 2^(x - max)) pairs of
// pass 1 into one (M, L) pair per row, so that pass 2 reads 8 bytes per row instead of chaining `parts` dependent updates
// in front of every tile's epilogue (measured: 705 us instead of ~200 for the 16384 x 16384 apply pass).
__global__ void __launch_bounds__(256) row_softmax_fold_kernel(const float2* __restrict__ parts, int n_parts, long long rows,
                                                                float2* __restrict__ out) {
  pdl_wait();
  const long long row = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row < rows) {
    float m = -INFINITY;
    for (int q = 0; q < n_parts; ++q) m = fmaxf(m, __ldg(&parts[q * rows + row]).x);   // independent loads
    float l = 0.f;
    for (int q = 0; q < n_parts; ++q) {
      const float2 t = __ldg(&parts[q * rows + row]);
      l += t.y * exp2f(t.x - m);
    }
    out[row] = make_float2(m, l);
  }
  pdl_launch_dependents();
}

}  // namespace b200sr

extern "C" int b200sr_row_softmax_fold(const float* parts, int32_t n_parts, int64_t rows, float* out,
                                       void* stream_ptr) {
  if (parts == nullptr || out == nullptr || n_parts <= 0 || rows <= 0) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  const unsigned grid = static_cast<unsigned>((rows + 255) / 256);
  return launch_k(row_softmax_fold_kernel, dim3(grid), dim3(256), 0, stream, 1, reinterpret_cast<const float2*>(parts), n_parts,
                  rows, reinterpret_cast<float2*>(out)) == cudaSuccess
             ? B200SR_OK
             : B200SR_ELAUNCH;
}

extern "C" int b200sr_softmax_rows(const float* x, void* y, int32_t rows, int32_t cols, int32_t valid, float scale,
                                   void* stream_ptr) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (rows <= 0 || cols <= 0 || valid <= 0 || valid > cols) return B200SR_EINVAL;
  if (cols > 1024 && cols <= 32768 && (cols % 4) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(y) & 7) == 0) {
    int threads = ((cols / 4 + 15) / 16 + 31) / 32 * 32;   // 16 float4 per thread
    if (threads < 64) threads = 64;
    __nv_bfloat16* yo = reinterpret_cast<__nv_bfloat16*>(y);
    const cudaError_t err =
        threads <= 256 ? launch_k(softmax_rows_block_kernel<256>, dim3(rows), dim3(threads), 0, stream, 1, x, yo, cols, valid, scale)
                       : launch_k(softmax_rows_block_kernel<512>, dim3(rows), dim3(threads), 0, stream, 1, x, yo, cols, valid, scale);
    return err == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
  }
  const int grid = (rows + 7) / 8;
  return launch_k(softmax_rows_kernel, dim3(grid), dim3(256), 0, stream, 1, x, reinterpret_cast<__nv_bfloat16*>(y), rows,
                  cols, valid, scale) == cudaSuccess
             ? B200SR_OK
             : B200SR_ELAUNCH;
}
