// b200sr — shared device helpers for the sm_100a kernels (PTX wrappers for mbarrier, TMA,
// tcgen05/TMEM, UMMA descriptors) and small host utilities.  Everything here is written
// for Blackwell only; there is no fallback path.
#pragma once
// The C ABI: every .cu file defines its extern "C" entry points against these prototypes.
#include "../../include/b200sr.h"
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef B200SR_HANG_GUARD
#define B200SR_HANG_GUARD 1  // trap instead of spinning forever on a lost mbarrier phase
#endif

#define B200SR_MAX_COPIES 8  // b200sr_copy_batch: copies per launch

namespace b200sr {

// ------------------------------------------------------------------------------------------
// error codes of the C-ABI (negative errno style, see include/b200sr.h)
// ------------------------------------------------------------------------------------------
enum : int {
  B200SR_OK = 0,
  B200SR_EINVAL = -22,   // bad shape / alignment / flag combination
  B200SR_ENODEV = -19,   // no sm_100 device / driver entry point missing
  B200SR_ELAUNCH = -5,   // CUDA launch error
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking probe (try_wait may sleep in hardware for a while before it reports "not yet")
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#if B200SR_HANG_GUARD
  long long t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins == 1024u) t0 = clock64();
    if (spins > 1024u && (spins & 1023u) == 0 && clock64() - t0 > 8000000000LL) __trap();
  }
#else
  while (!mbar_try_wait(bar, parity)) {
  }
#endif
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor), tile mode, completes on an mbarrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
          "r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// Explicit shared-space 16-byte accesses: pointers carved out of the dynamic shared memory by integer arithmetic lose their
// address space and compile to generic LD / ST otherwise.
__device__ __forceinline__ float4 lds128(const void* ptr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(ptr)));
  return v;
}
__device__ __forceinline__ void sts128(void* ptr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(ptr)), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// 256-bit global accesses (sm_100: LDG.256 / STG.256); the address must be 32-byte aligned
__device__ __forceinline__ void ldg256(const void* ptr, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
               : "l"(ptr));
}
__device__ __forceinline__ void stg256(void* ptr, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
               "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}

// TMA store: shared::cta tile -> global tensor (bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void tma_store_wait_read() {   // at most kPending groups still reading their source
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {  // whole warp
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; single thread issues.
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]; single thread issues.
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (base_lane + t).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// ------------------------------------------------------------------------------------------
// UMMA descriptors (bit layouts as in the PTX ISA "tcgen05 matrix / instruction descriptor")
// ------------------------------------------------------------------------------------------
// Shared-memory operand descriptor, 128-byte swizzle.
//   K-major : rows of 128 B (64 bf16 along K), 8-row groups 1024 B apart (SBO), LBO unused (=1)
//   MN-major: rows of 128 B (64 bf16 along M/N), 8 k-rows per 1024 B group (SBO),
//             LBO = byte distance between consecutive 64-element chunks along M/N
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                         uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);            // [0,14)  start address >> 4
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;       // [16,30) leading byte offset >> 4
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;       // [32,46) stride byte offset >> 4
  d |= static_cast<uint64_t>(1) << 46;                                // [46,48) descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                                // [61,64) SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32, M=128.
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(uint32_t m, uint32_t n, uint32_t a_mn_major,
                                                           uint32_t b_mn_major) {
  return (1u << 4)                 // c_format = F32
         | (1u << 7)               // a_format = BF16
         | (1u << 10)              // b_format = BF16
         | (a_mn_major << 15)      // a_major (0 = K)
         | (b_mn_major << 16)      // b_major (0 = K)
         | ((n >> 3) << 17)        // n_dim
         | ((m >> 4) << 24);       // m_dim
}

// ------------------------------------------------------------------------------------------
// Programmatic dependent launch: every kernel of the step is launched with the programmatic
// stream-serialisation attribute, lets its successor start launching immediately
// (pdl_launch_dependents) and waits for its predecessor's results (pdl_wait) only after its own
// prologue (barrier init, TMEM allocation, descriptor / weight prefetch).  pdl_wait must be
// executed by every thread before it touches memory written by earlier kernels.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// small numeric helpers
// ------------------------------------------------------------------------------------------
// x * sigmoid(x) with ex2.approx / rcp.approx (a full-precision divide is ~8 instructions; the GroupNorm
// apply pass is issue-bound on them).  exp(-x) -> inf for very negative x gives x * 0 = -0, as the exact form.
__device__ __forceinline__ float silu_f(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return x * r;
}
// x * sigmoid(1.702 x): the "quick_gelu" of the CLIP-L text tower (transformers' CLIPTextModel, hidden_act = quick_gelu).
__device__ __forceinline__ float quick_gelu_f(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * (-1.702f * 1.4426950408889634f)));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return x * r;
}
// Exact (erf) GELU, attention.py:84-91 via F.gelu.  erf by Abramowitz & Stegun 7.1.28,
//   erf(t) = 1 - (1 + a1 t + ... + a6 t^6)^-16,  |error| <= 3e-7 for t >= 0,
// branch-free and 11 instructions shorter than erff(): the GEGLU GEMM is bound by its epilogue's
// instruction count.  0.5 x (1 + sign(x) e) = 0.5 (x + |x| e).
__device__ __forceinline__ float gelu_erf_f(float x) {
  const float ax = fabsf(x);
  const float t = ax * 0.70710678118654752f;
  float p = fmaf(t, 0.0000430638f, 0.0002765672f);
  p = fmaf(p, t, 0.0001520143f);
  p = fmaf(p, t, 0.0092705272f);
  p = fmaf(p, t, 0.0422820123f);
  p = fmaf(p, t, 0.0705230784f);
  p = fmaf(p, t, 1.0f);
  p = p * p;
  p = p * p;
  p = p * p;
  p = p * p;
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));
  return 0.5f * fmaf(ax, 1.0f - r, x);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------
// host: driver entry point for tensor-map encoding (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();
int num_sms();
// true the first time it is called for (flags, current device): per-device one-time setup such as
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize), which is a per-device attribute
bool first_use_on_device(bool (&flags)[64]);
bool pdl_enabled();  // B200SR_PDL=0 disables programmatic dependent launch (debugging)

// Launch with the PDL attribute (and an optional cluster size along x).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                            int cluster, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Encode a bf16 tensor map with 128B swizzle. dims/strides innermost first; strides in bytes
// for dims 1..rank-1.  Returns 0 or a negative error code.
int make_tmap_f32(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                  const uint32_t* box);   // fp32 elements, 128B swizzle (box row = 32 floats)
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, int swizzle_bytes = 128);

}  // namespace b200sr
