// b200sr — tcgen05/TMEM GEMM and implicit-GEMM 3x3 convolution for sm_100a.
//
// One persistent, warp-specialised kernel serves every dense contraction on the denoiser path
// (reference call sites: nn.Linear in sgm/modules/attention.py:213-218,:87,:106,:587,:611 and
// openaimodel.py:283-287,:660-662; nn.Conv2d 3x3/1x1 in openaimodel.py:121,:190-197,:257,:294-300,:311
// and models/modules/SR_modules.py:76-84):
//
//   D[M, N] = A[M, K] * W[N, K]^T            bf16 operands, fp32 accumulation in TMEM
//
//   mode 0  GEMM      A is a row-major [M, K] matrix (tokens x channels / NHWC pixels x channels)
//   mode 1  conv3x3   A is an NHWC image; the K loop runs over 9 taps x Cin/64 chunks and each
//                     chunk is one 4-D TMA box shifted by the tap offset (zero fill = padding 1)
//                     (images smaller than one 8 x 16 tile)
//   mode 2  conv3x3 stride 2 (Downsample): the image is viewed as [N, H/2, 2, W/2, 2*C] so each
//                     tap is again one rectangular 5-D TMA box
//   mode 3  conv3x3 stride 1, "halo": per 64-channel chunk one (16+2) x (8+2)-pixel halo tile is staged and
//                     the nine taps read it as shifted windows of the same shared-memory tile, so the
//                     activation crosses L2 -> SM once instead of nine times; weights have their own ring
//
// Roles: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane) and TMEM owner,
// warps 2..5 = epilogue (TMEM -> registers -> fused epilogue -> global).  Two accumulator
// stages in TMEM (2 x 256 columns) let the epilogue of tile i overlap the mainloop of tile i+1.
//
// CTAs run as CTA pairs (kCluster = 2, tcgen05 cta_group::2): one 256 x BN UMMA spans both SMs, each
// CTA stages its own 128 rows of A and only HALF of the weight tile, and the leader CTA issues
// the MMAs for both.  Problems with a single M block use kCluster = 1 (cta_group::1).
//
// What bounds the mainloop (measured, see DESIGN.md section 3): the MMA issue thread pays 150-230 cycles per
// barrier wait + commit, more than the MMAs of one 64-wide chunk take at N <= 192, so a pipeline stage holds two
// K chunks (three taps in mode 3) and the next stage's barrier is probed before the current MMAs are issued;
// beyond that the mainloop is bound by shared-memory bandwidth (128 B/clk: TMA writes + UMMA operand reads, e.g.
// 80 KB per chunk at N = 256 -> 625 cycles against a 512-cycle MMA floor).
//
// Fused epilogues: +bias[N], +rowvec[group, N] (ResBlock timestep-embedding add, one group per
// image; may be a column window of a wider matrix), alpha scale, +residual[M, N], SiLU, GEGLU (value/gate
// interleaved in 16-column groups by the weight packer), per-head row softmax (folded text cross-attention),
// per-row-group weights (per-batch-element B operands), bf16 or fp32 output.
#include "common.cuh"
#include <cstdlib>

namespace b200sr {

static constexpr int BLOCK_M = 128;
static constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle-128B row
static constexpr int UMMA_K = 16;
static constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KiB
static constexpr int MAX_STAGES = 8;
// One pipeline stage = KSUB 64-wide K chunks (modes 0-2) or HALO_TAPS weight tiles (mode 3): the MMA issue thread
// pays ~150-230 cycles per barrier wait + commit (tools/micro/issue_overhead.cu), which at N <= 192 exceeds the
// MMAs' own time when it is paid per chunk.
static constexpr int KSUB = 2;
static constexpr int HALO_TAPS = 3;
// mode 3 ("halo" 3x3 convolution, stride 1): per 64-channel chunk ONE (16+2) x (8+2)-pixel halo tile of the input
// is staged and the nine taps read it as shifted windows (UMMA descriptor start + (kh * 10 + kw) * 128 B, 8-row
// groups 10 pixel rows = 1280 B apart; the 128B swizzle is a function of the absolute address, so shifted
// windows of a TMA-written tile are valid operands — tools/micro/shifted_desc.cu).  The activation tile then
// crosses L2 -> SM once instead of nine times; weights stream through their own ring.
static constexpr int HALO_TILE_W = 8, HALO_TILE_H = 16;
static constexpr int HALO_W = HALO_TILE_W + 2, HALO_H = HALO_TILE_H + 2;
static constexpr int A_HALO_TX_BYTES = HALO_W * HALO_H * BLOCK_K * 2;  // 23040 B written by the TMA box
static constexpr int A_HALO_BYTES = 23 * 1024;                         // stage stride (1024-aligned)
static constexpr int MAX_A_HALO_STAGES = 4;
static constexpr int MAX_B_STAGES = 16;
static constexpr int BAR_REGION_BYTES = 512;
static constexpr int GEMM_THREADS = 192;        // producer, MMA issuer, 4 epilogue warps
static constexpr int XFORM_WARPS = 6;   // 12 warps in all: the register file is allocated in 4-warp granules
static constexpr int GEMM_THREADS_XFORM = GEMM_THREADS + 32 * XFORM_WARPS;  // + warps that normalise the halo tile in place (fused GroupNorm)
static constexpr int TMEM_COLS = 512;
static constexpr int ACC_STAGE_COLS = 256;

struct GemmParams {
  int mode;
  int M, N, K;
  int BN;
  int num_m_blocks, num_n_blocks;  // num_m_blocks is rounded up to a multiple of the cluster size
  int k_iters;
  int kc_per_tap;
  int Cin;
  int pad_lo;  // mode 2: 1 = pad 1 on every side; 0 = pad (0, 1, 0, 1) (bottom / right only: the VAE Downsample)
  int OH, OW, NB;
  int bw_log2, bh_log2, bn_log2;
  int tiles_w, tiles_h, tiles_n;
  int stages;
  int a_stages;  // mode 3: halo-tile ring depth (stages = weight ring depth)
  int w_resident;  // mode 3, one N block whose 3 * kc_per_tap weight stages all fit: loaded once per CTA, never recycled
#ifdef B200SR_GEMM_TRACE
  long long* trace;  // [grid][32] (16..21: epilogue thread 64: cycles in tmem_ld wait / arithmetic / stores / tile prologue, chunks, tiles): 0 mainloop cycles, 1 cycles blocked on the full barrier, 2 chunks, 3 chunks found not ready,
                     // clock64 stamps: 4 entry, 5 set-up done, 6 producer past griddepcontrol.wait, 7 first stage landed,
                     // 8 last MMA committed, 9 accumulator visible to the epilogue, 10 last store issued, 11 exit;
                     // 12 / 13 globaltimer at entry / exit, 14 SM id
#endif
  // epilogue
  const float* bias;
  const float* rowvec;
  int rows_per_group;
  long long ld_rowvec;
  const __nv_bfloat16* residual;
  long long ldr;
  void* out;
  long long ldc;
  int out_fp32;
  int geglu;
  float alpha;
  int act;
  int softmax_valid;
  int w_dynamic;
  int w_rows_per_group;
  long long w_group_stride;
  // mode 3, fused GroupNorm(+SiLU) of the INPUT: y = silu(x * a[n, c] + b[n, c]) applied to the halo tile in shared memory
  // between TMA arrival and the MMAs (a = rstd * gamma, b = beta - mean * a); padding pixels stay zero
  const float* gn_stats;   // [NB][groups] (mean, rstd), nullptr = off
  const float* gn_weight;  // [Cin]
  const float* gn_bias;    // [Cin]
  int gn_groups, gn_silu;
  // mode 0, LayerNorm folded around the GEMM (see b200sr_epilogue in include/b200sr.h):
  //   consumer  v = rstd[m] * (acc[m, n] - mean[m] * colsum[g, n]) + shift[g, n]   with (mean, rstd) folded from ln_parts
  //             per-row partial (sum, sum of squares) written by the GEMM that produced A
  //   producer  ln_stats_out[n_blk][m] = (sum, sum of squares) of row m's fp32 values in this tile, before their rounding
  //             to the bf16 values it stores
  const float2* ln_stats;   // [ln_parts][M], nullptr = off
  int ln_parts;
  const float* ln_colsum;   // [weight groups][N]
  const float* ln_shift;    // [weight groups][N]
  float ln_eps;
  float2* ln_stats_out;     // [num_n_blocks][M], nullptr = off
  // mode 0, two-pass softmax over whole rows (single-head attention at widths the flash kernel cannot hold): 1 = statistics
  // pass (writes (max, sum of exp2) per row and N tile to ln_stats_out, no output matrix), 2 = apply pass (reads ln_stats)
  int row_softmax;
  int row_softmax_valid;    // columns >= this take no part (written as 0)
  // mode 0, fp32 output of a many-tile GEMM (attention scores): the epilogue stages 32 x 32 blocks in shared memory and
  // stores them with the TMA (tmO) so that whole 128-byte lines leave the SM
  int epi_tma;
  // out (and residual) rows are 32-byte aligned and N % 16 == 0: the epilogue moves 32 bytes per thread and instruction
  // (LDG.256 / STG.256, whole sectors) instead of 16
  int wide_io;
};

static constexpr int EPI_SLABS = 4;     // TMA-store epilogue: 32 x 32 fp32 staging blocks per epilogue warp
static constexpr int SOFTMAX_SEG = 80;  // columns per head segment in the softmax epilogue (77 text tokens, padded)

// Packed fp32 pairs (sm_100 FFMA2 / FADD2): the LayerNorm-fold epilogue's extra arithmetic at half the issue slots.
//   v = rstd * v + (nm * c + b)   for two columns
__device__ __forceinline__ void ln_apply2(float& v0, float& v1, float rstd, float nm, float c0, float c1, float b0, float b1) {
  asm("{\n\t.reg .b64 vv, rr, nn, cc, bb;\n\t"
      "mov.b64 vv, {%0, %1};\n\tmov.b64 rr, {%2, %2};\n\tmov.b64 nn, {%3, %3};\n\t"
      "mov.b64 cc, {%4, %5};\n\tmov.b64 bb, {%6, %7};\n\t"
      "fma.rn.f32x2 bb, nn, cc, bb;\n\tfma.rn.f32x2 vv, rr, vv, bb;\n\t"
      "mov.b64 {%0, %1}, vv;\n\t}"
      : "+f"(v0), "+f"(v1)
      : "f"(rstd), "f"(nm), "f"(c0), "f"(c1), "f"(b0), "f"(b1));
}
//   s1 += (v0, v1);  s2 += (v0^2, v1^2)
__device__ __forceinline__ void stats_acc2(float2& s1, float2& s2, float v0, float v1) {
  asm("{\n\t.reg .b64 vv, a1, a2;\n\t"
      "mov.b64 vv, {%4, %5};\n\tmov.b64 a1, {%0, %1};\n\tmov.b64 a2, {%2, %3};\n\t"
      "add.rn.f32x2 a1, a1, vv;\n\tfma.rn.f32x2 a2, vv, vv, a2;\n\t"
      "mov.b64 {%0, %1}, a1;\n\tmov.b64 {%2, %3}, a2;\n\t}"
      : "+f"(s1.x), "+f"(s1.y), "+f"(s2.x), "+f"(s2.y)
      : "f"(v0), "f"(v1));
}

__device__ __forceinline__ float ex2_approx_f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA tile loads of a CTA pair: data lands in the issuing CTA's smem, the bytes are counted on the
// mbarrier at `bar_addr`, which may live in the peer (leader) CTA.
__device__ __forceinline__ void tma2_load_2d(void* dst, const CUtensorMap* m, uint32_t bar_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma2_load_4d(void* dst, const CUtensorMap* m, uint32_t bar_addr, int c0, int c1, int c2,
                                             int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma2_load_5d(void* dst, const CUtensorMap* m, uint32_t bar_addr, int c0, int c1, int c2,
                                             int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6, %7}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void umma2_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit of the pair's MMAs: arrives on the mbarrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tmem2_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem2_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem2_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// kXform: the instantiation with the extra GroupNorm warps (320 threads, <= 204 registers); the plain one keeps 192
// threads and the full register budget its epilogues want.
// kEpi: the epilogue family.  One instantiation per family keeps the 32-column epilogue loop a few KB of straight code: with
// every variant in one body (GEGLU's erf, the softmax, fp32 / TMA stores, activations) the loop spanned 24 KB and ran at
// ~6 cycles per instruction on instruction fetch (tools/gemm_trace.py: 575 cycles for the ~100 instructions of bias + pack).
enum : int {
  EPI_GENERAL = 0,   // bias, alpha, rowvec, residual, activation; bf16 or fp32 (direct or TMA-staged) output
  EPI_XFORM,         // mode 3 with the GroupNorm transform warps; epilogue as EPI_GENERAL without fp32
  EPI_PLAIN,         // bias, alpha, residual; bf16
  EPI_GEGLU,         // bias, value * gelu(gate)
  EPI_SOFTMAX,       // per-head row softmax
  EPI_LN_PLAIN,      // EPI_PLAIN + LayerNorm fold (row statistics in and / or out)
  EPI_LN_GEGLU,
  EPI_LN_SOFTMAX,
  EPI_RS_STATS,      // row softmax over the WHOLE row, pass 1: per row and N tile (max, sum of exp2) of alpha * acc; no output
  EPI_RS_APPLY,      // pass 2: exp2(alpha * acc - M) / L as bf16, (M, L) folded from the pass-1 partials
};
template <int kCluster, int kEpi>
__global__ void __launch_bounds__(kEpi == EPI_XFORM ? GEMM_THREADS_XFORM : GEMM_THREADS, 1)
gemm_conv_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO, const GemmParams p) {
  constexpr bool kXform = kEpi == EPI_XFORM;
  constexpr bool kLn = kEpi == EPI_LN_PLAIN || kEpi == EPI_LN_GEGLU || kEpi == EPI_LN_SOFTMAX;
  constexpr bool kSoftmax = kEpi == EPI_SOFTMAX || kEpi == EPI_LN_SOFTMAX;
  constexpr bool kGeglu = kEpi == EPI_GEGLU || kEpi == EPI_LN_GEGLU;
  constexpr bool kRsStats = kEpi == EPI_RS_STATS;
  constexpr bool kRsApply = kEpi == EPI_RS_APPLY;
  constexpr bool kRs = kRsStats || kRsApply;
  constexpr bool kTail = !kSoftmax && !kGeglu && !kRs;               // alpha / residual / plain stores
  constexpr bool kExtras = kEpi == EPI_GENERAL || kEpi == EPI_XFORM;  // rowvec, activation
  constexpr bool kF32 = kEpi == EPI_GENERAL;                          // fp32 output
  constexpr int kResAhead = kXform ? 1 : 2;                           // residual prefetch distance in chunks (XFORM: 168 registers)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // Round the dynamic smem base up to 1024 B (swizzle-128B atoms are 1024 B aligned).  The
  // offset is identical in both CTAs of a cluster (same kernel, same static layout), which the
  // multicast relies on.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
#ifdef B200SR_GEMM_TRACE
#define GT(slot) do { if (p.trace != nullptr) p.trace[blockIdx.x * 32 + (slot)] = clock64(); } while (0)
  if (threadIdx.x == 0 && p.trace != nullptr) {
    long long gt;
    uint32_t smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    p.trace[blockIdx.x * 32 + 12] = gt;
    p.trace[blockIdx.x * 32 + 14] = smid;
    GT(4);
  }
#else
#define GT(slot) do { } while (0)
#endif
  // per-CTA stage: 128 rows of A and this CTA's BN / kCluster rows of the weight tile
  const int b_sub_bytes = (p.BN / kCluster) * (BLOCK_K * 2);      // one 64-wide weight tile of this CTA
  const int b_stage_bytes = HALO_TAPS * b_sub_bytes;               // mode 3 weight-ring stage
  const int stage_bytes = KSUB * (A_STAGE_BYTES + b_sub_bytes);    // modes 0-2: [A0 | A1 | B0 | B1]
  const int stages = p.stages;
  const bool halo = p.mode == 3;
  const uint32_t rank = kCluster > 1 ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  // modes 0-2: one ring of (A tile | weight tile) stages; mode 3: a ring of halo tiles, then a ring of weight tiles
  const int ring_bytes = halo ? p.a_stages * A_HALO_BYTES + stages * b_stage_bytes : stages * stage_bytes;
  uint8_t* smem_b = smem + p.a_stages * A_HALO_BYTES;  // mode 3 weight ring

  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + ring_bytes);   // [16]
  uint64_t* empty_bar = full_bar + MAX_B_STAGES;                          // [16]
  uint64_t* a_full = empty_bar + MAX_B_STAGES;                            // [4]  mode 3
  uint64_t* a_empty = a_full + MAX_A_HALO_STAGES;                         // [4]  mode 3
  uint64_t* a_land = a_empty + MAX_A_HALO_STAGES;                         // [4]  mode 3 + fused GN: this CTA's tile landed
  uint64_t* tmem_full = a_land + MAX_A_HALO_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* s_epi = reinterpret_cast<float*>(smem + ring_bytes + BAR_REGION_BYTES);  // [4 warps][256] staged bias
  float* s_ab = s_epi + 4 * 256;                                                  // fused GN: [Cin] a | [Cin] b of one image
  const bool xform = kXform && halo && p.gn_stats != nullptr;
  // TMA-store epilogue: [4 warps][EPI_SLABS] slabs of 32 rows x 128 B, 1024-byte aligned (128B swizzle atoms)
  uint8_t* s_out = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(s_ab) + 1023) & ~uintptr_t(1023));

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);   // leader's expect_tx arrive; bytes of both CTAs are counted here
      mbar_init(&empty_bar[s], 1);  // one (multicast) commit from the MMA issuer
    }
    if (halo) {
      for (int s = 0; s < p.a_stages; ++s) {
        // plain: TMA bytes of both CTAs land on the leader's barrier; fused GN: one arrive per CTA once its tile is
        // normalised (the TMA completes on the CTA-local a_land instead)
        mbar_init(&a_full[s], xform ? kCluster * XFORM_WARPS : 1);   // one arrive per transform warp of every CTA
        mbar_init(&a_empty[s], 1);
        mbar_init(&a_land[s], 1);
      }
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 4 * kCluster);  // one arrive per epilogue warp of every CTA in the pair
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (kCluster == 1) {
      tmem_alloc(tmem_base_slot, TMEM_COLS);
      tmem_relinquish();
    } else {
      tmem2_alloc(tmem_base_slot, TMEM_COLS);
      tmem2_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();  // peer barriers / TMEM must exist before remote arrives and pair MMAs
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  if (threadIdx.x == 0) GT(5);
  pdl_launch_dependents();  // the next kernel may start its own prologue now

  // Work = "cluster tiles": kCluster consecutive M blocks x one N block.
  const int m_groups = p.num_m_blocks / kCluster;
  const int num_work = m_groups * p.num_n_blocks;
  const int work0 = blockIdx.x / kCluster;
  const int work_stride = gridDim.x / kCluster;
  const int bw = 1 << p.bw_log2, bh = 1 << p.bh_log2;

  if (warp == 0 && halo) {
    // ================================ TMA producer, halo convolution ================================
    if (lane == 0) {
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      const int b_rows = p.BN / kCluster;
      const uint32_t a_tx = static_cast<uint32_t>(A_HALO_TX_BYTES) * kCluster;
      const uint32_t b_tx = static_cast<uint32_t>(b_stage_bytes) * kCluster;
      for (int work = work0; work < num_work; work += work_stride) {
        const int m_blk = (work % m_groups) * kCluster + static_cast<int>(rank);
        const int n_blk = work / m_groups;
        const int n0 = n_blk * p.BN + static_cast<int>(rank) * b_rows;
        const int tw = m_blk % p.tiles_w;
        const int th = (m_blk / p.tiles_w) % p.tiles_h;
        const int tn = m_blk / (p.tiles_w * p.tiles_h);
        const bool first = (work == work0);
        // weights do not depend on the previous kernel: the first tile's first weight tiles go out before the wait
        const int b_pre = first ? (stages < 3 ? stages : 3) : 0;
        // weight ring: one stage = the HALO_TAPS weight tiles of one kernel row (kh) of one channel chunk
        auto load_b = [&](int cc, int kh) {
          mbar_wait(&empty_bar[sb], pb ^ 1);
          uint8_t* dst = smem_b + sb * b_stage_bytes;
          if (leader) mbar_expect_tx(&full_bar[sb], b_tx);
#pragma unroll
          for (int kw = 0; kw < HALO_TAPS; ++kw) {
            const int kb = (kh * 3 + kw) * p.Cin + cc * BLOCK_K;
            if (kCluster == 1)
              tma_load_2d(dst + kw * b_sub_bytes, &tmB, &full_bar[sb], kb, n0);
            else
              tma2_load_2d(dst + kw * b_sub_bytes, &tmB, mapa_cluster(smem_u32(&full_bar[sb]), 0), kb, n0);
          }
          if (++sb == stages) {
            sb = 0;
            pb ^= 1;
          }
        };
        const bool stream_w = first || !p.w_resident;   // resident weights: the first tile's loads serve every tile
        for (int kh = 0; kh < b_pre; ++kh) load_b(0, kh);
        if (first) pdl_wait();
        for (int cc = 0; cc < p.kc_per_tap; ++cc) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          uint8_t* dst = smem + sa * A_HALO_BYTES;
          if (xform) {
            mbar_expect_tx(&a_land[sa], static_cast<uint32_t>(A_HALO_TX_BYTES));
            tma_load_4d(dst, &tmA, &a_land[sa], cc * BLOCK_K, tw * HALO_TILE_W - 1, th * HALO_TILE_H - 1, tn);
          } else if (kCluster == 1) {
            mbar_expect_tx(&a_full[sa], a_tx);
            tma_load_4d(dst, &tmA, &a_full[sa], cc * BLOCK_K, tw * HALO_TILE_W - 1, th * HALO_TILE_H - 1, tn);
          } else {
            if (leader) mbar_expect_tx(&a_full[sa], a_tx);
            tma2_load_4d(dst, &tmA, mapa_cluster(smem_u32(&a_full[sa]), 0), cc * BLOCK_K, tw * HALO_TILE_W - 1,
                         th * HALO_TILE_H - 1, tn);
          }
          if (++sa == p.a_stages) {
            sa = 0;
            pa ^= 1;
          }
          if (stream_w)
            for (int kh = (cc == 0 ? b_pre : 0); kh < 3; ++kh) load_b(cc, kh);
        }
      }
    }
  } else if (warp == 1 && halo) {
    // ================================ MMA issuer, halo convolution ================================
    if (lane == 0 && leader) {
      const uint32_t idesc = umma_idesc_bf16_f32(BLOCK_M * kCluster, static_cast<uint32_t>(p.BN), 0, 0);
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      bool ready = false;
      for (int work = work0; work < num_work; work += work_stride) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * ACC_STAGE_COLS;
        for (int cc = 0; cc < p.kc_per_tap; ++cc) {
          mbar_wait(&a_full[sa], pa);
          const uint32_t a_base = smem_u32(smem + sa * A_HALO_BYTES);
          for (int kh = 0; kh < 3; ++kh) {
            // resident weights: stage sb = cc * 3 + kh holds this row of this chunk for the whole kernel; only the first
            // tile waits for it to land
            const bool wait_w = !p.w_resident || work == work0;
            if (wait_w && !ready) mbar_wait(&full_bar[sb], pb);
            tc_fence_after();
            if (wait_w) {  // probe the next weight stage now, consume the answer after this row's MMAs are issued
              const int ns = sb + 1 == stages ? 0 : sb + 1;
              ready = mbar_test_wait(&full_bar[ns], ns == 0 ? pb ^ 1 : pb);
            }
            const uint32_t b_base = smem_u32(smem_b + sb * b_stage_bytes);
#pragma unroll
            for (int kw = 0; kw < HALO_TAPS; ++kw) {
              // window of tap (kh, kw): start (kh * 10 + kw) pixel rows in; 8-pixel groups one halo row (1280 B) apart
              const uint64_t adesc = umma_smem_desc_sw128(a_base + (kh * HALO_W + kw) * 128, 16, HALO_W * 128);
              const uint64_t bdesc = umma_smem_desc_sw128(b_base + kw * b_sub_bytes, 16, 1024);
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                if (kCluster == 1)
                  umma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (cc | kh | kw | k) != 0);
                else
                  umma2_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (cc | kh | kw | k) != 0);
              }
            }
            if (!p.w_resident) {
              if (kCluster == 1)
                umma_commit(&empty_bar[sb]);
              else
                umma2_commit_mc(&empty_bar[sb], 3);
            }
            if (++sb == stages) {
              sb = 0;
              pb ^= 1;
            }
          }
          if (kCluster == 1)
            umma_commit(&a_empty[sa]);
          else
            umma2_commit_mc(&a_empty[sa], 3);
          if (++sa == p.a_stages) {
            sa = 0;
            pa ^= 1;
          }
        }
        if (kCluster == 1)
          umma_commit(&tmem_full[acc]);
        else
          umma2_commit_mc(&tmem_full[acc], 3);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (!kXform && warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t sub_tx = static_cast<uint32_t>(A_STAGE_BYTES + b_sub_bytes) * kCluster;  // bytes of one K chunk, both CTAs
      const int b_rows = p.BN / kCluster;
      const int s_iters = (p.k_iters + KSUB - 1) / KSUB;  // pipeline stages per tile
      for (int work = work0; work < num_work; work += work_stride) {
        const int m_blk = (work % m_groups) * kCluster + static_cast<int>(rank);
        const int n_blk = work / m_groups;
        int n0 = n_blk * p.BN + static_cast<int>(rank) * b_rows;  // this CTA's rows of the weight tile
        if (p.w_rows_per_group > 0)  // per-batch-element weights stacked along the rows
          n0 += static_cast<int>((static_cast<long long>(m_blk) * BLOCK_M / p.w_rows_per_group) * p.w_group_stride);
        int w0 = 0, h0 = 0, i0 = 0;
        if (p.mode != 0) {
          const int tw = m_blk % p.tiles_w;
          const int th = (m_blk / p.tiles_w) % p.tiles_h;
          const int tn = m_blk / (p.tiles_w * p.tiles_h);
          w0 = tw * bw;
          h0 = th * bh;
          i0 = tn << p.bn_log2;
        }
        // Weights never depend on the previous kernel: on the first tile the weight chunks of the first `pre`
        // stages are requested before griddepcontrol.wait, the activation (A) chunks after it.
        const bool first = (work == work0);
        const int pre = (first && !p.w_dynamic) ? (s_iters < stages ? s_iters : stages) : 0;
        for (int it = 0; it < s_iters + pre; ++it) {
          // it in [0, pre): weights of stage `it` only; it in [pre, 2*pre): activations of stage it-pre only;
          // afterwards: both for stage it-pre.
          const bool w_only = it < pre, a_only = (it >= pre && it < 2 * pre);
          const int sit = w_only ? it : it - pre;
          if (it == pre && first) {
            pdl_wait();
            GT(6);
          }
          const int st = w_only || a_only ? sit : stage;
          if (!w_only && !a_only) mbar_wait(&empty_bar[stage], phase ^ 1);
          const int nsub = p.k_iters - sit * KSUB < KSUB ? p.k_iters - sit * KSUB : KSUB;
          uint8_t* sa0 = smem + st * stage_bytes;
          uint8_t* sb0 = sa0 + KSUB * A_STAGE_BYTES;
          if (leader && !a_only) mbar_expect_tx(&full_bar[st], sub_tx * nsub);
          const uint32_t bar = kCluster > 1 ? mapa_cluster(smem_u32(&full_bar[st]), 0) : 0u;  // the leader's barrier
          for (int j = 0; j < nsub; ++j) {
            const int kit = sit * KSUB + j;
            uint8_t* sa = sa0 + j * A_STAGE_BYTES;
            uint8_t* sb = sb0 + j * b_sub_bytes;
            int kb;  // K coordinate of the weight tile
            int tap = 0, c0 = 0, kh = 0, kw = 0;
            if (p.mode == 0) {
              kb = kit * BLOCK_K;
            } else {
              tap = kit / p.kc_per_tap;
              c0 = (kit - tap * p.kc_per_tap) * BLOCK_K;
              kh = tap / 3;
              kw = tap - kh * 3;
              kb = tap * p.Cin + c0;
            }
            // pad_lo = 1: input row 2*oh + kh - 1 -> (h2, parity): kh=0 -> (oh-1, 1), kh=1 -> (oh, 0), kh=2 -> (oh, 1)
            // pad_lo = 0: input row 2*oh + kh     ->               kh=0 -> (oh, 0),   kh=1 -> (oh, 1), kh=2 -> (oh+1, 0)
            const int hp = p.pad_lo ? ((kh == 1) ? 0 : 1) : (kh & 1), wp = p.pad_lo ? ((kw == 1) ? 0 : 1) : (kw & 1);
            const int dh = p.pad_lo ? -(kh == 0) : (kh == 2), dw = p.pad_lo ? -(kw == 0) : (kw == 2);
            if (kCluster == 1) {
              if (!w_only) {
                if (p.mode == 0)
                  tma_load_2d(sa, &tmA, &full_bar[st], kb, m_blk * BLOCK_M);
                else if (p.mode == 1)
                  tma_load_4d(sa, &tmA, &full_bar[st], c0, w0 + kw - 1, h0 + kh - 1, i0);
                else
                  tma_load_5d(sa, &tmA, &full_bar[st], wp * p.Cin + c0, w0 + dw, hp, h0 + dh, i0);
              }
              if (!a_only) tma_load_2d(sb, &tmB, &full_bar[st], kb, n0);
            } else {
              if (!w_only) {
                if (p.mode == 0)
                  tma2_load_2d(sa, &tmA, bar, kb, m_blk * BLOCK_M);
                else if (p.mode == 1)
                  tma2_load_4d(sa, &tmA, bar, c0, w0 + kw - 1, h0 + kh - 1, i0);
                else
                  tma2_load_5d(sa, &tmA, bar, wp * p.Cin + c0, w0 + dw, hp, h0 + dh, i0);
              }
              if (!a_only) tma2_load_2d(sb, &tmB, bar, kb, n0);
            }
          }
          if (w_only) continue;  // the ring position advances once per stage (with its activation loads)
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (!kXform && warp == 1) {
    // ================================ MMA issuer ================================
    if (lane == 0 && leader) {
      const uint32_t idesc = umma_idesc_bf16_f32(BLOCK_M * kCluster, static_cast<uint32_t>(p.BN), 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      // The issue thread is the mainloop's critical resource (tools/micro/issue_overhead.cu: wait + 4 MMAs + commit
      // = ~550 cycles per chunk against a 320-cycle MMA floor at N = 160), so the NEXT chunk's barrier is probed
      // before this chunk's MMAs are issued and the answer is consumed afterwards: the probe's latency hides
      // under the issue, and the blocking wait runs only when the data really is not there yet.
      bool ready = false;
#ifdef B200SR_GEMM_TRACE
      long long t_loop = 0, t_wait = 0, n_chunks = 0, n_late = 0;
#endif
      for (int work = work0; work < num_work; work += work_stride) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * ACC_STAGE_COLS;
#ifdef B200SR_GEMM_TRACE
        const long long t_begin = clock64();
#endif
        const int s_iters = (p.k_iters + KSUB - 1) / KSUB;
        for (int it = 0; it < s_iters; ++it) {
          const int nsub = p.k_iters - it * KSUB < KSUB ? p.k_iters - it * KSUB : KSUB;
#ifdef B200SR_GEMM_TRACE
          n_chunks += nsub;
          if (!ready) {
            const long long t0 = clock64();
            mbar_wait(&full_bar[stage], phase);
            t_wait += clock64() - t0;
            ++n_late;
          }
          if (it == 0 && work == work0) GT(7);
#else
          if (!ready) mbar_wait(&full_bar[stage], phase);
#endif
          tc_fence_after();
          {
            const int ns = stage + 1 == stages ? 0 : stage + 1;
            ready = mbar_test_wait(&full_bar[ns], ns == 0 ? phase ^ 1 : phase);
          }
          const uint32_t sa0 = smem_u32(smem + stage * stage_bytes);
          const uint32_t sb0 = sa0 + KSUB * A_STAGE_BYTES;
          for (int j = 0; j < nsub; ++j) {
            const uint64_t adesc = umma_smem_desc_sw128(sa0 + j * A_STAGE_BYTES, 16, 1024);
            const uint64_t bdesc = umma_smem_desc_sw128(sb0 + j * b_sub_bytes, 16, 1024);
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
              // advance 32 B (16 bf16) along K inside the 128 B swizzle row: +2 in 16-byte units
              if (kCluster == 1)
                umma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (it | j | k) != 0);
              else
                umma2_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (it | j | k) != 0);
            }
          }
          // free the smem slot (in both CTAs of a pair) once these MMAs retire
          if (kCluster == 1)
            umma_commit(&empty_bar[stage]);
          else
            umma2_commit_mc(&empty_bar[stage], 3);
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
#ifdef B200SR_GEMM_TRACE
        t_loop += clock64() - t_begin;
        if (p.trace != nullptr) {
          p.trace[blockIdx.x * 32 + 0] = t_loop;
          p.trace[blockIdx.x * 32 + 1] = t_wait;
          p.trace[blockIdx.x * 32 + 2] = n_chunks;
          p.trace[blockIdx.x * 32 + 3] = n_late;
          GT(8);
        }
#endif
        // accumulator complete -> epilogue warps (of both CTAs of a pair)
        if (kCluster == 1)
          umma_commit(&tmem_full[acc]);
        else
          umma2_commit_mc(&tmem_full[acc], 3);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp >= 6) {
    // ================================ fused GroupNorm(+SiLU) of the halo tile (2 warps) ================================
    // Mirrors the producer's tile order.  Per 64-channel chunk: thread t computes (a, b) of channel cc*64 + t from the
    // statistics of its group, the 64 threads wait for this CTA's tile (TMA, 128B swizzle: pixel row p holds its eight
    // 16-byte channel groups at chunk index j ^ (p & 7)), rewrite every in-image pixel in place and hand the tile to
    // the MMA issuer (of the pair's leader).  Pixels outside the image were zero-filled by the TMA and stay zero: the
    // convolution pads the NORMALISED tensor.
    if (xform) {
      constexpr int XT = 32 * XFORM_WARPS;
      const int t = threadIdx.x - 6 * 32;   // 0 .. XT-1
      const int xw = t >> 5;                 // transform warp 0 .. XFORM_WARPS-1: owns pixels xw, xw + XFORM_WARPS, ... of every tile
      const int cpg = p.Cin / p.gn_groups;
      float* ab = s_ab;                      // [Cin] a | [Cin] b of the image this CTA is working on
      int sa = 0, cur_n = -1;
      uint32_t pa = 0;
      pdl_wait();   // statistics come from the preceding kernel
      for (int work = work0; work < num_work; work += work_stride) {
        const int m_blk = (work % m_groups) * kCluster + static_cast<int>(rank);
        const int tw = m_blk % p.tiles_w;
        const int th = (m_blk / p.tiles_w) % p.tiles_h;
        const int tn = m_blk / (p.tiles_w * p.tiles_h);
        const bool img_ok = tn < p.NB;
        if (img_ok && tn != cur_n) {
          // per-channel scale / shift of this image, once per image (not per chunk: the loads would sit on every
          // chunk's path to the tensor core)
          asm volatile("bar.sync 2, %0;" ::"n"(XT) : "memory");   // previous image's table no longer read
          for (int c = t; c < p.Cin; c += XT) {
            const float2 st = __ldg(reinterpret_cast<const float2*>(p.gn_stats) + tn * p.gn_groups + c / cpg);
            const float a = st.y * __ldg(p.gn_weight + c);
            ab[c] = a;
            ab[p.Cin + c] = __ldg(p.gn_bias + c) - st.x * a;
          }
          asm volatile("bar.sync 2, %0;" ::"n"(XT) : "memory");
          cur_n = tn;
        }
        for (int cc = 0; cc < p.kc_per_tap; ++cc) {
          mbar_wait(&a_land[sa], pa);
          uint8_t* tile = smem + sa * A_HALO_BYTES;
          if (img_ok) {
            // lane = (pixel within a group of 4, LOGICAL 8-channel group j): the lane's 8 scales / shifts live in registers
            // for the whole chunk (reading them per element would cost 4x the tile's own shared-memory traffic, which
            // the tensor core's operand reads have no room for); a quarter-warp still covers one whole 128-byte pixel
            // row per access, its chunks permuted by the swizzle (physical chunk = j ^ (row & 7)).
            const int j = lane & 7;
            const float* ac = ab + cc * BLOCK_K + j * 8;
            const float* bc = ab + p.Cin + cc * BLOCK_K + j * 8;
            const float4 a0 = *reinterpret_cast<const float4*>(ac), a1 = *reinterpret_cast<const float4*>(ac + 4);
            const float4 b0 = *reinterpret_cast<const float4*>(bc), b1 = *reinterpret_cast<const float4*>(bc + 4);
            const float sc[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float sh[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
            for (int pix = xw * 4 + (lane >> 3); pix < HALO_W * HALO_H; pix += 4 * XFORM_WARPS) {
              const int hy = pix / HALO_W, hx = pix - hy * HALO_W;
              const int iy = th * HALO_TILE_H - 1 + hy, ix = tw * HALO_TILE_W - 1 + hx;
              if (iy < 0 || iy >= p.OH || ix < 0 || ix >= p.OW) continue;
              uint4* q = reinterpret_cast<uint4*>(tile + pix * 128 + ((j ^ (pix & 7)) << 4));
              const uint4 u = *q;
              const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
              float v[8];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 f = unpack_bf16x2(w4[e]);
                v[2 * e] = f.x * sc[2 * e] + sh[2 * e];
                v[2 * e + 1] = f.y * sc[2 * e + 1] + sh[2 * e + 1];
              }
              if (p.gn_silu) {
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = silu_f(v[e]);
              }
              *q = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
            }
          }
          // each warp hands over its own pixel rows: fence its generic-proxy writes for the tensor core's (async proxy)
          // reads, then one arrive per warp — no CTA-wide barrier on the tile's way to the MMAs
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (kCluster == 1)
              mbar_arrive(&a_full[sa]);
            else
              mbar_arrive_cluster(mapa_cluster(smem_u32(&a_full[sa]), 0));
          }
          if (++sa == p.a_stages) {
            sa = 0;
            pa ^= 1;
          }
        }
      }
    }
  } else {
    // ================================ epilogue (4 warps) ================================
    // Per tile: the tile's bias slice is staged in (warp-private) shared memory and the first residual
    // chunk is requested BEFORE waiting for the accumulator, so both overlap the mainloop; inside the
    // chunk loop the TMEM load and the residual load of chunk c+1 are in flight while chunk c is
    // processed and stored.
    const int sub = warp & 3;           // TMEM sub-partition this warp may access
    const int r = sub * 32 + lane;      // accumulator row == TMEM lane
    float* s_bias = s_epi + (warp - 2) * 256;
    const bool ln_in = kLn && p.ln_stats != nullptr;
    const bool ln_out = kEpi == EPI_LN_PLAIN && p.ln_stats_out != nullptr;
    const bool epi_tma = kF32 && p.epi_tma != 0;
    uint32_t slab_i = 0;                      // running slab counter of this warp (TMA-store epilogue)
    int staged_n_blk = -1;                    // N block whose bias slice this warp's s_bias holds
#ifdef B200SR_GEMM_TRACE
    long long e_ld = 0, e_math = 0, e_st = 0, e_pro = 0, e_chunks = 0, e_tiles = 0;
#define ET(var, since) do { const long long now_ = clock64(); var += now_ - since; since = now_; } while (0)
#else
#define ET(var, since) do { } while (0)
#endif
    float* s_col = s_ab + (warp - 2) * 256;   // LayerNorm fold: column sums of the weight tile (the fused-GN table is mode 3 only)
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int work = work0; work < num_work; work += work_stride) {
      const int m_blk = (work % m_groups) * kCluster + static_cast<int>(rank);
      const int n_blk = work / m_groups;
      const int n0 = n_blk * p.BN;
      long long row;
      int group;
      bool valid;
      if (p.mode == 0) {
        row = static_cast<long long>(m_blk) * BLOCK_M + r;
        valid = row < p.M;
        group = p.rows_per_group > 0 ? static_cast<int>(row / p.rows_per_group) : 0;
      } else {
        const int tw = m_blk % p.tiles_w;
        const int th = (m_blk / p.tiles_w) % p.tiles_h;
        const int tn = m_blk / (p.tiles_w * p.tiles_h);
        const int dw = r & (bw - 1);
        const int dh = (r >> p.bw_log2) & (bh - 1);
        const int dn = r >> (p.bw_log2 + p.bh_log2);
        const int ow = tw * bw + dw, oh = th * bh + dh, n = (tn << p.bn_log2) + dn;
        valid = (ow < p.OW) && (oh < p.OH) && (n < p.NB);
        row = (static_cast<long long>(n) * p.OH + oh) * p.OW + ow;
        group = n;
      }
      // stage bias[n0 .. n0+BN) (zero beyond N) — constant data, independent of earlier kernels
#ifdef B200SR_GEMM_TRACE
      long long et = clock64();
      ++e_tiles;
#endif
      __syncwarp();
      const bool has_res = kTail && p.residual != nullptr && valid;
      const __nv_bfloat16* res_row = has_res ? p.residual + row * p.ldr + n0 : nullptr;
      const float* rv_row = (kExtras && p.rowvec != nullptr) ? p.rowvec + static_cast<long long>(group) * p.ld_rowvec + n0 : nullptr;
      // residual chunks in flight: the loads of chunk c + kResAhead are issued at the top of chunk c (one chunk ahead left
      // ~650 cycles of L2 latency exposed per chunk: tools/gemm_trace.py, 944 vs 284 cycles with / without a residual)
      uint4 res[kResAhead + 1][4];
      auto load_res = [&](uint4 (&dst)[4], int cc) {   // cc: column offset of the chunk inside the tile
        if (p.wide_io) {
#pragma unroll
          for (int hq = 0; hq < 2; ++hq) {
            if (n0 + cc + hq * 16 < p.N)
              ldg256(res_row + cc + hq * 16, dst[2 * hq], dst[2 * hq + 1]);
            else
              dst[2 * hq] = dst[2 * hq + 1] = make_uint4(0, 0, 0, 0);
          }
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            dst[q] = (n0 + cc + q * 8 < p.N) ? __ldg(reinterpret_cast<const uint4*>(res_row + cc) + q) : make_uint4(0, 0, 0, 0);
        }
      };
      float ln_rstd = 1.f, ln_nm = 0.f;  // v = rstd * acc - mean * rstd * colsum + shift
      float rs_m = -INFINITY, rs_l = 0.f;   // row softmax: running (max, sum) of pass 1 / (M, 1 / L) of pass 2
      if (kRs) {
        if (work == work0) pdl_wait();
        if (kRsApply && valid) {
          // fold the pass-1 partials of this row: M = max m_q, L = sum l_q 2^(m_q - M); independent loads, one pass
          for (int q = 0; q < p.ln_parts; ++q) {
            const float2 t = __ldg(p.ln_stats + static_cast<long long>(q) * p.M + row);
            const float m_new = fmaxf(rs_m, t.x);
            if (m_new > -INFINITY) {
              rs_l = rs_l * ex2_approx_f(rs_m - m_new) + t.y * ex2_approx_f(t.x - m_new);
              rs_m = m_new;
            }
          }
          rs_l = rs_l > 0.f ? 1.0f / rs_l : 0.f;
        }
      } else if (!ln_in) {
        // consecutive tiles of a CTA usually share the N block (always, when there is only one): its bias slice is staged
        // once — the L2 round trip of this load otherwise sits in front of every tile's epilogue
        if (n_blk != staged_n_blk) {
          for (int j = lane; j < p.BN; j += 32)
            s_bias[j] = (p.bias != nullptr && n0 + j < p.N) ? __ldg(p.bias + n0 + j) : 0.f;
          staged_n_blk = n_blk;
        }
        __syncwarp();
        if (work == work0) pdl_wait();  // residual / rowvec come from earlier kernels
      } else {
        // Every global load of the tile's prologue is issued before the first use of any of them: with several tiles per
        // CTA the epilogue is the longer pipeline stage, and three dependent L2 round trips per tile showed as +25 %
        // kernel time (profiles/r02_ln_fold.txt).
        const long long wg =
            p.w_rows_per_group > 0 ? (static_cast<long long>(m_blk) * BLOCK_M / p.w_rows_per_group) * p.N : 0;
        float bb[8], cc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int j = lane + 32 * i;
          const bool in = j < p.BN && n0 + j < p.N;
          bb[i] = (in && p.bias != nullptr) ? __ldg(p.bias + n0 + j) : 0.f;
          cc[i] = in ? __ldg(p.ln_colsum + wg + n0 + j) : 0.f;
          bb[i] += in ? __ldg(p.ln_shift + wg + n0 + j) : 0.f;
        }
        if (work == work0) pdl_wait();  // residual / row statistics come from earlier kernels
        float s1 = 0.f, s2 = 0.f;
        if (valid) {
          for (int q = 0; q < p.ln_parts; ++q) {
            const float2 t = __ldg(p.ln_stats + static_cast<long long>(q) * p.M + row);
            s1 += t.x;
            s2 += t.y;
          }
        }
        if (has_res) {
#pragma unroll
          for (int d = 0; d < kResAhead; ++d)
            if (d * 32 < p.BN) load_res(res[d], d * 32);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int j = lane + 32 * i;
          if (j < p.BN) {
            s_bias[j] = bb[i];
            s_col[j] = cc[i];
          }
        }
        __syncwarp();
        const float inv_k = 1.0f / static_cast<float>(p.K);
        const float mean = s1 * inv_k;
        const float var = fmaxf(s2 * inv_k - mean * mean, 0.f);
        ln_rstd = rsqrtf(var + p.ln_eps);
        ln_nm = -mean * ln_rstd;
      }
      float2 ln_acc1 = make_float2(0.f, 0.f), ln_acc2 = make_float2(0.f, 0.f);  // producer side: (sum, sum of squares), 2 lanes
      if (has_res && !ln_in) {
#pragma unroll
        for (int d = 0; d < kResAhead; ++d)
          if (d * 32 < p.BN) load_res(res[d], d * 32);
      }
      ET(e_pro, et);
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (threadIdx.x == 64) GT(9);
#ifdef B200SR_GEMM_TRACE
      et = clock64();
#endif
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(sub * 32) << 16) + acc * ACC_STAGE_COLS;
      if (kSoftmax) {
        // Row softmax over each SOFTMAX_SEG-column head segment of the accumulator (logits already in log2
        // units), written as bf16 probabilities; columns >= softmax_valid of a segment are padding -> 0.
        for (int sg = 0; sg * SOFTMAX_SEG < p.BN; ++sg) {
          const int col0 = n0 + sg * SOFTMAX_SEG;
          if (col0 >= p.N) break;
          uint32_t a0[32], a1[32], a2[16];
          tmem_ld32(t_row + sg * SOFTMAX_SEG, a0);
          tmem_ld32(t_row + sg * SOFTMAX_SEG + 32, a1);
          tmem_ld16(t_row + sg * SOFTMAX_SEG + 64, a2);
          tmem_ld_wait();
          float v[SOFTMAX_SEG];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            v[j] = __uint_as_float(a0[j]);
            v[32 + j] = __uint_as_float(a1[j]);
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) v[64 + j] = __uint_as_float(a2[j]);
          if (ln_in) {
#pragma unroll
            for (int j = 0; j < SOFTMAX_SEG; j += 4) {
              const float4 c4 = lds128(s_col + sg * SOFTMAX_SEG + j);
              const float4 b4 = lds128(s_bias + sg * SOFTMAX_SEG + j);
              ln_apply2(v[j], v[j + 1], ln_rstd, ln_nm, c4.x, c4.y, b4.x, b4.y);
              ln_apply2(v[j + 2], v[j + 3], ln_rstd, ln_nm, c4.z, c4.w, b4.z, b4.w);
            }
          }
          float mx = -INFINITY;
#pragma unroll
          for (int j = 0; j < SOFTMAX_SEG; ++j) {
            if (j >= p.softmax_valid) v[j] = -INFINITY;
            mx = fmaxf(mx, v[j]);
          }
          float sum = 0.f;
#pragma unroll
          for (int j = 0; j < SOFTMAX_SEG; ++j) {
            float e;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v[j] - mx));
            v[j] = e;
            sum += e;
          }
          const float inv = 1.0f / sum;
          if (valid) {
            uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.ldc + col0);
#pragma unroll
            for (int q = 0; q < SOFTMAX_SEG / 8; q += 2) {
              uint4 u0, u1;
              u0.x = pack_bf16x2(v[q * 8 + 0] * inv, v[q * 8 + 1] * inv);
              u0.y = pack_bf16x2(v[q * 8 + 2] * inv, v[q * 8 + 3] * inv);
              u0.z = pack_bf16x2(v[q * 8 + 4] * inv, v[q * 8 + 5] * inv);
              u0.w = pack_bf16x2(v[q * 8 + 6] * inv, v[q * 8 + 7] * inv);
              u1.x = pack_bf16x2(v[q * 8 + 8] * inv, v[q * 8 + 9] * inv);
              u1.y = pack_bf16x2(v[q * 8 + 10] * inv, v[q * 8 + 11] * inv);
              u1.z = pack_bf16x2(v[q * 8 + 12] * inv, v[q * 8 + 13] * inv);
              u1.w = pack_bf16x2(v[q * 8 + 14] * inv, v[q * 8 + 15] * inv);
              if (p.wide_io) {
                stg256(dst + q, u0, u1);
              } else {
                dst[q] = u0;
                dst[q + 1] = u1;
              }
            }
          }
        }
      }
      uint32_t a_cur[32];
      if (!kSoftmax) tmem_ld32(t_row, a_cur);
      for (int c = 0; c < (kSoftmax ? 0 : p.BN); c += 32) {
        tmem_ld_wait();
        ET(e_ld, et);
#ifdef B200SR_GEMM_TRACE
        ++e_chunks;
#endif
        const bool more = c + 32 < p.BN;
        if (has_res && c + 32 * kResAhead < p.BN) load_res(res[kResAhead], c + 32 * kResAhead);
        const int col0 = n0 + c;
        // The accumulator chunk leaves its registers in the first arithmetic step (for every lane: rows beyond M compute
        // on zeros), so the next chunk's TMEM load can target the same registers and run under the rest of this chunk:
        // one 32-register buffer instead of two and no copy at the end of the chunk.
        float v[32];
        if (kRs) {
          const int left = p.row_softmax_valid - col0;   // columns of this chunk that take part
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = j < left ? __uint_as_float(a_cur[j]) * p.alpha : -INFINITY;
        } else {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b4 = lds128(s_bias + c + j);
            if (ln_in) {
              const float4 c4 = lds128(s_col + c + j);
              v[j] = __uint_as_float(a_cur[j]);
              v[j + 1] = __uint_as_float(a_cur[j + 1]);
              v[j + 2] = __uint_as_float(a_cur[j + 2]);
              v[j + 3] = __uint_as_float(a_cur[j + 3]);
              ln_apply2(v[j], v[j + 1], ln_rstd, ln_nm, c4.x, c4.y, b4.x, b4.y);
              ln_apply2(v[j + 2], v[j + 3], ln_rstd, ln_nm, c4.z, c4.w, b4.z, b4.w);
            } else {
              v[j] = __uint_as_float(a_cur[j]) + b4.x;
              v[j + 1] = __uint_as_float(a_cur[j + 1]) + b4.y;
              v[j + 2] = __uint_as_float(a_cur[j + 2]) + b4.z;
              v[j + 3] = __uint_as_float(a_cur[j + 3]) + b4.w;
            }
          }
        }
        if (more) tmem_ld32(t_row + c + 32, a_cur);
        if (kRs) {
          if (valid && col0 < p.N) {
            if (kRsStats) {
              float cmax = v[0];
#pragma unroll
              for (int j = 1; j < 32; ++j) cmax = fmaxf(cmax, v[j]);
              const float m_new = fmaxf(rs_m, cmax);
              if (m_new > -INFINITY) {
                float s0 = 0.f, s1 = 0.f;
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                  s0 += ex2_approx_f(v[j] - m_new);
                  s1 += ex2_approx_f(v[j + 1] - m_new);
                }
                rs_l = rs_l * ex2_approx_f(rs_m - m_new) + (s0 + s1);
                rs_m = m_new;
              }
            } else {
              __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.ldc + col0;
              uint4 uu[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                float e[8];
#pragma unroll
                for (int t = 0; t < 8; ++t) e[t] = ex2_approx_f(v[q * 8 + t] - rs_m) * rs_l;   // 2^-inf = 0 for masked columns
                uu[q].x = pack_bf16x2(e[0], e[1]);
                uu[q].y = pack_bf16x2(e[2], e[3]);
                uu[q].z = pack_bf16x2(e[4], e[5]);
                uu[q].w = pack_bf16x2(e[6], e[7]);
              }
              if (p.wide_io) {
#pragma unroll
                for (int hq = 0; hq < 2; ++hq)
                  if (col0 + hq * 16 < p.N) stg256(dst + hq * 16, uu[2 * hq], uu[2 * hq + 1]);
              } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                  if (col0 + q * 8 < p.N) reinterpret_cast<uint4*>(dst)[q] = uu[q];
              }
            }
          }
        } else if ((valid || epi_tma) && col0 < p.N) {   // the TMA clips rows >= M itself; its issue must not depend on the lane
          if (kGeglu) {
            // columns [0,16) = value, [16,32) = gate of the same 16 output features
            const long long ocol = col0 >> 1;
            float o[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = v[j] * gelu_erf_f(v[16 + j]);
            __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.ldc + ocol;
            uint4 q0, q1;
            q0.x = pack_bf16x2(o[0], o[1]);
            q0.y = pack_bf16x2(o[2], o[3]);
            q0.z = pack_bf16x2(o[4], o[5]);
            q0.w = pack_bf16x2(o[6], o[7]);
            q1.x = pack_bf16x2(o[8], o[9]);
            q1.y = pack_bf16x2(o[10], o[11]);
            q1.z = pack_bf16x2(o[12], o[13]);
            q1.w = pack_bf16x2(o[14], o[15]);
            if (p.wide_io) {
              stg256(dst, q0, q1);
            } else {
              reinterpret_cast<uint4*>(dst)[0] = q0;
              reinterpret_cast<uint4*>(dst)[1] = q1;
            }
          } else {
            if (p.alpha != 1.0f) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] *= p.alpha;
            }
            if (rv_row != nullptr) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                if (col0 + j < p.N) {
                  const float4 r4 = __ldg(reinterpret_cast<const float4*>(rv_row + c + j));
                  v[j] += r4.x;
                  v[j + 1] += r4.y;
                  v[j + 2] += r4.z;
                  v[j + 3] += r4.w;
                }
              }
            }
            if (has_res) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 f0 = unpack_bf16x2(res[0][q].x), f1 = unpack_bf16x2(res[0][q].y),
                             f2 = unpack_bf16x2(res[0][q].z), f3 = unpack_bf16x2(res[0][q].w);
                v[q * 8 + 0] += f0.x;
                v[q * 8 + 1] += f0.y;
                v[q * 8 + 2] += f1.x;
                v[q * 8 + 3] += f1.y;
                v[q * 8 + 4] += f2.x;
                v[q * 8 + 5] += f2.y;
                v[q * 8 + 6] += f3.x;
                v[q * 8 + 7] += f3.y;
              }
            }
            if (!kExtras) {
              // activations only in the general families
            } else if (p.act == 1) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = silu_f(v[j]);
            } else if (p.act == 2) {   // exact (erf) GELU: OpenCLIP text tower MLP
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = gelu_erf_f(v[j]);
            } else if (p.act == 3) {   // quick GELU x * sigmoid(1.702 x): CLIP-L text tower MLP
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = quick_gelu_f(v[j]);
            }
            ET(e_math, et);
            if (epi_tma) {
              // Row r of the warp's 32 x 32 block = 128 bytes; its 16-byte chunk q goes to chunk (q ^ (r & 7)), which is
              // what the tensor map's 128B swizzle reads back.  EPI_SLABS slabs per warp keep that many stores in flight.
              uint8_t* slab = s_out + ((warp - 2) * EPI_SLABS + (slab_i % EPI_SLABS)) * 4096;
              if (lane == 0) tma_store_wait_read<EPI_SLABS - 1>();   // the store that last used this slab has read it
              __syncwarp();
#pragma unroll
              for (int q = 0; q < 8; ++q)
                sts128(slab + lane * 128 + ((q ^ (lane & 7)) << 4), v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                tma_store_2d(&tmO, slab, col0, m_blk * BLOCK_M + sub * 32);
                tma_store_commit();
              }
              ++slab_i;
            } else if (kF32 && p.out_fp32) {
              float* dst = reinterpret_cast<float*>(p.out) + row * p.ldc + col0;
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                if (col0 + q * 4 < p.N)
                  reinterpret_cast<float4*>(dst)[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
              }
            } else {
              __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + row * p.ldc + col0;
              uint4 uu[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                uu[q].x = pack_bf16x2(v[q * 8 + 0], v[q * 8 + 1]);
                uu[q].y = pack_bf16x2(v[q * 8 + 2], v[q * 8 + 3]);
                uu[q].z = pack_bf16x2(v[q * 8 + 4], v[q * 8 + 5]);
                uu[q].w = pack_bf16x2(v[q * 8 + 6], v[q * 8 + 7]);
              }
              if (p.wide_io) {
#pragma unroll
                for (int hq = 0; hq < 2; ++hq)
                  if (col0 + hq * 16 < p.N) stg256(dst + hq * 16, uu[2 * hq], uu[2 * hq + 1]);
              }
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                if (col0 + q * 8 < p.N) {
                  if (!p.wide_io) reinterpret_cast<uint4*>(dst)[q] = uu[q];
                  if (ln_out) {
                    // Statistics of the fp32 values before their rounding to bf16 (the rounding errors average out over
                    // the row: the mean moves by ~2^-9 |x| / sqrt(N)), two columns per packed fp32 instruction.
#pragma unroll
                    for (int t = 0; t < 8; t += 2) stats_acc2(ln_acc1, ln_acc2, v[q * 8 + t], v[q * 8 + t + 1]);
                  }
                }
              }
            }
          }
        }
        ET(e_st, et);
        if (more) {
#pragma unroll
          for (int d = 0; d < kResAhead; ++d) {
#pragma unroll
            for (int q = 0; q < 4; ++q) res[d][q] = res[d + 1][q];
          }
        }
      }
      if (kRsStats && valid) p.ln_stats_out[static_cast<long long>(n_blk) * p.M + row] = make_float2(rs_m, rs_l);
      if (ln_out && valid)
        p.ln_stats_out[static_cast<long long>(n_blk) * p.M + row] = make_float2(ln_acc1.x + ln_acc1.y, ln_acc2.x + ln_acc2.y);
      // release this accumulator stage back to the MMA warp
      if (threadIdx.x == 64) GT(10);
#ifdef B200SR_GEMM_TRACE
      if (threadIdx.x == 64 && p.trace != nullptr) {
        long long* tr = p.trace + blockIdx.x * 32 + 16;
        tr[0] = e_ld; tr[1] = e_math; tr[2] = e_st; tr[3] = e_pro; tr[4] = e_chunks; tr[5] = e_tiles;
      }
#endif
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kCluster == 1)
          mbar_arrive(&tmem_empty[acc]);
        else
          mbar_arrive_cluster(mapa_cluster(smem_u32(&tmem_empty[acc]), 0));  // the leader's MMA thread waits on it
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  if (kF32 && p.epi_tma != 0 && warp >= 2 && lane == 0) tma_store_wait_all();  // slabs read, results written
  tc_fence_before();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();  // the pair's MMAs / remote arrives must be finished in both CTAs
  tc_fence_after();
  if (warp == 1) {
    if (kCluster == 1)
      tmem_dealloc(tmem_base, TMEM_COLS);
    else
      tmem2_dealloc(tmem_base, TMEM_COLS);
  }
#ifdef B200SR_GEMM_TRACE
  if (threadIdx.x == 0 && p.trace != nullptr) {
    long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.trace[blockIdx.x * 32 + 13] = gt;
    GT(11);
  }
#endif
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int ilog2_exact(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return ((1 << l) == v) ? l : -1;
}

// Pick the N tile: minimise waves x per-tile cost.  Per k-iteration (K = 64) a CTA is bounded by
// the MMA (4 x BN/2 cycles) and by shared-memory traffic: TMA writes + SS-mode operand reads of
// its A tile and its share of the weight tile, 2 x (16 KiB + BN*128/cluster B) at 128 B/cycle.
static int pick_bn(int m_blocks, int N, int k_iters, int sms, int cluster) {
  int best = 128;
  double best_cost = 1e30;
  const int slots = sms / cluster;
  const int m_groups = (m_blocks + cluster - 1) / cluster;
  for (int bn = 32; bn <= 256; bn += 32) {
    if (bn > ((N + 31) / 32) * 32 && bn != 32) continue;
    const int n_blocks = (N + bn - 1) / bn;
    const long long work = static_cast<long long>(m_groups) * n_blocks;
    const long long waves = (work + slots - 1) / slots;
    const double mma = 4.0 * (bn / 2.0);
    const double smem = 2.0 * (16384.0 + bn * 128.0 / cluster) / 128.0;
    const double tile_cost = fmax(mma, smem) * k_iters + 2500.0 + bn * 8.0;
    const double cost = waves * tile_cost;
    if (cost < best_cost - 1e-9) {
      best_cost = cost;
      best = bn;
    }
  }
  return best;
}

#ifdef B200SR_GEMM_TRACE
static long long* g_gemm_trace = nullptr;
#endif

template <int kCluster, int kEpi>
static cudaError_t launch_epi(int grid, size_t smem_bytes, cudaStream_t stream, const CUtensorMap& tmA, const CUtensorMap& tmB,
                              const CUtensorMap& tmO, const GemmParams& p) {
  static bool attr_set[64] = {false};  // per device and per instantiation
  if (first_use_on_device(attr_set)) {
    const cudaError_t e =
        cudaFuncSetAttribute(gemm_conv_kernel<kCluster, kEpi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
  }
  return launch_k(gemm_conv_kernel<kCluster, kEpi>, dim3(grid), dim3(kEpi == EPI_XFORM ? GEMM_THREADS_XFORM : GEMM_THREADS),
                  smem_bytes, stream, kCluster, tmA, tmB, tmO, p);
}

template <int kCluster>
static int launch_t(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, GemmParams& p,
                    cudaStream_t stream) {
  // per-channel (a, b) of one image (fused GroupNorm, mode 3) or the weight tile's column sums (LayerNorm fold, mode 0)
  const int xform_bytes = p.gn_stats != nullptr ? ((p.Cin * 8 + 1023) / 1024) * 1024
                          : (p.ln_stats != nullptr && p.row_softmax == 0) ? 4096
                          : p.epi_tma ? 4 * EPI_SLABS * 4096 + 1024   // TMA-store slabs + their alignment
                                      : 0;
  const int smem_budget = 227 * 1024 - 1024 /*align slack*/ - BAR_REGION_BYTES - 4096 /*epilogue bias staging*/ - xform_bytes;
  const int b_sub_bytes = (p.BN / kCluster) * BLOCK_K * 2;
  const int stage_bytes = KSUB * (A_STAGE_BYTES + b_sub_bytes);
  size_t ring_bytes;
  if (p.mode == 3) {
    const int b_stage_bytes = HALO_TAPS * b_sub_bytes;
    p.a_stages = p.kc_per_tap >= 2 ? 2 : 1;
    // fused input GroupNorm: TMA latency + the in-place transform sit between a tile's landing and its MMAs, so a third
    // halo stage pays — unless it squeezes the weight ring below three stages (BN = 256: a kernel row of weights is
    // 48 KB; two rows in flight no longer cover the TMA latency, measured +15 us per 1280-channel convolution)
    if (p.gn_stats != nullptr && (smem_budget - 3 * A_HALO_BYTES) / b_stage_bytes >= 3) p.a_stages = 3;
    int stages = (smem_budget - p.a_stages * A_HALO_BYTES) / b_stage_bytes;
    if (stages > MAX_B_STAGES) stages = MAX_B_STAGES;
    if (stages < 2) return B200SR_EINVAL;
    // Resident weights: a convolution with ONE N block (Cout <= the N tile) whose whole weight set — 3 * kc_per_tap ring
    // stages — fits next to the halo ring keeps it in shared memory for the life of the CTA.  The SR3 / first-stage
    // full-resolution convolutions (64 .. 192 -> 64 / 128 channels at 512^2 .. 1024^2, 55 tiles per SM) otherwise re-stream
    // 36 - 147 KB of weights for every 23 - 46 KB activation tile and wait on a weight barrier per kernel row.
    static const bool resident_enabled = [] {
      const char* e = getenv("B200SR_CONV_RESIDENT");
      return e == nullptr || e[0] != '0';
    }();
    p.w_resident = 0;
    if (resident_enabled && p.num_n_blocks == 1 && 3 * p.kc_per_tap <= stages && 3 * p.kc_per_tap <= MAX_B_STAGES) {
      p.w_resident = 1;
      stages = 3 * p.kc_per_tap;
      // the freed space goes to the halo ring (up to 4 tiles in flight)
      while (p.a_stages < MAX_A_HALO_STAGES && (smem_budget - (p.a_stages + 1) * A_HALO_BYTES) / b_stage_bytes >= stages)
        ++p.a_stages;
    }
    p.stages = stages;
    ring_bytes = static_cast<size_t>(p.a_stages) * A_HALO_BYTES + static_cast<size_t>(stages) * b_stage_bytes;
  } else {
    const int s_iters = (p.k_iters + KSUB - 1) / KSUB;
    int stages = smem_budget / stage_bytes;
    if (stages > MAX_STAGES) stages = MAX_STAGES;
    if (stages > s_iters + 1) stages = s_iters + 1;
    if (stages < 2) stages = 2;
    p.stages = stages;
    p.a_stages = 0;
    ring_bytes = static_cast<size_t>(stages) * stage_bytes;
  }
  const size_t smem_bytes = ring_bytes + 1024 + BAR_REGION_BYTES + 4096 + xform_bytes;
#ifdef B200SR_GEMM_TRACE
  p.trace = g_gemm_trace;
#endif
  const int work = (p.num_m_blocks / kCluster) * p.num_n_blocks;
  const int slots = num_sms() / kCluster;
  const int grid = (work < slots ? work : slots) * kCluster;
  const bool ln = p.row_softmax == 0 && (p.ln_stats != nullptr || p.ln_stats_out != nullptr);
  cudaError_t err;
  if (p.row_softmax == 1)
    err = launch_epi<kCluster, EPI_RS_STATS>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else if (p.row_softmax == 2)
    err = launch_epi<kCluster, EPI_RS_APPLY>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else if (p.gn_stats != nullptr)
    err = launch_epi<kCluster, EPI_XFORM>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else if (p.softmax_valid > 0)
    err = ln ? launch_epi<kCluster, EPI_LN_SOFTMAX>(grid, smem_bytes, stream, tmA, tmB, tmO, p)
             : launch_epi<kCluster, EPI_SOFTMAX>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else if (p.geglu)
    err = ln ? launch_epi<kCluster, EPI_LN_GEGLU>(grid, smem_bytes, stream, tmA, tmB, tmO, p)
             : launch_epi<kCluster, EPI_GEGLU>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else if (ln)
    err = launch_epi<kCluster, EPI_LN_PLAIN>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else if (p.rowvec != nullptr || p.act != 0 || p.out_fp32)
    err = launch_epi<kCluster, EPI_GENERAL>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  else
    err = launch_epi<kCluster, EPI_PLAIN>(grid, smem_bytes, stream, tmA, tmB, tmO, p);
  return err == cudaSuccess ? B200SR_OK : B200SR_ELAUNCH;
}

static int fill_epilogue(GemmParams& p, const b200sr_epilogue& e) {
  p.bias = e.bias;
  p.rowvec = e.rowvec;
  p.rows_per_group = e.rows_per_group;
  p.ld_rowvec = e.ld_rowvec != 0 ? e.ld_rowvec : p.N;
  if (e.rowvec != nullptr && ((p.ld_rowvec % 4) != 0 || p.ld_rowvec < p.N)) return B200SR_EINVAL;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(e.residual);
  p.ldr = e.ldr;
  p.out = e.out;
  p.ldc = e.ldc;
  p.out_fp32 = e.out_fp32;
  p.geglu = e.geglu;
  p.alpha = e.alpha;
  p.act = e.act;
  p.softmax_valid = e.softmax_valid;
  p.w_dynamic = e.w_dynamic;
  p.w_rows_per_group = e.w_rows_per_group;
  p.w_group_stride = e.w_group_stride;
  p.gn_stats = e.a_gn_stats;
  p.gn_weight = e.a_gn_weight;
  p.gn_bias = e.a_gn_bias;
  p.gn_groups = e.a_gn_groups;
  p.gn_silu = e.a_gn_silu;
  p.ln_stats = reinterpret_cast<const float2*>(e.ln_stats);
  p.ln_parts = e.ln_parts;
  p.ln_colsum = e.ln_colsum;
  p.ln_shift = e.ln_shift;
  p.ln_eps = e.ln_eps;
  p.ln_stats_out = reinterpret_cast<float2*>(e.ln_stats_out);
  p.row_softmax = e.row_softmax;
  p.row_softmax_valid = e.row_softmax_valid > 0 ? e.row_softmax_valid : p.N;
  // The epilogue moves out, residual and rowvec in 16-byte vectors (uint4 / float4) from row starts that the ld checks
  // keep 16-byte aligned relative to the base, and the row statistics in 8-byte float2 pairs.
  const auto misaligned = [](const void* ptr, uintptr_t bytes) { return (reinterpret_cast<uintptr_t>(ptr) & (bytes - 1)) != 0; };
  if (misaligned(e.out, 16) || misaligned(e.residual, 16) || misaligned(e.rowvec, 16) || misaligned(e.ln_stats, 8) ||
      misaligned(e.ln_stats_out, 8))
    return B200SR_EINVAL;
  if (e.row_softmax != 0) {
    // two-pass row softmax: plain GEMM, no other epilogue term; pass 1 writes statistics only, pass 2 bf16 probabilities
    if (p.mode != 0 || e.row_softmax < 0 || e.row_softmax > 2 || e.geglu || e.out_fp32 || e.residual != nullptr ||
        e.rowvec != nullptr || e.bias != nullptr || e.act != 0 || e.softmax_valid != 0 || e.a_gn_stats != nullptr ||
        e.ln_colsum != nullptr || e.ln_shift != nullptr)
      return B200SR_EINVAL;
    if (e.row_softmax == 1 && (e.ln_stats_out == nullptr || e.ln_stats != nullptr)) return B200SR_EINVAL;
    if (e.row_softmax == 2 && (e.ln_stats == nullptr || e.ln_parts <= 0 || e.ln_stats_out != nullptr || e.out == nullptr))
      return B200SR_EINVAL;
    if ((p.N % 8) != 0 || (e.row_softmax == 2 && ((e.ldc % 8) != 0 || e.ldc < p.N))) return B200SR_EINVAL;
    p.out = e.out;
    p.ldc = e.ldc;
    p.alpha = e.alpha;
    p.w_dynamic = e.w_dynamic;
    return B200SR_OK;
  }
  if (e.ln_stats != nullptr &&
      (p.mode != 0 || e.ln_parts <= 0 || e.ln_colsum == nullptr || e.ln_shift == nullptr || e.a_gn_stats != nullptr))
    return B200SR_EINVAL;
  if (e.ln_stats_out != nullptr && (p.mode != 0 || e.geglu || e.softmax_valid > 0)) return B200SR_EINVAL;
  // the LayerNorm-folding instantiation carries bias, alpha, residual, geglu and the softmax only
  if ((e.ln_stats != nullptr || e.ln_stats_out != nullptr) && (e.out_fp32 || e.rowvec != nullptr || e.act != 0))
    return B200SR_EINVAL;
  if (e.a_gn_stats != nullptr) {
    // fused input GroupNorm: halo convolution only, affine parameters required
    if (p.mode != 3 || e.a_gn_weight == nullptr || e.a_gn_bias == nullptr || e.a_gn_groups <= 0 ||
        (p.Cin % e.a_gn_groups) != 0)
      return B200SR_EINVAL;
  }
  if (e.softmax_valid < 0 || e.softmax_valid > SOFTMAX_SEG) return B200SR_EINVAL;
  if (e.softmax_valid > 0 && (e.geglu || e.out_fp32 || e.residual != nullptr || e.rowvec != nullptr || e.bias != nullptr ||
                              e.act != 0 || (p.N % SOFTMAX_SEG) != 0))
    return B200SR_EINVAL;
  if (e.w_rows_per_group < 0 || (e.w_rows_per_group % (2 * BLOCK_M)) != 0) return B200SR_EINVAL;
  if (e.geglu && e.act) return B200SR_EINVAL;
  if (e.act < 0 || e.act > 3) return B200SR_EINVAL;
  if (e.out == nullptr) return B200SR_EINVAL;
  if (e.geglu && (e.out_fp32 || e.residual != nullptr || e.rowvec != nullptr || (p.N % 32) != 0)) return B200SR_EINVAL;
  if (p.N % 8 != 0) return B200SR_EINVAL;
  if ((e.ldc % 8) != 0 || (e.residual != nullptr && (e.ldr % 8) != 0)) return B200SR_EINVAL;
  // rows must not overlap: out has N (GEGLU: N / 2) columns, the residual N
  if (e.ldc < (e.geglu ? p.N / 2 : p.N) || (e.residual != nullptr && e.ldr < p.N)) return B200SR_EINVAL;
  return B200SR_OK;
}

// Shared tail of both entry points: choose cluster / BN, encode the weight map, launch.
static int finish(const CUtensorMap& tmA, const void* W, GemmParams& p, int real_m_blocks, int force_bn,
                  cudaStream_t stream) {
  const int cluster = real_m_blocks >= 2 ? 2 : 1;
  p.num_m_blocks = ((real_m_blocks + cluster - 1) / cluster) * cluster;
  p.BN = force_bn > 0 ? force_bn : pick_bn(real_m_blocks, p.N, p.k_iters, num_sms(), cluster);
  if (p.softmax_valid > 0) p.BN = p.N >= 3 * SOFTMAX_SEG ? 3 * SOFTMAX_SEG : p.N;  // whole head segments per tile
  // halo convolution: two weight stages of three taps each must fit next to the halo ring
  if (p.mode == 3 && cluster == 1 && p.BN > 192 && force_bn <= 0) p.BN = 192;
  if (p.BN % (p.softmax_valid > 0 ? 16 : 32) != 0 || p.BN > 256 || p.BN <= 0) return B200SR_EINVAL;
  p.num_n_blocks = (p.N + p.BN - 1) / p.BN;
  CUtensorMap tmB;
  // stacked per-group weights: the map spans every group's rows
  const long long w_rows = p.w_rows_per_group > 0
                               ? ((static_cast<long long>(p.M) + p.w_rows_per_group - 1) / p.w_rows_per_group - 1) *
                                         p.w_group_stride + p.N
                               : p.N;
  uint64_t dims[2] = {static_cast<uint64_t>(p.K), static_cast<uint64_t>(w_rows)};
  uint64_t strides[1] = {static_cast<uint64_t>(p.K) * 2};
  uint32_t box[2] = {BLOCK_K, static_cast<uint32_t>(p.BN / cluster)};
  int rc = make_tmap_bf16(&tmB, W, 2, dims, strides, box);
  if (rc) return rc;
  // fp32 output of a GEMM with at least two tiles per CTA (SR3 / first-stage attention scores, 16384 x 16384): the
  // per-thread row stores of the plain epilogue (32 scattered 16-byte pieces per instruction) reach 1.9 TB/s and bound
  // the kernel; TMA stores of staged 32 x 32 blocks write whole lines.  One-tile launches keep the direct stores
  // (no shared-memory hop on their critical path).
  static const bool epi_tma_enabled = [] {
    const char* e = getenv("B200SR_EPI_TMA");
    return e == nullptr || e[0] != '0';
  }();
  {
    const long long n_out = p.geglu ? p.N / 2 : p.N;
    const long long esz = p.out_fp32 ? 4 : 2;
    p.wide_io = !p.out_fp32 && (n_out % 16) == 0 && (p.ldc * esz) % 32 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 31) == 0 &&
                (p.residual == nullptr || ((p.ldr * 2) % 32 == 0 && (reinterpret_cast<uintptr_t>(p.residual) & 31) == 0));
    static const bool wide_enabled = [] {
      const char* e = getenv("B200SR_WIDE_IO");
      return e == nullptr || e[0] != '0';
    }();
    if (!wide_enabled) p.wide_io = 0;
  }
  CUtensorMap tmO = tmA;
  p.epi_tma = 0;
  if (epi_tma_enabled && p.mode == 0 && p.out_fp32 && !p.geglu && p.softmax_valid <= 0 && p.ln_stats == nullptr &&
      p.ln_stats_out == nullptr && p.residual == nullptr && p.rowvec == nullptr && (p.ldc % 4) == 0 &&
      static_cast<long long>(p.num_m_blocks / cluster) * p.num_n_blocks >= 2LL * (num_sms() / cluster)) {
    uint64_t odims[2] = {static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.M)};
    uint64_t ostrides[1] = {static_cast<uint64_t>(p.ldc) * 4};
    uint32_t obox[2] = {32, 32};
    if (make_tmap_f32(&tmO, p.out, 2, odims, ostrides, obox) == B200SR_OK) p.epi_tma = 1;
  }
  return cluster == 2 ? launch_t<2>(tmA, tmB, tmO, p, stream) : launch_t<1>(tmA, tmB, tmO, p, stream);
}

}  // namespace b200sr

using namespace b200sr;

// The N tile b200sr_gemm_bf16 picks for a plain GEMM (no softmax epilogue, force_bn = 0): a GEMM that writes row
// statistics writes ceil(N / tile) partials per row, which the consuming GEMM has to be told.
extern "C" int b200sr_gemm_n_tile(int32_t M, int32_t N, int32_t K) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  const int m_blocks = (M + BLOCK_M - 1) / BLOCK_M;
  return pick_bn(m_blocks, N, (K + BLOCK_K - 1) / BLOCK_K, num_sms(), m_blocks >= 2 ? 2 : 1);
}

extern "C" int b200sr_gemm_bf16(const void* A, int64_t lda, const void* W, int32_t M, int32_t N, int32_t K,
                                const b200sr_epilogue* epi, int32_t force_bn, void* stream_ptr) {
  if (A == nullptr || W == nullptr || epi == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (M <= 0 || N <= 0 || K <= 0 || (K % 8) != 0 || (lda % 8) != 0) return B200SR_EINVAL;
  GemmParams p{};
  p.mode = 0;
  p.M = M;
  p.N = N;
  p.K = K;
  p.k_iters = (K + BLOCK_K - 1) / BLOCK_K;
  int rc = fill_epilogue(p, *epi);
  if (rc) return rc;
  CUtensorMap tmA;
  uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(M)};
  uint64_t strides[1] = {static_cast<uint64_t>(lda) * 2};
  uint32_t box[2] = {BLOCK_K, BLOCK_M};
  rc = make_tmap_bf16(&tmA, A, 2, dims, strides, box);
  if (rc) return rc;
  return finish(tmA, W, p, (M + BLOCK_M - 1) / BLOCK_M, force_bn, stream);
}

// x: NHWC bf16 [NB, H, W, Cin]; w: [Cout, 3, 3, Cin] bf16 (K = tap*Cin + c); stride 1 or 2, pad 1.
extern "C" int b200sr_conv3x3_bf16(const void* x, const void* w, int32_t NB, int32_t H, int32_t W, int32_t Cin,
                                   int32_t Cout, int32_t stride, int32_t pad_lo, const b200sr_epilogue* epi,
                                   int32_t force_bn, void* stream_ptr) {
  if (x == nullptr || w == nullptr || epi == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (NB <= 0 || H <= 0 || W <= 0 || Cin <= 0 || (Cin % BLOCK_K) != 0 || Cout <= 0) return B200SR_EINVAL;
  if (stride != 1 && stride != 2) return B200SR_EINVAL;
  if (pad_lo != 1 && !(pad_lo == 0 && stride == 2)) return B200SR_EINVAL;
  if (stride == 2 && ((H | W) & 1)) return B200SR_EINVAL;
  if (epi->geglu) return B200SR_EINVAL;
  const int OH = H / stride, OW = W / stride;
  // tile box: bw | OW, bw*bh*bn == 128, all powers of two
  int bw = 1;
  while (bw * 2 <= 128 && (OW % (bw * 2)) == 0) bw *= 2;
  int bh = 1;
  while (bw * bh * 2 <= 128 && bh < OH) bh *= 2;
  int bn = 128 / (bw * bh);
  // stride-1 convolutions on images at least one 8 x 16 tile large take the halo path (mode 3)
  static const bool halo_enabled = [] {
    const char* e = getenv("B200SR_CONV_HALO");
    return e == nullptr || e[0] != '0';
  }();
  const bool halo = halo_enabled && stride == 1 && (W % HALO_TILE_W) == 0 && H >= HALO_TILE_H;
  if (halo) {
    bw = HALO_TILE_W;
    bh = HALO_TILE_H;
    bn = 1;
  }
  GemmParams p{};
  p.mode = halo ? 3 : (stride == 1 ? 1 : 2);
  p.NB = NB;
  p.OH = OH;
  p.OW = OW;
  p.Cin = Cin;
  p.pad_lo = pad_lo;
  p.M = NB * OH * OW;
  p.N = Cout;
  p.K = 9 * Cin;
  p.bw_log2 = ilog2_exact(bw);
  p.bh_log2 = ilog2_exact(bh);
  p.bn_log2 = ilog2_exact(bn);
  p.tiles_w = OW / bw;
  p.tiles_h = (OH + bh - 1) / bh;
  p.tiles_n = (NB + bn - 1) / bn;
  p.kc_per_tap = Cin / BLOCK_K;
  p.k_iters = 9 * p.kc_per_tap;
  int rc = fill_epilogue(p, *epi);
  if (rc) return rc;
  CUtensorMap tmA;
  if (stride == 1) {
    uint64_t dims[4] = {static_cast<uint64_t>(Cin), static_cast<uint64_t>(W), static_cast<uint64_t>(H),
                        static_cast<uint64_t>(NB)};
    uint64_t strides[3] = {static_cast<uint64_t>(Cin) * 2, static_cast<uint64_t>(W) * Cin * 2,
                           static_cast<uint64_t>(H) * W * Cin * 2};
    uint32_t box[4] = {BLOCK_K, static_cast<uint32_t>(bw), static_cast<uint32_t>(bh), static_cast<uint32_t>(bn)};
    if (halo) {
      box[1] = HALO_W;
      box[2] = HALO_H;
    }
    rc = make_tmap_bf16(&tmA, x, 4, dims, strides, box);
  } else {
    // [NB, H/2, 2, W/2, 2*Cin]: (w parity, channel) merge into one contiguous dim of 2*Cin
    uint64_t dims[5] = {static_cast<uint64_t>(2 * Cin), static_cast<uint64_t>(W / 2), 2,
                        static_cast<uint64_t>(H / 2), static_cast<uint64_t>(NB)};
    uint64_t strides[4] = {static_cast<uint64_t>(2 * Cin) * 2, static_cast<uint64_t>(W) * Cin * 2,
                           static_cast<uint64_t>(2) * W * Cin * 2, static_cast<uint64_t>(H) * W * Cin * 2};
    uint32_t box[5] = {BLOCK_K, static_cast<uint32_t>(bw), 1, static_cast<uint32_t>(bh), static_cast<uint32_t>(bn)};
    rc = make_tmap_bf16(&tmA, x, 5, dims, strides, box);
  }
  if (rc) return rc;
  // Out-of-range spatial tiles (cluster round-up) decode to tn >= tiles_n: all rows masked, loads zero-filled.
  return finish(tmA, w, p, p.tiles_w * p.tiles_h * p.tiles_n, force_bn, stream);
}

#ifdef B200SR_GEMM_TRACE
extern "C" void b200sr_debug_set_gemm_trace(void* p) { b200sr::g_gemm_trace = reinterpret_cast<long long*>(p); }
#endif
