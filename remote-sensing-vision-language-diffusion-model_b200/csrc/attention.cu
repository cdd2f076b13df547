// b200sr — flash-style attention (online softmax) on tcgen05/TMEM for head_dim 64, non-causal.
//
// Reference semantics: softmax(Q K^T / sqrt(64)) V per head, heads = C / 64, no mask, no dropout
//   sgm/modules/attention.py:222-285 (CrossAttention -> F.scaled_dot_product_attention)
//   models/modules/SR_modules.py:135-149 (ZeroCrossAttn uses the same CrossAttention)
//
// One CTA = 128 query rows of one (batch, head).  Per 128-key block:
//   S[128x128] = Q K^T          tcgen05.mma SS  (Q, K tiles in smem, K-major, 128B swizzle)
//   P = exp2(S*c - m)           4 softmax warps, one thread per query row, S read from TMEM,
//                               P written back to TMEM as packed bf16 (never touches smem)
//   O[128x64] += P V            tcgen05.mma TS  (A = P in TMEM, B = V tile in smem, MN-major)
// O stays in TMEM for the whole KV loop; it is rescaled only when the running row maximum has
// grown by more than 2^8 since the last rescale (the softmax sum uses the same stale maximum, so
// the final O / l is exact).  Two CTAs are resident per SM (80 KiB smem, 256 TMEM columns each)
// so one CTA's exponentials overlap the other's MMAs.
//
// Wave quantisation: with 2 CTAs per SM the grid runs in waves of 296 tiles; the tiles of a last,
// partial wave are split over their key blocks (attention_plan) and merged by the last CTA to arrive.
//
// Q, K and V are addressed as column windows of row-major bf16 matrices ([B, N, ld] with a
// column offset), so the fused QKV GEMM output is consumed in place.
#include "common.cuh"

namespace b200sr {

static constexpr int ATT_BM = 128;   // query rows per CTA
static constexpr int ATT_BN = 128;   // keys per block
static constexpr int ATT_D = 64;     // head dim
static constexpr int ATT_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 softmax (two threads per query row)
static constexpr int ATT_STAGES = 2;
static constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // 16 KiB
static constexpr int ATT_TMEM_COLS = 256;
static constexpr int ATT_COL_S = 0;     // 128 fp32 columns
static constexpr int ATT_COL_P = 128;   // 64 columns of packed bf16 pairs
static constexpr int ATT_COL_O = 192;   // 64 fp32 columns
static constexpr int ATT_PART_FLOATS = 66 * 128;  // per split partial: O^T [64][128] fp32, m [128], l [128]
static constexpr int ATT_WS_COUNTERS = 512;       // uint32 arrival counters at the start of the workspace

struct AttnParams {
  int B, H, Nq, Nk;
  int q_col, k_col, v_col;  // column offsets (elements) of head 0 inside each matrix row
  __nv_bfloat16* out;
  long long ldo;  // elements per output row ([B*Nq, ldo], head h at columns h*64)
  float scale_log2;  // softmax scale * log2(e)
  int causal;        // != 0: key k takes part in query q only if k <= q (text towers of the conditioner)
  // Tail splitting (see attention_plan): CTAs [0, full_ctas) each own a whole 128-row tile; the
  // remaining tiles are each shared by `split` CTAs that take `blocks_per_split` key blocks apiece,
  // publish (O, m, l) partials to `partials` and the last to arrive merges them.
  int n_qtiles, full_ctas, split, blocks_per_split;
  float* partials;          // [tail tiles][split][ATT_PART_FLOATS]
  unsigned int* counters;   // [tail tiles], zero between launches
#ifdef B200SR_ATT_TRACE
  long long* trace;  // [4 CTAs][10 warps][64 blocks][8 events] clock64 stamps (debug builds only)
#endif
};

#ifdef B200SR_ATT_TRACE
static long long* g_att_trace = nullptr;
#define ATT_T(ev)                                                                                   \
  do {                                                                                              \
    if (p.trace != nullptr && lane == 0 && cta_lin < 4 && j < 64)                                   \
      p.trace[((cta_lin * 10 + warp) * 64 + j) * 8 + (ev)] = clock64();                             \
  } while (0)
__device__ __forceinline__ long long att_gtime() {
  long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define ATT_CTA(ev)                                                                                 \
  do {                                                                                              \
    if (p.trace != nullptr && threadIdx.x == 64 && cta_lin < 4096) {                                \
      p.trace[20480 + cta_lin * 3 + (ev)] = att_gtime();                                            \
      if ((ev) == 0) {                                                                              \
        uint32_t smid;                                                                              \
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));                                            \
        p.trace[20480 + cta_lin * 3 + 2] = smid;                                                    \
      }                                                                                             \
    }                                                                                               \
  } while (0)
#else
#define ATT_T(ev) do { } while (0)
#define ATT_CTA(ev) do { } while (0)
#endif

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(ATT_THREADS, 2)
attention_d64_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sKV = smem + ATT_TILE_BYTES;  // stage s: K at s*32K, V at s*32K + 16K
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + ATT_STAGES * 2 * ATT_TILE_BYTES);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;                 // [ATT_STAGES]
  uint64_t* kv_empty = kv_full + ATT_STAGES;    // [ATT_STAGES]
  uint64_t* s_full = kv_empty + ATT_STAGES;
  uint64_t* p_full = s_full + 1;
  uint64_t* o_done = p_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 1);
  float* s_xch = reinterpret_cast<float*>(tmem_slot + 2);  // [2][2][128] row-max / row-sum exchange

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // work decode: whole tile, or one key-block range of a tail tile
  int tile = blockIdx.x, jb0 = 0, split_idx = -1, tail_idx = 0;
  int nblk = (p.Nk + ATT_BN - 1) / ATT_BN;  // key blocks this CTA walks (global block = jb0 + j)
  if (static_cast<int>(blockIdx.x) >= p.full_ctas) {
    const int t = blockIdx.x - p.full_ctas;
    tail_idx = t / p.split;
    split_idx = t - tail_idx * p.split;
    tile = p.full_ctas + tail_idx;
    jb0 = split_idx * p.blocks_per_split;
    nblk = min(nblk - jb0, p.blocks_per_split);
  }
  const int q0 = (tile % p.n_qtiles) * ATT_BM;
  const int h = (tile / p.n_qtiles) % p.H, b = tile / (p.n_qtiles * p.H);
#ifdef B200SR_ATT_TRACE
  const int cta_lin = blockIdx.x;
#endif
  ATT_CTA(0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    mbar_init(q_full, 1);
    for (int s = 0; s < ATT_STAGES; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 8);  // one arrive per softmax warp
    mbar_init(o_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, ATT_TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_launch_dependents();

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      pdl_wait();  // Q, K, V are produced by the previous kernel
      mbar_expect_tx(q_full, ATT_TILE_BYTES);
      tma_load_3d(sQ, &tmQ, q_full, p.q_col + h * ATT_D, q0, b);
      int stage = 0;
      uint32_t phase = 0;
      for (int j = 0; j < nblk; ++j) {
        mbar_wait(&kv_empty[stage], phase ^ 1);
        ATT_T(0);
        uint8_t* sK = sKV + stage * 2 * ATT_TILE_BYTES;
        uint8_t* sV = sK + ATT_TILE_BYTES;
        mbar_expect_tx(&kv_full[stage], 2 * ATT_TILE_BYTES);
        tma_load_3d(sK, &tmK, &kv_full[stage], p.k_col + h * ATT_D, (jb0 + j) * ATT_BN, b);
        tma_load_3d(sV, &tmV, &kv_full[stage], p.v_col + h * ATT_D, (jb0 + j) * ATT_BN, b);
        if (++stage == ATT_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (lane == 0) {
      const uint32_t idesc_s = umma_idesc_bf16_f32(ATT_BM, ATT_BN, 0, 0);  // Q (K-major) x K^T (K-major)
      const uint32_t idesc_o = umma_idesc_bf16_f32(ATT_BM, ATT_D, 0, 1);   // P (tmem)  x V (MN-major)
      const uint64_t qdesc = umma_smem_desc_sw128(smem_u32(sQ), 16, 1024);
      mbar_wait(q_full, 0);
      int stage = 0;
      uint32_t phase = 0;
      // S(0)
      mbar_wait(&kv_full[0], 0);
      tc_fence_after();
      {
        const uint64_t kdesc = umma_smem_desc_sw128(smem_u32(sKV), 16, 1024);
#pragma unroll
        for (int k = 0; k < ATT_D / 16; ++k) umma_ss(tmem + ATT_COL_S, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
        umma_commit(s_full);
      }
      for (int j = 0; j < nblk; ++j) {
        // O += P(j) V(j)
        mbar_wait(p_full, j & 1);
        ATT_T(0);
        tc_fence_after();
        {
          const uint32_t sV = smem_u32(sKV + stage * 2 * ATT_TILE_BYTES + ATT_TILE_BYTES);
          // V tile: row = key (128 B of d), 8-key groups 1024 B apart; MN-major B operand.
          const uint64_t vdesc = umma_smem_desc_sw128(sV, 1024, 1024);
#pragma unroll
          for (int k = 0; k < ATT_BN / 16; ++k) {
            // 16 keys per MMA: P advances 8 packed columns, V advances 16 rows = 2048 B
            umma_ts(tmem + ATT_COL_O, tmem + ATT_COL_P + 8 * k, vdesc + (2048 >> 4) * k, idesc_o, (j | k) != 0);
          }
          umma_commit(&kv_empty[stage]);
          if (j + 1 == nblk) umma_commit(o_done);
        }
        ATT_T(1);
        if (++stage == ATT_STAGES) {
          stage = 0;
          phase ^= 1;
        }
        if (j + 1 < nblk) {
          mbar_wait(&kv_full[stage], phase);
          ATT_T(2);
          tc_fence_after();
          const uint64_t kdesc = umma_smem_desc_sw128(smem_u32(sKV + stage * 2 * ATT_TILE_BYTES), 16, 1024);
#pragma unroll
          for (int k = 0; k < ATT_D / 16; ++k)
            umma_ss(tmem + ATT_COL_S, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
          umma_commit(s_full);
          ATT_T(3);
        }
      }
    }
  } else {
    // ================================ softmax / correction / epilogue ================================
    // Two threads per query row: warp w owns TMEM lane quadrant (w & 3) and key columns
    // [64*half, 64*half + 64) of every S block, half = (w - 2) >> 2.  The row maximum is exchanged
    // through shared memory once per block; row sums stay per-thread until the epilogue.
    const int sub = warp & 3;
    const int half = (warp - 2) >> 2;
    const int r = sub * 32 + lane;  // query row inside the tile == TMEM lane
    const uint32_t lane_base = static_cast<uint32_t>(sub * 32) << 16;
    float m_used = -INFINITY;  // maximum the exponentials are currently taken against (log2 units)
    float l = 0.f;             // this thread's share of the running sum of exponentials
    for (int j = 0; j < nblk; ++j) {
      mbar_wait(s_full, j & 1);
      ATT_T(0);
      tc_fence_after();
      float s[64];
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t a[32];
        tmem_ld32(tmem + lane_base + ATT_COL_S + half * 64 + c * 32, a);
#pragma unroll
        for (int i = 0; i < 32; ++i) s[c * 32 + i] = __uint_as_float(a[i]);
      }
      tmem_ld_wait();
      ATT_T(1);
      int kv_left = p.Nk - (jb0 + j) * ATT_BN - half * 64;
      if (p.causal) kv_left = min(kv_left, q0 + r + 1 - (jb0 + j) * ATT_BN - half * 64);   // keys 0 .. q only
      if (kv_left < 64) {
#pragma unroll
        for (int i = 0; i < 64; ++i)
          if (i >= kv_left) s[i] = -INFINITY;
      }
      float mx = s[0];
#pragma unroll
      for (int i = 1; i < 64; ++i) mx = fmaxf(mx, s[i]);
      float* xch = s_xch + (j & 1) * 256;
      xch[half * 128 + r] = mx;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      ATT_T(2);
      mx = fmaxf(mx, xch[(half ^ 1) * 128 + r]) * p.scale_log2;
      // lazy rescale: only when the maximum grew by more than 8 (factor 256) since the last one
      const bool grow = mx > m_used + 8.0f;
      if (j == 0) {
        m_used = mx;
      } else if (__any_sync(0xffffffffu, grow)) {
        float alpha = 1.0f;
        if (grow) {
          alpha = ex2_approx(m_used - mx);
          m_used = mx;
          l *= alpha;
        }
        uint32_t o[32];
        tmem_ld32(tmem + lane_base + ATT_COL_O + half * 32, o);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
        tmem_st32(tmem + lane_base + ATT_COL_O + half * 32, o);
      }
      float sum0 = 0.f, sum1 = 0.f;
      uint32_t pk[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float e0 = ex2_approx(fmaf(s[2 * i], p.scale_log2, -m_used));
        const float e1 = ex2_approx(fmaf(s[2 * i + 1], p.scale_log2, -m_used));
        sum0 += e0;
        sum1 += e1;
        pk[i] = pack_bf16x2(e0, e1);
      }
      ATT_T(3);
      tmem_st32(tmem + lane_base + ATT_COL_P + half * 32, pk);
      l += sum0 + sum1;
      tmem_st_wait();
      ATT_T(4);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      ATT_T(5);
    }
    // epilogue: O / l -> bf16 -> global; each thread writes 32 of the 64 output columns of its row
    float* xch = s_xch + (nblk & 1) * 256;
    xch[half * 128 + r] = l;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    l += xch[(half ^ 1) * 128 + r];
    mbar_wait(o_done, 0);
    tc_fence_after();
    const int q = q0 + r;
    uint32_t o[32];
    tmem_ld32(tmem + lane_base + ATT_COL_O + half * 32, o);
    tmem_ld_wait();
    bool write_out = true;
    if (split_idx >= 0) {
      // publish this key range's partial: O (unnormalised, relative to m_used) transposed so that a warp
      // writes 128 contiguous bytes, then the running maximum and the sum
      float* part = p.partials + (static_cast<size_t>(tail_idx) * p.split + split_idx) * ATT_PART_FLOATS;
#pragma unroll
      for (int i = 0; i < 32; ++i) part[(half * 32 + i) * 128 + r] = __uint_as_float(o[i]);
      if (half == 0) {
        part[64 * 128 + r] = m_used;
        part[65 * 128 + r] = l;
      }
      __threadfence();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (threadIdx.x == 64) {
        const unsigned int prev = atomicAdd(&p.counters[tail_idx], 1u);
        tmem_slot[1] = (prev == static_cast<unsigned int>(p.split) - 1u) ? 1u : 0u;
        __threadfence();
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      write_out = tmem_slot[1] != 0u;
      if (write_out) {
        // last arriver: merge the partials in split order (fixed order -> deterministic)
        const float* base = p.partials + static_cast<size_t>(tail_idx) * p.split * ATT_PART_FLOATS;
        float m_all = -INFINITY;
        for (int s2 = 0; s2 < p.split; ++s2) m_all = fmaxf(m_all, __ldcg(base + s2 * ATT_PART_FLOATS + 64 * 128 + r));
        float acc[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = 0.f;
        l = 0.f;
        for (int s2 = 0; s2 < p.split; ++s2) {
          const float* ps = base + s2 * ATT_PART_FLOATS;
          const float w = ex2_approx(__ldcg(ps + 64 * 128 + r) - m_all);
          l = fmaf(w, __ldcg(ps + 65 * 128 + r), l);
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = fmaf(w, __ldcg(ps + (half * 32 + i) * 128 + r), acc[i]);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(acc[i]);
        if (threadIdx.x == 64) p.counters[tail_idx] = 0u;  // ready for the next launch / graph replay
      }
    }
    const float inv_l = 1.0f / l;
    if (write_out && q < p.Nq) {
      __nv_bfloat16* dst = p.out + (static_cast<long long>(b) * p.Nq + q) * p.ldo + h * ATT_D + half * 32;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        uint4 u;
        u.x = pack_bf16x2(__uint_as_float(o[v * 8 + 0]) * inv_l, __uint_as_float(o[v * 8 + 1]) * inv_l);
        u.y = pack_bf16x2(__uint_as_float(o[v * 8 + 2]) * inv_l, __uint_as_float(o[v * 8 + 3]) * inv_l);
        u.z = pack_bf16x2(__uint_as_float(o[v * 8 + 4]) * inv_l, __uint_as_float(o[v * 8 + 5]) * inv_l);
        u.w = pack_bf16x2(__uint_as_float(o[v * 8 + 6]) * inv_l, __uint_as_float(o[v * 8 + 7]) * inv_l);
        reinterpret_cast<uint4*>(dst)[v] = u;
      }
    }
  }

  ATT_CTA(1);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc(tmem, ATT_TMEM_COLS);
}

static int make_map3(CUtensorMap* m, const void* base, long long ld, int rows, int batch, int width_cols) {
  uint64_t dims[3] = {static_cast<uint64_t>(width_cols), static_cast<uint64_t>(rows), static_cast<uint64_t>(batch)};
  uint64_t strides[2] = {static_cast<uint64_t>(ld) * 2, static_cast<uint64_t>(rows) * ld * 2};
  uint32_t box[3] = {ATT_D, 128, 1};
  return make_tmap_bf16(m, base, 3, dims, strides, box);
}

// Work plan.  A tile = 128 query rows of one (batch, head); 2 CTAs are resident per SM, so the grid
// runs in waves of 2 * num_sms tiles and a last partial wave costs as much as a full one.  The tiles
// of that last wave are therefore split over the key blocks (`split` CTAs per tile, merged by the
// last CTA to finish) so that the tail wave is shorter by about that factor.
struct AttnPlan {
  int n_qtiles, tiles, full, tail, split, blocks_per_split;
  size_t workspace_bytes;
};

static AttnPlan attention_plan(int B, int H, int Nq, int Nk) {
  AttnPlan a;
  a.n_qtiles = (Nq + ATT_BM - 1) / ATT_BM;
  a.tiles = B * H * a.n_qtiles;
  const int nblk = (Nk + ATT_BN - 1) / ATT_BN;
  const int slots = 2 * num_sms();
  a.split = 1;
  a.blocks_per_split = nblk;
  a.full = a.tiles;
  a.tail = 0;
  if (slots <= 0) {  // no device visible (host-side size queries): plan without a split
    a.workspace_bytes = 0;
    return a;
  }
  a.full = (a.tiles / slots) * slots;
  a.tail = a.tiles - a.full;
  if (a.tail > 0 && a.tail <= ATT_WS_COUNTERS) {
    int s = 1;
    // at most 4 ranges: a CTA with a single key block spends more on its prologue and the merge than it saves
    // (N = 1024, 24 tail tiles: 31.7 us split 8 ways, 30.3 us split 4 ways, 32.7 us split 2 ways)
    while (s * 2 <= nblk && a.tail * s * 2 <= slots && s * 2 <= 4) s *= 2;
    if (s > 1) {
      a.blocks_per_split = (nblk + s - 1) / s;
      a.split = (nblk + a.blocks_per_split - 1) / a.blocks_per_split;  // no empty key ranges
    }
  }
  if (a.split == 1) {
    a.full = a.tiles;
    a.tail = 0;
  }
  a.workspace_bytes = a.tail == 0 ? 0
                                  : ATT_WS_COUNTERS * sizeof(unsigned int) +
                                        static_cast<size_t>(a.tail) * a.split * ATT_PART_FLOATS * sizeof(float);
  return a;
}

}  // namespace b200sr

using namespace b200sr;

extern "C" size_t b200sr_attention_d64_workspace_bytes(int32_t B, int32_t H, int32_t Nq, int32_t Nk) {
  if (B <= 0 || H <= 0 || Nq <= 0 || Nk <= 0) return 0;
  return attention_plan(B, H, Nq, Nk).workspace_bytes;
}

// q: [B, Nq, ldq] window at q_col; k, v: [B, Nk, ldk / ldv] windows; out: [B, Nq, ldo], head h at h*64.
// workspace: b200sr_attention_d64_workspace_bytes() bytes (may be null when that is 0); its first 2 KiB are
// arrival counters that must be zero before the first call and are left zero by every call.
extern "C" int b200sr_attention_d64(const void* q, int64_t ldq, int32_t q_col, const void* k, int64_t ldk, int32_t k_col,
                                    const void* v, int64_t ldv, int32_t v_col, void* out, int64_t ldo, int32_t B, int32_t H,
                                    int32_t Nq, int32_t Nk, float scale, int32_t causal, void* workspace,
                                    void* stream_ptr) {
  if (q == nullptr || k == nullptr || v == nullptr || out == nullptr) return B200SR_EINVAL;
  const cudaStream_t stream = static_cast<cudaStream_t>(stream_ptr);
  if (B <= 0 || H <= 0 || Nq <= 0 || Nk <= 0) return B200SR_EINVAL;
  if (causal && (Nq != Nk || Nk > ATT_BN)) return B200SR_EINVAL;   // causal: self-attention within one key block (77 tokens)
  if ((ldq % 8) || (ldk % 8) || (ldv % 8) || (ldo % 8) || (q_col % 8) || (k_col % 8) || (v_col % 8))
    return B200SR_EINVAL;
  if (q_col + H * ATT_D > ldq || k_col + H * ATT_D > ldk || v_col + H * ATT_D > ldv || H * ATT_D > ldo)
    return B200SR_EINVAL;
  const AttnPlan plan = attention_plan(B, H, Nq, Nk);
  if (plan.workspace_bytes != 0 && workspace == nullptr) return B200SR_EINVAL;
  CUtensorMap tmQ, tmK, tmV;
  int rc = make_map3(&tmQ, q, ldq, Nq, B, static_cast<int>(ldq));
  if (rc) return rc;
  rc = make_map3(&tmK, k, ldk, Nk, B, static_cast<int>(ldk));
  if (rc) return rc;
  rc = make_map3(&tmV, v, ldv, Nk, B, static_cast<int>(ldv));
  if (rc) return rc;
  AttnParams p;
  p.B = B;
  p.H = H;
  p.Nq = Nq;
  p.Nk = Nk;
  p.q_col = q_col;
  p.k_col = k_col;
  p.v_col = v_col;
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.ldo = ldo;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.causal = causal;
  p.n_qtiles = plan.n_qtiles;
  p.full_ctas = plan.full;
  p.split = plan.split;
  p.blocks_per_split = plan.blocks_per_split;
  p.counters = reinterpret_cast<unsigned int*>(workspace);
  p.partials = reinterpret_cast<float*>(reinterpret_cast<unsigned int*>(workspace) + ATT_WS_COUNTERS);
#ifdef B200SR_ATT_TRACE
  p.trace = g_att_trace;
#endif
  const size_t smem_bytes = ATT_TILE_BYTES * (1 + 2 * ATT_STAGES) + 1024 + 128 + 2048;
  static bool attr_set[64] = {false};  // per device
  if (first_use_on_device(attr_set)) {
    if (cudaFuncSetAttribute(attention_d64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(smem_bytes)) != cudaSuccess)
      return B200SR_ELAUNCH;
  }
  dim3 grid(plan.full + plan.tail * plan.split);
  return launch_k(attention_d64_kernel, grid, dim3(ATT_THREADS), smem_bytes, stream, 1, tmQ, tmK, tmV, p) == cudaSuccess
             ? B200SR_OK
             : B200SR_ELAUNCH;
}

#ifdef B200SR_ATT_TRACE
extern "C" void b200sr_debug_set_attn_trace(void* p) { b200sr::g_att_trace = reinterpret_cast<long long*>(p); }
#endif
