// b200sr — extern "C" entry points (include/b200sr.h) and shared host utilities.
#include "../../include/b200sr.h"
#include <stdlib.h>

#include "common.cuh"

namespace b200sr {

// ---- host utilities -----------------------------------------------------------------------
PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200SR_PDL");
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

bool first_use_on_device(bool (&flags)[64]) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
  if (flags[dev]) return false;
  flags[dev] = true;
  return true;
}

static int make_tmap_any(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, int swizzle_bytes) {
  return make_tmap_any(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rank, dims, strides_bytes, box, swizzle_bytes);
}

int make_tmap_f32(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                  const uint32_t* box) {
  return make_tmap_any(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, rank, dims, strides_bytes, box, 128);
}

static int make_tmap_any(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (enc == nullptr) return B200SR_ENODEV;
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return B200SR_EINVAL;
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
    if (box[i] == 0 || box[i] > 256) return B200SR_EINVAL;
  }
  for (int i = 0; i + 1 < rank; ++i) {
    gstr[i] = strides_bytes[i];
    if (gstr[i] % 16 != 0) return B200SR_EINVAL;
  }
  const CUresult r = enc(out, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(base),
                         gdim, gstr, bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? B200SR_OK : B200SR_EINVAL;
}

// ---- forward declarations of the kernel launchers -------------------------------------------
int gemm_bf16(const void* A, long long lda, const void* W, int M, int N, int K, const EpilogueArgs& e, int force_bn,
              cudaStream_t stream);
int conv3x3_bf16(const void* x, const void* w, int NB, int H, int W, int Cin, int Cout, int stride, int pad_lo,
                 const EpilogueArgs& e, int force_bn, cudaStream_t stream);
int gemm_n_tile(int M, int N, int K);
int pointwise_small(const void* x, const float* w, const float* bias, void* y, int Cin, int Cout, long long rows, int HW,
                    int out_nchw_f32, float scale, cudaStream_t stream);
int diag_gaussian(const float* moments, const float* noise, float* z, int N, int C, int HW, float scale,
                  cudaStream_t stream);
size_t group_norm_workspace_bytes(int N, int HW, int C, int groups);
int group_norm_launches(int N, int HW, int C, int groups);
int group_norm_nhwc(const void* x, void* y, const float* weight, const float* bias, int N, int HW, int C, int groups,
                    float eps, int silu, const void* sft_gamma, const void* sft_beta, const void* raw,
                    float control_scale, float* workspace, cudaStream_t stream);
int group_norm_stats(const void* x, int N, int HW, int C, int groups, float eps, float* stats_out, float* workspace,
                     cudaStream_t stream);
int layer_norm(const void* x, void* y, const float* weight, const float* bias, int M, int C, float eps,
               cudaStream_t stream);
int softmax_rows(const float* x, void* y, int rows, int cols, int valid, float scale, cudaStream_t stream);
int row_softmax_fold(const float* parts, int n_parts, long long rows, float* out, cudaStream_t stream);
int attention_d64(const void* q, long long ldq, int q_col, const void* k, long long ldk, int k_col, const void* v,
                  long long ldv, int v_col, void* out, long long ldo, int B, int H, int Nq, int Nk, float scale,
                  int causal, void* workspace, cudaStream_t stream);
int embed_tokens(const long long* ids, const float* tok, const float* pos, void* out, int B, int T, int C, int vocab,
                 cudaStream_t stream);
size_t attention_d64_workspace_bytes(int B, int H, int Nq, int Nk);
int nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int HW, float scale, cudaStream_t stream);
int nhwc_bf16_to_nchw_f32(const void* x, float* y, int N, int C, int Cs, int HW, cudaStream_t stream);
int upsample2x_nhwc(const void* x, void* y, int N, int H, int W, int C, cudaStream_t stream);
int concat_add(const void* a, int Ca, const void* b, int Cb, const void* c, void* out, long long rows,
               cudaStream_t stream);
int axpy_bf16(const void* a, const void* b, void* y, float alpha, long long n, cudaStream_t stream);
int silu_bf16(const void* x, void* y, long long n, cudaStream_t stream);
int pad_channels(const void* x, void* y, int C, int Cpad, long long rows, cudaStream_t stream);
int sinusoid_embedding(const float* t, void* out, int B, int dim, float max_period, int sin_first,
                       cudaStream_t stream);
int conv3x3_small(const void* x, const void* w, const float* bias, const void* addend, void* y, int N, int H, int W,
                  int Cin, int Cout, int out_nchw_f32, cudaStream_t stream);
int sampler_pre(const float* x, const float* noise, const float* scalars, float* x_hat, void* net_in, int B, int C,
                int HW, int cfg_copies, cudaStream_t stream);
int sampler_post(const float* eps, const float* x_hat, const float* scalars, float* denoised_out, float* x_next, int B,
                 int C, int HW, int use_cfg, cudaStream_t stream);
int euler_from_denoised(const float* denoised, const float* x_hat, const float* scalars, float* x_next, long long n,
                        cudaStream_t stream);
int tile_accumulate(const float* tile, const float* weight, float* acc, float* cnt, int BC, int th, int tw, int H, int W,
                    int h0, int w0, cudaStream_t stream);
int tile_normalize(const float* acc, const float* cnt, float* out, long long n, cudaStream_t stream);
int rel_l1_similarity(const void* prev, const void* cur, long long n, const float* threshold, double* workspace,
                      float* result, cudaStream_t stream);
int sr3_update(const float* x, const float* eps, const float* noise, const float* scalars, float* out, long long n,
               cudaStream_t stream);
int wavelet_level(const float* img, float* low, float* high, int first, int BC, int H, int W, int radius,
                  cudaStream_t stream);
int add_f32(const float* a, const float* b, float* out, long long n, cudaStream_t stream);
int image_to_u8(const float* x, void* out, int C, int H, int W, int OH, int OW, cudaStream_t stream);
int tensor2img_u8(const float* x, void* out, int C, int H, int W, cudaStream_t stream);
int resample_u8(const void* src, void* dst, int outer, int in_len, int out_len, int inner, const int* bounds,
                const int* coeffs, int ksize, cudaStream_t stream);
int img_u8_to_tensor(const void* in, float* out, int C, int H, int W, cudaStream_t stream);
int copy_batch(const void* const* src, void* const* dst, const long long* bytes, int n, cudaStream_t stream);
int tile_weighted_strip(const float* tile, const float* weight, float* strip, int BC, int th, int tw, int y0, int x0,
                        int sh, int sw, cudaStream_t stream);
int strip_add(const float* strip, float* acc, int BC, int sh, int sw, int H, int W, int h0, int w0, cudaStream_t stream);

static EpilogueArgs to_args(const b200sr_epilogue* e) {
  EpilogueArgs a;
  a.bias = e->bias;
  a.rowvec = e->rowvec;
  a.rows_per_group = e->rows_per_group;
  a.ld_rowvec = e->ld_rowvec;
  a.residual = e->residual;
  a.ldr = e->ldr;
  a.out = e->out;
  a.ldc = e->ldc;
  a.out_fp32 = e->out_fp32;
  a.geglu = e->geglu;
  a.alpha = e->alpha;
  a.act = e->act;
  a.softmax_valid = e->softmax_valid;
  a.w_dynamic = e->w_dynamic;
  a.w_rows_per_group = e->w_rows_per_group;
  a.w_group_stride = e->w_group_stride;
  a.a_gn_stats = e->a_gn_stats;
  a.a_gn_weight = e->a_gn_weight;
  a.a_gn_bias = e->a_gn_bias;
  a.a_gn_groups = e->a_gn_groups;
  a.a_gn_silu = e->a_gn_silu;
  a.ln_stats = e->ln_stats;
  a.ln_parts = e->ln_parts;
  a.ln_colsum = e->ln_colsum;
  a.ln_shift = e->ln_shift;
  a.ln_eps = e->ln_eps;
  a.ln_stats_out = e->ln_stats_out;
  a.row_softmax = e->row_softmax;
  a.row_softmax_valid = e->row_softmax_valid;
  return a;
}

}  // namespace b200sr

using namespace b200sr;
#define S(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int b200sr_abi_version(void) { return 6; }
int b200sr_num_sms(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return B200SR_ENODEV;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return B200SR_ENODEV;
  return n;
}

int b200sr_gemm_bf16(const void* A, int64_t lda, const void* W, int32_t M, int32_t N, int32_t K,
                     const b200sr_epilogue* epi, int32_t force_bn, void* stream) {
  if (A == nullptr || W == nullptr || epi == nullptr) return B200SR_EINVAL;
  return gemm_bf16(A, lda, W, M, N, K, to_args(epi), force_bn, S(stream));
}
int b200sr_gemm_n_tile(int32_t M, int32_t N, int32_t K) { return gemm_n_tile(M, N, K); }
int b200sr_conv3x3_bf16(const void* x, const void* w, int32_t N, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                        int32_t stride, int32_t pad_lo, const b200sr_epilogue* epi, int32_t force_bn, void* stream) {
  if (x == nullptr || w == nullptr || epi == nullptr) return B200SR_EINVAL;
  return conv3x3_bf16(x, w, N, H, W, Cin, Cout, stride, pad_lo, to_args(epi), force_bn, S(stream));
}
int b200sr_pointwise_small(const void* x, const float* w, const float* bias, void* y, int32_t Cin, int32_t Cout,
                           int64_t rows, int32_t HW, int32_t out_nchw_f32, float scale, void* stream) {
  if (x == nullptr || w == nullptr || y == nullptr) return B200SR_EINVAL;
  return pointwise_small(x, w, bias, y, Cin, Cout, rows, HW, out_nchw_f32, scale, S(stream));
}
int b200sr_diag_gaussian(const float* moments, const float* noise, float* z, int32_t N, int32_t C, int32_t HW,
                         float scale, void* stream) {
  if (moments == nullptr || z == nullptr) return B200SR_EINVAL;
  return diag_gaussian(moments, noise, z, N, C, HW, scale, S(stream));
}
int b200sr_conv3x3_small(const void* x, const void* w, const float* bias, const void* addend, void* y, int32_t N,
                         int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t out_nchw_f32, void* stream) {
  if (x == nullptr || w == nullptr || y == nullptr) return B200SR_EINVAL;
  return conv3x3_small(x, w, bias, addend, y, N, H, W, Cin, Cout, out_nchw_f32, S(stream));
}
size_t b200sr_group_norm_workspace_bytes(int32_t N, int32_t HW, int32_t C, int32_t groups) {
  if (N <= 0 || HW <= 0 || C < 8 || groups <= 0) return 0;
  return group_norm_workspace_bytes(N, HW, C, groups);
}
int b200sr_group_norm_launches(int32_t N, int32_t HW, int32_t C, int32_t groups) {
  return group_norm_launches(N, HW, C, groups);
}
int b200sr_group_norm_nhwc(const void* x, void* y, const float* weight, const float* bias, int32_t N, int32_t HW,
                           int32_t C, int32_t groups, float eps, int32_t silu, const void* sft_gamma,
                           const void* sft_beta, const void* raw, float control_scale, void* workspace, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return group_norm_nhwc(x, y, weight, bias, N, HW, C, groups, eps, silu, sft_gamma, sft_beta, raw, control_scale,
                         reinterpret_cast<float*>(workspace), S(stream));
}
int b200sr_group_norm_stats(const void* x, int32_t N, int32_t HW, int32_t C, int32_t groups, float eps, float* stats_out,
                            void* workspace, void* stream) {
  if (x == nullptr) return B200SR_EINVAL;
  return group_norm_stats(x, N, HW, C, groups, eps, stats_out, reinterpret_cast<float*>(workspace), S(stream));
}
int b200sr_layer_norm(const void* x, void* y, const float* weight, const float* bias, int32_t M, int32_t C, float eps,
                      void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return layer_norm(x, y, weight, bias, M, C, eps, S(stream));
}
int b200sr_row_softmax_fold(const float* parts, int32_t n_parts, int64_t rows, float* out, void* stream) {
  return row_softmax_fold(parts, n_parts, rows, out, S(stream));
}
int b200sr_softmax_rows(const float* x, void* y, int32_t rows, int32_t cols, int32_t valid_cols, float scale,
                        void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return softmax_rows(x, y, rows, cols, valid_cols, scale, S(stream));
}
int b200sr_attention_d64(const void* q, int64_t ldq, int32_t q_col, const void* k, int64_t ldk, int32_t k_col,
                         const void* v, int64_t ldv, int32_t v_col, void* out, int64_t ldo, int32_t B, int32_t H,
                         int32_t Nq, int32_t Nk, float scale, int32_t causal, void* workspace, void* stream) {
  if (q == nullptr || k == nullptr || v == nullptr || out == nullptr) return B200SR_EINVAL;
  return attention_d64(q, ldq, q_col, k, ldk, k_col, v, ldv, v_col, out, ldo, B, H, Nq, Nk, scale, causal, workspace,
                       S(stream));
}
int b200sr_embed_tokens(const int64_t* ids, const float* tok, const float* pos, void* out, int32_t B, int32_t T, int32_t C,
                        int32_t vocab, void* stream) {
  if (ids == nullptr || tok == nullptr || pos == nullptr || out == nullptr) return B200SR_EINVAL;
  return embed_tokens(reinterpret_cast<const long long*>(ids), tok, pos, out, B, T, C, vocab, S(stream));
}
size_t b200sr_attention_d64_workspace_bytes(int32_t B, int32_t H, int32_t Nq, int32_t Nk) {
  return attention_d64_workspace_bytes(B, H, Nq, Nk);
}
int b200sr_nchw_f32_to_nhwc_bf16(const float* x, void* y, int32_t N, int32_t C, int32_t HW, float scale, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return nchw_f32_to_nhwc_bf16(x, y, N, C, HW, scale, S(stream));
}
int b200sr_nhwc_bf16_to_nchw_f32(const void* x, float* y, int32_t N, int32_t C, int32_t HW, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return nhwc_bf16_to_nchw_f32(x, y, N, C, C, HW, S(stream));
}
int b200sr_nhwc_bf16_to_nchw_f32_strided(const void* x, float* y, int32_t N, int32_t C, int32_t Cs, int32_t HW, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return nhwc_bf16_to_nchw_f32(x, y, N, C, Cs, HW, S(stream));
}
int b200sr_upsample2x_nhwc(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return upsample2x_nhwc(x, y, N, H, W, C, S(stream));
}
int b200sr_concat_add(const void* a, int32_t Ca, const void* b, int32_t Cb, const void* c, void* out, int64_t rows,
                      void* stream) {
  if ((a == nullptr && Ca > 0) || b == nullptr || out == nullptr) return B200SR_EINVAL;
  return concat_add(a, Ca, b, Cb, c, out, rows, S(stream));
}
int b200sr_axpy_bf16(const void* a, const void* b, void* y, float alpha, int64_t n, void* stream) {
  if (a == nullptr || b == nullptr || y == nullptr) return B200SR_EINVAL;
  return axpy_bf16(a, b, y, alpha, n, S(stream));
}
int b200sr_pad_channels(const void* x, void* y, int32_t C, int32_t Cpad, int64_t rows, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return pad_channels(x, y, C, Cpad, rows, S(stream));
}
int b200sr_silu_bf16(const void* x, void* y, int64_t n, void* stream) {
  if (x == nullptr || y == nullptr) return B200SR_EINVAL;
  return silu_bf16(x, y, n, S(stream));
}
int b200sr_sinusoid_embedding(const float* t, void* out, int32_t B, int32_t dim, float max_period, int32_t sin_first,
                              void* stream) {
  if (t == nullptr || out == nullptr) return B200SR_EINVAL;
  return sinusoid_embedding(t, out, B, dim, max_period, sin_first, S(stream));
}
int b200sr_sampler_pre(const float* x, const float* noise, const float* scalars, float* x_hat, void* net_in, int32_t B,
                       int32_t C, int32_t HW, int32_t cfg_copies, void* stream) {
  if (x == nullptr || scalars == nullptr || x_hat == nullptr || net_in == nullptr) return B200SR_EINVAL;
  return sampler_pre(x, noise, scalars, x_hat, net_in, B, C, HW, cfg_copies, S(stream));
}
int b200sr_sampler_post(const float* eps, const float* x_hat, const float* scalars, float* denoised_out, float* x_next,
                        int32_t B, int32_t C, int32_t HW, int32_t use_cfg, void* stream) {
  if (eps == nullptr || x_hat == nullptr || scalars == nullptr || x_next == nullptr) return B200SR_EINVAL;
  return sampler_post(eps, x_hat, scalars, denoised_out, x_next, B, C, HW, use_cfg, S(stream));
}
int b200sr_euler_from_denoised(const float* denoised, const float* x_hat, const float* scalars, float* x_next,
                               int64_t n, void* stream) {
  if (denoised == nullptr || x_hat == nullptr || scalars == nullptr || x_next == nullptr) return B200SR_EINVAL;
  return euler_from_denoised(denoised, x_hat, scalars, x_next, n, S(stream));
}
int b200sr_tile_accumulate(const float* tile, const float* weight, float* acc, float* cnt, int32_t BC, int32_t th,
                           int32_t tw, int32_t H, int32_t W, int32_t h0, int32_t w0, void* stream) {
  if (tile == nullptr || weight == nullptr || acc == nullptr) return B200SR_EINVAL;  // cnt may be NULL
  return tile_accumulate(tile, weight, acc, cnt, BC, th, tw, H, W, h0, w0, S(stream));
}
int b200sr_tile_normalize(const float* acc, const float* cnt, float* out, int64_t n, void* stream) {
  if (acc == nullptr || cnt == nullptr || out == nullptr) return B200SR_EINVAL;
  return tile_normalize(acc, cnt, out, n, S(stream));
}
int b200sr_rel_l1_similarity(const void* prev, const void* cur, int64_t n, const float* threshold, void* workspace,
                             float* result, void* stream) {
  if (prev == nullptr || cur == nullptr || threshold == nullptr || workspace == nullptr || result == nullptr)
    return B200SR_EINVAL;
  return rel_l1_similarity(prev, cur, n, threshold, reinterpret_cast<double*>(workspace), result, S(stream));
}
int b200sr_sr3_update(const float* x, const float* eps, const float* noise, const float* scalars, float* out,
                      int64_t n, void* stream) {
  if (x == nullptr || eps == nullptr || scalars == nullptr || out == nullptr) return B200SR_EINVAL;
  return sr3_update(x, eps, noise, scalars, out, n, S(stream));
}

int b200sr_copy_batch(const b200sr_copy* copies, int32_t n, void* stream) {
  if (copies == nullptr || n <= 0 || n > B200SR_MAX_COPIES) return B200SR_EINVAL;
  const void* src[B200SR_MAX_COPIES];
  void* dst[B200SR_MAX_COPIES];
  long long bytes[B200SR_MAX_COPIES];
  for (int i = 0; i < n; ++i) {
    src[i] = copies[i].src;
    dst[i] = copies[i].dst;
    bytes[i] = copies[i].bytes;
  }
  return copy_batch(src, dst, bytes, n, S(stream));
}
int b200sr_tile_weighted_strip(const float* tile, const float* weight, float* strip, int32_t BC, int32_t th, int32_t tw,
                               int32_t y0, int32_t x0, int32_t sh, int32_t sw, void* stream) {
  if (tile == nullptr || weight == nullptr || strip == nullptr) return B200SR_EINVAL;
  return tile_weighted_strip(tile, weight, strip, BC, th, tw, y0, x0, sh, sw, S(stream));
}
int b200sr_strip_add(const float* strip, float* acc, int32_t BC, int32_t sh, int32_t sw, int32_t H, int32_t W,
                     int32_t h0, int32_t w0, void* stream) {
  if (strip == nullptr || acc == nullptr) return B200SR_EINVAL;
  return strip_add(strip, acc, BC, sh, sw, H, W, h0, w0, S(stream));
}

int b200sr_wavelet_level(const float* img, float* low, float* high, int32_t first, int32_t BC, int32_t H, int32_t W,
                         int32_t radius, void* stream) {
  if (img == nullptr || low == nullptr) return B200SR_EINVAL;
  return wavelet_level(img, low, high, first, BC, H, W, radius, S(stream));
}
int b200sr_add_f32(const float* a, const float* b, float* out, int64_t n, void* stream) {
  if (a == nullptr || b == nullptr || out == nullptr) return B200SR_EINVAL;
  return add_f32(a, b, out, n, S(stream));
}
int b200sr_image_to_u8(const float* x, void* out, int32_t C, int32_t H, int32_t W, int32_t OH, int32_t OW, void* stream) {
  if (x == nullptr || out == nullptr) return B200SR_EINVAL;
  return image_to_u8(x, out, C, H, W, OH, OW, S(stream));
}
int b200sr_tensor2img_u8(const float* x, void* out, int32_t C, int32_t H, int32_t W, void* stream) {
  if (x == nullptr || out == nullptr) return B200SR_EINVAL;
  return tensor2img_u8(x, out, C, H, W, S(stream));
}
int b200sr_resample_u8(const void* src, void* dst, int32_t outer, int32_t in_len, int32_t out_len, int32_t inner,
                       const int32_t* bounds, const int32_t* coeffs, int32_t ksize, void* stream) {
  if (src == nullptr || dst == nullptr || bounds == nullptr || coeffs == nullptr) return B200SR_EINVAL;
  return resample_u8(src, dst, outer, in_len, out_len, inner, bounds, coeffs, ksize, S(stream));
}
int b200sr_img_u8_to_tensor(const void* in, float* out, int32_t C, int32_t H, int32_t W, void* stream) {
  if (in == nullptr || out == nullptr) return B200SR_EINVAL;
  return img_u8_to_tensor(in, out, C, H, W, S(stream));
}

}  // extern "C"
