// b200sr — host utilities shared by the kernel files (tensor maps, SM count, PDL switch, per-device setup) and the
// library-wide entry points b200sr_abi_version / b200sr_num_sms.  Every other entry point is defined beside its kernel.
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

}  // namespace b200sr

using namespace b200sr;

extern "C" int b200sr_abi_version(void) { return B200SR_ABI_VERSION; }
extern "C" int b200sr_num_sms(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return B200SR_ENODEV;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return B200SR_ENODEV;
  return n;
}
