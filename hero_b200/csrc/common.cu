#include <cuda.h>
#include <cudaTypedefs.h>

#include <stdlib.h>

#include "common.h"

namespace hero {

char* error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}

int set_error(int status, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(error_buffer(), 512, fmt, ap);
  va_end(ap);
  return status;
}

bool serial_profiling() {
  static const bool on = [] {
    const char* v = getenv("HERO_SERIAL_PROFILE");
    return v != nullptr && v[0] == '1';
  }();
  return on;
}

int sm_count() {
  static int cached = 0;
  if (cached > 0) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -HERO_ERR_NO_DEVICE;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return -HERO_ERR_NO_DEVICE;
  cached = n;
  return cached;
}

int encode_tmap_2d_bf16(void* map, const void* ptr, long long inner, long long outer, long long ld,
                        int box_inner, int box_outer) {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
            cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return set_error(HERO_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
    fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(reinterpret_cast<CUtensorMap*>(map), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(HERO_ERR_CUDA, "cuTensorMapEncodeTiled(%lld x %lld, ld %lld) failed: %d", outer,
                     inner, ld, (int)r);
  return HERO_OK;
}

}  // namespace hero

extern "C" {

const char* hero_last_error(void) { return hero::error_buffer(); }

int hero_version(void) { return 100; }

int hero_sm_count(void) {
  int n = hero::sm_count();
  if (n < 0) hero::set_error(HERO_ERR_NO_DEVICE, "no CUDA device available");
  return n;
}

}  // extern "C"
