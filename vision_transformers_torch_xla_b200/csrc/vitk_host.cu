// vitk_host.cu — host-side support: thread-local error slot, CUtensorMap encoding, device props.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>

#include "vitk_common.cuh"
#include "vitk_internal.h"

namespace {
thread_local char g_err[512] = "";

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    // resolved through the runtime so libvitk.so does not link libcuda directly
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}
}  // namespace

int vitk_set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int vitk_check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    return vitk_set_error(VITK_ERR_CUDA, "%s: launch failed: %s", what, cudaGetErrorString(e));
  return VITK_OK;
}

int vitk_num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  return sms;
}

static int encode(CUtensorMap* out, const void* base, int elem_bytes, int rank, const cuuint64_t* dims,
                  const cuuint64_t* strides_bytes, const cuuint32_t* box,
                  CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = get_encode();
  if (!fn) return vitk_set_error(VITK_ERR_DRIVER, "cuTensorMapEncodeTiled not available from the driver");
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  CUresult r = fn(out, dt, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return vitk_set_error(VITK_ERR_DRIVER,
                          "cuTensorMapEncodeTiled failed (CUresult %d) rank=%d dims=[%llu,%llu,%llu] box=[%u,%u,%u]",
                          (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                          (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0,
                          rank > 2 ? box[2] : 0);
  return VITK_OK;
}

int vitk_make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t outer,
                      uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  return encode(out, base, elem_bytes, 2, dims, strides, box);
}

// 64-byte swizzle (box rows of 32 bf16): the layout of the GEMM epilogue's [32 rows][64 B] staging panels
int vitk_make_tmap_2d_sw64(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t outer,
                           uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  return encode(out, base, elem_bytes, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
}

int vitk_make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
                      uint64_t ld1_elems, uint64_t ld2_elems, uint32_t b0, uint32_t b1, uint32_t b2) {
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {ld1_elems * (uint64_t)elem_bytes, ld2_elems * (uint64_t)elem_bytes};
  cuuint32_t box[3] = {b0, b1, b2};
  return encode(out, base, elem_bytes, 3, dims, strides, box);
}

#ifndef VITK_BUILD_ID
#define VITK_BUILD_ID "unknown"
#endif
// sha256 over the sources this library was compiled from (csrc/Makefile passes it in); the Python binding recomputes
// it over the files on disk and refuses to run a stale binary
extern "C" const char* vitk_build_id(void) { return VITK_BUILD_ID; }
int vitk_make_tmap_4d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3,
                      uint64_t ld1_elems, uint64_t ld2_elems, uint64_t ld3_elems, uint32_t b0, uint32_t b1, uint32_t b2,
                      uint32_t b3, int swizzle_bytes) {
  cuuint64_t dims[4] = {d0, d1, d2, d3};
  cuuint64_t strides[3] = {ld1_elems * (uint64_t)elem_bytes, ld2_elems * (uint64_t)elem_bytes, ld3_elems * (uint64_t)elem_bytes};
  cuuint32_t box[4] = {b0, b1, b2, b3};
  return encode(out, base, elem_bytes, 4, dims, strides, box,
                swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                                        : CU_TENSOR_MAP_SWIZZLE_128B);
}

extern "C" int vitk_abi_version(void) { return VITK_ABI_VERSION; }
extern "C" const char* vitk_last_error(void) { return g_err; }
extern "C" const char* vitk_arch(void) { return "sm_100a"; }
