#include "include/b200_common.cuh"
#include "include/b200_ops.h"
#include "include/b200_tcgen05_host.h"
#include <stdio.h>
#include <string.h>

namespace b200 {
static thread_local char g_err[512] = {0};
static thread_local char g_err_out[512] = {0};
void set_last_error(const char* file, int line, const char* msg) {
  if (g_err[0] == 0) snprintf(g_err, sizeof(g_err), "%s:%d: %s", file, line, msg);
}
const char* take_last_error() {
  memcpy(g_err_out, g_err, sizeof(g_err));
  g_err[0] = 0;
  return g_err_out;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

bool encode_tiled(CUtensorMap* out, CUtensorMapDataType type, uint32_t rank, const void* ptr, const cuuint64_t* dims,
                  const cuuint64_t* strides, const cuuint32_t* box, const char* who) {
  char msg[128];
  bind_primary_context();
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled (%s) unavailable", who);
    set_last_error(__FILE__, __LINE__, msg);
    return false;
  }
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(out, type, rank, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled (%s) failed: %d", who, (int)r);
    set_last_error(__FILE__, __LINE__, msg);
    return false;
  }
  return true;
}
}  // namespace b200
