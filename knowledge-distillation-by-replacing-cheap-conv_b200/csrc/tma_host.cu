// Host-side TMA descriptor construction (cuTensorMapEncodeTiled resolved via the runtime so that
// libkdcc.so carries no link-time dependency on libcuda and still loads on a GPU-less build box).
#include <cuda_runtime.h>

#include <mutex>

#include "kdcc_common.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

static thread_local int g_last_driver_status = 0;

EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      (void)cudaGetLastError();
  });
  return fn;
}

static int make_tmap(CUtensorMapDataType type, CUtensorMap *out, const void *base, int rank, const uint64_t *dims,
                     const uint64_t *strides_bytes, const uint32_t *box, const uint32_t *elem_strides,
                     CUtensorMapSwizzle swizzle) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return KDCC_EDEVICE;
  // The encoder is a driver-API call and needs a current context on THIS thread.  Autograd runs backward
  // on its own worker thread whose first CUDA action may be this call, so bind the primary context once
  // per thread through the runtime.
  static thread_local bool context_bound = false;
  if (!context_bound) {
    (void)cudaFree(nullptr);
    context_bound = true;
  }
  cuuint64_t gdim[5], gstr[5];
  cuuint32_t bdim[5], estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = elem_strides ? elem_strides[i] : 1;
    if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
  }
  CUresult r = enc(out, type, (cuuint32_t)rank, const_cast<void *>(base), gdim, gstr, bdim,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  g_last_driver_status = (int)r;
  return r == CUDA_SUCCESS ? KDCC_OK : KDCC_ESHAPE;
}

int make_tmap_bf16(CUtensorMap *out, const void *base, int rank, const uint64_t *dims, const uint64_t *strides_bytes,
                   const uint32_t *box, const uint32_t *elem_strides, CUtensorMapSwizzle swizzle) {
  return make_tmap(CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, out, base, rank, dims, strides_bytes, box, elem_strides, swizzle);
}

int make_tmap_f32(CUtensorMap *out, const void *base, int rank, const uint64_t *dims, const uint64_t *strides_bytes,
                  const uint32_t *box, const uint32_t *elem_strides, CUtensorMapSwizzle swizzle) {
  return make_tmap(CU_TENSOR_MAP_DATA_TYPE_FLOAT32, out, base, rank, dims, strides_bytes, box, elem_strides, swizzle);
}

int last_driver_status() { return g_last_driver_status; }

}  // namespace kdcc
