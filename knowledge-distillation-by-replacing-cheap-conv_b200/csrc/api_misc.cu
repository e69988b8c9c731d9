// Version / error-string / dispatch-introspection entry points of the C ABI (include/kdcc.h).
#include "dw_kernels.cuh"
#include "pw_kernels.cuh"
#include "sm100_ptx.cuh"

using namespace kdcc;

KDCC_API int kdcc_version(void) { return KDCC_VERSION; }

KDCC_API int kdcc_last_driver_status(void) { return last_driver_status(); }

KDCC_API const char *kdcc_strerror(int code) {
  switch (code) {
    case KDCC_OK: return "success";
    case KDCC_EINVAL: return "kdcc: invalid argument (null pointer, non-positive dimension or bad enum)";
    case KDCC_ESHAPE: return "kdcc: shape not supported by the sm_100a kernels (no fallback exists)";
    case KDCC_EWORKSPACE: return "kdcc: workspace too small";
    case KDCC_EALIGN: return "kdcc: pointer not 16-byte aligned";
    case KDCC_EDEVICE: return "kdcc: device/driver lacks a required sm_100 feature (TMA descriptor encoder)";
    default: break;
  }
  if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
  return "kdcc: unknown error code";
}

KDCC_API const char *kdcc_dispatch_name(int op, int N, int H, int W, int C, int Cout, int k, int dil, int pad,
                                        int layout, int dtype) {
  const bool bf16 = dtype == KDCC_BF16;
  const long M = (long)N * H * W;
  const int Ho = H + 2 * pad - dil * (k - 1), Wo = W + 2 * pad - dil * (k - 1);
  const bool nchw = layout == KDCC_LAYOUT_NCHW;
  if (dtype == KDCC_F32_TF32X3) {
    // pointwise, NHWC only: the tf32x3 kernel, or the CUDA-core fp32 kernel for the shapes it does not take
    static const char *names[3] = {"pw_tf32x3_fwd", "pw_tf32x3_dx", "pw_tf32x3_dw"};
    if (op < 2 || op > 4 || layout != KDCC_LAYOUT_NHWC) return "unsupported";
    return pw_tf32x3_supported(M, C, Cout) ? names[op - 2] : "pw_simt";
  }
  switch (op) {
    case 0:
      if (nchw) return bf16 && dw_tc_supported(H, W, Ho, Wo, k, dil, pad) ? "dw_tc_conv" : "unsupported";
      return bf16 && dw_tma_supported(C, k, dil) ? dw_tma_name(k, dil, 0) : "dw_direct";
    case 1:
      if (nchw) return bf16 && dw_tc_supported(H, W, Ho, Wo, k, dil, pad) ? "dw_tc_wgrad" : "unsupported";
      return bf16 && dw_tma_supported(C, k, dil) ? dw_tma_name(k, dil, 1) : "dw_wgrad_direct";
    case 2: case 3: case 4: {
      static const char *names[3] = {"pw_gemm_sm100_fwd", "pw_gemm_sm100_dx", "pw_gemm_sm100_dw"};
      if (bf16 && pw_sm100_supported(M, C, Cout, N, layout)) return names[op - 2];
      return layout != KDCC_LAYOUT_NHWC ? "unsupported" : "pw_simt";
    }
    default: return "?";
  }
}
