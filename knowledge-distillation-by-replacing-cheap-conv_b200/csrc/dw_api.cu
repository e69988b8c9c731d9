// C-ABI entry points for the depthwise convolution (declared in include/kdcc.h) and their dispatch:
//   NCHW bf16                         -> tensor-core kernels (dw_tc.cu, dw_tc_wgrad.cu)
//   NHWC bf16, 3 x 3, dil 1, pad 1, C / 8 in {2, 4, 8, 16, 32 m} -> streaming 3 x 3 kernels (dw_nhwc3.cu)
//   NHWC bf16, k in {3, 9}, C % 16 == 0 -> TMA-staged CUDA-core kernels (dw_tma.cu)
//   NHWC anything else (fp32 parity path, odd kernel sizes) -> direct kernels (dw_direct.cu)
// There is no CPU or library fallback: unsupported combinations return KDCC_ESHAPE.
#include "dw_kernels.cuh"

using namespace kdcc;

enum NhwcKernel { NHWC_N3, NHWC_TMA, NHWC_DIRECT };

// the NHWC kernel family that runs for these arguments (a bias gradient always goes to the direct kernel)
static NhwcKernel nhwc_kernel(int C, int k, int dil, int pad, int dtype) {
  if (dtype != KDCC_BF16) return NHWC_DIRECT;
  if (dw_nhwc3_supported(C, k, dil, pad)) return NHWC_N3;
  return dw_tma_supported(C, k, dil) ? NHWC_TMA : NHWC_DIRECT;
}

static int check_geometry(int N, int H, int W, int C, int k, int dil, int pad, int layout, int dtype, int *Ho, int *Wo) {
  if (N < 0 || H <= 0 || W <= 0 || C <= 0 || k <= 0 || dil <= 0 || pad < 0) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16) return KDCC_EINVAL;
  if (layout != KDCC_LAYOUT_NHWC && layout != KDCC_LAYOUT_NCHW) return KDCC_EINVAL;
  *Ho = H + 2 * pad - dil * (k - 1);
  *Wo = W + 2 * pad - dil * (k - 1);
  if (*Ho <= 0 || *Wo <= 0) return KDCC_EINVAL;
  if (layout == KDCC_LAYOUT_NHWC) {
    if (C % (dtype == KDCC_F32 ? 4 : 8) != 0) return KDCC_ESHAPE;  // 16-byte channel vectors
  } else {
    if (dtype != KDCC_BF16 || !dw_tc_supported(H, W, *Ho, *Wo, k, dil, pad)) return KDCC_ESHAPE;
  }
  return KDCC_OK;
}

KDCC_API int kdcc_dw_fwd(const void *x, const float *w, const float *bias, void *y, int N, int H, int W, int C,
                         int k, int dil, int pad, int layout, int dtype, kdcc_stream_t stream) {
  int Ho, Wo;
  int rc = check_geometry(N, H, W, C, k, dil, pad, layout, dtype, &Ho, &Wo);
  if (rc) return rc;
  if (N == 0) return KDCC_OK;
  if (!x || !w || !y) return KDCC_EINVAL;
  if (!aligned16(x) || !aligned16(y)) return KDCC_EALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (layout == KDCC_LAYOUT_NCHW) return dw_tc_conv(x, w, bias, y, N, C, H, W, Ho, Wo, k, dil, pad, 0, st);
  const NhwcKernel kern = nhwc_kernel(C, k, dil, pad, dtype);
  if (kern == NHWC_N3) return dw_nhwc3_conv(x, w, bias, y, N, H, W, C, 0, st);
  if (kern == NHWC_TMA) return dw_tma_conv(x, w, bias, y, N, H, W, C, Ho, Wo, k, dil, pad, 0, st);
  if (dtype == KDCC_F32) return dw_direct_fwd<float>(x, w, bias, y, N, H, W, C, Ho, Wo, k, dil, pad, 0, st);
  return dw_direct_fwd<__nv_bfloat16>(x, w, bias, y, N, H, W, C, Ho, Wo, k, dil, pad, 0, st);
}

KDCC_API size_t kdcc_dw_bwd_workspace_bytes(int N, int H, int W, int C, int k, int dil, int pad, int layout,
                                            int dtype) {
  int Ho, Wo;
  if (check_geometry(N, H, W, C, k, dil, pad, layout, dtype, &Ho, &Wo) || N == 0) return 0;
  if (layout == KDCC_LAYOUT_NCHW) {
    const size_t a = dw_tc_wgrad_workspace(N, C, Ho, Wo, k), b = dw_tc_wgrad2_workspace(N, C, k), c = dw_tc_wgrad3_workspace(N, C);
    return a > b ? (a > c ? a : c) : (b > c ? b : c);
  }
  // bound over every weight-gradient kernel that may run: the direct one (bias gradients) for any shape, the TMA
  // one's splits for every TMA shape (each streaming 3 x 3 shape is one), the streaming one's CTAs
  const NhwcKernel kern = nhwc_kernel(C, k, dil, pad, dtype);
  const int vn = dtype == KDCC_F32 ? 4 : 8;
  size_t splits = (size_t)dw_direct_wgrad_splits(N, Ho, C, k, vn);
  if (kern != NHWC_DIRECT) {
    const size_t s2 = (size_t)dw_tma_wgrad_splits(N, Ho, Wo, C, k, dil);
    if (s2 > splits) splits = s2;
  }
  if (kern == NHWC_N3) {
    const size_t s3 = (size_t)dw_nhwc3_wgrad_ctas(N, H, W, C);
    if (s3 > splits) splits = s3;
  }
  return splits * (size_t)(k * k + 1) * (size_t)C * sizeof(float);
}

KDCC_API int kdcc_dw_bwd(const void *x, const float *w, const void *dy, void *dx, float *dw, float *dbias,
                         void *workspace, size_t workspace_bytes, int N, int H, int W, int C, int k, int dil,
                         int pad, int layout, int dtype, kdcc_stream_t stream) {
  int Ho, Wo;
  int rc = check_geometry(N, H, W, C, k, dil, pad, layout, dtype, &Ho, &Wo);
  if (rc) return rc;
  if (N == 0) return KDCC_OK;
  if (!dy || (dx && !w) || ((dw || dbias) && (!x || !workspace))) return KDCC_EINVAL;
  if (!aligned16(dy) || (dx && !aligned16(dx)) || (x && !aligned16(x))) return KDCC_EALIGN;
  if ((dw || dbias) && workspace_bytes < kdcc_dw_bwd_workspace_bytes(N, H, W, C, k, dil, pad, layout, dtype))
    return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // transposed correlation = the forward loop over dy with mirrored taps and pad' = dil*(k-1) - pad
  const int padt = dil * (k - 1) - pad;
  if (layout == KDCC_LAYOUT_NCHW) {
    if (dbias) return KDCC_ESHAPE;  // bias gradients go through kdcc_colsum on the NHWC path
    if (dx) {
      rc = dw_tc_conv(dy, w, nullptr, dx, N, C, Ho, Wo, H, W, k, dil, padt, 1, st);
      if (rc) return rc;
    }
    if (dw) {
      if (dw_tc_wgrad3_supported(H, W, Ho, Wo, k, dil, pad))
        return dw_tc_wgrad3(x, dy, dw, static_cast<float *>(workspace), N, C, H, W, st);
      if (dw_tc_wgrad2_supported(H, W, Ho, Wo, k, dil, pad))
        return dw_tc_wgrad2(x, dy, dw, static_cast<float *>(workspace), N, C, H, W, k, dil, pad, st);
      return dw_tc_wgrad(x, dy, dw, static_cast<float *>(workspace), N, C, H, W, Ho, Wo, k, dil, pad, st);
    }
    return KDCC_OK;
  }
  const NhwcKernel kern = nhwc_kernel(C, k, dil, pad, dtype);
  if (kern == NHWC_N3) {  // streaming 3 x 3 kernels: dX is the conv over dy with mirrored taps (pad' = 1), dW its own kernel
    if (dx) {
      rc = dw_nhwc3_conv(dy, w, nullptr, dx, N, H, W, C, 1, st);
      if (rc) return rc;
    }
    if (dw && !dbias) return dw_nhwc3_wgrad(x, dy, dw, static_cast<float *>(workspace), N, H, W, C, st);
    if (!dw && !dbias) return KDCC_OK;
    dx = nullptr;  // bias gradient requested: the direct weight-gradient kernel produces dw and dbias together
  }
  if (dx) {
    if (kern == NHWC_TMA && padt >= 0) rc = dw_tma_conv(dy, w, nullptr, dx, N, Ho, Wo, C, H, W, k, dil, padt, 1, st);
    else if (dtype == KDCC_F32) rc = dw_direct_fwd<float>(dy, w, nullptr, dx, N, Ho, Wo, C, H, W, k, dil, padt, 1, st);
    else rc = dw_direct_fwd<__nv_bfloat16>(dy, w, nullptr, dx, N, Ho, Wo, C, H, W, k, dil, padt, 1, st);
    if (rc) return rc;
  }
  if (dw || dbias) {
    float *part = static_cast<float *>(workspace);
    if (kern == NHWC_TMA && !dbias) rc = dw_tma_wgrad(x, dy, dw, part, N, H, W, C, Ho, Wo, k, dil, pad, st);
    else if (dtype == KDCC_F32) rc = dw_direct_wgrad<float>(x, dy, dw, dbias, part, N, H, W, C, Ho, Wo, k, dil, pad, st);
    else rc = dw_direct_wgrad<__nv_bfloat16>(x, dy, dw, dbias, part, N, H, W, C, Ho, Wo, k, dil, pad, st);
    if (rc) return rc;
  }
  return KDCC_OK;
}
