// C-ABI entry points for the pointwise (1x1) convolution (declared in include/kdcc.h).
// bf16 -> tcgen05/TMEM GEMM (pw_gemm_sm100.cu); KDCC_F32_TF32X3 -> fp32 as three tf32 tcgen05 products
// (pw_gemm_tf32x3.cu); fp32 (parity path) and channel counts the tensor-core kernels do not take -> CUDA-core GEMM
// (pw_gemm_simt.cu).  No CPU / library fallback.
#include "pw_kernels.cuh"

using namespace kdcc;

static bool use_sm100(long M, int K, int Nc, int batch, int layout, int dtype) {
  if (dtype != KDCC_BF16) return false;
  return pw_sm100_supported(M, K, Nc, batch, layout);
}

static int check(long M, int K, int Nc, int batch, int layout, int dtype) {
  if (M < 0 || K <= 0 || Nc <= 0) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16 && dtype != KDCC_F32_TF32X3) return KDCC_EINVAL;
  if (layout != KDCC_LAYOUT_NHWC && layout != KDCC_LAYOUT_NCHW && layout != KDCC_LAYOUT_PLANES_TO_NHWC) return KDCC_EINVAL;
  if (dtype == KDCC_F32_TF32X3 && layout != KDCC_LAYOUT_NHWC) return KDCC_ESHAPE;
  if (M >= (1L << 31)) return KDCC_ESHAPE;
  if (layout != KDCC_LAYOUT_NHWC) {
    if (batch <= 0 && M > 0) return KDCC_EINVAL;
    // the NCHW form exists on the tensor-core path only
    if (M > 0 && (dtype != KDCC_BF16 || !pw_sm100_supported(M, K, Nc, batch, layout))) return KDCC_ESHAPE;
  }
  return KDCC_OK;
}

static int pw_fwd_impl(const void *x, const void *w, const float *scale, const float *shift, const void *residual, int relu,
                       void *y_raw, void *y_act, long M, int K, int Nc, int batch, int layout, int dtype, kdcc_stream_t stream) {
  int rc = check(M, K, Nc, batch, layout, dtype);
  if (rc) return rc;
  if (M == 0) return KDCC_OK;
  if (!x || !w || (!y_raw && !y_act) || (residual && !y_act)) return KDCC_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (use_sm100(M, K, Nc, batch, layout, dtype)) {
    if (!aligned16(x) || !aligned16(w) || (y_raw && !aligned16(y_raw)) || (y_act && !aligned16(y_act)) ||
        (residual && !aligned16(residual)))
      return KDCC_EALIGN;
    return pw_sm100_fwd(x, w, scale, shift, residual, relu, y_raw, y_act, M, K, Nc, batch, layout, st);
  }
  if (dtype == KDCC_F32_TF32X3 && pw_tf32x3_supported(M, K, Nc)) {
    if (!aligned16(x) || !aligned16(w) || (y_raw && !aligned16(y_raw)) || (y_act && !aligned16(y_act)) ||
        (residual && !aligned16(residual)))
      return KDCC_EALIGN;
    return pw_tf32x3_fwd(x, w, scale, shift, residual, relu, y_raw, y_act, M, K, Nc, st);
  }
  if (layout != KDCC_LAYOUT_NHWC) return KDCC_ESHAPE;
  SimtGemm g{};
  g.I = (int)M; g.J = Nc; g.R = K;
  g.sai = K; g.sar = 1; g.sbj = K; g.sbr = 1; g.splits = 1;
  g.out_raw = y_raw; g.out_act = y_act; g.scale = scale; g.shift = shift; g.relu = relu; g.residual = residual;
  return dtype == KDCC_BF16 ? pw_simt_gemm<__nv_bfloat16>(x, w, g, st) : pw_simt_gemm<float>(x, w, g, st);
}

KDCC_API int kdcc_pw_fwd(const void *x, const void *w, const float *scale, const float *shift, int relu, void *y_raw,
                         void *y_act, long M, int K, int Nc, int batch, int layout, int dtype, kdcc_stream_t stream) {
  return pw_fwd_impl(x, w, scale, shift, nullptr, relu, y_raw, y_act, M, K, Nc, batch, layout, dtype, stream);
}

KDCC_API int kdcc_pw_fwd_residual(const void *x, const void *w, const float *scale, const float *shift, const void *residual,
                                  int relu, void *y_raw, void *y_act, long M, int K, int Nc, int batch, int layout, int dtype,
                                  kdcc_stream_t stream) {
  return pw_fwd_impl(x, w, scale, shift, residual, relu, y_raw, y_act, M, K, Nc, batch, layout, dtype, stream);
}

KDCC_API size_t kdcc_pw_bwd_workspace_bytes(int which, long M, int K, int Nc, int dtype) {
  if (M <= 0 || K <= 0 || Nc <= 0 || which != 1) return 0;
  size_t splits = (size_t)pw_simt_dw_splits(M, K, Nc);
  if (dtype == KDCC_BF16 && K % 8 == 0) {
    const size_t s2 = (size_t)pw_sm100_dw_splits(M, K, Nc);
    if (s2 > splits) splits = s2;
  }
  if (dtype == KDCC_F32_TF32X3 && pw_tf32x3_supported(M, K, Nc)) {
    const size_t s3 = (size_t)pw_tf32x3_dw_splits(M, K, Nc);
    if (s3 > splits) splits = s3;
  }
  return splits * (size_t)Nc * (size_t)K * sizeof(float);
}

KDCC_API int kdcc_pw_bwd_dx(const void *dy, const void *w, void *dx, void *workspace, size_t workspace_bytes, long M,
                            int K, int Nc, int batch, int layout, int dtype, kdcc_stream_t stream) {
  (void)workspace; (void)workspace_bytes;
  int rc = check(M, K, Nc, batch, layout, dtype);
  if (rc) return rc;
  if (M == 0) return KDCC_OK;
  if (!dy || !w || !dx) return KDCC_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (use_sm100(M, K, Nc, batch, layout, dtype)) {
    if (!aligned16(dy) || !aligned16(w) || !aligned16(dx)) return KDCC_EALIGN;
    return pw_sm100_bwd_dx(dy, w, dx, M, K, Nc, batch, layout, st);
  }
  if (dtype == KDCC_F32_TF32X3 && pw_tf32x3_supported(M, K, Nc)) {
    if (!aligned16(dy) || !aligned16(w) || !aligned16(dx)) return KDCC_EALIGN;
    return pw_tf32x3_bwd_dx(dy, w, dx, M, K, Nc, st);
  }
  if (layout != KDCC_LAYOUT_NHWC) return KDCC_ESHAPE;
  // dx[m][k] = sum_n dy[m][n] w[n][k]
  SimtGemm g{};
  g.I = (int)M; g.J = K; g.R = Nc;
  g.sai = Nc; g.sar = 1; g.sbj = 1; g.sbr = K; g.splits = 1;
  g.out_raw = dx;
  return dtype == KDCC_BF16 ? pw_simt_gemm<__nv_bfloat16>(dy, w, g, st) : pw_simt_gemm<float>(dy, w, g, st);
}

KDCC_API int kdcc_pw_bwd_dw(const void *dy, const void *x, float *dw, void *workspace, size_t workspace_bytes, long M,
                            int K, int Nc, int batch, int layout, int dtype, kdcc_stream_t stream) {
  int rc = check(M, K, Nc, batch, layout, dtype);
  if (rc) return rc;
  if (!dw) return KDCC_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (M == 0) return (int)cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)Nc * K, st);
  if (!dy || !x || !workspace) return KDCC_EINVAL;
  if (workspace_bytes < kdcc_pw_bwd_workspace_bytes(1, M, K, Nc, dtype)) return KDCC_EWORKSPACE;
  float *part = static_cast<float *>(workspace);
  if (use_sm100(M, K, Nc, batch, layout, dtype)) {
    if (!aligned16(dy) || !aligned16(x) || !aligned16(dw) || !aligned16(part)) return KDCC_EALIGN;
    return pw_sm100_bwd_dw(dy, x, dw, part, M, K, Nc, batch, layout, st);
  }
  if (dtype == KDCC_F32_TF32X3 && pw_tf32x3_supported(M, K, Nc)) {
    if (!aligned16(dy) || !aligned16(x) || !aligned16(dw) || !aligned16(part)) return KDCC_EALIGN;
    return pw_tf32x3_bwd_dw(dy, x, dw, part, M, K, Nc, st);
  }
  if (layout != KDCC_LAYOUT_NHWC) return KDCC_ESHAPE;
  // dw[n][k] = sum_m dy[m][n] x[m][k]
  SimtGemm g{};
  g.I = Nc; g.J = K; g.R = (int)M;
  g.sai = 1; g.sar = Nc; g.sbj = 1; g.sbr = K;
  g.splits = pw_simt_dw_splits(M, K, Nc);
  g.out_f32 = g.splits == 1 ? dw : part;
  rc = dtype == KDCC_BF16 ? pw_simt_gemm<__nv_bfloat16>(dy, x, g, st) : pw_simt_gemm<float>(dy, x, g, st);
  if (rc || g.splits == 1) return rc;
  const long count = (long)Nc * K;
  reduce_splits_kernel<<<(unsigned)ceil_div<long>(count, 4 * 256), 256, 0, st>>>(part, dw, g.splits, count);
  return launch_status();
}
