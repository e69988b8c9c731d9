// Internal interface between the pointwise C-ABI entry points (pw_api.cu) and the GEMM kernel files.
#pragma once
#include "kdcc_common.cuh"

namespace kdcc {

// ---- tcgen05 / TMEM / TMA bf16 GEMMs: pw_gemm_sm100.cu ---------------------------------------------
// layout NHWC: x [M][K]; layout NCHW: x [batch][K][M / batch] (the 1x1 conv then runs as W . X per image)
bool pw_sm100_supported(long M, int K, int Nc, int batch, int layout);
int pw_sm100_fwd(const void *x, const void *w, const float *scale, const float *shift, const void *residual, int relu, void *y_raw,
                 void *y_act, long M, int K, int Nc, int batch, int layout, cudaStream_t st);
int pw_sm100_bwd_dx(const void *dy, const void *w, void *dx, long M, int K, int Nc, int batch, int layout, cudaStream_t st);
int pw_sm100_dw_splits(long M, int K, int Nc);  // upper bound on the split count for either layout
int pw_sm100_bwd_dw(const void *dy, const void *x, float *dw, float *part, long M, int K, int Nc, int batch, int layout,
                    cudaStream_t st);
__global__ void reduce_splits_kernel(const float *__restrict__ part, float *__restrict__ out, int splits, long count);

// ---- fp32 as three tf32 tcgen05 products (KDCC_F32_TF32X3): pw_gemm_tf32x3.cu, NHWC only ---------------
bool pw_tf32x3_supported(long M, int K, int Nc);
int pw_tf32x3_fwd(const void *x, const void *w, const float *scale, const float *shift, const void *residual, int relu,
                  void *y_raw, void *y_act, long M, int K, int Nc, cudaStream_t st);
int pw_tf32x3_bwd_dx(const void *dy, const void *w, void *dx, long M, int K, int Nc, cudaStream_t st);
int pw_tf32x3_dw_splits(long M, int K, int Nc);
int pw_tf32x3_bwd_dw(const void *dy, const void *x, float *dw, float *part, long M, int K, int Nc, cudaStream_t st);

// ---- CUDA-core GEMM (fp32 parity path, shapes the tensor-core kernel does not take): pw_gemm_simt.cu -
// C[i][j] = sum_r A[i*sai + r*sar] * B[j*sbj + r*sbr]
struct SimtGemm {
  int I, J, R;
  long sai, sar, sbj, sbr;
  int splits;             // along r; > 1 only with out_f32 partials
  void *out_raw, *out_act;  // [I][J] in the input dtype, may be null
  const float *scale, *shift;
  const void *residual;     // [I][J] in the input dtype, added before the activation of out_act; may be null
  int relu;
  float *out_f32;         // [splits][I][J]
};
template <typename T>
int pw_simt_gemm(const void *a, const void *b, const SimtGemm &g, cudaStream_t st);
int pw_simt_dw_splits(long M, int K, int Nc);

}  // namespace kdcc
