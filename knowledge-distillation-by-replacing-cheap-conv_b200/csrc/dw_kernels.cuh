// Internal interface between the depthwise C-ABI entry points (dw_api.cu) and the kernel files.
#pragma once
#include "kdcc_common.cuh"

namespace kdcc {

// ---- direct (gather) kernels: dw_direct.cu --------------------------------------------------------
template <typename T>
int dw_direct_fwd(const void *x, const float *w, const float *bias, void *y, int N, int H, int W, int C, int Ho,
                  int Wo, int k, int dil, int pad, int flip, cudaStream_t st);
template <typename T>
int dw_direct_wgrad(const void *x, const void *dy, float *dw, float *dbias, float *part, int N, int H, int W,
                    int C, int Ho, int Wo, int k, int dil, int pad, cudaStream_t st);
int dw_direct_wgrad_splits(int N, int Ho, int C, int k, int vn);
__global__ void dw_wgrad_reduce_kernel(const float *__restrict__ part, float *__restrict__ dw,
                                       float *__restrict__ dbias, int splits, int C, int KK, int rows);

// ---- TMA-staged bf16 kernels: dw_tma.cu -------------------------------------------------------------
// A conv (or its transposed form when flip != 0) from `in` [N,Hi,Wi,C] to `out` [N,Ho,Wo,C] with
// effective padding `pad`:  out[i][j] = sum_{u,v} w'[u][v] in[i + u*dil - pad][j + v*dil - pad].
bool dw_tma_supported(int C, int k, int dil);
const char *dw_tma_name(int k, int dil, int which /*0 fwd, 1 wgrad*/);
int dw_tma_conv(const void *in, const float *w, const float *bias, void *out, int N, int Hi, int Wi, int C, int Ho,
                int Wo, int k, int dil, int pad, int flip, cudaStream_t st);
int dw_tma_wgrad_splits(int N, int Ho, int Wo, int C, int k, int dil);
int dw_tma_wgrad(const void *x, const void *dy, float *dw, float *part, int N, int H, int W, int C, int Ho, int Wo,
                 int k, int dil, int pad, cudaStream_t st);

// ---- streaming 3 x 3 (dil 1, pad 1) NHWC bf16 kernels: dw_nhwc3.cu ------------------------------------
bool dw_nhwc3_supported(int C, int k, int dil, int pad);
int dw_nhwc3_conv(const void *in, const float *w, const float *bias, void *out, int N, int H, int W, int C, int flip,
                  cudaStream_t st);
int dw_nhwc3_wgrad_ctas(int N, int H, int W, int C);
int dw_nhwc3_wgrad(const void *x, const void *dy, float *dw, float *part, int N, int H, int W, int C, cudaStream_t st);

// ---- tensor-core (tcgen05) bf16 kernels on NCHW planes: dw_tc.cu, dw_tc_wgrad.cu ---------------------
// pad <= dil * (k - 1): the input gradient is the same convolution with the transposed padding dil * (k - 1) - pad
bool dw_tc_supported(int Hi, int Wi, int Ho, int Wo, int k, int dil, int pad);
int dw_tc_conv(const void *in, const float *w, const float *bias, void *out, int N, int C, int Hi, int Wi, int Ho,
               int Wo, int k, int dil, int pad, int flip, cudaStream_t st);
int dw_tc_wgrad(const void *x, const void *dy, float *dw, float *part, int N, int C, int H, int W, int Ho, int Wo,
                int k, int dil, int pad, cudaStream_t st);
size_t dw_tc_wgrad_workspace(int N, int C, int Ho, int Wo, int k);
// whole-plane, column-phase variant of the convolution (H, W <= 128, same-size, pad % dil == 0): dw_tc2.cu
bool dw_tc_conv2_supported(int Hi, int Wi, int Ho, int Wo, int k, int dil, int pad);
int dw_tc_conv2(const void *in, const float *w, const float *bias, void *out, int N, int C, int H, int W, int k, int dil,
                int pad, int flip, cudaStream_t st);
// whole-plane variant (H, W <= 128, same-size convolution): dw_tc_wgrad2.cu
bool dw_tc_wgrad2_supported(int H, int W, int Ho, int Wo, int k, int dil, int pad);
int dw_tc_wgrad2(const void *x, const void *dy, float *dw, float *part, int N, int C, int H, int W, int k, int dil,
                 int pad, cudaStream_t st);
size_t dw_tc_wgrad2_workspace(int N, int C, int k);
int dw_tc_wgrad2_reduce(const float *part, float *dw, int splits, long count, cudaStream_t st);  // dw = sum over splits, fixed order
// column-phase variant for the 9 x 9, dilation 5, pad 20 geometry (H, W <= 128): dw_tc_wgrad3.cu
bool dw_tc_wgrad3_supported(int H, int W, int Ho, int Wo, int k, int dil, int pad);
int dw_tc_wgrad3(const void *x, const void *dy, float *dw, float *part, int N, int C, int H, int W, cudaStream_t st);
size_t dw_tc_wgrad3_workspace(int N, int C);

}  // namespace kdcc
