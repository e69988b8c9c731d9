// Helpers shared by the per-pixel loss kernels (loss_kernels.cu, ce_kernels.cu): launch geometry, base-2 constants and
// the pixel-group loads / stores that serve both NCHW (pixel_stride 1) and channels_last logits.
#pragma once
#include "kdcc_common.cuh"

namespace kdcc {

constexpr int kLossThreads = 256;
constexpr int kMaxLossBlocks = kNumSMs * 8;  // 1184 partial sums at most
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// ------------------------------------------------------------------------------------------------
// pixel-group loads: PIX consecutive pixels of one class plane (pixel_stride == 1) or one pixel
// ------------------------------------------------------------------------------------------------
template <typename T, int PIX>
__device__ __forceinline__ void load_pix(const T *p, float (&v)[PIX]);
template <>
__device__ __forceinline__ void load_pix<float, 1>(const float *p, float (&v)[1]) { v[0] = __ldg(p); }
template <>
__device__ __forceinline__ void load_pix<float, 2>(const float *p, float (&v)[2]) {
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  v[0] = r.x; v[1] = r.y;
}
template <>
__device__ __forceinline__ void load_pix<__nv_bfloat16, 1>(const __nv_bfloat16 *p, float (&v)[1]) {
  v[0] = __bfloat162float(*p);
}
template <>
__device__ __forceinline__ void load_pix<__nv_bfloat16, 2>(const __nv_bfloat16 *p, float (&v)[2]) {
  uint32_t w;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(w) : "l"(p));
  v[0] = bf16lo(w); v[1] = bf16hi(w);
}
template <typename T, int PIX>
__device__ __forceinline__ void store_pix(T *p, const float (&v)[PIX]);
template <>
__device__ __forceinline__ void store_pix<float, 1>(float *p, const float (&v)[1]) { *p = v[0]; }
template <>
__device__ __forceinline__ void store_pix<float, 2>(float *p, const float (&v)[2]) {
  asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" :: "l"(p), "f"(v[0]), "f"(v[1]) : "memory");
}
template <>
__device__ __forceinline__ void store_pix<__nv_bfloat16, 1>(__nv_bfloat16 *p, const float (&v)[1]) {
  *p = __float2bfloat16_rn(v[0]);
}
template <>
__device__ __forceinline__ void store_pix<__nv_bfloat16, 2>(__nv_bfloat16 *p, const float (&v)[2]) {
  const uint32_t w = pack_bf16x2(v[0], v[1]);
  asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" :: "l"(p), "r"(w) : "memory");
}

}  // namespace kdcc
