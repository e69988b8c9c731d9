// Shared device/host helpers for libkdcc.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/kdcc.h"

#define KDCC_API extern "C" __attribute__((visibility("default")))

namespace kdcc {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

static inline int launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? KDCC_OK : (int)e;
}

// ---- programmatic dependent launch (PDL) ----------------------------------------------------------
// Kernels launched through launch_pdl may become resident while their predecessor in the stream is still running:
// their prologue (shared-memory fills, barrier init, TMEM allocation, descriptor prefetch) overlaps its tail.  Every
// such kernel calls pdl_prologue_done() before its first global-memory access: it lets ITS dependents start early and
// then waits until the predecessor grid has completed and flushed.
__device__ __forceinline__ void pdl_prologue_done() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <typename... KArgs, typename... Args>
static inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Opt a kernel in to `bytes` of dynamic shared memory on the CURRENT device.  Function attributes are per device,
// so the cache is per (call site, device); a benign race only repeats the idempotent call.
template <typename F>
static inline int ensure_dynamic_smem(F *kernel, int bytes, int (&cache)[16]) {
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 15;
  if (bytes > cache[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return (int)e;
    cache[dev] = bytes;
  }
  return 0;
}

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <typename T>
static inline T ceil_div(T a, T b) {
  return (a + b - 1) / b;
}

// ---- element <-> float conversion -------------------------------------------------------------
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) {
  return v;
}
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

// numpy's / torch's float -> uint8 on x86-64: cvttss2si to int32 (out of range / NaN -> INT_MIN, whose low byte is 0),
// low byte.  PTX cvt.rzi saturates instead, hence the explicit range check.
__device__ __forceinline__ uint8_t cast_u8_like_numpy(float v) {
  const float t = truncf(v);
  return (t >= -2147483648.f && t < 2147483648.f) ? (uint8_t)(int)t : (uint8_t)0;
}

// bf16x2 word -> two floats (low element first) with one ALU op each
__device__ __forceinline__ float bf16lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&v);
}

// 16-byte vector of elements: 4 floats or 8 bf16
template <typename T>
struct Vec16;
template <>
struct Vec16<float> {
  static constexpr int N = 4;
  float4 raw;
  __device__ __forceinline__ void unpack(float (&f)[4]) const {
    f[0] = raw.x; f[1] = raw.y; f[2] = raw.z; f[3] = raw.w;
  }
  __device__ __forceinline__ void pack(const float (&f)[4]) { raw = make_float4(f[0], f[1], f[2], f[3]); }
};
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  uint4 raw;
  __device__ __forceinline__ void unpack(float (&f)[8]) const {
    f[0] = bf16lo(raw.x); f[1] = bf16hi(raw.x); f[2] = bf16lo(raw.y); f[3] = bf16hi(raw.y);
    f[4] = bf16lo(raw.z); f[5] = bf16hi(raw.z); f[6] = bf16lo(raw.w); f[7] = bf16hi(raw.w);
  }
  __device__ __forceinline__ void pack(const float (&f)[8]) {
    raw.x = pack_bf16x2(f[0], f[1]); raw.y = pack_bf16x2(f[2], f[3]);
    raw.z = pack_bf16x2(f[4], f[5]); raw.w = pack_bf16x2(f[6], f[7]);
  }
};

// streaming 16-byte global accesses (read-once / write-once data: keep it out of L1)
template <typename V>
__device__ __forceinline__ V ld_stream(const void *p) {
  V v;
  uint32_t a, b, c, d;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p));
  uint4 u = make_uint4(a, b, c, d);
  v.raw = *reinterpret_cast<decltype(v.raw) *>(&u);
  return v;
}
template <typename V>
__device__ __forceinline__ void st_stream(void *p, const V &v) {
  const uint4 u = *reinterpret_cast<const uint4 *>(&v.raw);
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w) : "memory");
}

// ---- reductions ---------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the CTA in a fixed order (deterministic).  Result valid in thread 0.  `scratch` >= 32 floats.
__device__ __forceinline__ float block_sum(float v, float *scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  float r = 0.f;
  if (wid == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? scratch[lane] : 0.f;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;
}

// ---- stage-skipping switches of the timing experiments (tools/gpu_nhwc3_probe.sh, DESIGN.md 4.1) --------------------
// They make kernels skip MMAs / stores, i.e. produce WRONG results on purpose, so the shipped library does not contain
// them: without -DKDCC_DEBUG every test is the constant `false` (the branches fold away) and KDCC_TC_DEBUG in the
// environment is ignored.  tools/build_variant.sh builds an instrumented copy with -DKDCC_DEBUG.
#ifdef KDCC_DEBUG
#define KDCC_DBG(p, bit) (((p).dbg & (bit)) != 0)
static inline int tc_debug_bits() {
  const char *e = getenv("KDCC_TC_DEBUG");
  return e ? atoi(e) : 0;
}
#else
#define KDCC_DBG(p, bit) false
static inline int tc_debug_bits() { return 0; }
#endif

}  // namespace kdcc
