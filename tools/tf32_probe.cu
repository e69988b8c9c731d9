// Correctness probe (measurement tooling, not product): single 128 x 128 x 8 `tcgen05.mma.cta_group::1.kind::tf32`
// products on known data against a host reference, before pw_gemm_tf32x3.cu relies on them.  It answers:
//   (a) are K-major fp32 operands in the 128-byte swizzle read as expected (including the 32-byte step to the next
//       8-deep reduction slice inside the swizzle atom)?
//   (b) are MN-major (transposed) operand descriptors honoured for kind::tf32 (32-element MN groups 4096 bytes apart,
//       8-row reduction groups 1024 bytes apart)?
//   (c) how does the tensor core treat the 13 mantissa bits below tf32: truncated or rounded?
//   (d) how is the fp32 accumulator rounded, within one MMA and from one MMA to the next: to nearest, or toward zero?
//       (With truncation a long reduction drifts toward zero by about half an ulp per rounding, which is why
//       pw_gemm_tf32x3.cu keeps the number of roundings per accumulator small.)
// The operand tiles are written into shared memory by the threads themselves, in the swizzled layout TMA produces.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/tf32_probe tools/tf32_probe.cu && tools/tf32_probe
#include <cstdio>
#include <cstdint>
#include <cmath>
#include <vector>
#include <cuda_runtime.h>
#include "../knowledge-distillation-by-replacing-cheap-conv_b200/csrc/sm100_ptx.cuh"

using namespace kdcc;

constexpr int TM = 128, TN = 128, TK = 32;  // operand tiles: 128 rows x 32 reduction elements (one swizzle atom deep)

__host__ __device__ inline uint32_t sw_offset(int mn, int k, bool mn_major) {
  if (!mn_major) return mn * 128 + ((((k >> 2) ^ (mn & 7)) & 7) << 4) + (k & 3) * 4;
  const int c = mn & 31;
  return (mn >> 5) * 4096 + k * 128 + ((((c >> 2) ^ (k & 7)) & 7) << 4) + (c & 3) * 4;
}

__device__ inline uint64_t desc(uint32_t addr, uint32_t lbo) {
  return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

// out[m][n] = sum_{k in slice} A[m][k] B[n][k] for the 8-deep reduction slice `ks`
// two != 0: a second MMA on slice ks + 1 accumulates onto the first
__global__ void probe_kernel(const float *A, const float *B, float *out, int a_mn, int b_mn, int ks, int two) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *gen = smem_raw + (base - ptx::smem_u32(smem_raw));
  const uint32_t a_s = base, b_s = base + TM * TK * 4, bar = b_s + TN * TK * 4, slot = bar + 8;
  for (int e = threadIdx.x; e < TM * TK; e += blockDim.x) {
    const int m = e / TK, k = e % TK;
    *reinterpret_cast<float *>(gen + sw_offset(m, k, a_mn)) = A[e];
    *reinterpret_cast<float *>(gen + TM * TK * 4 + sw_offset(m, k, b_mn)) = B[e];
  }
  ptx::fence_proxy_async_smem();
  if (threadIdx.x == 0) { ptx::mbar_init(bar, 1); ptx::fence_barrier_init(); }
  if (threadIdx.x < 32) ptx::tmem_alloc<128>(slot);
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t *>(gen + (slot - base));
  if (threadIdx.x == 0) {
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
                           ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
    const uint64_t da = desc(a_s + ks * (a_mn ? 1024 : 32), a_mn ? 4096 : 16);
    const uint64_t db = desc(b_s + ks * (b_mn ? 1024 : 32), b_mn ? 4096 : 16);
    ptx::umma_tf32(tmem, da, db, idesc, 0u);
    if (two)
      ptx::umma_tf32(tmem, desc(a_s + (ks + 1) * (a_mn ? 1024 : 32), a_mn ? 4096 : 16),
                     desc(b_s + (ks + 1) * (b_mn ? 1024 : 32), b_mn ? 4096 : 16), idesc, 1u);
    ptx::umma_commit(bar);
  }
  ptx::mbar_wait(bar, 0);
  ptx::tcgen05_fence_after();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int c = 0; c < TN; c += 32) {
    uint32_t v[32];
    ptx::tmem_ld_32x32b_x32(tmem + ((uint32_t)(warp * 32) << 16) + c, v);
    ptx::tmem_ld_wait();
    for (int j = 0; j < 32; ++j) out[(warp * 32 + lane) * TN + c + j] = __uint_as_float(v[j]);
  }
  ptx::tcgen05_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) ptx::tmem_dealloc<128>(tmem);
}

static int run(const std::vector<float> &A, const std::vector<float> &B, std::vector<float> &out, int a_mn, int b_mn, int ks,
               int two = 0) {
  float *dA, *dB, *dO;
  cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dO, TM * TN * 4);
  cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
  const int smem = TM * TK * 4 + TN * TK * 4 + 64 + 1024;
  cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  probe_kernel<<<1, 128, smem>>>(dA, dB, dO, a_mn, b_mn, ks, two);
  cudaError_t e = cudaDeviceSynchronize();
  out.resize(TM * TN);
  cudaMemcpy(out.data(), dO, TM * TN * 4, cudaMemcpyDeviceToHost);
  cudaFree(dA); cudaFree(dB); cudaFree(dO);
  return (int)e;
}

int main() {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, 0) != cudaSuccess) { printf("no device\n"); return 1; }
  printf("device: %s (sm_%d%d)\n", prop.name, prop.major, prop.minor);
  // small integers: every product and sum is exact in tf32 / fp32, so any layout error shows as a mismatch
  std::vector<float> A(TM * TK), B(TN * TK);
  for (int m = 0; m < TM; ++m)
    for (int k = 0; k < TK; ++k) A[m * TK + k] = (float)((m * 7 + k * 3) % 17 - 8);
  for (int n = 0; n < TN; ++n)
    for (int k = 0; k < TK; ++k) B[n * TK + k] = (float)((n * 5 + k * 11) % 13 - 6);
  const char *names[2] = {"K-major", "MN-major"};
  int bad_kk = 0, bad_mn = 0;   // K-major x K-major cases / cases with an MN-major operand that miss
  for (int a_mn = 0; a_mn < 2; ++a_mn)
    for (int b_mn = 0; b_mn < 2; ++b_mn)
      for (int ks = 0; ks < TK / 8; ++ks) {
        std::vector<float> out;
        const int rc = run(A, B, out, a_mn, b_mn, ks);
        long bad = 0;
        double maxerr = 0;
        for (int m = 0; m < TM; ++m)
          for (int n = 0; n < TN; ++n) {
            double ref = 0;
            for (int k = ks * 8; k < ks * 8 + 8; ++k) ref += (double)A[m * TK + k] * B[n * TK + k];
            const double err = std::fabs(out[m * TN + n] - ref);
            maxerr = std::fmax(maxerr, err);
            bad += err != 0.0;
          }
        (a_mn || b_mn ? bad_mn : bad_kk) += bad != 0 || rc != 0;
        printf("A %-8s B %-8s k-slice %d: cuda=%d mismatches %ld / %d, max |err| %g -> %s\n", names[a_mn], names[b_mn], ks, rc,
               bad, TM * TN, maxerr, (bad == 0 && rc == 0) ? "OK" : "FAIL");
      }
  // (c) low mantissa bits: A = 1 + 3*2^-12 (between the tf32 neighbours 1 and 1 + 2^-10), B = 1, one term
  std::fill(A.begin(), A.end(), 0.f);
  std::fill(B.begin(), B.end(), 0.f);
  for (int m = 0; m < TM; ++m) A[m * TK] = 1.f + 3.f * std::ldexp(1.f, -12);
  for (int n = 0; n < TN; ++n) B[n * TK] = 1.f;
  std::vector<float> out;
  const int rc = run(A, B, out, 0, 0, 0);
  printf("low-bit treatment: (1 + 3*2^-12) * 1 = %.10f (truncated: 1.0, rounded: %.10f), cuda=%d\n", out[0],
         1.0 + std::ldexp(1.0, -10), rc);
  // (d) 1 + 0.75 ulp(1) (ulp(1) = 2^-23): nearest gives 1 + 2^-23, toward zero gives 1; the same negated
  const float small = 3.f * std::ldexp(1.f, -25);
  for (int sign = 1; sign >= -1; sign -= 2)
    for (int two = 0; two < 2; ++two) {
      std::fill(A.begin(), A.end(), 0.f);
      for (int m = 0; m < TM; ++m) { A[m * TK] = (float)sign; A[m * TK + (two ? 8 : 1)] = sign * small; }
      for (int n = 0; n < TN; ++n) { B[n * TK] = 1.f; B[n * TK + (two ? 8 : 1)] = 1.f; }
      const int r2 = run(A, B, out, 0, 0, 0, two);
      const double got = out[0], up = sign * (1.0 + std::ldexp(1.0, -23));
      printf("accumulate %s: %+.1f + %+g = %.9f -> %s, cuda=%d\n", two ? "across two MMAs" : "inside one MMA ", (double)sign,
             (double)(sign * small), got, got == up ? "nearest" : (got == (double)sign ? "toward zero" : "other"), r2);
    }
  printf("(a) K-major x K-major products: %s\n", bad_kk ? "WRONG" : "exact");
  printf("(b) MN-major operand descriptors for kind::tf32: %s\n", bad_mn ? "NOT honoured (transpose to K-major)" : "honoured");
  return bad_kk ? 1 : 0;
}
