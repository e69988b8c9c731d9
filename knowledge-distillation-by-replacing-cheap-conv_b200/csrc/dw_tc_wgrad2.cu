// Depthwise weight gradient on the tensor cores, whole-plane variant (H, W <= 128, same-size convolution).
//
//   dw[c][u][v] = sum_{n,i,j} dy[n][c][i][j] * x[n][c][i + u*d - p][j + v*d - p]
//
// Same algebra as dw_tc_wgrad.cu -- P_u = dy^T * x[u*d - p ...] on tcgen05, dw[u][v] = sum_j P_u[j][j + v*d - p] --
// re-planned around what bounds these MMAs on a B200 (tools/mma_probe.cu: an M=128, K=16 MMA with A in TMEM costs
// ~10 + N/2 clocks, its B operand streams from shared memory at 128 B/clk):
//  * the planes are not padded with a halo.  TMA lands the bare 128-row plane between always-zero gap rows, the
//    tap-row shift u*d - p moves the B descriptor into the gap, and columns outside the plane are simply never
//    extracted.  N drops from 128+halo (176) to 128 columns: 74 instead of 98 clocks per MMA;
//  * the two images of a pair accumulate into the SAME P_u in TMEM (16 MMAs per tap row), so the diagonal
//    extraction -- TMEM -> registers -> a private shared-memory scratch row -> k dynamic reads -- runs once per
//    pair instead of once per plane; its shared-memory traffic was the limiter of the first kernel;
//  * dy^T lives in TMEM (A operand), transposed once per plane by four dedicated warps; the other four non-issuing
//    warps only extract, keeping the k*k partial sums of the channel in registers.
// Shared memory: 2 pair stages x [gap | plane | gap | plane | gap] x 2 swizzled 64-column boxes (164 KB), one dy
// landing tile (32 KB), scratch (18 KB).  TMEM: dy^T of 2 stages x 2 planes (256 columns) + 2 x P_u (256 columns).
// Deterministic: fixed-order sums, no atomics; splits are reduced by dw_tc_wgrad_reduce (dw_tc_wgrad.cu).
// Reference semantics: autograd of models/students/transform_blocks/depthwise_separable_conv.py:12.
#include "dw_kernels.cuh"
#include "dw_tc_common.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int W2_THREADS = 320;            // warp 0 TMA, warp 1 MMA, warps 2-5 extraction, warps 6-9 dy transposers
constexpr int W2_GAP = 24;                 // zero rows around every plane slot (>= pad and >= halo - pad, multiple of 8)
constexpr int W2_SLOT = 128 + W2_GAP;      // rows from one plane slot to the next
constexpr int W2_ROWS = W2_GAP + 2 * W2_SLOT;   // rows of one box of a pair stage
constexpr int W2_BOX = W2_ROWS * 128;      // bytes: 128-byte swizzled rows of 64 columns
constexpr int W2_STAGE = 2 * W2_BOX;       // two boxes = 128 columns
constexpr int W2_DYBOX = 128 * 128;
constexpr int W2_SCR_PITCH = 36;           // floats per scratch row: conflict-free 128-bit stores
constexpr uint32_t W2_TMEM_P = 256;        // P_u accumulators at TMEM columns [256,384) and [384,512)

struct W2Params {
  int N, C, H, W, k, dil, pad;
  int npairs, splits;
  long units;   // C * splits
  float *out;   // [splits][C][k*k] (dw itself when splits == 1)
  int dbg;      // KDCC_TC_DEBUG (timing experiments only): 1 skip extraction, 2 skip MMAs, 4 skip transposition
};

template <int K>
__global__ void __launch_bounds__(W2_THREADS, 1)
dw_tc_wgrad2_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_dy, const W2Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  constexpr uint32_t dy_off = 2 * W2_STAGE;
  constexpr uint32_t scr_off = dy_off + 2 * W2_DYBOX;
  constexpr uint32_t bar_off = scr_off + 4 * 32 * W2_SCR_PITCH * 4;
  const uint32_t bar_base = smem_base + bar_off;
  auto x_full = [&](int s) { return bar_base + 8u * s; };
  auto x_empty = [&](int s) { return bar_base + 8u * (2 + s); };
  auto a_full = [&](int s) { return bar_base + 8u * (4 + s); };    // dy^T of both planes of a pair is in TMEM
  auto a_empty = [&](int s) { return bar_base + 8u * (6 + s); };
  auto t_full = [&](int s) { return bar_base + 8u * (8 + s); };
  auto t_empty = [&](int s) { return bar_base + 8u * (10 + s); };
  const uint32_t dy_full = bar_base + 8u * 12, dy_empty = bar_base + 8u * 13;
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + bar_off + 128);
  float *red = reinterpret_cast<float *>(smem_gen + bar_off + 192);  // [4 warps][K*K]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // the gap rows (and everything else) start as zeros; TMA only ever rewrites the plane slots
  for (int i = threadIdx.x; i < (int)(dy_off / 16); i += W2_THREADS)
    reinterpret_cast<uint4 *>(smem_gen)[i] = make_uint4(0, 0, 0, 0);
  ptx::fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(x_full(s), 1);
      ptx::mbar_init(x_empty(s), 1);
      ptx::mbar_init(a_full(s), 8);
      ptx::mbar_init(a_empty(s), 1);
      ptx::mbar_init(t_full(s), 1);
      ptx::mbar_init(t_empty(s), 4);
    }
    ptx::mbar_init(dy_full, 1);
    ptx::mbar_init(dy_empty, 4);
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_x);
    ptx::prefetch_tensormap(&tm_dy);
  }
  if (warp == 1) ptx::tmem_alloc<512>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();  // everything above overlapped the previous kernel's tail; global memory from here on

  if (warp == 0) {
    if (ptx::elect_one()) {
      // ===== TMA producer: the pair's x planes into their slots, its dy planes one after the other =====
      int it = 0, pit = 0;
      for (PlaneWalk w(p.units, p.npairs, p.splits, p.C); w.valid(); w.next(), ++it) {
        const int s = it & 1;
        const uint32_t ph = (it >> 1) & 1;
        const int c = w.channel(), n0 = 2 * w.pl;
        const int np = min(2, p.N - n0);
        ptx::mbar_wait(x_empty(s), ph ^ 1);
        ptx::mbar_arrive_expect_tx(x_full(s), (uint32_t)(np * 2 * W2_DYBOX));
        for (int pl = 0; pl < np; ++pl)
          for (int b = 0; b < 2; ++b)
            ptx::tma_load_4d(smem_base + s * W2_STAGE + b * W2_BOX + (W2_GAP + pl * W2_SLOT) * 128, &tm_x, x_full(s),
                             64 * b, 0, c, n0 + pl);
        for (int pl = 0; pl < np; ++pl, ++pit) {
          ptx::mbar_wait(dy_empty, (uint32_t)(pit & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(dy_full, 2 * W2_DYBOX);
          for (int b = 0; b < 2; ++b)
            ptx::tma_load_4d(smem_base + dy_off + b * W2_DYBOX, &tm_dy, dy_full, 64 * b, 0, c, n0 + pl);
        }
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      // ===== MMA issuer: P_u (128 dy columns x 128 x columns) += dy_n^T [TMEM] * x_n[u*d - p ...] [smem, MN-major] =====
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
      constexpr uint32_t b_hi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO 1024, version 1, SWIZZLE_128B
      int it = 0, tit = 0;
      for (PlaneWalk w(p.units, p.npairs, p.splits, p.C); w.valid(); w.next(), ++it) {
        const int s = it & 1;
        const uint32_t ph = (it >> 1) & 1;
        const int np = min(2, p.N - 2 * w.pl);
        ptx::mbar_wait(a_full(s), ph);
        ptx::mbar_wait(x_full(s), ph);
#pragma unroll 1
        for (int u = 0; u < K; ++u, ++tit) {
          const int tb = tit & 1;
          ptx::mbar_wait(t_empty(tb), ((tit >> 1) & 1) ^ 1);
          ptx::tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + W2_TMEM_P + (uint32_t)tb * 128u;
          if (!KDCC_DBG(p, 2)) {
            for (int pl = 0; pl < np; ++pl) {
              // tap row u: the B window starts u*d - p rows from the plane's first row, inside the zero gap if negative
              const uint32_t xa = smem_base + s * W2_STAGE + (uint32_t)(W2_GAP + pl * W2_SLOT + u * p.dil - p.pad) * 128u;
              const uint32_t b_lo = ((xa & 0x3FFFF) >> 4) | ((uint32_t)(W2_BOX >> 4) << 16);
              const uint32_t a_tmem = tmem_base + (uint32_t)((s * 2 + pl) * 64);
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)  // 16 reduction rows per MMA: 8 TMEM columns of A, 2 KB of B
                ptx::umma_f16_ts(d_tmem, a_tmem + ks * 8, b_lo + ks * 128, b_hi, idesc, (pl | ks) ? 1u : 0u);
            }
          }
          ptx::umma_commit(t_full(tb));
        }
        ptx::umma_commit(x_empty(s));
        ptx::umma_commit(a_empty(s));
      }
    }
  } else if (warp >= 6) {
    // ===== dy transposers (128 threads; thread = dy column j = TMEM lane) =====
    const int quad = warp & 3;
    const int j = quad * 32 + lane;
    const uint8_t *tile = smem_gen + dy_off + (size_t)(j >> 6) * W2_DYBOX;
    const int chunk = (j & 63) >> 3, within = (j & 7) * 2;
    int it = 0, pit = 0;
    for (PlaneWalk w(p.units, p.npairs, p.splits, p.C); w.valid(); w.next(), ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int np = min(2, p.N - 2 * w.pl);
      ptx::mbar_wait(a_empty(s), ph ^ 1);  // the MMAs that read this TMEM stage two pairs ago are done
      ptx::tcgen05_fence_after();
      __syncwarp();  // lanes leave the polling loop one by one; the TMEM accesses below are .sync.aligned
      for (int pl = 0; pl < 2; ++pl) {
        if (pl < np) {
          ptx::mbar_wait(dy_full, (uint32_t)(pit & 1));
          __syncwarp();
          const uint32_t t_dst = tmem_base + (uint32_t)((s * 2 + pl) * 64) + ((uint32_t)(quad * 32) << 16);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t regs[32];
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              const int r = half * 64 + 2 * q;  // TMEM column r/2 = (dy[r][j], dy[r+1][j])
              const uint32_t lo = *reinterpret_cast<const uint16_t *>(tile + r * 128 + ((chunk ^ (r & 7)) << 4) + within);
              const uint32_t hi = *reinterpret_cast<const uint16_t *>(tile + (r + 1) * 128 + ((chunk ^ ((r + 1) & 7)) << 4) + within);
              regs[q] = KDCC_DBG(p, 4) ? 0u : (lo | (hi << 16));
            }
            ptx::tmem_st_32x32b_x32(t_dst + half * 32, regs);
          }
          ptx::tmem_st_wait();
          ++pit;
        }
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (pl < np) ptx::mbar_arrive(dy_empty);  // the landing tile can be refilled
          ptx::mbar_arrive(a_full(s));
        }
      }
    }
  } else {
    // ===== diagonal extraction (128 threads; thread = dy column j = TMEM lane) =====
    const int quad = warp & 3;
    const int halo = p.dil * (K - 1);
    float *scr = reinterpret_cast<float *>(smem_gen + scr_off) + ((warp - 2) * 32 + lane) * W2_SCR_PITCH;
    // x columns this warp's rows reach: [32*quad - pad, 32*quad + 31 + halo - pad], walked in aligned chunks of 32
    const int c_first = ((32 * quad - p.pad + 128) / 32) * 32 - 128;  // floor to a multiple of 32 (may be negative)
    const int c_last = 32 * quad + 31 + halo - p.pad;
    float acc[K][K];
    int tit = 0;
    for (PlaneWalk w(p.units, p.npairs, p.splits, p.C); w.valid(); w.next()) {
      if (w.first_of_unit()) {
#pragma unroll
        for (int u = 0; u < K; ++u)
#pragma unroll
          for (int v = 0; v < K; ++v) acc[u][v] = 0.f;
      }
#pragma unroll
      for (int u = 0; u < K; ++u, ++tit) {
        const int tb = tit & 1;
        ptx::mbar_wait(t_full(tb), (tit >> 1) & 1);
        ptx::tcgen05_fence_after();
        __syncwarp();  // lanes leave the polling loop one by one; the TMEM accesses below are .sync.aligned
        const uint32_t t_row = tmem_base + W2_TMEM_P + (uint32_t)tb * 128u + ((uint32_t)(quad * 32) << 16);
        for (int col0 = c_first; col0 <= c_last && !KDCC_DBG(p, 1); col0 += 32) {
          if (col0 < 0 || col0 >= 128) continue;
          uint32_t vr[32];
          ptx::tmem_ld_32x32b_x32(t_row + col0, vr);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4 *>(scr + 4 * q) = make_uint4(vr[4 * q], vr[4 * q + 1], vr[4 * q + 2], vr[4 * q + 3]);
#pragma unroll
          for (int v = 0; v < K; ++v) {
            const int e = 32 * quad + lane + v * p.dil - p.pad - col0;  // x column of tap v for row j, relative to this chunk
            if (e >= 0 && e < 32) acc[u][v] += scr[e];
          }
        }
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(t_empty(tb));
      }
      if (w.last_of_unit()) {
        // channel finished: sum the 128 rows -- inside the warp by recursive halving (each exchange step also halves
        // the number of values a lane is responsible for: 93 shuffles for 81 sums instead of 5 x 81), fixed order
        // across the four warps
        warp_sum_taps<K>(acc, lane, red + (warp - 2) * K * K);
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int et = threadIdx.x - 64;
        if (et < K * K) {
          float sum = 0.f;
#pragma unroll
          for (int q = 0; q < 4; ++q) sum += red[q * K * K + et];
          p.out[((long)w.split() * p.C + w.channel()) * (K * K) + et] = sum;
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
    }
  }

  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool dw_tc_wgrad2_supported(int H, int W, int Ho, int Wo, int k, int dil, int pad) {
  const int halo = dil * (k - 1);
  return H == Ho && W == Wo && H <= 128 && W <= 128 && W % 8 == 0 && k % 2 == 1 && k <= 9 && pad <= W2_GAP &&
         halo - pad >= 0 && halo - pad <= W2_GAP;
}

static int w2_splits(int N, int C) { return tc_unit_splits(C, (N + 1) / 2); }

size_t dw_tc_wgrad2_workspace(int N, int C, int k) { return (size_t)w2_splits(N, C) * C * k * k * sizeof(float) + 16; }

__global__ void dw_tc_wgrad2_reduce_kernel(const float *__restrict__ part, float *__restrict__ dw, int splits, long count) {
  pdl_prologue_done();
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += part[(long)s * count + i];
  dw[i] = acc;
}

int dw_tc_wgrad2_reduce(const float *part, float *dw, int splits, long count, cudaStream_t st) {
  launch_pdl(dw_tc_wgrad2_reduce_kernel, dim3((unsigned)ceil_div<long>(count, 256)), dim3(256), 0, st, part, dw, splits, count);
  return launch_status();
}

template <int K>
static int wgrad2_launch(const void *x, const void *dy, float *dw, float *part, W2Params p, cudaStream_t st) {
  CUtensorMap tm_x, tm_dy;
  const uint64_t dims[4] = {(uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.C, (uint64_t)p.N};
  const uint64_t strides[3] = {(uint64_t)p.W * 2, (uint64_t)p.H * p.W * 2, (uint64_t)p.C * p.H * p.W * 2};
  const uint32_t box[4] = {64, 128, 1, 1};
  int rc = make_tmap_bf16(&tm_x, x, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = make_tmap_bf16(&tm_dy, dy, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  p.out = p.splits == 1 ? dw : part;
  const int smem = 2 * W2_STAGE + 2 * W2_DYBOX + 4 * 32 * W2_SCR_PITCH * 4 + 192 + 4 * K * K * 4 + 64 + 1024;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tc_wgrad2_kernel<K>, smem, attr_cache)) return e;
  const int grid = (int)min(p.units, (long)kNumSMs);
  launch_pdl(dw_tc_wgrad2_kernel<K>, dim3(grid), dim3(W2_THREADS), (size_t)smem, st, tm_x, tm_dy, p);
  rc = launch_status();
  if (rc || p.splits == 1) return rc;
  return dw_tc_wgrad2_reduce(part, dw, p.splits, (long)p.C * K * K, st);
}

int dw_tc_wgrad2(const void *x, const void *dy, float *dw, float *part, int N, int C, int H, int W, int k, int dil,
                 int pad, cudaStream_t st) {
  W2Params p{};
  p.N = N; p.C = C; p.H = H; p.W = W; p.k = k; p.dil = dil; p.pad = pad;
  p.npairs = (N + 1) / 2;
  p.splits = w2_splits(N, C);
  p.units = (long)C * p.splits;
  p.dbg = tc_debug_bits();
  switch (k) {
    case 1: return wgrad2_launch<1>(x, dy, dw, part, p, st);
    case 3: return wgrad2_launch<3>(x, dy, dw, part, p, st);
    case 5: return wgrad2_launch<5>(x, dy, dw, part, p, st);
    case 7: return wgrad2_launch<7>(x, dy, dw, part, p, st);
    case 9: return wgrad2_launch<9>(x, dy, dw, part, p, st);
    default: return KDCC_ESHAPE;
  }
}

}  // namespace kdcc
