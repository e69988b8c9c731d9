// Depthwise weight gradient ON THE TENSOR CORES (tcgen05 + TMEM + TMA), bf16, NCHW planes.
//
//   dw[c][u][v] = sum_{n,i,j} dy[n][c][i][j] * x[n][c][i + u*d - p][j + v*d - p]
//
// For one channel plane and one 128 x 128 dy tile, with xw the (128+halo)^2 input window whose origin is
// (i0 - p, j0 - p) and zero outside the image:
//     P_u[j][q] = sum_i dy[i][j] * xw[i + u*d][q]           (a 128 x (128+halo) matrix, reduction over rows)
//     dw[u][v] += sum_j P_u[j][j + v*d]                      (k diagonals of P_u)
// P_u is one tcgen05.mma chain per tap row u.  B = xw[u*d ...] is an "MN-major" view of the 128B-swizzled
// window TMA landed once per plane (no transpose; the tap-row shift u*d is a +128*u*d byte bump of the
// descriptor start address).  A = dy^T is the same for all k tap rows, so the epilogue warps transpose
// the landed dy tile ONCE per plane into tensor memory (lane = dy column, 64 columns of bf16 pairs) and
// the MMAs take A from TMEM: the shared-memory operand feed -- the limiter of these small MMAs -- then
// only carries B.
// Only k of the 128+halo columns of each P_u row are needed, so the FFMA-bound CUDA-core formulation
// (dw_tma.cu: ~14 TFMA/s) is replaced by ~5 % efficient but 50x faster tensor-core work.
// The epilogue warps pull P_u out of TMEM 32 columns at a time, pick the k diagonal entries of their row
// through a private shared-memory scratch row (dynamic column index), and keep the k*k partial sums in
// registers across all planes of the channel; a warp-shuffle + fixed-order cross-warp sum finishes the
// channel.  Deterministic: no atomics, splits (if any) are reduced by dw_wgrad_reduce_kernel.
// Reference semantics: autograd of models/students/transform_blocks/depthwise_separable_conv.py:12.
#include "dw_kernels.cuh"
#include "dw_tc_common.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int WG_TILE = 128;
constexpr int WG_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2-5 / 6-9: epilogue groups for TMEM accumulator 0 / 1
constexpr int WG_SCR_PITCH = 36;  // floats per scratch row: 16-byte aligned rows, conflict-free 128-bit stores

struct DwTcWgradParams {
  int N, C, H, W, Ho, Wo, k, dil, pad;
  int halo, nbox, x_stages;         // 64-column boxes per x tile, x tiles in flight
  int rows, box_bytes;              // rows per box: the (128+halo)-row window of one plane; bytes per box
  int extra;                        // zero columns on the left so that the TMA column origin is 16-byte aligned
  int nq;                           // P_u columns: (128 + halo) rounded up to 16
  int tiles_h, tiles_w, planes;     // planes = N * tiles_h * tiles_w (per channel)
  int splits;                       // CTAs sharing one channel
  long pairs;                       // C * splits
  float *out;                       // [splits][C][k*k] (or dw itself when splits == 1)
  int dbg;                          // KDCC_TC_DEBUG (timing experiments only): 1 skip diagonal extraction, 2 skip MMAs, 4 skip transposition
};

// MN-major SWIZZLE_128B operands: 64-element groups LBO bytes apart, 8-row (reduction) groups 1024 B apart.
// Descriptors are assembled from 32-bit halves inside the asm: one integer add per operand per MMA for the
// single issuing thread.
__device__ __forceinline__ void wg_mma(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "mov.b64 da, {%1, %3};\n"
      "mov.b64 db, {%2, %3};\n"
      "setp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n"
      "}\n"
      ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

constexpr int WG_BOX = WG_TILE * 128;  // 128 rows x 64 columns, swizzled

// TMEM map (512 columns allocated): P_u accumulators at columns [0,192) and [256,448) (nq <= 192), the
// transposed dy operand (128 reduction rows packed as 64 columns of bf16 pairs) at [192,256) and [448,512).
constexpr uint32_t WG_TMEM_D1 = 256, WG_TMEM_A0 = 192, WG_TMEM_A1 = 448;

// A from TMEM, B from shared memory
__device__ __forceinline__ void wg_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 db;\n"
      "mov.b64 db, {%2, %3};\n"
      "setp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n"
      "}\n"
      ::"r"(tmem_d), "r"(tmem_a), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

template <int K>
__global__ void __launch_bounds__(WG_THREADS, 1)
dw_tc_wgrad_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_dy,
                   const DwTcWgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  const int x_bytes = p.nbox * p.box_bytes;
  const int XS = p.x_stages;
  const uint32_t dy_off = XS * x_bytes;                     // one stage = 2 boxes of dy (consumed at once by the transposers)
  const uint32_t scr_off = dy_off + 2 * WG_BOX;
  const uint32_t bar_off = scr_off + 8 * 32 * WG_SCR_PITCH * 4;
  const uint32_t bar_base = smem_base + bar_off;
  auto dy_full = [&](int s) { return bar_base + 8u * s; };
  auto dy_empty = [&](int s) { return bar_base + 8u * (2 + s); };
  auto t_full = [&](int s) { return bar_base + 8u * (4 + s); };
  auto t_empty = [&](int s) { return bar_base + 8u * (6 + s); };
  auto a_full = [&](int s) { return bar_base + 8u * (8 + s); };   // dy^T of a plane is in TMEM
  auto x_full = [&](int s) { return bar_base + 8u * (10 + s); };
  auto x_empty = [&](int s) { return bar_base + 8u * (14 + s); };  // room for 4 x stages (2 in use)
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + bar_off + 160);
  float *red = reinterpret_cast<float *>(smem_gen + bar_off + 192);  // [8 warps][K*K]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(dy_full(s), 1);
      ptx::mbar_init(dy_empty(s), 8);
      ptx::mbar_init(t_full(s), 1);
      ptx::mbar_init(t_empty(s), 4);
      ptx::mbar_init(a_full(s), 8);
    }
    for (int s = 0; s < XS; ++s) {
      ptx::mbar_init(x_full(s), 1);
      ptx::mbar_init(x_empty(s), 1);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_x);
    ptx::prefetch_tensormap(&tm_dy);
  }
  if (warp == 1) ptx::tmem_alloc<512>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto decode_plane = [&](int pl, int &n, int &i0, int &j0) {
    const int tj = pl % p.tiles_w; pl /= p.tiles_w;
    const int ti = pl % p.tiles_h;
    n = pl / p.tiles_h;
    i0 = ti * WG_TILE;
    j0 = tj * WG_TILE;
  };

  if (warp == 0 && lane == 0) {
    // ===== TMA producer: dy tile and x window once per plane =====
    int it = 0;
    int xs = 0; uint32_t xph = 0;
    for (PlaneWalk w(p.pairs, p.planes, p.splits, p.C); w.valid(); w.next(), ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int c = w.channel();
      int n, i0, j0;
      decode_plane(w.pl, n, i0, j0);
      ptx::mbar_wait(dy_empty(0), (uint32_t)(it & 1) ^ 1);
      ptx::mbar_arrive_expect_tx(dy_full(0), 2 * WG_BOX);
      for (int b = 0; b < 2; ++b)
        ptx::tma_load_4d(smem_base + dy_off + b * WG_BOX, &tm_dy, dy_full(0), j0 + 64 * b, i0, c, n);
      ptx::mbar_wait(x_empty(xs), xph ^ 1);
      ptx::mbar_arrive_expect_tx(x_full(xs), (uint32_t)(p.nbox * p.rows * 128));
      for (int b = 0; b < p.nbox; ++b)
        ptx::tma_load_4d(smem_base + xs * x_bytes + b * p.box_bytes, &tm_x, x_full(xs),
                         j0 - p.pad - p.extra + 64 * b, i0 - p.pad, c, n);
      if (++xs == XS) { xs = 0; xph ^= 1; }
    }
  } else if (warp == 1 && lane == 0) {
    // ===== MMA issuer: P_u (128 dy columns x nq window columns) = dy^T [TMEM] * x_u [smem, MN-major] =====
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) |
                           ((uint32_t)(p.nq >> 3) << 17) | ((uint32_t)(WG_TILE >> 4) << 24);
    const uint32_t b_hi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO 1024, version 1, SWIZZLE_128B
    int it = 0, tit = 0;
    int xs = 0; uint32_t xph = 0;
    for (PlaneWalk w(p.pairs, p.planes, p.splits, p.C); w.valid(); w.next(), ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      ptx::mbar_wait(a_full(s), ph);
      const uint32_t a_tmem = tmem_base + (s ? WG_TMEM_A1 : WG_TMEM_A0);
      for (int u = 0; u < K; ++u, ++tit) {
        const int tb = tit & 1;
        if (u == 0) ptx::mbar_wait(x_full(xs), xph);  // inside the loop: hoisted, it costs the K = 9 instance a spill
        ptx::mbar_wait(t_empty(tb), ((tit >> 1) & 1) ^ 1);
        ptx::tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (tb ? WG_TMEM_D1 : 0u);
        // tap row u starts u*dil rows (128 B each) further down the window
        const uint32_t xa = smem_base + xs * x_bytes + (uint32_t)(u * p.dil) * 128u;
        const uint32_t b_lo = ((xa & 0x3FFFF) >> 4) | ((uint32_t)(p.box_bytes >> 4) << 16);
        if (!KDCC_DBG(p, 2)) {
#pragma unroll
          for (int ks = 0; ks < WG_TILE / 16; ++ks)  // 16 reduction rows per MMA: 8 TMEM columns of A, 2 KB of B
            wg_mma_ts(d_tmem, a_tmem + ks * 8, b_lo + ks * 128, b_hi, idesc, ks ? 1u : 0u);
        }
        ptx::umma_commit(t_full(tb));
        if (u == K - 1) {
          ptx::umma_commit(x_empty(xs));  // window free once the last tap row's MMAs have read it
          if (++xs == XS) { xs = 0; xph ^= 1; }
        }
      }
    }
  } else if (warp >= 2) {
    // ===== operand transposer + epilogue (128 threads; thread = dy column j = TMEM lane) =====
    const int quad = warp & 3;
    const int grp = (warp - 2) >> 2;  // 0: TMEM accumulator 0 and dy rows 0-63, 1: accumulator 1 and dy rows 64-127
    const int j = quad * 32 + lane;
    float *scr = reinterpret_cast<float *>(smem_gen + scr_off) + (grp * 128 + j) * WG_SCR_PITCH;
    const int nch = (31 + p.halo + p.extra) / 32 + 1;  // 32-column chunks a warp's rows reach into

    // dy tile (two 128B-swizzled boxes of 64 columns) -> TMEM lane j, column r/2 = (dy[r][j], dy[r+1][j])
    auto transpose_dy = [&](int it) {
      const int s = it & 1;
      ptx::mbar_wait(dy_full(0), (uint32_t)(it & 1));
      const uint8_t *tile = smem_gen + dy_off + (size_t)(j >> 6) * WG_BOX;
      const int chunk = (j & 63) >> 3, within = (j & 7) * 2;
      const uint32_t t_dst = tmem_base + (s ? WG_TMEM_A1 : WG_TMEM_A0) + ((uint32_t)(quad * 32) << 16);
      {
        const int half = grp;  // each group packs 64 reduction rows = 32 TMEM columns
        uint32_t regs[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          const int r = half * 64 + 2 * q;  // rows r (even) and r + 1 share the 8-row swizzle phase pair (r & 7, r & 7 + 1)
          const uint32_t lo = *reinterpret_cast<const uint16_t *>(tile + r * 128 + ((chunk ^ (r & 7)) << 4) + within);
          const uint32_t hi = *reinterpret_cast<const uint16_t *>(tile + (r + 1) * 128 + ((chunk ^ ((r + 1) & 7)) << 4) + within);
          regs[q] = lo | (hi << 16);
        }
        tmem_st_32x32b_x32(t_dst + half * 32, regs);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(a_full(s));    // operand ready for the MMA thread
        ptx::mbar_arrive(dy_empty(0));  // the smem tile can be refilled
      }
    };

    int it = 0, tit = 0;
    PlaneWalk cur(p.pairs, p.planes, p.splits, p.C), nxt(p.pairs, p.planes, p.splits, p.C);
    if (nxt.valid()) nxt.next();
    if (cur.valid()) transpose_dy(0);
    float acc[K][K];
    for (; cur.valid(); ++it) {
      // the other TMEM A buffer was last read by the MMAs of plane it-1, all observed complete through t_full
      if (nxt.valid()) transpose_dy(it + 1);
      if (cur.first_of_unit()) {
#pragma unroll
        for (int u = 0; u < K; ++u)
#pragma unroll
          for (int v = 0; v < K; ++v) acc[u][v] = 0.f;
      }
#pragma unroll
      for (int u = 0; u < K; ++u, ++tit) {
        const int tb = tit & 1;
        if (tb != grp) continue;  // the other group drains this accumulator
        ptx::mbar_wait(t_full(tb), (tit >> 1) & 1);
        ptx::tcgen05_fence_after();
        __syncwarp();  // lanes leave the polling loop one by one; the TMEM accesses below are .sync.aligned
        const uint32_t t_row = tmem_base + (tb ? WG_TMEM_D1 : 0u) + ((uint32_t)(quad * 32) << 16);
        for (int c3 = 0; c3 < (KDCC_DBG(p, 1) ? 0 : nch); ++c3) {
          const int col0 = 32 * (quad + c3);
          if (col0 >= p.nq) break;
          uint32_t vr[32];
          ptx::tmem_ld_32x32b_x32(t_row + col0, vr);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4 *>(scr + 4 * q) = make_uint4(vr[4 * q], vr[4 * q + 1], vr[4 * q + 2], vr[4 * q + 3]);
#pragma unroll
          for (int v = 0; v < K; ++v) {
            const int e = lane + v * p.dil + p.extra - 32 * c3;  // window column of tap v for row j, relative to this chunk
            if (e >= 0 && e < 32) acc[u][v] += scr[e];
          }
        }
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(t_empty(tb));
      }
      if (cur.last_of_unit()) {
        // channel (pair) finished: sum the 128 rows -- reduce-scatter inside the warp, fixed order across warps
        warp_sum_taps<K>(acc, lane, red + (grp * 4 + quad) * K * K);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const int et = threadIdx.x - 64;
        if (et < K * K) {
          float sum = 0.f;
#pragma unroll
          for (int q = 0; q < 8; ++q) sum += red[q * K * K + et];  // fixed order: group, then quadrant
          p.out[((long)cur.split() * p.C + cur.channel()) * (K * K) + et] = sum;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      cur.next();
      if (nxt.valid()) nxt.next();
    }
  }

  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc<512>(tmem_base);
}

// dw[c][tap] = sum_s part[s][c][tap]
__global__ void dw_tc_wgrad_reduce_kernel(const float *__restrict__ part, float *__restrict__ dw, int splits, long count) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += part[(long)s * count + i];
  dw[i] = acc;
}

static int wg_splits(int C, int planes) { return tc_unit_splits(C, planes); }

size_t dw_tc_wgrad_workspace(int N, int C, int Ho, int Wo, int k) {
  const int planes = N * ceil_div(Ho, WG_TILE) * ceil_div(Wo, WG_TILE);
  return (size_t)wg_splits(C, planes) * C * k * k * sizeof(float) + 16;
}

template <int K>
static int wgrad_launch(const void *x, const void *dy, float *dw, float *part, const DwTcWgradParams &p0, cudaStream_t st) {
  DwTcWgradParams p = p0;
  CUtensorMap tm_x, tm_dy;
  {
    const uint64_t dims[4] = {(uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.C, (uint64_t)p.N};
    const uint64_t strides[3] = {(uint64_t)p.W * 2, (uint64_t)p.H * p.W * 2, (uint64_t)p.C * p.H * p.W * 2};
    const uint32_t box[4] = {64, (uint32_t)p.rows, 1, 1};
    int rc = make_tmap_bf16(&tm_x, x, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  {
    const uint64_t dims[4] = {(uint64_t)p.Wo, (uint64_t)p.Ho, (uint64_t)p.C, (uint64_t)p.N};
    const uint64_t strides[3] = {(uint64_t)p.Wo * 2, (uint64_t)p.Ho * p.Wo * 2, (uint64_t)p.C * p.Ho * p.Wo * 2};
    const uint32_t box[4] = {64, WG_TILE, 1, 1};
    int rc = make_tmap_bf16(&tm_dy, dy, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  p.out = p.splits == 1 ? dw : part;
  const int fixed = 2 * WG_BOX + 8 * 32 * WG_SCR_PITCH * 4 + 192 + 8 * K * K * 4 + 64 + 1024;  // dy, scratch, barriers, red, slack
  p.x_stages = min(2, (220 * 1024 - fixed) / (p.nbox * p.box_bytes));
  if (p.x_stages < 2) return KDCC_ESHAPE;
  const int smem = p.x_stages * p.nbox * p.box_bytes + fixed;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tc_wgrad_kernel<K>, smem, attr_cache)) return e;
  const int grid = (int)min(p.pairs, (long)kNumSMs);
  dw_tc_wgrad_kernel<K><<<grid, WG_THREADS, smem, st>>>(tm_x, tm_dy, p);
  int rc = launch_status();
  if (rc || p.splits == 1) return rc;
  const long count = (long)p.C * K * K;
  dw_tc_wgrad_reduce_kernel<<<(unsigned)ceil_div<long>(count, 256), 256, 0, st>>>(part, dw, p.splits, count);
  return launch_status();
}

int dw_tc_wgrad(const void *x, const void *dy, float *dw, float *part, int N, int C, int H, int W, int Ho, int Wo,
                int k, int dil, int pad, cudaStream_t st) {
  DwTcWgradParams p{};
  p.N = N; p.C = C; p.H = H; p.W = W; p.Ho = Ho; p.Wo = Wo; p.k = k; p.dil = dil; p.pad = pad;
  p.halo = dil * (k - 1);
  p.dbg = tc_debug_bits();
  p.extra = (8 - pad % 8) % 8;
  p.nq = (WG_TILE + p.halo + p.extra + 15) / 16 * 16;
  p.nbox = ceil_div(p.nq, 64);
  p.rows = WG_TILE + p.halo;
  p.box_bytes = (p.rows + 7) / 8 * 8 * 128;
  p.tiles_h = ceil_div(Ho, WG_TILE);
  p.tiles_w = ceil_div(Wo, WG_TILE);
  p.planes = N * p.tiles_h * p.tiles_w;
  p.splits = wg_splits(C, p.planes);
  p.pairs = (long)C * p.splits;
  if (p.nq > 192) return KDCC_ESHAPE;  // TMEM map: two P_u buffers of <= 192 columns + two dy^T operands of 64
  switch (k) {
    case 1: return wgrad_launch<1>(x, dy, dw, part, p, st);
    case 3: return wgrad_launch<3>(x, dy, dw, part, p, st);
    case 5: return wgrad_launch<5>(x, dy, dw, part, p, st);
    case 7: return wgrad_launch<7>(x, dy, dw, part, p, st);
    case 9: return wgrad_launch<9>(x, dy, dw, part, p, st);
    default: return KDCC_ESHAPE;
  }
}

}  // namespace kdcc
