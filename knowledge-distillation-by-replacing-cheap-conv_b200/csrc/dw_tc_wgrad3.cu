// Depthwise weight gradient on the tensor cores, column-phase variant (bf16 NCHW planes, 9 x 9 taps, dilation 5, pad 20,
// H, W <= 128): the Cityscapes geometry of the reference's students.
//
//   dw[c][u][v] = sum_{n,i,j} dy[n][c][i][j] * x[n][c][i + 5u - 20][j + 5v - 20]
//
// dw_tc_wgrad2.cu forms P_u = dy^T x (128 x 128 per tap row) and keeps 9 of its 255 diagonals: 93 % of its MMA work is
// junk.  Here both planes are first regrouped by column phase b = j mod 5 (q = j div 5), where the dilated filter is dense:
//
//   dw[u][v] = sum_{n,b} sum_q P_{u,b}[q][q + v - 4],        P_{u,b} = dy_b^T (32 x rows) . x_b[rows + 5u - 20] (rows x 32)
//
// and FOUR tap rows share one MMA: the 128 TMEM lanes of the A operand hold four copies of dy_b^T, copy jj shifted down by
// 5*jj rows, so lane (jj, q) of the product against the x_b window of tap row u0 is P_{u0+jj,b}[q][.].  Per plane that is
// 5 phases x 3 tap-row groups x 9 K-steps of M = 128, N = 32, K = 16 (16 clk each, 1 KB of B from shared memory) instead
// of 72 MMAs of N = 128 (64 clk, 4 KB): 2.2 instead of 4.6 kclk of tensor time and 135 instead of 288 KB of operand reads,
// and the three 128 x 32 accumulators simply keep summing over phases, images and K -- the diagonals are extracted once
// per channel, not once per tap row.
//
// The four shifted copies of dy_b^T cannot be written by address arithmetic (a shift of 5 rows is 10 bytes; TMEM lanes
// belong to warp quadrants), and transposing 2-byte elements through the load/store unit four times would cost more than
// it saves.  The tensor core transposes instead: S . dy_b^T with the selection matrix S[(jj, q)][k] = (k == q) (a constant
// A operand in TMEM, K = 32) lands dy_b^T in all four lane quadrants at once as fp32; eight converter warps read their
// quadrant (tcgen05.ld), keep the upper 16 bits (the values are bf16 already: exact), pair the rows with their quadrant's
// shift and write the bf16 A operand (tcgen05.st).  Zero rows above / below come for free: x_b has 20 zero gap rows on
// both sides (written once), the A slots have zero columns outside each quadrant's data range (written once).
//
// Roles (576 threads): warp 0 TMA (x and dy planes into one landing buffer each), warp 1 MMA issue, warps 2-5 regroup both
// planes into [phase][8-column chunk][row][16 B] (the layout of dw_tc2.cu: K-major for the transposing MMA, MN-major for
// the product), warps 6-9 diagonal extraction, warps 10-17 converters.
// Shared memory: 2 x 32 KB landing, 2 x 52.5 KB x operand, 40 KB dy operand.  TMEM: 2 x 64 columns transposed dy (halves of
// a phase), 2 x 3 x 32 accumulators, 2 x 72 columns A slots, 16 columns S.
// Deterministic: fixed-order sums, no atomics; splits are reduced by dw_tc_wgrad2's reduce kernel.
//
// Measured (4096 channels x 4 images, same box): 0.298 ms against 0.46 ms for dw_tc_wgrad2 -- 5.0 kclk per plane where the
// tensor work is 2.8 and shared memory 3.3.  What is left is hand-off latency: a phase is only ~550 clocks of tensor work, and
// on this chip an mbarrier hand-off between two warps costs ~180 clocks, one through tcgen05.commit ~240, a tcgen05.ld + wait
// ~160 when idle and ~340 under these MMAs (tools/hop_probe.cu, the hand-off trace of a debug build): the chain transposing MMA
// -> commit -> converters load -> release -> store -> product MMA runs once per phase.  Variants that were built and measured
// on the same box (DESIGN.md 4.1): a second issuing thread for the transposing MMAs (equal), a ring of three half-phase tiles
// with the third tap-row group single-buffered to pay for it in TMEM (slower: 0.317), per-phase hand-over of single operand
// buffers behind double landing buffers (slower: ten fence.proxy.async + hops per plane on the regrouping warps), two sets of
// converter warps alternating phases at 72 registers (equal), two transposed tiles with the transposition two phases ahead
// and one accumulator set (0.303 vs 0.293), sixteen converter warps of 32 rows each (0.351 vs 0.303).  tcgen05.ld does not slow
// the MMAs down, but beside them a warp gets one x32 load per ~240 clk (tools/tc_probe2 "ts 128 32 3 1 8": 134 B/clk/SM for
// eight warps, 239 idle): the converters' 320 KB per plane are latency-, not bandwidth-bound.
// Reference semantics: autograd of models/students/transform_blocks/depthwise_separable_conv.py:12.
#include "dw_kernels.cuh"
#include "dw_tc_common.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int W3_THREADS = 576;
constexpr int W3_D = 5, W3_K = 9, W3_PAD = 20;
constexpr uint32_t W3_LAND = 2 * 128 * 128;      // one landed plane: two boxes of 128 rows x 128 bytes
constexpr uint32_t W3_XROWS = 128 + 2 * W3_PAD;  // operand rows of x: zero gap, plane, zero gap
constexpr uint32_t W3_XLBO = W3_XROWS * 16;      // bytes between 8-column chunks of the x operand
constexpr uint32_t W3_XO = W3_D * 4 * W3_XLBO;   // one x operand buffer
constexpr uint32_t W3_DLBO = 128 * 16;
constexpr uint32_t W3_DO = W3_D * 4 * W3_DLBO;   // the dy operand
constexpr uint32_t W3_OFF_XL = 0, W3_OFF_DL = W3_LAND, W3_OFF_XO = 2 * W3_LAND, W3_OFF_DO = W3_OFF_XO + 2 * W3_XO;
constexpr uint32_t W3_OFF_BAR = W3_OFF_DO + W3_DO;
constexpr int W3_SMEM = W3_OFF_BAR + 256 + 1024;
constexpr uint32_t W3_T_DT = 0;     // transposed dy_b, fp32: rows [0, 64) and [64, 128) of the plane
constexpr uint32_t W3_T_ACC = 128;  // [2 units][3 tap-row groups][32]
constexpr uint32_t W3_T_A = 320;    // [2 slots][72]: bf16 pairs of K rows
constexpr uint32_t W3_T_SEL = 464;  // selection matrix, K = 32 -> 16 columns
constexpr uint32_t W3_A_COLS = 72;  // 144 K rows: 128 + 3 * 5 shift, rounded up to the K step

struct W3Params {
  int N, C, H, W;
  int splits;
  long units;  // C * splits
  float *out;  // [splits][C][81] (dw itself when splits == 1)
  int dbg;     // KDCC_TC_DEBUG (timing experiments only): 1 skip extraction, 2 skip product MMAs, 4 skip conversion, 8 skip regrouping
};

// 8*5 consecutive columns of landed row r -> one 16-byte chunk (8 phase-columns) of each of the 5 phases
__device__ __forceinline__ void w3_regroup_row(const uint8_t *stg, uint8_t *dst, uint32_t lbo, int r, int nchunks) {
  constexpr int D = W3_D;
#pragma unroll 1
  for (int g = 0; g < 4; ++g) {
    uint32_t in[4 * D];
#pragma unroll
    for (int j = 0; j < D; ++j) {
      const int c = g * D + j;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (c < nchunks) v = *reinterpret_cast<const uint4 *>(stg + (c >> 3) * (W3_LAND / 2) + r * 128 + (((c & 7) ^ (r & 7)) << 4));
      in[4 * j] = v.x; in[4 * j + 1] = v.y; in[4 * j + 2] = v.z; in[4 * j + 3] = v.w;
    }
#pragma unroll
    for (int b = 0; b < D; ++b) {
      uint32_t o[4];
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int x0 = D * (2 * m) + b, x1 = D * (2 * m + 1) + b;  // elements of the 40-column group
        const uint32_t sel = ((x0 & 1) ? 0x32u : 0x10u) | ((x1 & 1) ? 0x7600u : 0x5400u);
        o[m] = __byte_perm(in[x0 >> 1], in[x1 >> 1], sel);
      }
      *reinterpret_cast<uint4 *>(dst + (size_t)(b * 4 + g) * lbo) = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}

// rotate a lane's 32 registers left by its lane index: afterwards r[k] holds what was r[(k + lane) % 32]
template <int S>
__device__ __forceinline__ void w3_rotate(float (&r)[32], int lane) {
  const bool on = (lane & S) != 0;
  float t[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) t[k] = on ? r[(k + S) & 31] : r[k];
#pragma unroll
  for (int k = 0; k < 32; ++k) r[k] = t[k];
}

__global__ void __launch_bounds__(W3_THREADS, 1)
dw_tc_wgrad3_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_dy, const W3Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + W3_OFF_BAR;
  const uint32_t xl_full = bar_base, xl_empty = bar_base + 8, dl_full = bar_base + 16, dl_empty = bar_base + 24;
  auto xo_full = [&](int s) { return bar_base + 32u + 8u * s; };
  auto xo_empty = [&](int s) { return bar_base + 48u + 8u * s; };
  auto dt_full = [&](int h) { return bar_base + 64u + 8u * h; };
  auto dt_empty = [&](int h) { return bar_base + 80u + 8u * h; };
  auto a_full = [&](int s) { return bar_base + 96u + 8u * s; };
  auto a_empty = [&](int s) { return bar_base + 112u + 8u * s; };
  auto acc_full = [&](int s) { return bar_base + 128u + 8u * s; };
  auto acc_empty = [&](int s) { return bar_base + 144u + 8u * s; };
  auto do_full = [&](int b) { return bar_base + 160u + 8u * b; };   // one per phase: the dy operand is single-buffered and
  auto do_empty = [&](int b) { return bar_base + 200u + 8u * b; };  // handed over phase by phase
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + W3_OFF_BAR + 240);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // the gap rows of the x operand (and the phase-columns past the plane) start as zeros and are never written again
  for (uint32_t i = threadIdx.x; i < 2 * W3_XO / 16; i += W3_THREADS)
    reinterpret_cast<uint4 *>(smem_gen + W3_OFF_XO)[i] = make_uint4(0, 0, 0, 0);
  ptx::fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    ptx::mbar_init(xl_full, 1);
    ptx::mbar_init(xl_empty, 4);
    ptx::mbar_init(dl_full, 1);
    ptx::mbar_init(dl_empty, 4);
    for (int b = 0; b < W3_D; ++b) {
      ptx::mbar_init(do_full(b), 4);
      ptx::mbar_init(do_empty(b), 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(xo_full(s), 4);
      ptx::mbar_init(xo_empty(s), 1);
      ptx::mbar_init(dt_full(s), 1);
      ptx::mbar_init(a_full(s), 8);
      ptx::mbar_init(a_empty(s), 1);
      ptx::mbar_init(acc_full(s), 1);
      ptx::mbar_init(acc_empty(s), 4);
    }
    ptx::mbar_init(dt_empty(0), 6);  // the four converters of rows [0, 64) + the two odd-shift converters of rows [64, 128) (row 63)
    ptx::mbar_init(dt_empty(1), 4);
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_x);
    ptx::prefetch_tensormap(&tm_dy);
  }
  if (warp == 1) ptx::tmem_alloc<512>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp >= 6 && warp <= 9) {
    // constant TMEM contents: zero A slots (each quadrant's data columns are rewritten every phase, the rest stays zero)
    // and the selection matrix: lane (jj, q) holds 1.0 at k = q
    const uint32_t quad = ((uint32_t)((warp & 3) * 32)) << 16;
    uint32_t z[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) z[k] = 0u;
#pragma unroll
    for (int c = 0; c < 2 * (int)W3_A_COLS; c += 16) ptx::tmem_st_32x32b_x16(tmem_base + W3_T_A + quad + c, z);
#pragma unroll
    for (int k = 0; k < 16; ++k) z[k] = (k == (lane >> 1)) ? ((lane & 1) ? 0x3F800000u : 0x00003F80u) : 0u;
    ptx::tmem_st_32x32b_x16(tmem_base + W3_T_SEL + quad, z);
    ptx::tmem_st_wait();
  }
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  pdl_prologue_done();  // everything above overlapped the previous kernel's tail; global memory from here on

  if (warp == 0) {
    if (ptx::elect_one()) {
      // ===== TMA producer: the x plane and the dy plane of every item, one landing buffer each =====
      int t = 0;
      for (PlaneWalk w(p.units, p.N, p.splits, p.C); w.valid(); w.next(), ++t) {
        const int c = w.channel(), n = w.pl;
        ptx::mbar_wait(xl_empty, (uint32_t)(t & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(xl_full, W3_LAND);
        for (int b = 0; b < 2; ++b)  // rows / columns past the plane are zero-filled by the hardware
          ptx::tma_load_4d(smem_base + W3_OFF_XL + b * (W3_LAND / 2), &tm_x, xl_full, 64 * b, 0, c, n);
        ptx::mbar_wait(dl_empty, (uint32_t)(t & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(dl_full, W3_LAND);
        for (int b = 0; b < 2; ++b)
          ptx::tma_load_4d(smem_base + W3_OFF_DL + b * (W3_LAND / 2), &tm_dy, dl_full, 64 * b, 0, c, n);
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      // ===== MMA issuer =====
      constexpr uint32_t idesc_sel = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
      constexpr uint32_t idesc_main = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((32u >> 3) << 17) | ((128u >> 4) << 24);
      // dy operand, K-major: 8-row groups 128 B apart (SBO), K chunks W3_DLBO apart (LBO); no swizzle, descriptor version 1
      constexpr uint32_t sel_hi = (128u >> 4) | (1u << 14);
      const uint32_t sel_lo = (((smem_base + W3_OFF_DO) & 0x3FFFF) >> 4) | ((W3_DLBO >> 4) << 16);
      // x operand, MN-major: 8-column chunks W3_XLBO apart (SBO), 8-row K groups 128 B apart (LBO)
      constexpr uint32_t main_hi = (W3_XLBO >> 4) | (1u << 14);
      const uint32_t main_lo0 = (((smem_base + W3_OFF_XO) & 0x3FFFF) >> 4) | ((128u >> 4) << 16);
      const uint32_t t_sel = tmem_base + W3_T_SEL;
      uint32_t n = 0;  // phase counter: 5 * plane + phase
      // transposing MMAs of phase b of plane t (phase counter m): S (128 x 32) . dy_b^T -> rows [0, 64) and [64, 128)
      auto issue_sel = [&](int t, int b, long m) {
        ptx::mbar_wait(do_full(b), (uint32_t)(t & 1));
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          ptx::mbar_wait(dt_empty(h), (uint32_t)(m & 1) ^ 1);
          ptx::tcgen05_fence_after();
          const uint32_t b_lo = sel_lo + (uint32_t)b * (4u * (W3_DLBO >> 4)) + (uint32_t)h * 64u;
          ptx::umma_f16_ts(tmem_base + W3_T_DT + 64u * h, t_sel, b_lo, sel_hi, idesc_sel, 0u);
          ptx::umma_f16_ts(tmem_base + W3_T_DT + 64u * h, t_sel + 8u, b_lo + 2u * (W3_DLBO >> 4), sel_hi, idesc_sel, 1u);
          ptx::umma_commit(dt_full(h));
        }
        ptx::umma_commit(do_empty(b));  // phase b of the dy operand may be overwritten with the next plane
      };
      int t = 0, unit = -1;
      PlaneWalk w(p.units, p.N, p.splits, p.C);
      if (w.valid()) issue_sel(0, 0, 0);
      for (; w.valid(); w.next(), ++t) {
        PlaneWalk nx = w;
        nx.next();
        const bool has_next = nx.valid(), first = w.first_of_unit(), last = w.last_of_unit();
        const int s = t & 1;
        if (first) {
          ++unit;
          ptx::mbar_wait(acc_empty(unit & 1), (uint32_t)((unit >> 1) & 1) ^ 1);
        }
        ptx::mbar_wait(xo_full(s), (uint32_t)(t >> 1) & 1);
        const uint32_t acc0 = tmem_base + W3_T_ACC + (uint32_t)(unit & 1) * 96u;
        const uint32_t x_lo = main_lo0 + (uint32_t)s * (W3_XO >> 4);
#pragma unroll
        for (int b = 0; b < W3_D; ++b, ++n) {
          if (b < W3_D - 1) issue_sel(t, b + 1, n + 1);
          else if (has_next) issue_sel(t + 1, 0, n + 1);
          const int as = (int)(n & 1);
          ptx::mbar_wait(a_full(as), (uint32_t)(n >> 1) & 1);
          ptx::tcgen05_fence_after();
          if (!KDCC_DBG(p, 2)) {
            const uint32_t a0 = tmem_base + W3_T_A + (uint32_t)as * W3_A_COLS;
            const uint32_t b0 = x_lo + (uint32_t)b * (4u * (W3_XLBO >> 4));
            const uint32_t fresh = (first && b == 0) ? 0u : 1u;
#pragma unroll
            for (int g = 0; g < 3; ++g) {
              // tap rows 4g .. 4g+3: K row kappa of the A slot meets operand row kappa + 20g (plane row kappa + 20g - 20)
#pragma unroll
              for (int ks = 0; ks < (g == 2 ? 8 : 9); ++ks)
                ptx::umma_f16_ts(acc0 + 32u * g, a0 + 8u * ks, b0 + (uint32_t)(16 * ks + 20 * g), main_hi, idesc_main, ks ? 1u : fresh);
            }
          }
          ptx::umma_commit(a_empty(as));
        }
        ptx::umma_commit(xo_empty(s));
        if (last) ptx::umma_commit(acc_full(unit & 1));
      }
    }
  } else if (warp <= 5) {
    // ===== regrouping (128 threads, thread = plane row): x into its double-buffered operand, dy into its single one =====
    const int r = threadIdx.x - 64;
    const int nchunks = p.W >> 3;
    int t = 0;
    for (PlaneWalk w(p.units, p.N, p.splits, p.C); w.valid(); w.next(), ++t) {
      const int s = t & 1;
      ptx::mbar_wait(xo_empty(s), (uint32_t)((t >> 1) & 1) ^ 1);  // the product MMAs of plane t-2 are done
      ptx::mbar_wait(xl_full, (uint32_t)(t & 1));
      if (!KDCC_DBG(p, 8))
        w3_regroup_row(smem_gen + W3_OFF_XL, smem_gen + W3_OFF_XO + (size_t)s * W3_XO + (size_t)(r + W3_PAD) * 16, W3_XLBO, r, nchunks);
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(xo_full(s));
        ptx::mbar_arrive(xl_empty);
      }
      // dy: the row goes to registers (the landing buffer is free again at once), then phase by phase into the single
      // operand buffer as the transposing MMAs of the previous plane release it
      ptx::mbar_wait(dl_full, (uint32_t)(t & 1));
      uint32_t row[80];  // 128 columns + the zeros the last phase-columns (q >= 26) read
#pragma unroll
      for (int c = 64; c < 80; ++c) row[c] = 0u;
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (c < nchunks) v = *reinterpret_cast<const uint4 *>(smem_gen + W3_OFF_DL + (c >> 3) * (W3_LAND / 2) + r * 128 + (((c & 7) ^ (r & 7)) << 4));
        row[4 * c] = v.x; row[4 * c + 1] = v.y; row[4 * c + 2] = v.z; row[4 * c + 3] = v.w;
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(dl_empty);
      uint8_t *dyo = smem_gen + W3_OFF_DO + (size_t)r * 16;
#pragma unroll
      for (int b = 0; b < W3_D; ++b) {
        ptx::mbar_wait(do_empty(b), (uint32_t)(t & 1) ^ 1);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t o[4];
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int x0 = b + W3_D * (8 * g + 2 * m), x1 = x0 + W3_D;  // columns of phase-columns 8g + 2m, 8g + 2m + 1
            const uint32_t sel = ((x0 & 1) ? 0x32u : 0x10u) | ((x1 & 1) ? 0x7600u : 0x5400u);
            o[m] = __byte_perm(row[x0 >> 1], row[x1 >> 1], sel);
          }
          if (!KDCC_DBG(p, 8)) *reinterpret_cast<uint4 *>(dyo + (size_t)(b * 4 + g) * W3_DLBO) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(do_full(b));
      }
    }
  } else if (warp <= 9) {
    // ===== diagonal extraction, once per unit (128 threads; thread = TMEM lane (jj, q)): dw[4g + jj][v] = sum_q D_g[(jj, q)][q + v - 4] =====
    const int jj = warp & 3;
    const uint32_t quad = ((uint32_t)(jj * 32)) << 16;
    int unit = -1;
    for (PlaneWalk w(p.units, p.N, p.splits, p.C); w.valid(); w.next()) {
      if (w.first_of_unit()) ++unit;
      if (!w.last_of_unit()) continue;
      const int ab = unit & 1;
      ptx::mbar_wait(acc_full(ab), (uint32_t)(unit >> 1) & 1);
      ptx::tcgen05_fence_after();
      __syncwarp();
      float *out = p.out + ((long)w.split() * p.C + w.channel()) * (W3_K * W3_K);
#pragma unroll 1
      for (int g = 0; g < 3; ++g) {
        const int u = 4 * g + jj;
        if (u >= W3_K || KDCC_DBG(p, 1)) continue;  // warp-uniform
        uint32_t raw[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + W3_T_ACC + (uint32_t)ab * 96u + 32u * g + quad, raw);
        ptx::tmem_ld_wait();
        float r[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) r[k] = __uint_as_float(raw[k]);
        w3_rotate<16>(r, lane);
        w3_rotate<8>(r, lane);
        w3_rotate<4>(r, lane);
        w3_rotate<2>(r, lane);
        w3_rotate<1>(r, lane);
#pragma unroll
        for (int v = 0; v < W3_K; ++v) {
          const int col = lane + v - 4;
          float val = (col >= 0 && col < 32) ? r[(v - 4) & 31] : 0.f;
#pragma unroll
          for (int m = 16; m >= 1; m >>= 1) val += __shfl_xor_sync(0xffffffffu, val, m);
          if (lane == 0) out[u * W3_K + v] = val;
        }
      }
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(acc_empty(ab));
    }
  } else {
    // ===== converters (256 threads; thread = TMEM lane (jj, q), two warps per quadrant: rows [0, 64) and [64, 128)) =====
    // fp32 dy_b[i][q] in the transposed tile -> bf16 pair (kappa, kappa + 1) of the A slot, kappa = i + 5 jj
    const int jj = warp & 3, h = (warp - 10) >> 2;
    const uint32_t quad = ((uint32_t)(jj * 32)) << 16;
    const int sh = W3_D * jj;
    const bool odd = (jj & 1) != 0, edge = odd && h == 1;
    uint32_t n = 0;
    for (PlaneWalk w(p.units, p.N, p.splits, p.C); w.valid(); w.next()) {
#pragma unroll 1
      for (int b = 0; b < W3_D; ++b, ++n) {
        const int as = (int)(n & 1);
        ptx::mbar_wait(dt_full(h), (uint32_t)(n & 1));
        if (edge) ptx::mbar_wait(dt_full(0), (uint32_t)(n & 1));
        ptx::tcgen05_fence_after();
        __syncwarp();
        uint32_t r0[32], r1[32];
        uint32_t carry = 0u;
        const uint32_t src = tmem_base + W3_T_DT + quad + 64u * h;
        ptx::tmem_ld_32x32b_x32(src, r0);
        ptx::tmem_ld_32x32b_x32(src + 32u, r1);
        if (edge) carry = ptx::tmem_ld_32x32b_x1(tmem_base + W3_T_DT + quad + 63u);
        ptx::tmem_ld_wait();
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive(dt_empty(h));
          if (edge) ptx::mbar_arrive(dt_empty(0));
        }
        ptx::mbar_wait(a_empty(as), (uint32_t)((n >> 1) & 1) ^ 1);  // the product MMAs of phase n-2 are done
        ptx::tcgen05_fence_after();
        __syncwarp();
        const uint32_t dst = tmem_base + W3_T_A + (uint32_t)as * W3_A_COLS + quad;
        if (!KDCC_DBG(p, 4)) {
          uint32_t o[16];
          if (!odd) {
            const uint32_t c0 = (uint32_t)(64 * h + sh) >> 1;
#pragma unroll
            for (int k = 0; k < 16; ++k) o[k] = __byte_perm(r0[2 * k], r0[2 * k + 1], 0x7632);
            ptx::tmem_st_32x32b_x16(dst + c0, o);
#pragma unroll
            for (int k = 0; k < 16; ++k) o[k] = __byte_perm(r1[2 * k], r1[2 * k + 1], 0x7632);
            ptx::tmem_st_32x32b_x16(dst + c0 + 16u, o);
          } else {
            // odd shift: pairs (i, i + 1) with i odd; the first pair of a chunk starts with the last row of the chunk before
            const uint32_t c0 = (uint32_t)(64 * h + sh - 1) >> 1;
            o[0] = __byte_perm(carry, r0[0], 0x7632);
#pragma unroll
            for (int k = 1; k < 16; ++k) o[k] = __byte_perm(r0[2 * k - 1], r0[2 * k], 0x7632);
            ptx::tmem_st_32x32b_x16(dst + c0, o);
            o[0] = __byte_perm(r0[31], r1[0], 0x7632);
#pragma unroll
            for (int k = 1; k < 16; ++k) o[k] = __byte_perm(r1[2 * k - 1], r1[2 * k], 0x7632);
            ptx::tmem_st_32x32b_x16(dst + c0 + 16u, o);
            if (h == 1) ptx::tmem_st_32x32b_x1(dst + c0 + 32u, __byte_perm(r1[31], 0u, 0x7632));  // (row 127, zero)
          }
          ptx::tmem_st_wait();
        }
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(a_full(as));
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
bool dw_tc_wgrad3_supported(int H, int W, int Ho, int Wo, int k, int dil, int pad) {
  return H == Ho && W == Wo && H <= 128 && W <= 128 && W % 8 == 0 && k == W3_K && dil == W3_D && pad == W3_PAD;
}

static int w3_splits(int N, int C) { return tc_unit_splits(C, N); }

size_t dw_tc_wgrad3_workspace(int N, int C) { return (size_t)w3_splits(N, C) * C * W3_K * W3_K * sizeof(float) + 16; }

int dw_tc_wgrad3(const void *x, const void *dy, float *dw, float *part, int N, int C, int H, int W, cudaStream_t st) {
  W3Params p{};
  p.N = N; p.C = C; p.H = H; p.W = W;
  p.splits = w3_splits(N, C);
  p.units = (long)C * p.splits;
  p.dbg = tc_debug_bits();
  p.out = p.splits == 1 ? dw : part;
  CUtensorMap tm_x, tm_dy;
  const uint64_t dims[4] = {(uint64_t)W, (uint64_t)H, (uint64_t)C, (uint64_t)N};
  const uint64_t strides[3] = {(uint64_t)W * 2, (uint64_t)H * W * 2, (uint64_t)C * H * W * 2};
  const uint32_t box[4] = {64, 128, 1, 1};
  int rc = make_tmap_bf16(&tm_x, x, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = make_tmap_bf16(&tm_dy, dy, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tc_wgrad3_kernel, W3_SMEM, attr_cache)) return e;
  const int grid = (int)min(p.units, (long)kNumSMs);
  launch_pdl(dw_tc_wgrad3_kernel, dim3(grid), dim3(W3_THREADS), (size_t)W3_SMEM, st, tm_x, tm_dy, p);
  rc = launch_status();
  if (rc || p.splits == 1) return rc;
  return dw_tc_wgrad2_reduce(part, dw, p.splits, (long)C * W3_K * W3_K, st);
}

}  // namespace kdcc
