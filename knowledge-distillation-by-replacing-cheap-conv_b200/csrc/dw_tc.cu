// Depthwise k x k convolution ON THE TENSOR CORES (tcgen05 + TMEM + TMA), bf16, NCHW planes.
//
// Why: a 9x9 depthwise tap set is 81 MAC per output element -- 20 MAC per HBM byte -- which is far past
// the CUDA-core FFMA ridge of a B200 (dw_tma.cu measures ~14 TFMA/s, FFMA-issue-bound at ~10 % of HBM
// speed).  Per channel the convolution along a row is a banded (Toeplitz) matrix product, so it can be
// fed to tcgen05.mma; even at ~12 % structural efficiency the tensor pipe outruns the FFMA pipe by an
// order of magnitude and the kernel becomes HBM/L2-bound again, as the north star asks.
//
// Formulation for one channel plane and a 128 x 128 output tile (i rows, j cols), dilation d, taps k:
//     out[i][j] = sum_u  sum_{j'}  X[i + u*d][j'] * T_u[j'][j],      T_u[j'][j] = w[u][(j'-j)/d] (banded)
//   = sum_u  A_u (128 x K) * B_u (K x 16)   per 16-column output slice, K = 16 + d(k-1) rounded to 16.
//  * A_u is the SAME shared-memory tile for every u: TMA lands the (128+halo)-row input window once
//    (128B-swizzled rows of 64 columns, out-of-bounds = zero = the conv padding); the tap-row shift u*d is
//    a +128*u*d byte bump of the UMMA descriptor start address, the column slice of an output N-tile a
//    +32 byte bump.  No im2col, no data movement.  (TMA needs a 16-byte aligned column origin, so the window
//    starts up to 7 columns left of j0 - pad and the Toeplitz band is shifted right by the same amount.)
//  * B_u (16 x 64 bf16, 2 KB) is the Toeplitz band of one tap row; the band positions are identical for
//    every channel, so the buffers are zeroed once and only the k*16*k band values are rewritten per plane.
//  * D (128 x 128 fp32) lives in TMEM, double buffered: the epilogue of plane n overlaps the MMAs of n+1.
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 build B for the NEXT plane then drain TMEM
// for the current one (tcgen05.ld -> bf16 -> global).
// The input-gradient form is the same kernel over dy with mirrored taps (flip) and pad' = d(k-1) - pad.
// Reference semantics: models/students/transform_blocks/depthwise_separable_conv.py:7-8,12 (+ autograd).
#include "dw_kernels.cuh"
#include "dw_tc_common.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int TC_TILE = 128;     // output rows and columns per tile (UMMA M = 128)
constexpr int TC_THREADS = 288;  // warp 0 TMA, warps 1,6,7,8 MMA issuers (N-tiles round-robin), warps 2-5 epilogue
constexpr int TC_ISSUERS = 4;    // MMA-issuing threads: lane 0 of warps 1, 6, 7, 8

struct DwTcParams {
  int N, C, Hi, Wi, Ho, Wo, k, dil, pad, flip;
  int halo;       // dil * (k - 1)
  int nbox;       // 64-column boxes per A tile
  int a_stages;   // A tiles in flight
  int rows;       // rows per A tile: 128 + halo, the input window of one item
  int box_bytes;  // ceil8(rows) * 128
  int extra;      // zero columns added on the left so that the TMA column origin is 16-byte aligned
  int ksteps;     // ceil((NT + halo) / 16)
  int tiles_h, tiles_w;
  int planes, splits;  // planes per channel (N * tiles), CTAs sharing a channel
  long pairs;          // units = C * splits
  const float *w, *bias;
  __nv_bfloat16 *out;
  int dbg;  // KDCC_TC_DEBUG (timing experiments only): 1 skip Toeplitz rebuild, 2 skip MMAs, 4 skip epilogue stores
};

// K-major, SWIZZLE_128B operand tile: 128-byte rows, 8-row groups 1024 B apart, tile base 1024-byte aligned;
// the start address may advance by 32-byte K slices inside the swizzle row.
__device__ __forceinline__ uint64_t tc_desc(uint32_t addr, int base_mode = 1) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;                    // LBO (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;          // SBO
  d |= (uint64_t)1 << 46;                    // descriptor version
  // The start may sit on any 128-byte row of the tile: the hardware derives the swizzle phase from the
  // address bits, so the base-offset field stays 0 (measured on B200; setting it to the row phase breaks
  // the results).  Modes 1/2 exist only to reproduce that measurement.
  if (base_mode == 1) d |= (uint64_t)((addr >> 7) & 7) << 49;
  else if (base_mode == 2) d |= (uint64_t)((8 - ((addr >> 7) & 7)) & 7) << 49;
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
  return d;
}

// 64-bit descriptors are assembled from 32-bit halves inside the asm so that the single issuing thread spends
// one integer add per operand per MMA (the MMAs are small -- N = 16/32 -- and would otherwise be issue-bound).
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                       uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "mov.b64 da, {%1, %2};\n"
      "mov.b64 db, {%3, %4};\n"
      "setp.ne.b32 p, %6, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
      "}\n"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

template <int NT, int KS>
__global__ void __launch_bounds__(TC_THREADS, 1)
dw_tc_conv_kernel(const __grid_constant__ CUtensorMap tm_in, const DwTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  const int a_stage_bytes = p.nbox * p.box_bytes;
  // one tap row's Toeplitz tile, un-swizzled K-major core matrices: [K chunk of 8][NT rows][16 bytes]
  constexpr int BU_BYTES = KS * 2 * NT * 16;
  const int b_stage_bytes = p.k * BU_BYTES;
  const int AS = p.a_stages;
  const uint32_t b_base = smem_base + AS * a_stage_bytes;
  const uint32_t bar_base = b_base + 2 * b_stage_bytes;
  auto b_full = [&](int s) { return bar_base + 8u * s; };
  auto t_full = [&](int s) { return bar_base + 8u * (2 + s); };
  auto t_empty = [&](int s) { return bar_base + 8u * (4 + s); };
  auto a_full = [&](int s) { return bar_base + 8u * (6 + s); };
  auto a_empty = [&](int s) { return bar_base + 8u * (6 + 8 + s); };  // room for 8 A stages (2 in use)
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + (bar_base - smem_base) + 8 * 22);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(b_full(s), 128);
      ptx::mbar_init(t_full(s), TC_ISSUERS);   // one commit per issuing thread
      ptx::mbar_init(t_empty(s), 4);
    }
    for (int s = 0; s < AS; ++s) {
      ptx::mbar_init(a_full(s), 1);
      ptx::mbar_init(a_empty(s), TC_ISSUERS);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_in);
  }
  if (warp == 1) ptx::tmem_alloc<2 * TC_TILE>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto decode = [&](int pl, int &n, int &i0, int &j0) {
    const int tj = pl % p.tiles_w; pl /= p.tiles_w;
    const int ti = pl % p.tiles_h;
    n = pl / p.tiles_h;
    i0 = ti * TC_TILE;
    j0 = tj * TC_TILE;
  };

  if (warp == 0 && lane == 0) {
    // ===== TMA producer: the input window of an item, once =====
    int as = 0; uint32_t aph = 0;
    for (PlaneWalk w(p.pairs, p.planes, p.splits, p.C); w.valid(); w.next()) {
      const int c = w.channel();
      int n, i0, j0;
      decode(w.pl, n, i0, j0);
      ptx::mbar_wait(a_empty(as), aph ^ 1);
      ptx::mbar_arrive_expect_tx(a_full(as), (uint32_t)(p.nbox * p.rows * 128));
      for (int b = 0; b < p.nbox; ++b)
        ptx::tma_load_4d(smem_base + as * a_stage_bytes + b * p.box_bytes, &tm_in, a_full(as),
                         j0 - p.pad - p.extra + 64 * b, i0 - p.pad, c, n);
      if (++as == AS) { as = 0; aph ^= 1; }
    }
  } else if ((warp == 1 || warp >= 6) && lane == 0) {
    // ===== MMA issuers: N-tile t belongs to issuer t % TC_ISSUERS (each tile has its own TMEM columns) =====
    const int t_first = warp == 1 ? 0 : warp - 5;
    // instruction descriptor: fp32 accumulate, bf16 x bf16, both K-major, N = NT, M = 128
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(TC_TILE >> 4) << 24);
    constexpr int T = TC_TILE / NT;
    // A: K-major SWIZZLE_128B (SBO 1024, version 1); the start may sit on any 128-byte row / 32-byte K slice of the
    // window: the hardware derives the swizzle phase from the address bits, the base-offset field stays 0.
    const uint32_t a_hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    // B: K-major, no swizzle: 8-row groups 128 B apart (SBO), K chunks NT*16 B apart (LBO)
    const uint32_t b_hi = (128u >> 4) | (1u << 14);
    const uint32_t b_lbo = (uint32_t)((NT * 16) >> 4) << 16;
    uint32_t a_off[T][KS];  // descriptor start-address increments (16-byte units) of every (N-tile, K slice)
#pragma unroll
    for (int t = 0; t < T; ++t)
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        const int q0 = t * NT + kk * 16;  // first window column of this 16-wide reduction slice
        a_off[t][kk] = ((uint32_t)(q0 >> 6) * (uint32_t)p.box_bytes + (uint32_t)(q0 & 63) * 2u) >> 4;
      }
    int it = 0, unit = -1;
    int as = 0; uint32_t aph = 0;
    for (PlaneWalk w(p.pairs, p.planes, p.splits, p.C); w.valid(); w.next(), ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      ptx::mbar_wait(t_empty(s), ph ^ 1);
      if (w.first_of_unit()) {  // the Toeplitz operand is per channel: one build per unit
        ++unit;
        ptx::mbar_wait(b_full(unit & 1), (unit >> 1) & 1);
      }
      const uint32_t b0 = b_base + (unit & 1) * b_stage_bytes;
      const uint32_t d0 = tmem_base + (uint32_t)(s * TC_TILE);
      ptx::mbar_wait(a_full(as), aph);
      ptx::tcgen05_fence_after();
#pragma unroll 1
      for (int u = 0; u < p.k; ++u) {
        // tap row u starts u*dil rows (128 B each) further down the window
        const uint32_t a0 = smem_base + as * a_stage_bytes + (uint32_t)(u * p.dil) * 128u;
        const uint32_t a_lo = ((a0 & 0x3FFFF) >> 4) | (1u << 16);
        const uint32_t b_lo = (((b0 + (uint32_t)u * BU_BYTES) & 0x3FFFF) >> 4) | b_lbo;
        const uint32_t acc0 = u ? 1u : 0u;
#pragma unroll
        for (int t = 0; t < T; ++t) {
          if (t % TC_ISSUERS != t_first || KDCC_DBG(p, 2)) continue;
#pragma unroll
          for (int kk = 0; kk < KS; ++kk)
            tc_mma(d0 + (uint32_t)(t * NT), a_lo + a_off[t][kk], a_hi, b_lo + (uint32_t)(kk * 2 * NT), b_hi, idesc,
                   kk ? 1u : acc0);
        }
      }
      ptx::umma_commit(a_empty(as));  // window free once these MMAs have read it
      if (++as == AS) { as = 0; aph ^= 1; }
      ptx::umma_commit(t_full(s));
    }
  } else if (warp >= 2 && warp <= 5) {
    // ===== Toeplitz builder + epilogue (128 threads) =====
    const int et = threadIdx.x - 64;  // 0..127
    const int quad = warp & 3;
    // zero both B stages once: the band positions never change, only their values
    for (int i = et; i < 2 * b_stage_bytes / 16; i += 128)
      *reinterpret_cast<uint4 *>(smem_gen + (b_base - smem_base) + (size_t)i * 16) = make_uint4(0, 0, 0, 0);
    asm volatile("bar.sync 1, 128;" ::: "memory");

    auto build_b = [&](int c, int s) {
      const float *wc = p.w + (long)c * p.k * p.k;
      uint8_t *bs = smem_gen + (b_base - smem_base) + (size_t)s * b_stage_bytes;
      // (tap row u, output column j) pairs; the k taps of a pair land on the band j' = j + v*dil + extra
      for (int idx = et; idx < (KDCC_DBG(p, 1) ? 0 : p.k * NT); idx += 128) {
        const int u = idx / NT, j = idx % NT;
        const float *wr = wc + (p.flip ? (p.k - 1 - u) * p.k : u * p.k);
        uint8_t *row = bs + u * BU_BYTES + j * 16;
        for (int v = 0; v < p.k; ++v) {
          const int jp = j + v * p.dil + p.extra;
          const float wv = __ldg(wr + (p.flip ? p.k - 1 - v : v));
          *reinterpret_cast<__nv_bfloat16 *>(row + (jp >> 3) * (NT * 16) + (jp & 7) * 2) = __float2bfloat16_rn(wv);
        }
      }
      ptx::fence_proxy_async_smem();
      ptx::mbar_arrive(b_full(s));
    };

    PlaneWalk cur(p.pairs, p.planes, p.splits, p.C), ahead(p.pairs, p.planes, p.splits, p.C);
    if (ahead.valid()) ahead.next_unit();
    if (cur.valid()) build_b(cur.channel(), 0);
    int it = 0, unit = -1;
    for (; cur.valid(); cur.next(), ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      if (cur.first_of_unit()) {
        ++unit;
        // build the NEXT unit's operand now: its buffer was last read by the MMAs of unit-1, all of which we
        // observed complete (t_full of that unit's last plane) before getting here
        if (ahead.valid()) { build_b(ahead.channel(), (unit + 1) & 1); ahead.next_unit(); }
      }
      const int c = cur.channel();
      int n, i0, j0;
      decode(cur.pl, n, i0, j0);
      ptx::mbar_wait(t_full(s), ph);
      ptx::tcgen05_fence_after();
      __syncwarp();  // lanes leave the polling loop one by one; the TMEM accesses below are .sync.aligned
      const int gi = i0 + quad * 32 + lane;
      const float bias = p.bias ? __ldg(p.bias + c) : 0.f;
      __nv_bfloat16 *orow = p.out + (((long)n * p.C + c) * p.Ho + gi) * p.Wo + j0;
      const uint32_t t_row = tmem_base + (uint32_t)(s * TC_TILE) + ((uint32_t)(quad * 32) << 16);
#pragma unroll 1
      for (int ch = 0; ch < TC_TILE / 32; ++ch) {
        uint32_t vr[32];
        ptx::tmem_ld_32x32b_x32(t_row + ch * 32, vr);
        ptx::tmem_ld_wait();
        if (gi < p.Ho && !KDCC_DBG(p, 4)) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int col = j0 + ch * 32 + q * 8;
            if (col < p.Wo) {
              uint4 o;
              o.x = pack_bf16x2(__uint_as_float(vr[8 * q + 0]) + bias, __uint_as_float(vr[8 * q + 1]) + bias);
              o.y = pack_bf16x2(__uint_as_float(vr[8 * q + 2]) + bias, __uint_as_float(vr[8 * q + 3]) + bias);
              o.z = pack_bf16x2(__uint_as_float(vr[8 * q + 4]) + bias, __uint_as_float(vr[8 * q + 5]) + bias);
              o.w = pack_bf16x2(__uint_as_float(vr[8 * q + 6]) + bias, __uint_as_float(vr[8 * q + 7]) + bias);
              *reinterpret_cast<uint4 *>(orow + ch * 32 + q * 8) = o;
            }
          }
        }
      }
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(t_empty(s));
    }
  }

  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc<2 * TC_TILE>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int tc_extra(int pad) { return (8 - pad % 8) % 8; }
// output columns per MMA (N): 32 halves both the MMA count and the A re-reads; the Toeplitz K extent
// (N + halo + alignment columns) must stay within the instantiated K-slice counts
static int tc_nt(int reach) { return reach + 32 <= 80 ? 32 : 16; }

bool dw_tc_supported(int Hi, int Wi, int Ho, int Wo, int k, int dil, int pad) {
  (void)Hi; (void)Ho;
  const int halo = dil * (k - 1);
  if (k > 9 || k % 2 == 0) return false;      // wgrad keeps k*k register partials: instantiated for k = 1,3,5,7,9
  if (pad > halo) return false;               // the input gradient runs this kernel with pad' = halo - pad >= 0
  if (halo + 7 + 16 > 80) return false;       // Toeplitz K extent (incl. alignment columns) <= 5 slices of 16
  if (Wi % 8 != 0 || Wo % 8 != 0) return false;  // 16-byte rows for TMA strides and epilogue stores
  return true;
}

template <int NT, int KS>
static int tc_conv_launch(const void *in, const DwTcParams &p0, cudaStream_t st) {
  DwTcParams p = p0;
  p.ksteps = KS;
  p.nbox = ceil_div((TC_TILE - NT) + KS * 16, 64);  // the last N-tile's last reduction slice ends here
  p.rows = TC_TILE + p.halo;
  p.box_bytes = (p.rows + 7) / 8 * 8 * 128;
  const int b_bytes = 2 * p.k * KS * 2 * NT * 16;
  p.a_stages = min(2, (int)((226 * 1024 - b_bytes - 2048) / (p.nbox * p.box_bytes)));
  if (p.a_stages < 2) return KDCC_ESHAPE;
  CUtensorMap tm;
  const uint64_t dims[4] = {(uint64_t)p.Wi, (uint64_t)p.Hi, (uint64_t)p.C, (uint64_t)p.N};
  const uint64_t strides[3] = {(uint64_t)p.Wi * 2, (uint64_t)p.Hi * p.Wi * 2, (uint64_t)p.C * p.Hi * p.Wi * 2};
  const uint32_t box[4] = {64, (uint32_t)p.rows, 1, 1};
  int rc = make_tmap_bf16(&tm, in, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  const int smem = p.a_stages * p.nbox * p.box_bytes + b_bytes + 256 + 1024;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tc_conv_kernel<NT, KS>, smem, attr_cache)) return e;
  const int grid = (int)min(p.pairs, (long)kNumSMs);
  dw_tc_conv_kernel<NT, KS><<<grid, TC_THREADS, smem, st>>>(tm, p);
  return launch_status();
}

template <int NT>
static int tc_conv_dispatch_ks(const void *in, const DwTcParams &p, cudaStream_t st) {
  switch (ceil_div(NT + p.halo + p.extra, 16)) {
    case 1: case 2: return tc_conv_launch<NT, 2>(in, p, st);
    case 3: return tc_conv_launch<NT, 3>(in, p, st);
    case 4: return tc_conv_launch<NT, 4>(in, p, st);
    case 5: return tc_conv_launch<NT, 5>(in, p, st);
    default: return KDCC_ESHAPE;
  }
}

int dw_tc_conv(const void *in, const float *w, const float *bias, void *out, int N, int C, int Hi, int Wi, int Ho,
               int Wo, int k, int dil, int pad, int flip, cudaStream_t st) {
  if (dw_tc_conv2_supported(Hi, Wi, Ho, Wo, k, dil, pad)) return dw_tc_conv2(in, w, bias, out, N, C, Hi, Wi, k, dil, pad, flip, st);
  DwTcParams p{};
  p.N = N; p.C = C; p.Hi = Hi; p.Wi = Wi; p.Ho = Ho; p.Wo = Wo; p.k = k; p.dil = dil; p.pad = pad; p.flip = flip;
  p.halo = dil * (k - 1);
  p.tiles_h = ceil_div(Ho, TC_TILE);
  p.tiles_w = ceil_div(Wo, TC_TILE);
  p.planes = N * p.tiles_h * p.tiles_w;
  p.splits = tc_unit_splits(C, p.planes);
  p.pairs = (long)C * p.splits;
  p.w = w; p.bias = bias;
  p.out = static_cast<__nv_bfloat16 *>(out);
  if (p.planes == 0 || C == 0) return KDCC_OK;
  p.dbg = tc_debug_bits();
  p.extra = tc_extra(pad);
  if (tc_nt(p.halo + p.extra) == 32) return tc_conv_dispatch_ks<32>(in, p, st);
  return tc_conv_dispatch_ks<16>(in, p, st);
}

}  // namespace kdcc
