// Depthwise k x k convolution on the tensor cores, whole-plane / column-phase variant (bf16, NCHW planes,
// H, W <= 128, same-size convolution, pad % dil == 0).
//
// dw_tc.cu multiplies the 128-row image window by a banded Toeplitz matrix whose band, for a dilated tap set,
// is mostly zeros: with d = 5 only every fifth input column of a 72-column reduction slice meets a tap.  Here the
// columns are first regrouped by their residue b = j mod d ("phase").  Inside one phase the dilated row filter is
// a DENSE k-tap filter over q = j div d, so per phase b and tap row u
//         out_b[i][q] += sum_{q'} X_b[i + u*d - p][q'] * T_u[q'][q],      T_u[q'][q] = w[u][q' - q + p/d]
// is one 128 x 32 x 32 product (two K=16 tcgen05.mma): 2*d*k = 90 MMAs per plane instead of 180, and every
// plane is read from shared memory 9 instead of ~11 times.  tools/mma_probe.cu: these SS MMAs cost 43 + N/2 = 59
// clocks each whatever the layout, so the plane costs ~5.3 kclk -- the kernel is tensor-issue bound, not HBM bound.
//  * TMA lands the bare plane (no halo) as two 128B-swizzled 64-column boxes.
//  * Four warps regroup it into the phase-major operand X_b: [phase][16-byte K chunk][row][8 phase-columns], an
//    un-swizzled K-major layout whose rows are 16 bytes apart, so the tap-row shift u*d is a +16*u*d byte bump of the
//    descriptor start address.  The pad rows above / below the plane are zeros written once; pad columns do not
//    exist at all (T_u simply has no entry for them).  X_b is double buffered.
//  * The same warps rebuild the k Toeplitz tiles (32 x 32 bf16 each) once per channel.
//  * D = d accumulators of 128 x 32 fp32 in TMEM, double buffered; four epilogue warps re-interleave the phases in
//    registers (thread = output row) and store bf16 rows.
// The input-gradient form is the same kernel over dy with mirrored taps.
//
// Planes of 129 .. 256 columns (Gated-SCNN sites on a 1024 x 2048 input: 128 x 256) run as TWO column halves, each a
// "virtual channel" with its own landing window and Toeplitz offset (9x9, dilation 5 only): the left half produces
// columns [0, 120) from input columns [0, 160), the right half columns [120, W) from input columns [100, 260) (landed from
// column 96: TMA wants a 16-byte aligned origin, the regrouping starts 4 columns in) -- both
// windows are 32 phase-columns wide, so a half costs exactly what a 128-column plane costs (90 MMAs) instead of the
// 180 of the tiled kernel (dw_tc.cu).  Split points are multiples of 5 (phases line up) and of 8 (16-byte store rows).
// Reference semantics: models/students/transform_blocks/depthwise_separable_conv.py:7-8,12 (+ autograd).
#include "dw_kernels.cuh"
#include "dw_tc_common.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int C2_THREADS = 320;        // warp 0 TMA, warp 1 MMA, warps 2-5 regroup + Toeplitz, warps 6-9 epilogue
constexpr int C2_STG = 2 * 128 * 128;  // one landed plane: two boxes of 128 rows x 128 bytes
constexpr int C2_TZ_CHUNK = 512;       // one Toeplitz K chunk: [32 output columns][16 bytes]
constexpr int C2_MAXROWS = 128 + 48;   // operand rows: plane + halo

struct C2Params {
  int N, C, H, W, k, dil, pad, flip;
  int rows_p;     // 128 + dil*(k-1): rows of the phase-major operand
  int ks;         // K slices of 16 phase-columns per N-tile
  int qoff;       // pad / dil
  int nt;         // N-tiles (32 output phase-columns) per phase: 1 when a phase is at most 32 columns wide
  int zpad;       // nt > 1: always-zero K chunks in front of chunk 0 (the first tile's window starts at 8*floor(-qoff/8))
  int chunks_p;   // K chunk slots per phase of the operand
  int planes, splits;
  long pairs;
  int halves;     // 1; 2 = planes wider than 128 columns as two column halves (virtual channel = channel * halves + half)
  int VC;         // C * halves
  int in_x0[2], in_shift[2], out_x0[2], half_qoff[2], out_groups[2];  // per half: landing window start (a multiple of 8 columns:
                  // TMA wants a 16-byte aligned origin) and whether the half's phase grid starts 4 columns into it, first output column, pad / dil seen
                  // by its Toeplitz tiles, store tiles (groups of 8 * D columns)
  int nbox;       // 64-column landing boxes per (half) plane
  int nstg;       // landing stages: 2; 1 for the wide planes (their three boxes per stage would not fit twice)
  int in_chunks;  // 16-byte chunks of a landed row the regrouping visits
  const float *w, *bias;
  __nv_bfloat16 *out;
  int dbg;  // KDCC_TC_DEBUG (timing experiments only): 1 skip Toeplitz rebuild, 2 skip MMAs, 4 skip stores, 8 skip regrouping
};

// NT / KS: N-tiles per phase and K slices per N-tile known at compile time (0 = read them from the parameters): the
// single issuing thread then runs a straight line of MMAs, one integer add per operand each.
template <int D, int NT, int KS>
__global__ void __launch_bounds__(C2_THREADS, 1)
dw_tc_conv2_kernel(const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out, const C2Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  const uint32_t lbo = (uint32_t)p.rows_p * 16u;       // bytes between K chunks of the operand
  const uint32_t xp_bytes = (uint32_t)(D * p.chunks_p) * lbo;  // one operand buffer
  const uint32_t stg_bytes = (uint32_t)p.nbox * (C2_STG / 2);     // one landing stage: nbox boxes of 128 rows x 128 bytes
  const uint32_t xp_off = (uint32_t)p.nstg * stg_bytes;
  const uint32_t tz_off = xp_off + 2 * xp_bytes;
  const uint32_t tz_u = (uint32_t)(2 * p.ks) * C2_TZ_CHUNK;  // one tap row's Toeplitz tile: [2*ks K chunks][32][16 B]
  const uint32_t tz_bytes = (uint32_t)p.k * tz_u;
  constexpr int G = D == 1 ? 4 : (D == 2 ? 2 : 1);      // column groups per store tile
  constexpr uint32_t OB = 32 * 16 * D * G;             // one epilogue staging tile: 32 rows x 8*D*G bf16 columns
  const uint32_t ob_off = (tz_off + 2 * tz_bytes + 127u) & ~127u;
  const uint32_t bar_off = ob_off + 4 * 2 * OB;
  const uint32_t bar_base = smem_base + bar_off;
  auto stg_full = [&](int s) { return bar_base + 8u * s; };
  auto stg_empty = [&](int s) { return bar_base + 8u * (2 + s); };
  auto xp_full = [&](int s) { return bar_base + 8u * (4 + s); };
  auto xp_empty = [&](int s) { return bar_base + 8u * (6 + s); };
  auto b_full = [&](int s) { return bar_base + 8u * (8 + s); };
  auto t_full = [&](int s) { return bar_base + 8u * (10 + s); };
  auto t_empty = [&](int s) { return bar_base + 8u * (12 + s); };
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + bar_off + 128);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // operand buffers and Toeplitz tiles start as zeros: pad rows, unused phase-columns and everything off the band
  // are never written again
  for (uint32_t i = threadIdx.x; i < (ob_off - xp_off) / 16; i += C2_THREADS)
    reinterpret_cast<uint4 *>(smem_gen + xp_off)[i] = make_uint4(0, 0, 0, 0);
  ptx::fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(stg_full(s), 1);
      ptx::mbar_init(stg_empty(s), 4);
      ptx::mbar_init(xp_full(s), 4);
      ptx::mbar_init(xp_empty(s), 1);
      ptx::mbar_init(b_full(s), 4);
      ptx::mbar_init(t_full(s), 1);
      ptx::mbar_init(t_empty(s), 4);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_in);
    ptx::prefetch_tensormap(&tm_out);
  }
  if (warp == 1) ptx::tmem_alloc<512>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();  // everything above overlapped the previous kernel's tail; global memory from here on

  if (warp == 0) {
    if (ptx::elect_one()) {
      // ===== TMA producer: one bare (half) plane per item =====
      int it = 0;
      for (PlaneWalk w(p.pairs, p.planes, p.splits, p.VC); w.valid(); w.next(), ++it) {
        const int sl = it % p.nstg;
        const int vc = w.channel(), c = vc / p.halves, h = vc % p.halves;
        ptx::mbar_wait(stg_empty(sl), ((it / p.nstg) & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(stg_full(sl), stg_bytes);
        for (int b = 0; b < p.nbox; ++b)   // columns past the plane are zero-filled by the hardware
          ptx::tma_load_4d(smem_base + sl * stg_bytes + b * (C2_STG / 2), &tm_in, stg_full(sl), p.in_x0[h] + 64 * b, 0, c, w.pl);
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      // ===== MMA issuer: D_b (128 rows x 32 phase-columns) += X_b[u*d ...] (128 x 16) * T_u (16 x 32) =====
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((32u >> 3) << 17) | ((128u >> 4) << 24);
      constexpr uint32_t hi = (128u >> 4) | (1u << 14);  // 8-row groups 128 B apart, descriptor version 1, no swizzle
      const uint32_t a_lbo = (lbo >> 4) << 16;
      constexpr uint32_t b_lbo = (512u >> 4) << 16;      // Toeplitz K chunks: 32 columns x 16 B apart
      const uint32_t chunk16 = lbo >> 4;  // one K chunk of the operand, in descriptor units
      uint32_t a_phase[D];                // operand offset of every phase: the issue loop below only adds
#pragma unroll
      for (int b = 0; b < D; ++b) a_phase[b] = (uint32_t)(b * p.chunks_p) * chunk16;
      const uint32_t a_tile = 4u * chunk16, a_slice = 2u * chunk16;
      int it = 0, unit = -1;
      for (PlaneWalk w(p.pairs, p.planes, p.splits, p.VC); w.valid(); w.next(), ++it) {
        const int s = it & 1;
        const uint32_t ph = (it >> 1) & 1;
        if (w.first_of_unit()) {
          ++unit;
          ptx::mbar_wait(b_full(unit & 1), (unit >> 1) & 1);
        }
        ptx::mbar_wait(xp_full(s), ph);
        ptx::mbar_wait(t_empty(s), ph ^ 1);
        ptx::tcgen05_fence_after();
        const uint32_t a_base = (((smem_base + xp_off + s * xp_bytes) & 0x3FFFF) >> 4) | a_lbo;
        const uint32_t b_base = (((smem_base + tz_off + (unit & 1) * tz_bytes) & 0x3FFFF) >> 4) | b_lbo;
        const uint32_t d0 = tmem_base + (uint32_t)s * 256u;
        if (!KDCC_DBG(p, 2)) {
#pragma unroll 1
          for (int u = 0; u < p.k; ++u) {
            const uint32_t a_u = a_base + (uint32_t)(u * p.dil);       // tap row u: u*d rows of 16 bytes further down
            const uint32_t b_u = b_base + (uint32_t)u * (tz_u >> 4);
            const int nt = NT ? NT : p.nt, ks = KS ? KS : p.ks;
#pragma unroll
            for (int b = 0; b < D; ++b) {
              // N-tile t of phase b: its K window starts at chunk slot 4t (the zero chunks in front make that uniform)
              uint32_t a_t = a_u + a_phase[b];
              uint32_t d_t = d0 + (uint32_t)(b * nt) * 32u;
#pragma unroll
              for (int t = 0; t < nt; ++t, a_t += a_tile, d_t += 32u) {
                ptx::umma_f16_ss(d_t, a_t, hi, b_u, hi, idesc, u ? 1u : 0u);
                uint32_t a_s = a_t + a_slice, b_s = b_u + (1024u >> 4);
#pragma unroll
                for (int ss = 1; ss < ks; ++ss, a_s += a_slice, b_s += (1024u >> 4))
                  ptx::umma_f16_ss(d_t, a_s, hi, b_s, hi, idesc, 1u);
              }
            }
          }
        }
        ptx::umma_commit(xp_empty(s));
        ptx::umma_commit(t_full(s));
      }
    }
  } else if (warp <= 5) {
    // ===== regrouping (128 threads, thread = plane row) + Toeplitz tiles =====
    const int r = threadIdx.x - 64;
    const int nchunks = p.in_chunks;  // 16-byte chunks of a landed row
    auto build_t = [&](int vc, int s) {
      const float *wc = p.w + (long)(vc / p.halves) * p.k * p.k;
      const int qoff = p.half_qoff[vc % p.halves];
      uint8_t *ts = smem_gen + tz_off + (size_t)s * tz_bytes;
      // (tap row u, output phase-column q): tap v sits at reduction index q' = q - p/d + v
      for (int idx = r; idx < (KDCC_DBG(p, 1) ? 0 : p.k * 32); idx += 128) {
        const int u = idx >> 5, q = idx & 31;
        const float *wr = wc + (p.flip ? (p.k - 1 - u) * p.k : u * p.k);
        float wv[9];
#pragma unroll
        for (int v = 0; v < 9; ++v) wv[v] = v < p.k ? __ldg(wr + (p.flip ? p.k - 1 - v : v)) : 0.f;
#pragma unroll
        for (int v = 0; v < 9; ++v) {
          const int qp = q - qoff + v + 8 * p.zpad;  // reduction index inside the N-tile's K window
          if (v < p.k && qp >= 0 && qp < 16 * p.ks)
            *reinterpret_cast<__nv_bfloat16 *>(ts + u * tz_u + (qp >> 3) * C2_TZ_CHUNK + q * 16 + (qp & 7) * 2) = __float2bfloat16_rn(wv[v]);
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(b_full(s));
    };
    int it = 0, unit = -1, built = 0;
    PlaneWalk ahead(p.pairs, p.planes, p.splits, p.VC);  // first plane of the next unit whose tiles are not built yet
    for (PlaneWalk w(p.pairs, p.planes, p.splits, p.VC); w.valid(); w.next(), ++it) {
      const int s = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      const int sl = it % p.nstg;
      // the MMAs of plane it-2 are done: operand buffer s is free
      ptx::mbar_wait(xp_empty(s), ph ^ 1);
      if (w.first_of_unit()) {
        ++unit;
        if (built == unit) {  // not built ahead (first unit, or the previous unit had a single plane)
          build_t(w.channel(), unit & 1);
          ++built;
          ahead.next_unit();
        }
      } else if (built == unit + 1 && ahead.valid()) {
        // second or later plane of the unit: plane it-2 was the last one that read the other Toeplitz buffer, so
        // the next unit's tiles are built here, off the critical path
        build_t(ahead.channel(), (unit + 1) & 1);
        ++built;
        ahead.next_unit();
      }
      ptx::mbar_wait(stg_full(sl), (it / p.nstg) & 1);
      const uint8_t *stg = smem_gen + sl * stg_bytes;
      const int shift = p.in_shift[w.channel() % p.halves];
      uint8_t *xp = smem_gen + xp_off + (size_t)s * xp_bytes + (size_t)(r + p.pad) * 16;
      if (!KDCC_DBG(p, 8)) {
#pragma unroll 1
        for (int g = 0; g * D < nchunks; ++g) {
          // 8*D consecutive columns of row r -> 8 phase-columns (one 16-byte chunk) of each of the D phases
          uint32_t in[4 * D];
#pragma unroll
          for (int j = 0; j < D; ++j) {
            const int c = g * D + j;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (c < nchunks) {
              if (!shift) {
                v = *reinterpret_cast<const uint4 *>(stg + (c >> 3) * (C2_STG / 2) + r * 128 + (((c & 7) ^ (r & 7)) << 4));
              } else {  // the 8 columns start 4 columns (8 bytes) into landed chunk c: upper half of c, lower half of c + 1
                const int c1 = c + 1;
                const uint2 lo = *reinterpret_cast<const uint2 *>(stg + (c >> 3) * (C2_STG / 2) + r * 128 + (((c & 7) ^ (r & 7)) << 4) + 8);
                const uint2 hi = *reinterpret_cast<const uint2 *>(stg + (c1 >> 3) * (C2_STG / 2) + r * 128 + (((c1 & 7) ^ (r & 7)) << 4));
                v = make_uint4(lo.x, lo.y, hi.x, hi.y);
              }
            }
            in[4 * j] = v.x; in[4 * j + 1] = v.y; in[4 * j + 2] = v.z; in[4 * j + 3] = v.w;
          }
#pragma unroll
          for (int b = 0; b < D; ++b) {
            uint32_t o[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              const int x0 = D * (2 * m) + b, x1 = D * (2 * m + 1) + b;  // elements of the 8*D-column group
              const uint32_t sel = ((x0 & 1) ? 0x32u : 0x10u) | ((x1 & 1) ? 0x7600u : 0x5400u);
              o[m] = __byte_perm(in[x0 >> 1], in[x1 >> 1], sel);
            }
            *reinterpret_cast<uint4 *>(xp + (size_t)(b * p.chunks_p + p.zpad + g) * lbo) = make_uint4(o[0], o[1], o[2], o[3]);
          }
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(xp_full(s));
        ptx::mbar_arrive(stg_empty(sl));
      }
    }
  } else {
    // ===== epilogue (128 threads, thread = output row = TMEM lane): re-interleave the phases in registers, stage
    // 32 rows x 8*D columns per warp in shared memory and let TMA store them (coalesced, clips ragged edges) =====
    const int quad = warp & 3;
    const uint32_t ob = ob_off + (uint32_t)(warp - 6) * 2 * OB;
    int it = 0, gi = 0;
    for (PlaneWalk w(p.pairs, p.planes, p.splits, p.VC); w.valid(); w.next(), ++it) {
      const int s = it & 1;
      ptx::mbar_wait(t_full(s), (it >> 1) & 1);
      ptx::tcgen05_fence_after();
      __syncwarp();  // lanes leave the polling loop one by one; the TMEM accesses below are .sync.aligned
      const int c = w.channel() / p.halves, h = w.channel() % p.halves;
      const int ngroups = p.out_groups[h], x0 = p.out_x0[h];
      const float bias = p.bias ? __ldg(p.bias + c) : 0.f;
      const uint32_t t_row = tmem_base + (uint32_t)s * 256u + ((uint32_t)(quad * 32) << 16);
      // a store tile = G groups of 8*D output columns (G chosen so that a tile row is 64-128 bytes)
#pragma unroll 1
      for (int g0 = 0; g0 < ngroups; g0 += G, ++gi) {
        if (gi >= 2) {  // the store that read this staging tile two tiles ago has finished reading it
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          __syncwarp();
        }
        const uint32_t tile = ob + (uint32_t)(gi & 1) * OB;
#pragma unroll
        for (int gg = 0; gg < G; ++gg) {
          const int g = g0 + gg;
          if (g >= ngroups) break;
          uint32_t v[D][8];
#pragma unroll
          for (int b = 0; b < D; ++b) ptx::tmem_ld_32x32b_x8(t_row + (uint32_t)((b * p.nt + (g >> 2)) * 32 + (g & 3) * 8), v[b]);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < D; ++j) {
            uint32_t o[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              const int x0 = 8 * j + 2 * m, x1 = x0 + 1;  // output columns of the group: column x = phase x % D, index x / D
              o[m] = pack_bf16x2(__uint_as_float(v[x0 % D][x0 / D]) + bias, __uint_as_float(v[x1 % D][x1 / D]) + bias);
            }
            *reinterpret_cast<uint4 *>(smem_gen + tile + lane * (16 * D * G) + 16 * (gg * D + j)) = make_uint4(o[0], o[1], o[2], o[3]);
          }
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && !KDCC_DBG(p, 4)) {
          ptx::tma_store_4d(&tm_out, smem_base + tile, x0 + 8 * D * g0, 32 * quad, c, w.pl);
          ptx::tma_store_commit();
        }
      }
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(t_empty(s));
    }
    if (lane == 0) ptx::tma_store_wait_all();
  }

  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// planes of 129 .. 256 columns as two column halves: derived for the 9 x 9, dilation 5, pad 20 geometry (split at column 120)
static bool conv2_wide(int Hi, int Wi, int Ho, int Wo, int k, int dil, int pad) {
  return Hi == Ho && Wi == Wo && Hi <= 128 && Wi > 128 && Wi <= 256 && Wi % 8 == 0 && k == 9 && dil == 5 && pad == 20;
}

bool dw_tc_conv2_supported(int Hi, int Wi, int Ho, int Wo, int k, int dil, int pad) {
  if (conv2_wide(Hi, Wi, Ho, Wo, k, dil, pad)) return true;
  const int halo = dil * (k - 1);
  if (Hi != Ho || Wi != Wo || Hi > 128 || Wi > 128 || Wi % 8 != 0) return false;
  if (k % 2 == 0 || k > 9 || halo > 48 || 2 * pad != halo || pad % dil != 0) return false;
  if (dil != 1 && dil != 2 && dil != 5) return false;   // instantiated phase counts
  const int nt = ((Wi + dil - 1) / dil + 31) / 32;       // N-tiles per phase: the d accumulators of a plane must fit 256 TMEM columns
  if (dil * nt * 32 > 256) return false;
  if (nt > 1) {                                          // operand with zero chunks around every phase: must fit shared memory twice
    const int qoff = pad / dil, zpad = (qoff + 7) / 8;
    const int ks = ((31 + k - 1 - qoff + 8 * zpad) / 8 + 2) / 2;
    const int chunks_p = 4 * (nt - 1) + 2 * ks;
    if (2 * C2_STG + 2 * dil * chunks_p * (128 + halo) * 16 + 2 * k * 2 * ks * C2_TZ_CHUNK + 8 * 32 * 16 * dil * (dil == 1 ? 4 : (dil == 2 ? 2 : 1)) + 2048 > 227 * 1024) return false;
  }
  return true;
}

template <int D, int NT, int KS>
static int conv2_launch(const void *in, C2Params p, cudaStream_t st) {
  CUtensorMap tm;
  const uint64_t dims[4] = {(uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.C, (uint64_t)p.N};
  const uint64_t strides[3] = {(uint64_t)p.W * 2, (uint64_t)p.H * p.W * 2, (uint64_t)p.C * p.H * p.W * 2};
  const uint32_t box[4] = {64, 128, 1, 1};
  int rc = make_tmap_bf16(&tm, in, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  CUtensorMap tm_out;
  const uint32_t obox[4] = {8 * D * (D == 1 ? 4 : (D == 2 ? 2 : 1)), 32, 1, 1};
  rc = make_tmap_bf16(&tm_out, p.out, 4, dims, strides, obox, nullptr, CU_TENSOR_MAP_SWIZZLE_NONE);
  if (rc) return rc;
  const int smem = p.nstg * p.nbox * (C2_STG / 2) + 2 * D * p.chunks_p * p.rows_p * 16 + 2 * p.k * 2 * p.ks * C2_TZ_CHUNK + 128 + 8 * 32 * 16 * D * (D == 1 ? 4 : (D == 2 ? 2 : 1)) + 256 + 1024;
  if (smem > 227 * 1024 || D * p.nt * 32 > 256) return KDCC_ESHAPE;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tc_conv2_kernel<D, NT, KS>, smem, attr_cache)) return e;
  const int grid = (int)min(p.pairs, (long)kNumSMs);
  launch_pdl(dw_tc_conv2_kernel<D, NT, KS>, dim3(grid), dim3(C2_THREADS), (size_t)smem, st, tm, tm_out, p);
  return launch_status();
}

int dw_tc_conv2(const void *in, const float *w, const float *bias, void *out, int N, int C, int H, int W, int k, int dil,
                int pad, int flip, cudaStream_t st) {
  C2Params p{};
  p.N = N; p.C = C; p.H = H; p.W = W; p.k = k; p.dil = dil; p.pad = pad; p.flip = flip;
  p.rows_p = 128 + dil * (k - 1);
  p.qoff = pad / dil;
  const bool wide = W > 128;
  const int Q = ((wide ? 160 : W) + dil - 1) / dil;  // columns of one phase (of one half's window)
  p.nt = (Q + 31) / 32;
  if (p.nt == 1) {  // the whole phase is one N-tile: its K window is the phase itself (pad columns do not exist)
    p.zpad = 0;
    p.ks = (Q + 15) / 16;
    p.chunks_p = 4;
  } else {          // N-tile t reduces over q' in [32t - qoff, 32t + 31 + k - 1 - qoff], walked from the aligned chunk below
    p.zpad = (p.qoff + 7) / 8;
    p.ks = ((31 + k - 1 - p.qoff + 8 * p.zpad) / 8 + 1 + 1) / 2;
    p.chunks_p = 4 * (p.nt - 1) + 2 * p.ks;
  }
  p.halves = wide ? 2 : 1;
  p.VC = C * p.halves;
  if (!wide) {
    p.in_x0[0] = 0; p.in_shift[0] = 0; p.out_x0[0] = 0; p.half_qoff[0] = p.qoff;
    p.out_groups[0] = ((W >> 3) + dil - 1) / dil;
    p.nbox = 2; p.nstg = 2; p.in_chunks = W >> 3;
  } else {
    // left half: outputs q in [0, 24) of every phase = columns [0, 120), inputs q' in [0, 32) = columns [0, 160);
    // right half: outputs q in [24, 52) = columns [120, W), inputs q' in [20, 52) = columns [100, 260): the window starts
    // qoff = 4 phase-columns before its first output, so its Toeplitz tiles see pad / dil = 0.  TMA needs a 16-byte aligned
    // column origin: the right window is landed from column 96 and regrouped from 4 columns in.
    p.in_x0[0] = 0;  p.in_shift[0] = 0; p.out_x0[0] = 0;   p.half_qoff[0] = p.qoff; p.out_groups[0] = 3;
    p.in_x0[1] = 96; p.in_shift[1] = 1; p.out_x0[1] = 120; p.half_qoff[1] = 0;      p.out_groups[1] = ((W - 120) + 39) / 40;
    p.nbox = 3; p.nstg = 1; p.in_chunks = 20;
  }
  p.planes = N;
  p.splits = tc_unit_splits(p.VC, N);
  p.pairs = (long)p.VC * p.splits;
  p.w = w; p.bias = bias;
  p.out = static_cast<__nv_bfloat16 *>(out);
  if (N == 0 || C == 0) return KDCC_OK;
  p.dbg = tc_debug_bits();
  // compile-time MMA schedules for the shapes that matter; every other supported shape takes the run-time loops
  if (dil == 5 && p.nt == 1 && p.ks == 2) return conv2_launch<5, 1, 2>(in, p, st);  // Cityscapes: 9x9, dilation 5, 128 columns
  if (dil == 1 && p.nt == 4 && p.ks == 3) return conv2_launch<1, 4, 3>(in, p, st);  // 3x3 on a 128-column plane
  switch (dil) {
    case 1: return conv2_launch<1, 0, 0>(in, p, st);
    case 2: return conv2_launch<2, 0, 0>(in, p, st);
    case 5: return conv2_launch<5, 0, 0>(in, p, st);
    default: return KDCC_ESHAPE;
  }
}

}  // namespace kdcc
