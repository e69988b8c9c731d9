// Pointwise (1x1) convolution as a dense bf16 GEMM on the sm_100a tensor cores:
// TMA (128B-swizzled tiles) -> shared memory -> tcgen05.mma with the fp32 accumulator in TMEM ->
// tcgen05.ld epilogue -> TMA store of swizzled 32 x 64 tiles (plain bf16 output) or direct 16-byte stores
// (fp32 split partials; BN scale/shift + ReLU + residual, dual output).  256-wide tiles run as CTA pairs
// (cta_group::2: each CTA holds half of B, see GemmCfg).
//
// Reference semantics: models/students/transform_blocks/depthwise_separable_conv.py:9,13 (nn.Conv2d 1x1)
// and its autograd backward (dX = dY.W, dW = dY^T.X).
//
// One kernel template covers the three GEMMs of the block:
//     D[i][j] = sum_r A(i,r) * B(j,r)
//   forward   i = pixel m, j = out channel, r = in channel : A = X  (r-contiguous, "K-major"),
//                                                            B = W  [Co][Ci]      (K-major)
//   dX        i = pixel m, j = in channel,  r = out channel: A = dY (K-major),
//                                                            B = W  [Co][Ci] read as (j contiguous, "MN-major")
//   dW        i = out channel, j = in channel, r = pixel m : A = dY (MN-major), B = X (MN-major); the pixel
//             reduction is split over CTAs into fp32 partials (deterministic second-stage sum).
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer (one lane),
// warps 2..5 = epilogue (one TMEM lane quadrant each).  Persistent CTAs walk work items round-robin;
// the accumulator is double-buffered in TMEM so the epilogue of item n overlaps the MMAs of item n+1.
#include "kdcc_common.cuh"
#include "pw_kernels.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int GEMM_BI = 128;   // UMMA M
constexpr int GEMM_BR = 64;    // reduction elements per stage = one 128-byte swizzle atom of bf16
#ifndef KDCC_GEMM_EPI_WARPS
#define KDCC_GEMM_EPI_WARPS 4
#endif
// Epilogue warps: 4 = one per TMEM lane quadrant; 8 = two per quadrant, each draining every other 64-column chunk.
// Measured equal (same box, whole step: pw fwd 0.761 vs 0.758 ms, dX 0.855 vs 0.843): the short-K GEMMs whose tensor
// pipe is only 50 % active (4096<-256 dX: 128 FLOP per L2 byte with 256-deep tiles) wait on operand traffic, not on the
// drain, so the default stays 4 (tools/build_variant.sh builds the other one).
constexpr int GEMM_EPI_WARPS = KDCC_GEMM_EPI_WARPS;
constexpr int GEMM_EPI_HALVES = GEMM_EPI_WARPS / 4;
#ifndef KDCC_GEMM_EPI_TILES
#define KDCC_GEMM_EPI_TILES (KDCC_GEMM_EPI_WARPS == 4 ? 2 : 1)
#endif
#ifndef KDCC_GEMM_PAIR_STAGES
#define KDCC_GEMM_PAIR_STAGES 6
#endif
constexpr int GEMM_EPI_TILES = KDCC_GEMM_EPI_TILES;   // staging tiles (4 KB) per epilogue warp: TMA stores in flight per warp
constexpr int GEMM_THREADS = 64 + 32 * GEMM_EPI_WARPS;

struct GemmParams {
  int I, J, R;          // logical extents (R per batch entry)
  int batch;            // independent GEMMs (NCHW images); 1 for the NHWC forms
  int a_batched, b_batched;  // operand has a batch dimension (else it is shared, e.g. the weights)
  int r_spans_batch;    // dW on NCHW: the reduction runs over (batch, r) and the output is not batched
  long out_batch_stride;     // elements between batch entries of the output
  int affine_rows;      // scale/shift indexed by output row i (NCHW: channel = row) instead of column j
  int tiles_i, tiles_j; // output tiling
  int splits;           // CTAs sharing one output tile along r (dW only)
  int rblocks;          // reduction blocks of 64: ceil(R / 64) (* batch when r_spans_batch)
  int rblocks_per_batch;
  // epilogue
  __nv_bfloat16 *out_raw, *out_act;  // [I][J] bf16, either may be null
  const float *scale, *shift;        // per j, may be null
  const __nv_bfloat16 *residual;     // [I][J] like out_act, added before the activation (the block's shortcut); may be null
  int relu;
  float *out_f32;                    // [splits][I][J] fp32 partials (dW) -- exclusive with the bf16 outputs
  int tma_out;                       // out_raw only: the epilogue stages 32 x 64 tiles in smem and TMA stores them
};

// PAIR: two CTAs of a cluster (one TPC) work on one 256 x BJ tile with cta_group::2 MMAs: each loads its own 128 rows of
// A and HALF of B, the tensor core reads the other half from the partner's shared memory.  Per CTA and reduction block
// that is 32 KB instead of 48 KB from L2 -- the 1-CTA kernel is L2-bandwidth bound (9.7 TB/s of L2 traffic per step).
template <int BJ, bool PAIR>
struct GemmCfg {
  static constexpr int A_BYTES = GEMM_BI * GEMM_BR * 2;  // 16 KB
  static constexpr int BJ_CTA = PAIR ? BJ / 2 : BJ;       // B rows held by one CTA
  static constexpr int B_BYTES = BJ_CTA * GEMM_BR * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = PAIR ? KDCC_GEMM_PAIR_STAGES : (BJ == 256 ? 4 : (BJ == 128 ? 6 : 8));
  static constexpr int TMEM_COLS = 2 * BJ;  // double-buffered accumulator (power of two >= 32)
  static constexpr int OUT_OFF = STAGES * STAGE_BYTES;   // epilogue staging: tiles of 32 rows x 128 bytes per warp
  static constexpr int BAR_OFF = OUT_OFF + GEMM_EPI_WARPS * GEMM_EPI_TILES * 4096;
  static constexpr int SMEM = BAR_OFF + 256 + 1024;  // barriers + slack for manual 1024-byte alignment
};

// UMMA shared-memory descriptors (SWIZZLE_128B, bf16), cf. the canonical layouts of the PTX ISA:
//  K-major : rows of 128 bytes (64 reduction elements); 8-row groups 1024 bytes apart (SBO).
//  MN-major: rows of 128 bytes (64 i/j elements) indexed by r; 8-r groups 1024 bytes apart (SBO),
//            64-element i/j groups `lbo_bytes` apart (LBO).
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

template <int BJ, bool A_MN, bool B_MN, int BI = GEMM_BI>
__device__ __forceinline__ constexpr uint32_t umma_idesc() {
  // c_format F32 (bits 4-5 = 1), a/b format BF16 (bits 7-9 / 10-12 = 1), majors (bits 15, 16),
  // N >> 3 (bits 17-22), M >> 4 (bits 24-28)
  return (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
         ((uint32_t)(BJ >> 3) << 17) | ((uint32_t)(BI >> 4) << 24);
}

template <int BJ, bool A_MN, bool B_MN, bool PAIR>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
pw_gemm_sm100_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                     const __grid_constant__ CUtensorMap tm_out, const GemmParams p) {
  using Cfg = GemmCfg<BJ, PAIR>;
  const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0u;  // 0 = leader: issues the MMAs, owns the full / tempty barriers
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + Cfg::BAR_OFF;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + Cfg::BAR_OFF + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (PAIR) ptx::cluster_sync();  // both CTAs are resident before the pair-wide TMEM allocation
  if (threadIdx.x == 0) {
    // pair: the leader's full barrier collects one arrival per CTA and the bytes of both; its tempty barrier the
    // epilogue warps of both CTAs; empty / tfull are signalled in both CTAs by multicast commits
    for (int s = 0; s < STAGES; ++s) { ptx::mbar_init(full_bar(s), PAIR ? 2 : 1); ptx::mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), (PAIR ? 2 : 1) * GEMM_EPI_WARPS); }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_a);
    ptx::prefetch_tensormap(&tm_b);
    if (p.tma_out) ptx::prefetch_tensormap(&tm_out);
  }
  if (warp == 1) {
    if (PAIR) ptx::tmem_alloc_pair<Cfg::TMEM_COLS>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
    else ptx::tmem_alloc<Cfg::TMEM_COLS>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  }
  ptx::tcgen05_fence_before();
  if (PAIR) ptx::cluster_sync(); else __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();  // the prologue overlapped the previous kernel's tail; global memory from here on

  const int out_batches = p.r_spans_batch ? 1 : p.batch;
  const int tiles_iw = PAIR ? p.tiles_i / 2 : p.tiles_i;   // work items along i: tiles, or pairs of tiles
  const long items = (long)tiles_iw * p.tiles_j * p.splits * out_batches;
  const int rb_per_split = (p.rblocks + p.splits - 1) / p.splits;
  const long item0 = PAIR ? (long)(blockIdx.x >> 1) : (long)blockIdx.x;
  const long item_step = PAIR ? (long)(gridDim.x >> 1) : (long)gridDim.x;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    int s = 0; uint32_t ph = 0;
    for (long item = item0; item < items; item += item_step) {
      const int split = (int)(item % p.splits);
      long tile = item / p.splits;
      // i fastest: CTAs running side by side share the (large) B tile and differ in the (small, L2-resident) A tile
      const int ti = (int)(tile % tiles_iw) * (PAIR ? 2 : 1) + (int)rank; tile /= tiles_iw;
      const int tj = (int)(tile % p.tiles_j);
      const int bo = (int)(tile / p.tiles_j);  // output batch entry
      const int rb0 = split * rb_per_split, rb1 = min(p.rblocks, rb0 + rb_per_split);
      for (int rb = rb0; rb < rb1; ++rb) {
        // reduction block -> (batch entry, block inside the entry)
        const int bz = p.r_spans_batch ? rb / p.rblocks_per_batch : bo;
        const int rl = p.r_spans_batch ? rb % p.rblocks_per_batch : rb;
        const int za = p.a_batched ? bz : 0, zb = p.b_batched ? bz : 0;
        ptx::mbar_wait(empty_bar(s), ph ^ 1);
        const uint32_t a_dst = smem_base + s * Cfg::STAGE_BYTES;
        const uint32_t b_dst = a_dst + Cfg::A_BYTES;
        auto load = [&](uint32_t dst, const CUtensorMap *m, int c0, int c1, int c2) {
          if (PAIR) ptx::tma_load_3d_pair(dst, m, full_bar(s), c0, c1, c2);  // bytes are credited to the leader's barrier
          else ptx::tma_load_3d(dst, m, full_bar(s), c0, c1, c2);
        };
        if (!PAIR) ptx::mbar_arrive_expect_tx(full_bar(s), Cfg::STAGE_BYTES);
        else if (rank == 0) ptx::mbar_arrive_expect_tx(full_bar(s), 2 * Cfg::STAGE_BYTES);
        else ptx::mbar_arrive_cluster(full_bar(s), 0);
        const int jb = tj * BJ + (int)rank * Cfg::BJ_CTA;  // this CTA's part of the B tile
        if (!A_MN) {
          load(a_dst, &tm_a, rl * GEMM_BR, ti * GEMM_BI, za);
        } else {
#pragma unroll
          for (int b = 0; b < GEMM_BI / 64; ++b) load(a_dst + b * 8192, &tm_a, ti * GEMM_BI + b * 64, rl * GEMM_BR, za);
        }
        if (!B_MN) {
          load(b_dst, &tm_b, rl * GEMM_BR, jb, zb);
        } else {
#pragma unroll
          for (int b = 0; b < Cfg::BJ_CTA / 64; ++b) load(b_dst + b * 8192, &tm_b, jb + b * 64, rl * GEMM_BR, zb);
        }
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1 && lane == 0 && rank == 0) {
    // ===== MMA issuer (pair: the leader CTA issues for both) =====
    constexpr uint32_t idesc = umma_idesc<BJ, A_MN, B_MN, PAIR ? 2 * GEMM_BI : GEMM_BI>();
    int s = 0; uint32_t ph = 0;
    int as = 0; uint32_t aph = 0;
    for (long item = item0; item < items; item += item_step) {
      const int split = (int)(item % p.splits);
      const int rb0 = split * rb_per_split, rb1 = min(p.rblocks, rb0 + rb_per_split);
      ptx::mbar_wait(tempty_bar(as), aph ^ 1);
      ptx::tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * BJ);
      for (int rb = rb0; rb < rb1; ++rb) {
        ptx::mbar_wait(full_bar(s), ph);
        ptx::tcgen05_fence_after();
        const uint32_t a_addr = smem_base + s * Cfg::STAGE_BYTES;
        const uint32_t b_addr = a_addr + Cfg::A_BYTES;
#pragma unroll
        for (int k = 0; k < GEMM_BR / 16; ++k) {
          // K-major: step 16 elements (32 bytes) inside the swizzle atom; MN-major: step 16 r-rows (2 KB)
          const uint64_t da = A_MN ? umma_desc(a_addr + k * 2048, 8192, 1024) : umma_desc(a_addr + k * 32, 16, 1024);
          const uint64_t db = B_MN ? umma_desc(b_addr + k * 2048, 8192, 1024) : umma_desc(b_addr + k * 32, 16, 1024);
          if (PAIR) ptx::umma_f16_pair(d_tmem, da, db, idesc, (rb > rb0 || k > 0) ? 1u : 0u);
          else ptx::umma_f16(d_tmem, da, db, idesc, (rb > rb0 || k > 0) ? 1u : 0u);
        }
        // frees the smem stage (in both CTAs of a pair) once these MMAs have read it
        if (PAIR) ptx::umma_commit_pair(empty_bar(s)); else ptx::umma_commit(empty_bar(s));
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
      if (PAIR) ptx::umma_commit_pair(tfull_bar(as)); else ptx::umma_commit(tfull_bar(as));   // accumulator complete -> epilogue
      if (++as == 2) { as = 0; aph ^= 1; }
    }
  } else if (warp >= 2) {
    // ===== epilogue: TMEM -> registers -> global =====
    const int quad = warp & 3;  // TMEM lanes [32*quad, 32*quad+32) are accessible to this warp
    const int half = (warp - 2) >> 2;  // which of the quadrant's warps: column chunks half, half + HALVES, ...
    int as = 0; uint32_t aph = 0;
    const uint32_t stage_tiles = Cfg::OUT_OFF + (uint32_t)(warp - 2) * GEMM_EPI_TILES * 4096;
    int tn = 0;  // staging tiles written by this warp
    for (long item = item0; item < items; item += item_step) {
      const int split = (int)(item % p.splits);
      long tile = item / p.splits;
      const int ti = (int)(tile % tiles_iw) * (PAIR ? 2 : 1) + (int)rank; tile /= tiles_iw;
      const int tj = (int)(tile % p.tiles_j);
      const long tile_batch = tile / p.tiles_j;
      const long obase = tile_batch * p.out_batch_stride;
      ptx::mbar_wait(tfull_bar(as), aph);
      ptx::tcgen05_fence_after();
      __syncwarp();  // lanes leave the polling loop one by one; the TMEM accesses below are .sync.aligned
      const int row = ti * GEMM_BI + quad * 32 + lane;
      const uint32_t t_row = tmem_base + (uint32_t)(as * BJ) + ((uint32_t)(quad * 32) << 16);
      if (p.tma_out) {
        // bf16 output through shared memory: 32 rows x 64 columns per warp and chunk, 128B-swizzled, stored by TMA
        // (coalesced 128-byte rows; ragged edges are clipped by the tensor map)
#pragma unroll 1
        for (int ch = half; ch < BJ / 64; ch += GEMM_EPI_HALVES) {
          const int col0 = tj * BJ + ch * 64;
          if (col0 >= p.J) break;
          uint32_t v[64];
          ptx::tmem_ld_32x32b_x32(t_row + ch * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
          ptx::tmem_ld_32x32b_x32(t_row + ch * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
          ptx::tmem_ld_wait();
          if (tn >= GEMM_EPI_TILES) {  // the store that last read this staging tile has finished reading it
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(GEMM_EPI_TILES - 1) : "memory");
            __syncwarp();
          }
          const uint32_t tile = stage_tiles + (uint32_t)(tn % GEMM_EPI_TILES) * 4096;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(v[8 * c + 0]), __uint_as_float(v[8 * c + 1]));
            o.y = pack_bf16x2(__uint_as_float(v[8 * c + 2]), __uint_as_float(v[8 * c + 3]));
            o.z = pack_bf16x2(__uint_as_float(v[8 * c + 4]), __uint_as_float(v[8 * c + 5]));
            o.w = pack_bf16x2(__uint_as_float(v[8 * c + 6]), __uint_as_float(v[8 * c + 7]));
            *reinterpret_cast<uint4 *>(smem_gen + tile + lane * 128 + ((c ^ (lane & 7)) << 4)) = o;
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_3d(&tm_out, smem_base + tile, col0, ti * GEMM_BI + quad * 32, (int)(tile_batch));
            ptx::tma_store_commit();
          }
          ++tn;
        }
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) { if (PAIR) ptx::mbar_arrive_cluster(tempty_bar(as), 0); else ptx::mbar_arrive(tempty_bar(as)); }
        if (++as == 2) { as = 0; aph ^= 1; }
        continue;
      }
#pragma unroll 1
      for (int ch = half; ch < BJ / 32; ch += GEMM_EPI_HALVES) {
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(t_row + ch * 32, v);
        ptx::tmem_ld_wait();
        const int col0 = tj * BJ + ch * 32;
        if (row < p.I && col0 < p.J) {
          if (p.out_f32 != nullptr) {
            float *dst = p.out_f32 + ((long)split * p.I + row) * p.J + col0;
#pragma unroll
            for (int q = 0; q < 8; ++q)
              if (col0 + q * 4 < p.J)
                *reinterpret_cast<uint4 *>(dst + q * 4) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          } else {
            if (p.out_raw != nullptr) {
              __nv_bfloat16 *dst = p.out_raw + obase + (long)row * p.J + col0;
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (col0 + q * 8 < p.J) {
                  uint4 o;
                  o.x = pack_bf16x2(__uint_as_float(v[8 * q + 0]), __uint_as_float(v[8 * q + 1]));
                  o.y = pack_bf16x2(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3]));
                  o.z = pack_bf16x2(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5]));
                  o.w = pack_bf16x2(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7]));
                  *reinterpret_cast<uint4 *>(dst + q * 8) = o;
                }
            }
            if (p.out_act != nullptr) {
              __nv_bfloat16 *dst = p.out_act + obase + (long)row * p.J + col0;
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (col0 + q * 8 < p.J) {
                  float f[8], r[8];
                  if (p.residual) {
                    const uint4 rv = __ldg(reinterpret_cast<const uint4 *>(p.residual + obase + (long)row * p.J + col0 + q * 8));
                    r[0] = bf16lo(rv.x); r[1] = bf16hi(rv.x); r[2] = bf16lo(rv.y); r[3] = bf16hi(rv.y);
                    r[4] = bf16lo(rv.z); r[5] = bf16hi(rv.z); r[6] = bf16lo(rv.w); r[7] = bf16hi(rv.w);
                  }
#pragma unroll
                  for (int e = 0; e < 8; ++e) {
                    const int ch = p.affine_rows ? row : col0 + q * 8 + e;
                    float x = __uint_as_float(v[8 * q + e]);
                    if (p.scale) x *= __ldg(p.scale + ch);
                    if (p.shift) x += __ldg(p.shift + ch);
                    if (p.residual) x += r[e];
                    if (p.relu) x = fmaxf(x, 0.f);
                    f[e] = x;
                  }
                  uint4 o;
                  o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
                  o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
                  *reinterpret_cast<uint4 *>(dst + q * 8) = o;
                }
            }
          }
        }
      }
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) { if (PAIR) ptx::mbar_arrive_cluster(tempty_bar(as), 0); else ptx::mbar_arrive(tempty_bar(as)); }
      if (++as == 2) { as = 0; aph ^= 1; }
    }
    if (p.tma_out && lane == 0) ptx::tma_store_wait_all();
  }

  ptx::tcgen05_fence_before();
  if (PAIR) ptx::cluster_sync(); else __syncthreads();  // pair: the partner may still read this CTA's shared memory / signal its barriers
  if (warp == 1) {
    if (PAIR) ptx::tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base); else ptx::tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// out[i] = sum_s part[s][i]   (fixed order); four elements per thread, as float4 when count % 4 == 0 keeps them aligned
__global__ void reduce_splits_kernel(const float *__restrict__ part, float *__restrict__ out, int splits, long count) {
  pdl_prologue_done();
  const long i4 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= count) return;
  if (count % 4 != 0) {  // the CUDA-core fp32 / odd-channel weight gradient: Nc * K of any value
    for (long i = i4; i < i4 + 4 && i < count; ++i) {
      float acc = 0.f;
      for (int s = 0; s < splits; ++s) acc += part[(long)s * count + i];
      out[i] = acc;
    }
    return;
  }
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < splits; ++s) {
    const float4 v = *reinterpret_cast<const float4 *>(part + (long)s * count + i4);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4 *>(out + i4) = acc;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// 3-D bf16 map, 128B swizzle: inner extent `inner` (contiguous), outer extent `outer`, `batch` entries of
// inner*outer elements; box (64, box_outer, 1)
static int gemm_map(CUtensorMap *m, const void *base, long inner, long outer, int batch, int box_outer) {
  const uint64_t dims[3] = {(uint64_t)inner, (uint64_t)outer, (uint64_t)batch};
  const uint64_t strides[2] = {(uint64_t)inner * 2, (uint64_t)inner * (uint64_t)outer * 2};
  const uint32_t box[3] = {64, (uint32_t)box_outer, 1};
  return make_tmap_bf16(m, base, 3, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int BJ, bool A_MN, bool B_MN, bool PAIR>
static int gemm_launch(const void *a, const void *b, const GemmParams &p0, cudaStream_t st) {
  using Cfg = GemmCfg<BJ, PAIR>;
  GemmParams p = p0;
  p.tiles_i = ceil_div(p.I, GEMM_BI);
  p.tiles_j = ceil_div(p.J, BJ);
  if (p.batch < 1) p.batch = 1;
  p.rblocks_per_batch = ceil_div(p.R, GEMM_BR);
  p.rblocks = p.rblocks_per_batch * (p.r_spans_batch ? p.batch : 1);
  CUtensorMap tm_a, tm_b;
  const int ba = p.a_batched ? p.batch : 1, bb = p.b_batched ? p.batch : 1;
  int rc = A_MN ? gemm_map(&tm_a, a, p.I, p.R, ba, 64) : gemm_map(&tm_a, a, p.R, p.I, ba, GEMM_BI);
  if (rc) return rc;
  rc = B_MN ? gemm_map(&tm_b, b, p.J, p.R, bb, 64) : gemm_map(&tm_b, b, p.R, p.J, bb, Cfg::BJ_CTA);
  if (rc) return rc;
  // bf16 raw output only: TMA-store epilogue over out[batch][I][J]
  CUtensorMap tm_out = tm_a;
  p.tma_out = 0;
  if (p.out_raw && !p.out_act && !p.out_f32) {
    const int ob = p.r_spans_batch ? 1 : p.batch;
    const uint64_t dims[3] = {(uint64_t)p.J, (uint64_t)p.I, (uint64_t)ob};
    const uint64_t strides[2] = {(uint64_t)p.J * 2, (uint64_t)(ob > 1 ? p.out_batch_stride : (long)p.I * p.J) * 2};
    const uint32_t box[3] = {64, 32, 1};
    rc = make_tmap_bf16(&tm_out, p.out_raw, 3, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    p.tma_out = 1;
  }
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(pw_gemm_sm100_kernel<BJ, A_MN, B_MN, PAIR>, Cfg::SMEM, attr_cache)) return e;
  const long items = (long)(PAIR ? p.tiles_i / 2 : p.tiles_i) * p.tiles_j * p.splits * (p.r_spans_batch ? 1 : p.batch);
  if (!PAIR) {
    const int grid = (int)min(items, (long)kNumSMs);
    launch_pdl(pw_gemm_sm100_kernel<BJ, A_MN, B_MN, PAIR>, dim3(grid), dim3(GEMM_THREADS), (size_t)Cfg::SMEM, st, tm_a, tm_b, tm_out, p);
    return launch_status();
  }
  // one cluster of two CTAs (one TPC) per work item
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * (unsigned)min(items, (long)(kNumSMs / 2)));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaLaunchKernelEx(&cfg, pw_gemm_sm100_kernel<BJ, A_MN, B_MN, PAIR>, tm_a, tm_b, tm_out, p);
  return launch_status();
}

template <bool A_MN, bool B_MN>
static int gemm_dispatch_bj(const void *a, const void *b, const GemmParams &p, cudaStream_t st) {
  if (p.J >= 256 && p.J % 256 == 0) {
    // CTA pairs need an even number of 128-row tiles
    if (ceil_div(p.I, GEMM_BI) % 2 == 0) return gemm_launch<256, A_MN, B_MN, true>(a, b, p, st);
    return gemm_launch<256, A_MN, B_MN, false>(a, b, p, st);
  }
  if (p.J > 64) return gemm_launch<128, A_MN, B_MN, false>(a, b, p, st);
  return gemm_launch<64, A_MN, B_MN, false>(a, b, p, st);
}

bool pw_sm100_supported(long M, int K, int Nc, int batch, int layout) {
  // 16-byte global strides for TMA and 16-byte epilogue stores
  if (M <= 0 || M >= (1L << 31) || K % 8 != 0) return false;
  if (layout == KDCC_LAYOUT_NCHW) return batch > 0 && M % batch == 0 && (M / batch) % 8 == 0;
  if (layout == KDCC_LAYOUT_PLANES_TO_NHWC) return batch > 0 && M % batch == 0 && (M / batch) % 8 == 0 && Nc % 8 == 0;
  return Nc % 8 == 0;
}

int pw_sm100_fwd(const void *x, const void *w, const float *scale, const float *shift, const void *residual, int relu,
                 void *y_raw, void *y_act, long M, int K, int Nc, int batch, int layout, cudaStream_t st) {
  GemmParams p{};
  p.out_raw = static_cast<__nv_bfloat16 *>(y_raw);
  p.out_act = static_cast<__nv_bfloat16 *>(y_act);
  p.scale = scale; p.shift = shift; p.relu = relu; p.splits = 1;
  p.residual = static_cast<const __nv_bfloat16 *>(residual);
  if (layout == KDCC_LAYOUT_NHWC) {
    // y[m][n] = sum_k x[m][k] w[n][k]
    p.I = (int)M; p.J = Nc; p.R = K; p.batch = 1;
    return gemm_dispatch_bj<false, false>(x, w, p, st);
  }
  const int P = (int)(M / batch);
  if (layout == KDCC_LAYOUT_PLANES_TO_NHWC) {
    // x planes, y channels_last: y_b[pix][n] = sum_k x_b[k][pix] w[n][k] : A = x_b (pixel-contiguous: MN-major), B = w (K-major)
    p.I = P; p.J = Nc; p.R = K; p.batch = batch; p.a_batched = 1; p.b_batched = 0;
    p.out_batch_stride = (long)P * Nc;
    return gemm_dispatch_bj<true, false>(x, w, p, st);
  }
  // NCHW: y_b[n][pix] = sum_k w[n][k] x_b[k][pix] : A = w (shared, K-major), B = x_b (pixel-contiguous, MN-major)
  p.I = Nc; p.J = P; p.R = K; p.batch = batch; p.a_batched = 0; p.b_batched = 1;
  p.out_batch_stride = (long)Nc * P; p.affine_rows = 1;
  return gemm_dispatch_bj<false, true>(w, x, p, st);
}

int pw_sm100_bwd_dx(const void *dy, const void *w, void *dx, long M, int K, int Nc, int batch, int layout, cudaStream_t st) {
  GemmParams p{};
  p.out_raw = static_cast<__nv_bfloat16 *>(dx);
  p.splits = 1;
  if (layout == KDCC_LAYOUT_NHWC) {
    // dx[m][k] = sum_n dy[m][n] w[n][k] : j = k, r = n; W [Nc][K] is j-contiguous -> MN-major B
    p.I = (int)M; p.J = K; p.R = Nc; p.batch = 1;
    return gemm_dispatch_bj<false, true>(dy, w, p, st);
  }
  // NCHW: dx_b[k][pix] = sum_n w[n][k] dy_b[n][pix] : A(i = k, r = n) = w (i-contiguous, MN-major, shared), B = dy_b (MN-major)
  const int P = (int)(M / batch);
  p.I = K; p.J = P; p.R = Nc; p.batch = batch; p.a_batched = 0; p.b_batched = 1;
  p.out_batch_stride = (long)K * P;
  // dy channels_last, dx planes: B = dy_b [pix][n] is r-contiguous (K-major)
  if (layout == KDCC_LAYOUT_PLANES_TO_NHWC) return gemm_dispatch_bj<true, false>(w, dy, p, st);
  return gemm_dispatch_bj<true, true>(w, dy, p, st);
}

static int dw_bj(int K) { return (K >= 256 && K % 256 == 0) ? 256 : (K > 64 ? 128 : 64); }

// Splits of the weight-gradient reduction: one reduction block (64 pixels, never across images in the NCHW form) is
// the unit, every split owns at least one.  `rblocks` differs by layout -- ceil(M / 64) for NHWC, batch * ceil(P / 64) for
// NCHW -- so the launch and the workspace bound below share this one formula.
static int dw_splits_for(long rblocks, int K, int Nc) {
  const long tiles = (long)ceil_div(Nc, GEMM_BI) * ceil_div(K, dw_bj(K));
  const long s = min(max(1L, (long)kNumSMs / tiles), rblocks);
  const long per = ceil_div<long>(rblocks, s);
  return (int)ceil_div<long>(rblocks, per);
}

// Upper bound on the split count for either layout and any batch (what kdcc_pw_bwd_workspace_bytes sizes for): the
// split count never exceeds kNumSMs / tiles, nor the number of reduction blocks, of which there are at most M / 8
// (an image contributes at least one block and at least 8 pixels).
int pw_sm100_dw_splits(long M, int K, int Nc) {
  const long tiles = (long)ceil_div(Nc, GEMM_BI) * ceil_div(K, dw_bj(K));
  return (int)min(max(1L, (long)kNumSMs / tiles), max(1L, ceil_div<long>(M, 8)));
}

int pw_sm100_bwd_dw(const void *dy, const void *x, float *dw, float *part, long M, int K, int Nc, int batch, int layout,
                    cudaStream_t st) {
  // dw[n][k] = sum_m dy[m][n] x[m][k] : i = n, j = k, r = pixels
  GemmParams p{};
  p.I = Nc; p.J = K;
  int rc;
  if (layout == KDCC_LAYOUT_NHWC) {
    p.R = (int)M; p.batch = 1;
    p.splits = dw_splits_for(ceil_div<long>(M, GEMM_BR), K, Nc);
    if (p.splits > pw_sm100_dw_splits(M, K, Nc)) return KDCC_EWORKSPACE;
    p.out_f32 = p.splits == 1 ? dw : part;
    rc = gemm_dispatch_bj<true, true>(dy, x, p, st);   // both operands are MN-major views
  } else {
    // NCHW: the pixel axis is contiguous in both dy_b [Nc][P] and x_b [K][P]: two K-major operands, the
    // reduction runs over (image, pixel block)
    const int P = (int)(M / batch);
    p.R = P; p.batch = batch; p.a_batched = 1; p.b_batched = 1; p.r_spans_batch = 1;
    p.splits = dw_splits_for((long)batch * ceil_div(P, GEMM_BR), K, Nc);
    if (p.splits > pw_sm100_dw_splits(M, K, Nc)) return KDCC_EWORKSPACE;  // the caller's workspace is sized by that bound
    p.out_f32 = p.splits == 1 ? dw : part;
    // dy channels_last [pix][n] (n-contiguous: MN-major A), x planes [k][pix] (K-major B)
    if (layout == KDCC_LAYOUT_PLANES_TO_NHWC) rc = gemm_dispatch_bj<true, false>(dy, x, p, st);
    else rc = gemm_dispatch_bj<false, false>(dy, x, p, st);
  }
  if (rc || p.splits == 1) return rc;
  const long count = (long)Nc * K;  // multiple of 4 because K % 8 == 0
  launch_pdl(reduce_splits_kernel, dim3((unsigned)ceil_div<long>(count / 4, 256)), dim3(256), 0, st, part, dw, p.splits, count);
  return launch_status();
}

}  // namespace kdcc
