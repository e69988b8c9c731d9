// fp32 pointwise (1x1) convolution on the sm_100a tensor cores at fp32 accuracy (KDCC_F32_TF32X3, DESIGN.md 4.3g).
// Every fp32 operand x is split into two tf32 values, hi = rna(x) and lo = rna(x - hi), and a product a.b is formed as
// lo(a).hi(b) + hi(a).lo(b) + hi(a).hi(b) -- three kind::tf32 MMAs (the dropped lo.lo term is below 2^-21 relative).
// NHWC only; the three GEMMs of the block, D[i][j] = sum_r A(i,r) B(j,r):
//   forward  i = pixel, j = out channel, r = in channel  : A = X [M][K] (K-major), B = W [Co][K] (K-major)
//   dX       i = pixel, j = in channel,  r = out channel : A = dY (K-major),       B = W read j-contiguous (MN-major)
//   dW       i = out channel, j = in channel, r = pixel  : A = dY, B = X, both MN-major; the pixel reduction is split
//            over CTAs into fp32 partials summed in fixed order by reduce_splits_kernel.
// Two properties of kind::tf32 on sm_100a shape the kernel (tools/tf32_probe.cu, profiles/r06_tf32_probe.txt):
//   - MN-major operand descriptors are not honoured, so the converter warps transpose an MN-major tile into the K-major
//     layout while they split it; the MMAs read K-major operands only.
//   - The tensor core rounds its fp32 accumulator toward zero, so a long reduction drifts toward zero by about half an
//     ulp per MMA.  The MMAs therefore accumulate X3_CHUNK_RB * 32 = 256-deep chunks, and the epilogue adds each chunk
//     into a running fp32 sum kept in tensor memory, rounded to nearest.
// Warp roles (448 threads): warp 0 = TMA producer (fp32 tiles, 128B swizzle, 32-deep reduction blocks), warp 1 = TMEM
// owner + MMA issuer, warps 2..5 = epilogue (one TMEM lane quadrant each), warps 6..13 = converters.  A converter rewrites
// each landed element as hi in place and writes lo into a sibling buffer of the same layout; a K-major tile keeps its
// swizzle untouched, an MN-major one is read whole by the converters before any of them writes it back transposed.
// Persistent CTAs walk the output tiles round-robin (i fastest); the chunk accumulator is double-buffered so the
// epilogue's fold of one chunk overlaps the next chunk's MMAs.
#include "kdcc_common.cuh"
#include "pw_kernels.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

constexpr int X3_BI = 128;        // UMMA M
constexpr int X3_BR = 32;         // reduction elements per stage = one 128-byte swizzle atom of fp32
constexpr int X3_CONV_WARPS = 8;
constexpr int X3_THREADS = 64 + 128 + 32 * X3_CONV_WARPS;
constexpr int X3_CHUNK_RB = 8;    // reduction blocks per TMEM chunk: 96 toward-zero roundings before a round-to-nearest add

template <int BJ>
struct X3Cfg {
  static constexpr int A_BYTES = X3_BI * X3_BR * 4;      // 16 KB
  static constexpr int B_BYTES = BJ * X3_BR * 4;
  static constexpr int HI_BYTES = A_BYTES + B_BYTES;     // [A hi | B hi] as loaded, then [A lo | B lo]
  static constexpr int STAGE_BYTES = 2 * HI_BYTES;
  static constexpr int STAGES = BJ == 128 ? 3 : 4;       // 192 KB either way
  static constexpr int TMEM_COLS = BJ == 128 ? 512 : 256;  // two chunk accumulators + the running sum (3 * BJ, power of 2)
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int SMEM = BAR_OFF + 256 + 1024;      // barriers + slack for the manual 1024-byte alignment
};

struct X3Params {
  int I, J, R;
  int tiles_i, tiles_j, splits, rblocks;
  float *out_raw, *out_act;          // [I][J], either may be null
  const float *scale, *shift;        // per j, may be null
  const float *residual;             // [I][J], added before the activation of out_act; may be null
  int relu;
  float *out_f32;                    // [splits][I][J] partials (dW) -- exclusive with the outputs above
};

// K-major SWIZZLE_128B shared-memory descriptor: 128-byte rows of 32 reduction elements, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t x3_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;  // LBO (unused by swizzled K-major layouts)
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

template <int BJ>
__device__ __forceinline__ constexpr uint32_t x3_idesc() {
  // c_format F32 (bits 4-5 = 1), a/b format TF32 (bits 7-9 / 10-12 = 2), both K-major (bits 15, 16 = 0), N >> 3, M >> 4
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BJ >> 3) << 17) | ((uint32_t)(X3_BI >> 4) << 24);
}

// hi = rna(x), lo = rna(x - hi); lo = 0 where hi is not finite, so inf and NaN inputs reach the output through hi.hi
__device__ __forceinline__ void x3_split(float x, float &hi, float &lo) {
  hi = ptx::cvt_rna_tf32(x);
  lo = isfinite(hi) ? ptx::cvt_rna_tf32(x - hi) : 0.f;
}

// Split a K-major region (`n16` 16-byte vectors) in place: hi over x, lo at the same offset in `lo`.
__device__ __forceinline__ void x3_split_kmajor(float4 *hi, float4 *lo, int n16, int ct) {
#pragma unroll 4
  for (int i = ct; i < n16; i += 32 * X3_CONV_WARPS) {
    const float4 x = hi[i];
    float4 h, l;
    x3_split(x.x, h.x, l.x); x3_split(x.y, h.y, l.y); x3_split(x.z, h.z, l.z); x3_split(x.w, h.w, l.w);
    hi[i] = h;
    lo[i] = l;
  }
}

// An MN-major region as TMA lands it: 32-element i/j groups of 4096 bytes, each 32 r-rows of 128 bytes, swizzled.  The
// 16-byte vector at byte offset o holds r = (o >> 7) & 31 and i/j = 32 * (o >> 12) + 4 * (((o >> 4) & 7) ^ (r & 7)) + 0..3.
// Its elements go to row i/j, column r of the K-major layout (128-byte rows of 32 r, swizzled).
template <int N>
__device__ __forceinline__ void x3_split_transposed(uint8_t *hi, uint8_t *lo, const float4 (&v)[N], int ct) {
#pragma unroll
  for (int j = 0; j < N; ++j) {
    const int o = (ct + j * 32 * X3_CONV_WARPS) * 16;
    const int r = (o >> 7) & 31;
    const int mn0 = 32 * (o >> 12) + 4 * (((o >> 4) & 7) ^ (r & 7));
    const float x[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int mn = mn0 + e;
      const int dst = mn * 128 + ((((r >> 2) ^ mn) & 7) << 4) + (r & 3) * 4;
      float h, l;
      x3_split(x[e], h, l);
      *reinterpret_cast<float *>(hi + dst) = h;
      *reinterpret_cast<float *>(lo + dst) = l;
    }
  }
}

template <int BJ, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(X3_THREADS, 1)
pw_gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const X3Params p) {
  using Cfg = X3Cfg<BJ>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem_gen = smem_raw + (smem_base - ptx::smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + Cfg::BAR_OFF;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };                  // TMA landed
  auto conv_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };       // split into hi / lo
  auto empty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };  // MMAs done reading
  auto tfull_bar = [&](int s) { return bar_base + 8u * (3 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (3 * STAGES + 2 + s); };
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem_gen + Cfg::BAR_OFF + 8 * (3 * STAGES + 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(conv_bar(s), X3_CONV_WARPS); ptx::mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), 4); }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_a);
    ptx::prefetch_tensormap(&tm_b);
  }
  if (warp == 1) ptx::tmem_alloc<Cfg::TMEM_COLS>(ptx::smem_u32(const_cast<uint32_t *>(tmem_slot)));
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();

  const long items = (long)p.tiles_i * p.tiles_j * p.splits;
  const int rb_per_split = (p.rblocks + p.splits - 1) / p.splits;

  if (warp == 0) {
    // ===== TMA producer =====
    if (ptx::elect_one()) {
      int s = 0; uint32_t ph = 0;
      for (long item = blockIdx.x; item < items; item += gridDim.x) {
        const int split = (int)(item % p.splits);
        const long tile = item / p.splits;
        const int ti = (int)(tile % p.tiles_i), tj = (int)(tile / p.tiles_i);
        const int rb0 = split * rb_per_split, rb1 = min(p.rblocks, rb0 + rb_per_split);
        for (int rb = rb0; rb < rb1; ++rb) {
          ptx::mbar_wait(empty_bar(s), ph ^ 1);
          const uint32_t a_dst = smem_base + s * Cfg::STAGE_BYTES, b_dst = a_dst + Cfg::A_BYTES;
          ptx::mbar_arrive_expect_tx(full_bar(s), Cfg::HI_BYTES);
          if (!A_MN) {
            ptx::tma_load_2d(a_dst, &tm_a, full_bar(s), rb * X3_BR, ti * X3_BI);
          } else {
#pragma unroll
            for (int b = 0; b < X3_BI / 32; ++b) ptx::tma_load_2d(a_dst + b * 4096, &tm_a, full_bar(s), ti * X3_BI + b * 32, rb * X3_BR);
          }
          if (!B_MN) {
            ptx::tma_load_2d(b_dst, &tm_b, full_bar(s), rb * X3_BR, tj * BJ);
          } else {
#pragma unroll
            for (int b = 0; b < BJ / 32; ++b) ptx::tma_load_2d(b_dst + b * 4096, &tm_b, full_bar(s), tj * BJ + b * 32, rb * X3_BR);
          }
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = x3_idesc<BJ>();
      int s = 0; uint32_t ph = 0;
      int as = 0; uint32_t aph = 0;
      for (long item = blockIdx.x; item < items; item += gridDim.x) {
        const int split = (int)(item % p.splits);
        const int rb0 = split * rb_per_split, rb1 = min(p.rblocks, rb0 + rb_per_split);
        for (int c0 = rb0; c0 < rb1; c0 += X3_CHUNK_RB) {
          ptx::mbar_wait(tempty_bar(as), aph ^ 1);
          ptx::tcgen05_fence_after();
          const uint32_t d = tmem_base + (uint32_t)(as * BJ);
          for (int rb = c0; rb < min(rb1, c0 + X3_CHUNK_RB); ++rb) {
            ptx::mbar_wait(conv_bar(s), ph);
            ptx::tcgen05_fence_after();
            const uint32_t a_hi = smem_base + s * Cfg::STAGE_BYTES, b_hi = a_hi + Cfg::A_BYTES;
            const uint32_t a_lo = a_hi + Cfg::HI_BYTES, b_lo = b_hi + Cfg::HI_BYTES;
#pragma unroll
            for (int k = 0; k < X3_BR / 8; ++k) {
              // 8 reduction elements = 32 bytes inside the swizzle atom; small terms first
              ptx::umma_tf32(d, x3_desc(a_lo + k * 32), x3_desc(b_hi + k * 32), idesc, (rb > c0 || k > 0) ? 1u : 0u);
              ptx::umma_tf32(d, x3_desc(a_hi + k * 32), x3_desc(b_lo + k * 32), idesc, 1u);
              ptx::umma_tf32(d, x3_desc(a_hi + k * 32), x3_desc(b_hi + k * 32), idesc, 1u);
            }
            ptx::umma_commit(empty_bar(s));
            if (++s == STAGES) { s = 0; ph ^= 1; }
          }
          ptx::umma_commit(tfull_bar(as));   // chunk complete -> epilogue
          if (++as == 2) { as = 0; aph ^= 1; }
        }
      }
    }
  } else if (warp < 6) {
    // ===== epilogue: TMEM -> registers -> global =====
    const int quad = warp & 3;  // TMEM lanes [32*quad, 32*quad+32) are accessible to this warp
    int as = 0; uint32_t aph = 0;
    const uint32_t t_lane = (uint32_t)(quad * 32) << 16;
    const uint32_t t_sum = tmem_base + 2 * BJ + t_lane;   // running sum over the chunks of the current tile
    for (long item = blockIdx.x; item < items; item += gridDim.x) {
      const int split = (int)(item % p.splits);
      const long tile = item / p.splits;
      const int ti = (int)(tile % p.tiles_i), tj = (int)(tile / p.tiles_i);
      const int rb0 = split * rb_per_split, rb1 = min(p.rblocks, rb0 + rb_per_split);
      const int row = ti * X3_BI + quad * 32 + lane;
      for (int c0 = rb0; c0 < rb1; c0 += X3_CHUNK_RB) {
        const bool first = c0 == rb0, last = c0 + X3_CHUNK_RB >= rb1;
        ptx::mbar_wait(tfull_bar(as), aph);
        ptx::tcgen05_fence_after();
        __syncwarp();
        const uint32_t t_acc = tmem_base + (uint32_t)(as * BJ) + t_lane;
#pragma unroll 1
        for (int ch = 0; ch < BJ / 32; ++ch) {
          const int col0 = tj * BJ + ch * 32;
          if (col0 >= p.J) break;  // warp-uniform
          uint32_t v[32];
          ptx::tmem_ld_32x32b_x32(t_acc + ch * 32, v);
          if (!first) {
            uint32_t w[32];
            ptx::tmem_ld_32x32b_x32(t_sum + ch * 32, w);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(w[e]) + __uint_as_float(v[e]));
          } else {
            ptx::tmem_ld_wait();
          }
          if (!last) {
            ptx::tmem_st_32x32b_x32(t_sum + ch * 32, v);
            continue;
          }
          if (row >= p.I) continue;
          const long off = (long)row * p.J + col0;
          if (p.out_f32 != nullptr) {
            float *dst = p.out_f32 + (long)split * p.I * p.J + off;
#pragma unroll
            for (int q = 0; q < 8; ++q)
              if (col0 + q * 4 < p.J)
                *reinterpret_cast<uint4 *>(dst + q * 4) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            continue;
          }
          if (p.out_raw != nullptr) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              if (col0 + q * 4 < p.J)
                *reinterpret_cast<uint4 *>(p.out_raw + off + q * 4) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          }
          if (p.out_act != nullptr) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              if (col0 + q * 4 >= p.J) continue;
              float r[4] = {0.f, 0.f, 0.f, 0.f}, f[4];
              if (p.residual) {
                const float4 rv = __ldg(reinterpret_cast<const float4 *>(p.residual + off + q * 4));
                r[0] = rv.x; r[1] = rv.y; r[2] = rv.z; r[3] = rv.w;
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int c = col0 + q * 4 + e;
                float x = __uint_as_float(v[4 * q + e]);
                if (p.scale) x *= __ldg(p.scale + c);
                if (p.shift) x += __ldg(p.shift + c);
                if (p.residual) x += r[e];
                if (p.relu) x = fmaxf(x, 0.f);
                f[e] = x;
              }
              *reinterpret_cast<float4 *>(p.out_act + off + q * 4) = make_float4(f[0], f[1], f[2], f[3]);
            }
          }
        }
        if (!last) ptx::tmem_st_wait();
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(tempty_bar(as));
        if (++as == 2) { as = 0; aph ^= 1; }
      }
    }
  } else {
    // ===== converters: x -> (hi in place, lo in the sibling buffer) =====
    const int ct = threadIdx.x - 192;
    int s = 0; uint32_t ph = 0;
    for (long item = blockIdx.x; item < items; item += gridDim.x) {
      const int split = (int)(item % p.splits);
      const int rb0 = split * rb_per_split, rb1 = min(p.rblocks, rb0 + rb_per_split);
      for (int rb = rb0; rb < rb1; ++rb) {
        ptx::mbar_wait(full_bar(s), ph);
        uint8_t *a_hi = smem_gen + s * Cfg::STAGE_BYTES, *b_hi = a_hi + Cfg::A_BYTES;
        uint8_t *a_lo = a_hi + Cfg::HI_BYTES, *b_lo = b_hi + Cfg::HI_BYTES;
        constexpr int NA = Cfg::A_BYTES / 16 / (32 * X3_CONV_WARPS), NB = Cfg::B_BYTES / 16 / (32 * X3_CONV_WARPS);
        float4 va[A_MN ? NA : 1], vb[B_MN ? NB : 1];
        if (A_MN) {
#pragma unroll
          for (int j = 0; j < NA; ++j) va[j] = reinterpret_cast<const float4 *>(a_hi)[ct + j * 32 * X3_CONV_WARPS];
        }
        if (B_MN) {
#pragma unroll
          for (int j = 0; j < NB; ++j) vb[j] = reinterpret_cast<const float4 *>(b_hi)[ct + j * 32 * X3_CONV_WARPS];
        }
        // an MN-major tile is rewritten in a different order: every converter has read it before any writes
        if (A_MN || B_MN) asm volatile("bar.sync 1, %0;" ::"n"(32 * X3_CONV_WARPS) : "memory");
        if (A_MN) x3_split_transposed(a_hi, a_lo, va, ct);
        else x3_split_kmajor(reinterpret_cast<float4 *>(a_hi), reinterpret_cast<float4 *>(a_lo), Cfg::A_BYTES / 16, ct);
        if (B_MN) x3_split_transposed(b_hi, b_lo, vb, ct);
        else x3_split_kmajor(reinterpret_cast<float4 *>(b_hi), reinterpret_cast<float4 *>(b_lo), Cfg::B_BYTES / 16, ct);
        ptx::fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's operand reads
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(conv_bar(s));
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  }

  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// 2-D fp32 map over a row-major [outer][inner] tensor, 128B swizzle, box (32, box_outer)
static int x3_map(CUtensorMap *m, const void *base, long inner, long outer, int box_outer) {
  const uint64_t dims[2] = {(uint64_t)inner, (uint64_t)outer};
  const uint64_t strides[1] = {(uint64_t)inner * 4};
  const uint32_t box[2] = {32, (uint32_t)box_outer};
  return make_tmap_f32(m, base, 2, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_128B);
}

static int x3_bj(int J) { return J > 64 ? 128 : 64; }

template <int BJ, bool A_MN, bool B_MN>
static int x3_launch(const void *a, const void *b, const X3Params &p0, cudaStream_t st) {
  using Cfg = X3Cfg<BJ>;
  X3Params p = p0;
  p.tiles_i = ceil_div(p.I, X3_BI);
  p.tiles_j = ceil_div(p.J, BJ);
  p.rblocks = ceil_div(p.R, X3_BR);
  CUtensorMap tm_a, tm_b;
  int rc = A_MN ? x3_map(&tm_a, a, p.I, p.R, 32) : x3_map(&tm_a, a, p.R, p.I, X3_BI);
  if (rc) return rc;
  rc = B_MN ? x3_map(&tm_b, b, p.J, p.R, 32) : x3_map(&tm_b, b, p.R, p.J, BJ);
  if (rc) return rc;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(pw_gemm_tf32x3_kernel<BJ, A_MN, B_MN>, Cfg::SMEM, attr_cache)) return e;
  const long items = (long)p.tiles_i * p.tiles_j * p.splits;
  const int grid = (int)min(items, (long)kNumSMs);
  launch_pdl(pw_gemm_tf32x3_kernel<BJ, A_MN, B_MN>, dim3(grid), dim3(X3_THREADS), (size_t)Cfg::SMEM, st, tm_a, tm_b, p);
  return launch_status();
}

template <bool A_MN, bool B_MN>
static int x3_dispatch(const void *a, const void *b, const X3Params &p, cudaStream_t st) {
  if (x3_bj(p.J) == 128) return x3_launch<128, A_MN, B_MN>(a, b, p, st);
  return x3_launch<64, A_MN, B_MN>(a, b, p, st);
}

bool pw_tf32x3_supported(long M, int K, int Nc) {
  // 16-byte TMA rows and 16-byte epilogue stores
  return M > 0 && M < (1L << 31) && K > 0 && Nc > 0 && K % 4 == 0 && Nc % 4 == 0;
}

int pw_tf32x3_fwd(const void *x, const void *w, const float *scale, const float *shift, const void *residual, int relu,
                  void *y_raw, void *y_act, long M, int K, int Nc, cudaStream_t st) {
  // y[m][n] = sum_k x[m][k] w[n][k]
  X3Params p{};
  p.I = (int)M; p.J = Nc; p.R = K; p.splits = 1;
  p.out_raw = static_cast<float *>(y_raw); p.out_act = static_cast<float *>(y_act);
  p.scale = scale; p.shift = shift; p.residual = static_cast<const float *>(residual); p.relu = relu;
  return x3_dispatch<false, false>(x, w, p, st);
}

int pw_tf32x3_bwd_dx(const void *dy, const void *w, void *dx, long M, int K, int Nc, cudaStream_t st) {
  // dx[m][k] = sum_n dy[m][n] w[n][k] : W [Nc][K] is j-contiguous -> MN-major B
  X3Params p{};
  p.I = (int)M; p.J = K; p.R = Nc; p.splits = 1;
  p.out_raw = static_cast<float *>(dx);
  return x3_dispatch<false, true>(dy, w, p, st);
}

// Splits of the weight-gradient pixel reduction (to fill the SMs): one 32-pixel block is the unit, every split owns at
// least one.
int pw_tf32x3_dw_splits(long M, int K, int Nc) {
  const long tiles = (long)ceil_div(Nc, X3_BI) * ceil_div(K, x3_bj(K));
  const long rblocks = ceil_div<long>(M, X3_BR);
  const long s = min(max(1L, (long)kNumSMs / tiles), rblocks);
  const long per = ceil_div<long>(rblocks, s);
  return (int)ceil_div<long>(rblocks, per);
}

int pw_tf32x3_bwd_dw(const void *dy, const void *x, float *dw, float *part, long M, int K, int Nc, cudaStream_t st) {
  // dw[n][k] = sum_m dy[m][n] x[m][k] : i = n, j = k, r = pixels; both operands are MN-major views
  X3Params p{};
  p.I = Nc; p.J = K; p.R = (int)M;
  p.splits = pw_tf32x3_dw_splits(M, K, Nc);
  p.out_f32 = p.splits == 1 ? dw : part;
  const int rc = x3_dispatch<true, true>(dy, x, p, st);
  if (rc || p.splits == 1) return rc;
  const long count = (long)Nc * K;  // multiple of 4 because K % 4 == 0
  launch_pdl(reduce_splits_kernel, dim3((unsigned)ceil_div<long>(count / 4, 256)), dim3(256), 0, st, part, dw, p.splits, count);
  return launch_status();
}

}  // namespace kdcc
