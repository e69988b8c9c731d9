// Depthwise 3 x 3 (dilation 1, pad 1) for NHWC bf16: the HBM-bound stencil of the north star, on the CUDA cores.
//
// Reference semantics: models/students/transform_blocks/depthwise_separable_conv.py:7-8,12 with the CIFAR geometry
// (cfg/cifar10/resnet44/config1.json:84-89: k = 3, d = 1, p = 1) and its autograd backward.
//
// 2.25 MAC per HBM byte: the kernel has to stream.  No shared-memory tile, no widening pass:
//  * a lane owns 8 channels (one 16-byte vector) of one pixel column, a warp 32 adjacent vectors of the NHWC row
//    (512 contiguous bytes: fully coalesced), a CTA 6 adjacent column groups x 32 rows; CTAs are persistent (two per
//    SM, 168 registers each) and walk their tiles with one continuous ring;
//  * TMA streams the tile row by row (columns j0-1 .. j0+8, out-of-bounds zero fill = the conv padding, so there are
//    no edge predicates) through a 16-deep shared-memory ring: ~60 KB in flight per CTA independent of registers
//    (a register-prefetch version with one row in flight per thread reached only 2.4 TB/s, an 8-deep ring 3.0);
//  * each thread walks down its column: the input row r is read as three 16-byte LDS (left, centre, right), widened
//    ONCE to fp32 and scattered into the three output rows it touches (r-1, r, r+1), whose accumulators rotate
//    through registers; 72 FMAs per arrival as 36 packed fma.rn.f32x2 (half the issue slots; tools/fma_probe.cu: the
//    packed form does not raise fp32 throughput), the 9 x 8 taps of the lane's channels stay in registers;
//  * the input-gradient is the same kernel over dy with mirrored taps;
//  * weight gradient: same walk, the arriving x row meets the three dy rows around it; 9 x 8 partial sums per
//    thread over ALL the tiles of a persistent CTA, then a fixed-order shared-memory sum over the CTA's columns and
//    one partial per CTA (deterministic two-stage reduction, no atomics).
#include "dw_kernels.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

#ifndef KDCC_N3_WARPS
#define KDCC_N3_WARPS 6
#endif
#ifndef KDCC_N3_OCC
#define KDCC_N3_OCC 2
#endif
constexpr int N3_WARPS = KDCC_N3_WARPS;     // pixel-column groups per CTA tile
constexpr int N3_THREADS = 32 * N3_WARPS;
constexpr int N3_CH = 8;                    // channels per thread (one 16-byte vector; 4 = 8-byte vectors, more warps, measured slower)
constexpr int N3_OCC = KDCC_N3_OCC;                 // CTAs per SM (launch bounds): 192 threads x 168 registers
constexpr int N3_PAIRS = N3_CH / 2;
constexpr int N3_VB = 2 * N3_CH;            // bytes of one thread's vector
constexpr int N3_TH = 32;                   // rows per CTA tile
constexpr int N3_STAGES = 16;               // rows in flight per CTA: ~80 KB per CTA, 160 KB per SM (8 stages starve the ring)
constexpr int N3_BAR = 8 * N3_STAGES;       // byte offset of the empty barriers behind the full barriers
constexpr int N3_WSTAGES = 12;              // weight gradient: a stage holds an x row and a dy row (7 KB); 2 CTAs per SM stay resident
constexpr int N3_WBAR = 8 * N3_WSTAGES;

struct N3Params {
  __nv_bfloat16 *out;
  const float *w, *bias;
  float *part;               // wgrad: [ctas_per_group][9][C]
  int N, H, W, C;
  int Vb, Jb;                // vectors (N3_CH channels) per warp along C, pixel columns per warp: Vb * Jb == 32
  int vgroups;               // C / (N3_CH * Vb)
  int tiles_h, tiles_w;      // tile = N3_TH rows x N3_WARPS * Jb columns
  int flip;
  int ctas_per_group;        // persistent CTAs per channel group
  int prefill;               // ring stages filled ahead: stages - 1 (the producer refills a stage one arrival after it was read)
  int dbg;                   // KDCC_TC_DEBUG (timing experiments): 1 skip the FMAs, 2 skip the TMA ring (compute on stale smem), 4 skip stores
};

// Blackwell packed fp32 FMA: two FFMAs per instruction on 64-bit register pairs (halves the FMA issue slots)
__device__ __forceinline__ float2 ffma2(const float2 a, const float2 b, const float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(*reinterpret_cast<unsigned long long *>(&d))
      : "l"(*reinterpret_cast<const unsigned long long *>(&a)), "l"(*reinterpret_cast<const unsigned long long *>(&b)),
        "l"(*reinterpret_cast<const unsigned long long *>(&c)));
  return d;
}
struct N3Vec {  // one thread's N3_CH bf16 channels
  uint32_t w[N3_PAIRS];
};
__device__ __forceinline__ N3Vec n3_lds(const uint8_t *p) {
  N3Vec v;
  if constexpr (N3_CH == 8) {
    const uint4 q = *reinterpret_cast<const uint4 *>(p);
    v.w[0] = q.x; v.w[1] = q.y; v.w[N3_PAIRS - 2] = q.z; v.w[N3_PAIRS - 1] = q.w;
  } else {
    const uint2 q = *reinterpret_cast<const uint2 *>(p);
    v.w[0] = q.x; v.w[1] = q.y;
  }
  return v;
}
__device__ __forceinline__ void n3_stg(__nv_bfloat16 *p, const float2 (&a)[N3_PAIRS]) {
  if constexpr (N3_CH == 8) {
    *reinterpret_cast<uint4 *>(p) = make_uint4(pack_bf16x2(a[0].x, a[0].y), pack_bf16x2(a[1].x, a[1].y),
                                               pack_bf16x2(a[N3_PAIRS - 2].x, a[N3_PAIRS - 2].y),
                                               pack_bf16x2(a[N3_PAIRS - 1].x, a[N3_PAIRS - 1].y));
  } else {
    *reinterpret_cast<uint2 *>(p) = make_uint2(pack_bf16x2(a[0].x, a[0].y), pack_bf16x2(a[1].x, a[1].y));
  }
}
__device__ __forceinline__ void unpackv(const N3Vec &v, float2 (&f)[N3_PAIRS]) {
#pragma unroll
  for (int e = 0; e < N3_PAIRS; ++e) f[e] = make_float2(bf16lo(v.w[e]), bf16hi(v.w[e]));
}

// One tile = N3_TH rows x (N3_WARPS * Jb) columns of one image; arrivals = its input rows i0-1 .. i1.
struct N3Tile {
  int n, i0, i1, j0;
};
__device__ __forceinline__ N3Tile n3_tile(const N3Params &p, long tile) {
  N3Tile t;
  const int tw = (int)(tile % p.tiles_w); tile /= p.tiles_w;
  const int th = (int)(tile % p.tiles_h);
  t.n = (int)(tile / p.tiles_h);
  t.i0 = th * N3_TH; t.i1 = min(t.i0 + N3_TH, p.H); t.j0 = tw * N3_WARPS * p.Jb;
  return t;
}

// ------------------------------------------------------------------------------------------------
// forward / input gradient
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(N3_THREADS, N3_OCC)
dw_nhwc3_conv_kernel(const __grid_constant__ CUtensorMap tm_in, const N3Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int vb = lane % p.Vb, jl = lane / p.Vb;
  const int vg = blockIdx.x % p.vgroups;
  const int slot = blockIdx.x / p.vgroups;
  const int jt = warp * p.Jb + jl;       // column inside the tile
  const int c0 = (vg * p.Vb + vb) * N3_CH;
  const int px_bytes = p.Vb * N3_VB;                              // one pixel of the channel group
  const int row_bytes = (N3_WARPS * p.Jb + 2) * px_bytes;      // tile row with one halo column on each side
  const int row_stride = (row_bytes + 127) & ~127;             // TMA destinations are 128-byte aligned
  const uint32_t ring = ptx::smem_u32(smem);
  const uint32_t bars = ring + N3_STAGES * row_stride;         // full[s] at bars + 8 s, empty[s] at bars + N3_BAR + 8 s
  if (threadIdx.x == 0) {
    for (int s = 0; s < N3_STAGES; ++s) { ptx::mbar_init(bars + 8u * s, 1); ptx::mbar_init(bars + N3_BAR + 8u * s, N3_WARPS); }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_in);
  }
  // taps of this lane's 8 channels as fp32 pairs: wr[u*3+v][pair]; the bias starts every output row
  float2 wr[9][N3_PAIRS], b2[N3_PAIRS];
#pragma unroll
  for (int e = 0; e < N3_PAIRS; ++e) {
#pragma unroll
    for (int tap = 0; tap < 9; ++tap)
      wr[tap][e] = make_float2(__ldg(p.w + (long)(c0 + 2 * e) * 9 + (p.flip ? 8 - tap : tap)),
                               __ldg(p.w + (long)(c0 + 2 * e + 1) * 9 + (p.flip ? 8 - tap : tap)));
    b2[e] = p.bias ? make_float2(__ldg(p.bias + c0 + 2 * e), __ldg(p.bias + c0 + 2 * e + 1)) : make_float2(0.f, 0.f);
  }
  __syncthreads();
  pdl_prologue_done();
  const long tiles = (long)p.N * p.tiles_h * p.tiles_w;
  const long rowp = (long)p.W * p.C;
  // producer (thread 0): arrivals are numbered across all the tiles of this CTA, the ring never drains between tiles
  long ptile = slot; int pa = 0; uint32_t pcount = 0;
  N3Tile pt = n3_tile(p, ptile < tiles ? ptile : 0);
  auto issue_next = [&]() {
    if (ptile >= tiles) return;
    const uint32_t s = pcount % N3_STAGES;
    ptx::mbar_wait(bars + N3_BAR + 8u * s, ((pcount / N3_STAGES) & 1) ^ 1);
    ptx::mbar_arrive_expect_tx(bars + 8u * s, (uint32_t)row_bytes);
    // rows -1 / H and columns -1 / W are zero-filled by the hardware: that IS the conv padding
    ptx::tma_load_4d(ring + s * row_stride, &tm_in, bars + 8u * s, vg * p.Vb * N3_CH, pt.j0 - 1, pt.i0 - 1 + pa, pt.n);
    ++pcount;
    if (++pa == pt.i1 - pt.i0 + 2) {
      pa = 0;
      ptile += p.ctas_per_group;
      if (ptile < tiles) pt = n3_tile(p, ptile);
    }
  };
  if (threadIdx.x == 0 && !KDCC_DBG(p, 2))
    for (int k = 0; k < p.prefill; ++k) issue_next();
  uint32_t count = 0;  // arrivals consumed
  const uint8_t *mine = smem + jt * px_bytes + vb * N3_VB;   // left neighbour of this thread's column inside a ring row
  for (long tile = slot; tile < tiles; tile += p.ctas_per_group) {
    const N3Tile t = n3_tile(p, tile);
    const bool active = t.j0 + jt < p.W;
    const int arrivals = t.i1 - t.i0 + 2;
    __nv_bfloat16 *optr = p.out + (((long)t.n * p.H + t.i0) * p.W + t.j0 + jt) * p.C + c0;  // next output row to store
    int skip = 2;  // the first two arrivals complete rows i0-2 and i0-1, which belong to other tiles
    // the arriving input row r adds tap row 2 to output row r-1, tap row 1 to r, and starts output row r+1 with tap row 0
    auto arrive = [&](float2 (&prev)[N3_PAIRS], float2 (&cur)[N3_PAIRS], float2 (&next)[N3_PAIRS]) {
      const uint32_t s = count % N3_STAGES;
      if (!KDCC_DBG(p, 2)) {
        if (threadIdx.x == 0) issue_next();
        ptx::mbar_wait(bars + 8u * s, (count / N3_STAGES) & 1);
      }
      ++count;
      const uint8_t *row = mine + s * row_stride;
      const N3Vec vl = n3_lds(row), vc = n3_lds(row + px_bytes), vr = n3_lds(row + 2 * px_bytes);
      if (!KDCC_DBG(p, 2)) {
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bars + N3_BAR + 8u * s);
      }
      float2 x[N3_PAIRS];
      if (KDCC_DBG(p, 1)) {
        unpackv(vl, x);
#pragma unroll
        for (int e = 0; e < N3_PAIRS; ++e) { prev[e].x += x[e].x + __uint_as_float(vc.w[e]) + __uint_as_float(vr.w[e]); }
        if (skip > 0) { --skip; return; }
        if (active && !KDCC_DBG(p, 4)) n3_stg(optr, prev);
        optr += rowp;
        return;
      }
      unpackv(vl, x);
#pragma unroll
      for (int e = 0; e < N3_PAIRS; ++e) {
        prev[e] = ffma2(wr[6][e], x[e], prev[e]); cur[e] = ffma2(wr[3][e], x[e], cur[e]); next[e] = ffma2(wr[0][e], x[e], b2[e]);
      }
      unpackv(vc, x);
#pragma unroll
      for (int e = 0; e < N3_PAIRS; ++e) {
        prev[e] = ffma2(wr[7][e], x[e], prev[e]); cur[e] = ffma2(wr[4][e], x[e], cur[e]); next[e] = ffma2(wr[1][e], x[e], next[e]);
      }
      unpackv(vr, x);
#pragma unroll
      for (int e = 0; e < N3_PAIRS; ++e) {
        prev[e] = ffma2(wr[8][e], x[e], prev[e]); cur[e] = ffma2(wr[5][e], x[e], cur[e]); next[e] = ffma2(wr[2][e], x[e], next[e]);
      }
      // `prev` is complete: output row r-1
      if (skip > 0) { --skip; return; }
      if (active && !KDCC_DBG(p, 4)) n3_stg(optr, prev);
      optr += rowp;
    };
    float2 a0[N3_PAIRS], a1[N3_PAIRS], a2[N3_PAIRS];
#pragma unroll
    for (int e = 0; e < N3_PAIRS; ++e) a0[e] = a1[e] = b2[e];  // (never stored: rows i0-2 and i0-1)
    for (int a = 0; a < arrivals; a += 3) {
      arrive(a0, a1, a2);
      if (a + 1 >= arrivals) break;
      arrive(a1, a2, a0);
      if (a + 2 >= arrivals) break;
      arrive(a2, a0, a1);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// weight gradient: dw[c][u][v] = sum dy[n][i][j][c] * x[n][i+u-1][j+v-1][c]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(N3_THREADS, N3_OCC)
dw_nhwc3_wgrad_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_dy, const N3Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int vb = lane % p.Vb, jl = lane / p.Vb;
  const int vg = blockIdx.x % p.vgroups;
  const int slot = blockIdx.x / p.vgroups;
  const int jt = warp * p.Jb + jl;
  const int px_bytes = p.Vb * N3_VB;
  const int xrow_bytes = (N3_WARPS * p.Jb + 2) * px_bytes;   // x row with halo columns
  const int grow_bytes = N3_WARPS * p.Jb * px_bytes;         // dy row
  const int xrow_stride = (xrow_bytes + 127) & ~127;         // TMA destinations are 128-byte aligned
  const int stage_bytes = xrow_stride + ((grow_bytes + 127) & ~127);
  const uint32_t ring = ptx::smem_u32(smem);
  const uint32_t bars = ring + N3_WSTAGES * stage_bytes;
  float *red = reinterpret_cast<float *>(smem + N3_WSTAGES * stage_bytes + 2 * N3_WBAR);  // [threads][N3_CH] per tap
  if (threadIdx.x == 0) {
    for (int s = 0; s < N3_WSTAGES; ++s) { ptx::mbar_init(bars + 8u * s, 1); ptx::mbar_init(bars + N3_WBAR + 8u * s, N3_WARPS); }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_x);
    ptx::prefetch_tensormap(&tm_dy);
  }
  float2 acc[9][N3_PAIRS];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap)
#pragma unroll
    for (int e = 0; e < N3_PAIRS; ++e) acc[tap][e] = make_float2(0.f, 0.f);
  __syncthreads();
  pdl_prologue_done();
  const long tiles = (long)p.N * p.tiles_h * p.tiles_w;
  long ptile = slot; int pa = 0; uint32_t pcount = 0;
  N3Tile pt = n3_tile(p, ptile < tiles ? ptile : 0);
  auto issue_next = [&]() {
    if (ptile >= tiles) return;
    const uint32_t s = pcount % N3_WSTAGES;
    ptx::mbar_wait(bars + N3_WBAR + 8u * s, ((pcount / N3_WSTAGES) & 1) ^ 1);
    const bool has_g = pa < pt.i1 - pt.i0;  // stage = x row i0-1+pa and, while there is one, dy row i0+pa
    ptx::mbar_arrive_expect_tx(bars + 8u * s, (uint32_t)(xrow_bytes + (has_g ? grow_bytes : 0)));
    ptx::tma_load_4d(ring + s * stage_bytes, &tm_x, bars + 8u * s, vg * p.Vb * N3_CH, pt.j0 - 1, pt.i0 - 1 + pa, pt.n);
    if (has_g) ptx::tma_load_4d(ring + s * stage_bytes + xrow_stride, &tm_dy, bars + 8u * s, vg * p.Vb * N3_CH, pt.j0, pt.i0 + pa, pt.n);
    ++pcount;
    if (++pa == pt.i1 - pt.i0 + 2) {
      pa = 0;
      ptile += p.ctas_per_group;
      if (ptile < tiles) pt = n3_tile(p, ptile);
    }
  };
  if (threadIdx.x == 0)
    for (int k = 0; k < p.prefill; ++k) issue_next();
  uint32_t count = 0;
  const uint8_t *mine = smem + jt * px_bytes + vb * N3_VB;
  for (long tile = slot; tile < tiles; tile += p.ctas_per_group) {
    const N3Tile t = n3_tile(p, tile);
    const bool active = t.j0 + jt < p.W;
    const int nrows = t.i1 - t.i0, arrivals = nrows + 2;
    // the arriving x row r meets dy row r+1 through tap row 0, dy row r through tap row 1, dy row r-1 through tap row 2
    auto arrive = [&](int a, const float2 (&gm)[N3_PAIRS], const float2 (&g0)[N3_PAIRS], float2 (&gp)[N3_PAIRS]) {
      if (threadIdx.x == 0) issue_next();
      const uint32_t s = count % N3_WSTAGES;
      ptx::mbar_wait(bars + 8u * s, (count / N3_WSTAGES) & 1);
      ++count;
      const uint8_t *row = mine + s * stage_bytes;
      const N3Vec vl = n3_lds(row), vc = n3_lds(row + px_bytes), vr = n3_lds(row + 2 * px_bytes);
      N3Vec vg4 = {};  // dy row r+1 = i0+a (zeros once the tile's rows are exhausted)
      if (a < nrows) vg4 = n3_lds(row + xrow_stride);
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(bars + N3_WBAR + 8u * s);
      unpackv(vg4, gp);
      if (!active) return;
      float2 x[N3_PAIRS];
      unpackv(vl, x);
#pragma unroll
      for (int e = 0; e < N3_PAIRS; ++e) {
        acc[0][e] = ffma2(gp[e], x[e], acc[0][e]); acc[3][e] = ffma2(g0[e], x[e], acc[3][e]); acc[6][e] = ffma2(gm[e], x[e], acc[6][e]);
      }
      unpackv(vc, x);
#pragma unroll
      for (int e = 0; e < N3_PAIRS; ++e) {
        acc[1][e] = ffma2(gp[e], x[e], acc[1][e]); acc[4][e] = ffma2(g0[e], x[e], acc[4][e]); acc[7][e] = ffma2(gm[e], x[e], acc[7][e]);
      }
      unpackv(vr, x);
#pragma unroll
      for (int e = 0; e < N3_PAIRS; ++e) {
        acc[2][e] = ffma2(gp[e], x[e], acc[2][e]); acc[5][e] = ffma2(g0[e], x[e], acc[5][e]); acc[8][e] = ffma2(gm[e], x[e], acc[8][e]);
      }
    };
    float2 ga[N3_PAIRS], gb[N3_PAIRS], gc[N3_PAIRS];  // dy rows r-1, r, r+1 (roles rotate); rows outside the tile are zeros
#pragma unroll
    for (int e = 0; e < N3_PAIRS; ++e) ga[e] = gb[e] = gc[e] = make_float2(0.f, 0.f);
    for (int a = 0; a < arrivals; a += 3) {
      arrive(a, ga, gb, gc);
      if (a + 1 >= arrivals) break;
      arrive(a + 1, gb, gc, ga);
      if (a + 2 >= arrivals) break;
      arrive(a + 2, gc, ga, gb);
    }
  }
  // fixed-order sum over the CTA's N3_WARPS * Jb pixel columns, tap by tap
  float *out = p.part + (long)slot * 9 * p.C;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    __syncthreads();
#pragma unroll
    for (int e = 0; e < N3_PAIRS; ++e) {
      red[(warp * 32 + lane) * N3_CH + 2 * e] = acc[tap][e].x;
      red[(warp * 32 + lane) * N3_CH + 2 * e + 1] = acc[tap][e].y;
    }
    __syncthreads();
    // Vb * N3_CH channels to produce; each is summed over the N3_WARPS * Jb columns in (warp, column) order
    for (int i = threadIdx.x; i < p.Vb * N3_CH; i += N3_THREADS) {
      const int v = i / N3_CH, e = i % N3_CH;
      float sum = 0.f;
      for (int w = 0; w < N3_WARPS; ++w)
        for (int q = 0; q < p.Jb; ++q) sum += red[(w * 32 + q * p.Vb + v) * N3_CH + e];
      out[(long)tap * p.C + (vg * p.Vb + v) * N3_CH + e] = sum;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool dw_nhwc3_supported(int C, int k, int dil, int pad) {
  if (k != 3 || dil != 1 || pad != 1 || C % 8 != 0) return false;
  const int V = C / N3_CH;
  return V % 32 == 0 || V == 2 || V == 4 || V == 8 || V == 16;  // (V == 1 would need a TMA box wider than 256 columns)
}

static void n3_geometry(N3Params &p) {
  const int V = p.C / N3_CH;
  p.Vb = V >= 32 ? 32 : V;
  p.Jb = 32 / p.Vb;
  p.vgroups = V / p.Vb;
  p.tiles_h = ceil_div(p.H, N3_TH);
  p.tiles_w = ceil_div(p.W, N3_WARPS * p.Jb);
  const long tiles = (long)p.N * p.tiles_h * p.tiles_w;
  // every CTA must be resident at once (a second wave of persistent CTAs doubles the run time): round DOWN
  p.ctas_per_group = (int)max(1L, min(tiles, (long)(kNumSMs * N3_OCC / p.vgroups)));
}

static int n3_map(CUtensorMap *m, const void *base, const N3Params &p, int cols) {
  const uint64_t dims[4] = {(uint64_t)p.C, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.N};
  const uint64_t strides[3] = {(uint64_t)p.C * 2, (uint64_t)p.W * p.C * 2, (uint64_t)p.H * p.W * p.C * 2};
  const uint32_t box[4] = {(uint32_t)(p.Vb * N3_CH), (uint32_t)cols, 1, 1};
  return make_tmap_bf16(m, base, 4, dims, strides, box, nullptr, CU_TENSOR_MAP_SWIZZLE_NONE);
}

int dw_nhwc3_conv(const void *in, const float *w, const float *bias, void *out, int N, int H, int W, int C, int flip,
                  cudaStream_t st) {
  N3Params p{};
  p.out = static_cast<__nv_bfloat16 *>(out);
  p.w = w; p.bias = bias; p.N = N; p.H = H; p.W = W; p.C = C; p.flip = flip;
  n3_geometry(p);
  if ((long)N * H * W == 0) return KDCC_OK;
  p.dbg = tc_debug_bits();
  CUtensorMap tm;
  p.prefill = N3_STAGES - 1;
  int rc = n3_map(&tm, in, p, N3_WARPS * p.Jb + 2);
  if (rc) return rc;
  const int smem = N3_STAGES * (((N3_WARPS * p.Jb + 2) * p.Vb * N3_VB + 127) & ~127) + 2 * N3_BAR;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_nhwc3_conv_kernel, smem, attr_cache)) return e;
  launch_pdl(dw_nhwc3_conv_kernel, dim3(p.ctas_per_group * p.vgroups), dim3(N3_THREADS), (size_t)smem, st, tm, p);
  return launch_status();
}

int dw_nhwc3_wgrad_ctas(int N, int H, int W, int C) {
  N3Params p{};
  p.N = N; p.H = H; p.W = W; p.C = C;
  n3_geometry(p);
  return p.ctas_per_group;
}

int dw_nhwc3_wgrad(const void *x, const void *dy, float *dw, float *part, int N, int H, int W, int C, cudaStream_t st) {
  N3Params p{};
  p.part = part; p.N = N; p.H = H; p.W = W; p.C = C;
  n3_geometry(p);
  p.prefill = N3_WSTAGES - 1;
  CUtensorMap tm_x, tm_dy;
  int rc = n3_map(&tm_x, x, p, N3_WARPS * p.Jb + 2);
  if (rc) return rc;
  rc = n3_map(&tm_dy, dy, p, N3_WARPS * p.Jb);
  if (rc) return rc;
  const int smem = N3_WSTAGES * ((((N3_WARPS * p.Jb + 2) * p.Vb * N3_VB + 127) & ~127) + ((N3_WARPS * p.Jb * p.Vb * N3_VB + 127) & ~127)) + 2 * N3_WBAR +
                   N3_THREADS * N3_CH * (int)sizeof(float);
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_nhwc3_wgrad_kernel, smem, attr_cache)) return e;
  launch_pdl(dw_nhwc3_wgrad_kernel, dim3(p.ctas_per_group * p.vgroups), dim3(N3_THREADS), (size_t)smem, st, tm_x, tm_dy, p);
  rc = launch_status();
  if (rc) return rc;
  dw_wgrad_reduce_kernel<<<ceil_div(9 * C, 256), 256, 0, st>>>(part, dw, nullptr, p.ctas_per_group, C, 9, 9);
  return launch_status();
}

}  // namespace kdcc
