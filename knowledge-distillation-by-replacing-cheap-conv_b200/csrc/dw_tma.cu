// Depthwise k x k convolution for sm_100a, bf16 NHWC, TMA-staged.
//
// Reference semantics: models/students/transform_blocks/depthwise_separable_conv.py:7-8,12 and its
// autograd backward (input gradient = the same kernel run on dy with mirrored taps; weight gradient =
// dw_tma_wgrad_kernel).
//
// Design (see DESIGN.md "depthwise"):
//  * A dilated depthwise conv splits into dil*dil independent DENSE k x k convs on the sub-images
//    {x[ri + a*dil][rj + b*dil]}.  One CTA tile = one (image, row residue, col residue, channel block)
//    sub-image tile.  TMA's element strides fetch exactly that sub-image (traversal stride = dil) and
//    its out-of-bounds zero fill IS the conv padding, so the halo costs no HBM traffic and there is no
//    read amplification: every input element is fetched by exactly one CTA.
//  * Persistent CTAs, two landing stages: the TMA load of tile i+1/i+2 overlaps the FMA work of tile i.
//  * The landing tile (bf16) is widened once to an fp32 smem tile; the inner loop is then LDS.64 + FFMA
//    with a register sliding window: T outputs per thread reuse each loaded input K times, so the
//    k=9 case (81 MAC per output, FFMA-bound, not HBM-bound) runs at ~85 % FFMA issue density.
//  * Results go back through a bf16 smem tile and one strided TMA store (out-of-range rows/cols are
//    clipped by the hardware).
//  * Weight gradient: same staging for x, dy read straight from its bf16 landing tile; each thread owns
//    (channel pair, tap row u) and keeps K x 2 partial sums in registers across ALL the tiles of its
//    CTA; cross-thread / cross-CTA reduction is a fixed-order two-stage sum (deterministic, no atomics).
#include "dw_kernels.cuh"
#include "sm100_ptx.cuh"

namespace kdcc {

__host__ __device__ constexpr int align128(int v) { return (v + 127) / 128 * 128; }

template <int K_, int TH_, int TW_, int T_, int CB_, int RG_, int OCC_>
struct DwCfg {
  static constexpr int K = K_, TH = TH_, TW = TW_, T = T_, CB = CB_, RG = RG_, OCC = OCC_;
  static constexpr int CP = CB / 2;          // channel pairs (one bf16x2 word / one float2)
  static constexpr int IH = TH + K - 1, IW = TW + K - 1;
  static constexpr int STRIPS = TW / T;
  static_assert(TW % T == 0, "strip width must divide the tile width");
  static_assert(CP == 8, "lane mapping assumes 8 channel pairs per pixel");
  // fp32 tile: pixel pitch CB floats, row pitch padded to 16 (mod 32) words so that the two rows a
  // half-warp touches with LDS.64 fall into disjoint bank halves
  static constexpr int ROWP = IW * CB + ((IW * CB) % 32 == 16 ? 0 : 16);
  static constexpr int LAND_BYTES = IH * IW * CB * 2;
  static constexpr int F32_BYTES = IH * ROWP * 4;
  static constexpr int OUT_BYTES = TH * TW * CB * 2;
  static constexpr int W_BYTES = (K * K + 1) * CB * 4;  // taps + bias row
  // conv kernel
  static constexpr int CONV_TASKS = CP * TH * STRIPS;
  static constexpr int CONV_NT = (CONV_TASKS + 31) / 32 * 32;
  static constexpr int CONV_OFF_F32 = 2 * align128(LAND_BYTES);
  static constexpr int CONV_OFF_OUT = CONV_OFF_F32 + align128(F32_BYTES);
  static constexpr int CONV_OFF_W = CONV_OFF_OUT + align128(OUT_BYTES);
  static constexpr int CONV_OFF_BAR = CONV_OFF_W + align128(W_BYTES);
  static constexpr int CONV_SMEM = CONV_OFF_BAR + 64;
  // wgrad kernel
  static constexpr int WG_TASKS = CP * K * STRIPS * RG;
  static constexpr int WG_NT = (WG_TASKS + 31) / 32 * 32;
  static constexpr int WG_OFF_DY = 2 * align128(LAND_BYTES);
  static constexpr int WG_OFF_F32 = WG_OFF_DY + 2 * align128(OUT_BYTES);
  static constexpr int WG_RED_BYTES = STRIPS * RG * K * K * CB * 4;
  static constexpr int WG_F32_REGION = F32_BYTES > WG_RED_BYTES ? F32_BYTES : WG_RED_BYTES;
  static constexpr int WG_OFF_BAR = WG_OFF_F32 + align128(WG_F32_REGION);
  static constexpr int WG_SMEM = WG_OFF_BAR + 64;
};

//                    K  TH  TW   T  CB RG OCC
using Cfg9 = DwCfg<9, 26, 26, 13, 16, 3, 1>;  // Cityscapes cfgs: k=9, dil=5, pad=20 on 128x128 -> 26x26 sub-images
using Cfg3 = DwCfg<3, 16, 32, 8, 16, 4, 2>;   // CIFAR / north-star 3x3

struct DwTmaParams {
  int N, C, dil, pad, flip;
  int tiles_h, tiles_w, ncb;
  long total;  // conv: all tiles; wgrad: spatial tiles (without the channel-block factor)
  int splits;  // wgrad: CTAs per channel block
  const float *w, *bias;
  float *part;
};

struct TileCoord {
  int n, i0, j0, cb;
};

template <class Cfg>
__device__ __forceinline__ TileCoord decode_tile(const DwTmaParams &p, long tile, bool with_cb) {
  TileCoord t;
  if (with_cb) { t.cb = (int)(tile % p.ncb); tile /= p.ncb; } else { t.cb = 0; }
  const int tb = (int)(tile % p.tiles_w); tile /= p.tiles_w;
  const int ta = (int)(tile % p.tiles_h); tile /= p.tiles_h;
  const int rj = (int)(tile % p.dil); tile /= p.dil;
  const int ri = (int)(tile % p.dil);
  t.n = (int)(tile / p.dil);
  t.i0 = ta * Cfg::TH * p.dil + ri;
  t.j0 = tb * Cfg::TW * p.dil + rj;
  return t;
}

// bf16 landing tile [IH][IW][CB] -> fp32 tile [IH][ROWP]
template <class Cfg, int NT>
__device__ __forceinline__ void widen_tile(const uint8_t *land, float *f32, int tid) {
  constexpr int CHUNKS = Cfg::IH * Cfg::IW * (Cfg::CB / 8);
  for (int i = tid; i < CHUNKS; i += NT) {
    const uint4 raw = *reinterpret_cast<const uint4 *>(land + (size_t)i * 16);
    const int px = i / (Cfg::CB / 8), ch = i % (Cfg::CB / 8);
    const int r = px / Cfg::IW, c = px % Cfg::IW;
    float *dst = f32 + r * Cfg::ROWP + c * Cfg::CB + ch * 8;
    *reinterpret_cast<float4 *>(dst) = make_float4(bf16lo(raw.x), bf16hi(raw.x), bf16lo(raw.y), bf16hi(raw.y));
    *reinterpret_cast<float4 *>(dst + 4) = make_float4(bf16lo(raw.z), bf16hi(raw.z), bf16lo(raw.w), bf16hi(raw.w));
  }
}

// ------------------------------------------------------------------------------------------------
// forward / input-gradient kernel
// ------------------------------------------------------------------------------------------------
template <class Cfg>
__global__ void __launch_bounds__(Cfg::CONV_NT, Cfg::OCC)
dw_tma_conv_kernel(const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out,
                   const DwTmaParams p) {
  constexpr int K = Cfg::K, T = Cfg::T, CB = Cfg::CB, CP = Cfg::CP, NT = Cfg::CONV_NT;
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t *land[2] = {smem, smem + align128(Cfg::LAND_BYTES)};
  float *f32 = reinterpret_cast<float *>(smem + Cfg::CONV_OFF_F32);
  uint32_t *outs = reinterpret_cast<uint32_t *>(smem + Cfg::CONV_OFF_OUT);
  float *wsm = reinterpret_cast<float *>(smem + Cfg::CONV_OFF_W);
  const uint32_t bar0 = ptx::smem_u32(smem + Cfg::CONV_OFF_BAR);
  const int tid = threadIdx.x;

  if (tid == 0) {
    ptx::mbar_init(bar0, 1);
    ptx::mbar_init(bar0 + 8, 1);
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_in);
    ptx::prefetch_tensormap(&tm_out);
  }
  __syncthreads();

  auto issue_load = [&](long tile, int stage) {
    const TileCoord tc = decode_tile<Cfg>(p, tile, true);
    const uint32_t bar = bar0 + 8 * stage;
    ptx::mbar_arrive_expect_tx(bar, Cfg::LAND_BYTES);
    ptx::tma_load_4d(ptx::smem_u32(land[stage]), &tm_in, bar, tc.cb * CB, tc.j0 - p.pad, tc.i0 - p.pad, tc.n);
  };
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      const long tile = (long)blockIdx.x + (long)s * gridDim.x;
      if (tile < p.total) issue_load(tile, s);
    }
  }

  // this thread's share of a tile: channel pair, output row, strip of T consecutive outputs
  const int cp = tid % CP;
  const int orow = (tid / CP) % Cfg::TH;
  const int strip = tid / (CP * Cfg::TH);
  const bool worker = tid < Cfg::CONV_TASKS;

  int it = 0;
  for (long tile = blockIdx.x; tile < p.total; tile += gridDim.x, ++it) {
    const int st = it & 1;
    const uint32_t phase = (it >> 1) & 1;
    const TileCoord tc = decode_tile<Cfg>(p, tile, true);

    // taps of this channel block: wsm[tap][c] (mirrored for the input-gradient form), bias row last
    for (int i = tid; i < (K * K + 1) * CB; i += NT) {
      const int tap = i / CB, c = i % CB;
      float v;
      if (tap < K * K) v = __ldg(p.w + (long)(tc.cb * CB + c) * (K * K) + (p.flip ? K * K - 1 - tap : tap));
      else v = p.bias ? __ldg(p.bias + tc.cb * CB + c) : 0.f;
      wsm[i] = v;
    }
    ptx::mbar_wait(bar0 + 8 * st, phase);
    widen_tile<Cfg, NT>(land[st], f32, tid);
    if (tid == 0) ptx::tma_store_wait_read();  // the previous tile's store has drained the out tile
    __syncthreads();

    if (worker) {
      float acc[T][2];
      {
        const float2 b = *reinterpret_cast<const float2 *>(wsm + K * K * CB + 2 * cp);
#pragma unroll
        for (int t = 0; t < T; ++t) { acc[t][0] = b.x; acc[t][1] = b.y; }
      }
      const float *xrow = f32 + orow * Cfg::ROWP + strip * T * CB + 2 * cp;
#pragma unroll 1
      for (int u = 0; u < K; ++u) {
        float2 wv[K];
#pragma unroll
        for (int v = 0; v < K; ++v) wv[v] = *reinterpret_cast<const float2 *>(wsm + (u * K + v) * CB + 2 * cp);
        const float *xr = xrow + u * Cfg::ROWP;
#pragma unroll
        for (int m = 0; m < T + K - 1; ++m) {
          const float2 xv = *reinterpret_cast<const float2 *>(xr + m * CB);
#pragma unroll
          for (int v = 0; v < K; ++v) {
            const int t = m - v;
            if (t >= 0 && t < T) {
              acc[t][0] = fmaf(wv[v].x, xv.x, acc[t][0]);
              acc[t][1] = fmaf(wv[v].y, xv.y, acc[t][1]);
            }
          }
        }
      }
      uint32_t *orow_ptr = outs + (orow * Cfg::TW + strip * T) * CP + cp;
#pragma unroll
      for (int t = 0; t < T; ++t) orow_ptr[t * CP] = pack_bf16x2(acc[t][0], acc[t][1]);
    }
    ptx::fence_proxy_async_smem();
    __syncthreads();

    if (tid == 0) {
      ptx::tma_store_4d(&tm_out, ptx::smem_u32(outs), tc.cb * CB, tc.j0, tc.i0, tc.n);
      ptx::tma_store_commit();
      const long next = tile + 2L * gridDim.x;
      if (next < p.total) issue_load(next, st);
    }
  }
  if (tid == 0) ptx::tma_store_wait_all();
}

// ------------------------------------------------------------------------------------------------
// weight-gradient kernel: part[split][tap][c] = sum over this CTA's tiles of dy * shifted x
// ------------------------------------------------------------------------------------------------
template <class Cfg>
__global__ void __launch_bounds__(Cfg::WG_NT, Cfg::OCC)
dw_tma_wgrad_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_dy,
                    const DwTmaParams p) {
  constexpr int K = Cfg::K, T = Cfg::T, CB = Cfg::CB, CP = Cfg::CP, NT = Cfg::WG_NT;
  constexpr int STRIPS = Cfg::STRIPS, RG = Cfg::RG;
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t *landx[2] = {smem, smem + align128(Cfg::LAND_BYTES)};
  uint8_t *landg[2] = {smem + Cfg::WG_OFF_DY, smem + Cfg::WG_OFF_DY + align128(Cfg::OUT_BYTES)};
  float *f32 = reinterpret_cast<float *>(smem + Cfg::WG_OFF_F32);
  const uint32_t bar0 = ptx::smem_u32(smem + Cfg::WG_OFF_BAR);
  const int tid = threadIdx.x;
  const int cb = blockIdx.x % p.ncb;
  const int split = blockIdx.x / p.ncb;

  if (tid == 0) {
    ptx::mbar_init(bar0, 1);
    ptx::mbar_init(bar0 + 8, 1);
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tm_x);
    ptx::prefetch_tensormap(&tm_dy);
  }
  __syncthreads();

  auto issue_load = [&](long tile, int stage) {
    const TileCoord tc = decode_tile<Cfg>(p, tile, false);
    const uint32_t bar = bar0 + 8 * stage;
    ptx::mbar_arrive_expect_tx(bar, Cfg::LAND_BYTES + Cfg::OUT_BYTES);
    ptx::tma_load_4d(ptx::smem_u32(landx[stage]), &tm_x, bar, cb * CB, tc.j0 - p.pad, tc.i0 - p.pad, tc.n);
    ptx::tma_load_4d(ptx::smem_u32(landg[stage]), &tm_dy, bar, cb * CB, tc.j0, tc.i0, tc.n);
  };
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      const long tile = (long)split + (long)s * p.splits;
      if (tile < p.total) issue_load(tile, s);
    }
  }

  // task: channel pair, tap row u, strip, row group
  const int cp = tid % CP;
  const int u = (tid / CP) % K;
  const int strip = (tid / (CP * K)) % STRIPS;
  const int rg = tid / (CP * K * STRIPS);
  const bool worker = tid < Cfg::WG_TASKS;
  constexpr int ROWS_PER = (Cfg::TH + RG - 1) / RG;
  const int rb = rg * ROWS_PER;
  const int re = min(Cfg::TH, rb + ROWS_PER);

  float acc[K][2];
#pragma unroll
  for (int v = 0; v < K; ++v) acc[v][0] = acc[v][1] = 0.f;

  int it = 0;
  for (long tile = split; tile < p.total; tile += p.splits, ++it) {
    const int st = it & 1;
    const uint32_t phase = (it >> 1) & 1;
    ptx::mbar_wait(bar0 + 8 * st, phase);
    widen_tile<Cfg, NT>(landx[st], f32, tid);
    __syncthreads();

    if (worker) {
      const uint32_t *gbase = reinterpret_cast<const uint32_t *>(landg[st]) + strip * T * CP + cp;
      const float *xbase = f32 + u * Cfg::ROWP + strip * T * CB + 2 * cp;
#pragma unroll 1
      for (int r = rb; r < re; ++r) {
        float g[T][2];
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const uint32_t wd = gbase[(r * Cfg::TW + t) * CP];
          g[t][0] = bf16lo(wd);
          g[t][1] = bf16hi(wd);
        }
        const float *xr = xbase + r * Cfg::ROWP;
#pragma unroll
        for (int m = 0; m < T + K - 1; ++m) {
          const float2 xv = *reinterpret_cast<const float2 *>(xr + m * CB);
#pragma unroll
          for (int v = 0; v < K; ++v) {
            const int t = m - v;
            if (t >= 0 && t < T) {
              acc[v][0] = fmaf(g[t][0], xv.x, acc[v][0]);
              acc[v][1] = fmaf(g[t][1], xv.y, acc[v][1]);
            }
          }
        }
      }
    }
    __syncthreads();
    if (tid == 0) {
      const long next = tile + 2L * p.splits;
      if (next < p.total) issue_load(next, st);
    }
  }

  // fixed-order reduction over the STRIPS*RG threads that share (cp, u), then one store per (tap, c)
  float *red = f32;  // [STRIPS*RG][K*K][CB]
  if (worker) {
    float *dst = red + ((rg * STRIPS + strip) * K * K + u * K) * CB + 2 * cp;
#pragma unroll
    for (int v = 0; v < K; ++v) *reinterpret_cast<float2 *>(dst + v * CB) = make_float2(acc[v][0], acc[v][1]);
  }
  __syncthreads();
  for (int o = tid; o < K * K * CB; o += NT) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < STRIPS * RG; ++q) s += red[q * K * K * CB + o];
    const int tap = o / CB, c = o % CB;
    p.part[((long)split * (K * K) + tap) * p.C + cb * CB + c] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// 4-D map over an NHWC bf16 tensor; box = (CB, cols*dil, rows*dil, 1) traversed with stride dil
static int nhwc_map(CUtensorMap *m, const void *base, int N, int H, int W, int C, int cb, int rows, int cols, int dil) {
  const uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
  const uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)W * C * 2, (uint64_t)H * W * C * 2};
  const uint32_t box[4] = {(uint32_t)cb, (uint32_t)(cols * dil), (uint32_t)(rows * dil), 1};
  const uint32_t es[4] = {1, (uint32_t)dil, (uint32_t)dil, 1};
  return make_tmap_bf16(m, base, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_NONE);
}

template <class Cfg>
static bool cfg_fits(int dil) {
  return Cfg::IW * dil <= 256 && Cfg::IH * dil <= 256 && dil <= 8;
}

bool dw_tma_supported(int C, int k, int dil) {
  if (C % 16 != 0 || dil < 1) return false;
  if (k == 9) return cfg_fits<Cfg9>(dil);
  if (k == 3) return cfg_fits<Cfg3>(dil);
  return false;
}

const char *dw_tma_name(int k, int dil, int which) {
  (void)dil;
  if (k == 9) return which ? "dw_wgrad_tma_k9" : "dw_conv_tma_k9";
  return which ? "dw_wgrad_tma_k3" : "dw_conv_tma_k3";
}

template <class Cfg>
static void fill_geometry(DwTmaParams &p, int N, int C, int Ho, int Wo, int dil, int pad) {
  p.N = N; p.C = C; p.dil = dil; p.pad = pad;
  p.tiles_h = ceil_div(ceil_div(Ho, dil), Cfg::TH);
  p.tiles_w = ceil_div(ceil_div(Wo, dil), Cfg::TW);
  p.ncb = C / Cfg::CB;
}

template <class Cfg>
static int conv_launch(const void *in, const float *w, const float *bias, void *out, int N, int Hi, int Wi, int C,
                       int Ho, int Wo, int dil, int pad, int flip, cudaStream_t st) {
  DwTmaParams p{};
  fill_geometry<Cfg>(p, N, C, Ho, Wo, dil, pad);
  p.flip = flip; p.w = w; p.bias = bias;
  p.total = (long)N * dil * dil * p.tiles_h * p.tiles_w * p.ncb;
  if (p.total == 0) return KDCC_OK;
  CUtensorMap tm_in, tm_out;
  int rc = nhwc_map(&tm_in, in, N, Hi, Wi, C, Cfg::CB, Cfg::IH, Cfg::IW, dil);
  if (rc) return rc;
  rc = nhwc_map(&tm_out, out, N, Ho, Wo, C, Cfg::CB, Cfg::TH, Cfg::TW, dil);
  if (rc) return rc;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tma_conv_kernel<Cfg>, Cfg::CONV_SMEM, attr_cache)) return e;
  const int grid = (int)min(p.total, (long)kNumSMs * Cfg::OCC);
  dw_tma_conv_kernel<Cfg><<<grid, Cfg::CONV_NT, Cfg::CONV_SMEM, st>>>(tm_in, tm_out, p);
  return launch_status();
}

int dw_tma_conv(const void *in, const float *w, const float *bias, void *out, int N, int Hi, int Wi, int C, int Ho,
                int Wo, int k, int dil, int pad, int flip, cudaStream_t st) {
  if (k == 9) return conv_launch<Cfg9>(in, w, bias, out, N, Hi, Wi, C, Ho, Wo, dil, pad, flip, st);
  if (k == 3) return conv_launch<Cfg3>(in, w, bias, out, N, Hi, Wi, C, Ho, Wo, dil, pad, flip, st);
  return KDCC_ESHAPE;
}

template <class Cfg>
static int wgrad_splits(int N, int Ho, int Wo, int C, int dil) {
  const long spatial = (long)N * dil * dil * ceil_div(ceil_div(Ho, dil), Cfg::TH) * ceil_div(ceil_div(Wo, dil), Cfg::TW);
  const int ncb = C / Cfg::CB;
  long want = ceil_div<long>(2L * kNumSMs * Cfg::OCC, ncb);  // about two waves of CTAs
  return (int)max(1L, min(want, spatial));
}

int dw_tma_wgrad_splits(int N, int Ho, int Wo, int C, int k, int dil) {
  return k == 9 ? wgrad_splits<Cfg9>(N, Ho, Wo, C, dil) : wgrad_splits<Cfg3>(N, Ho, Wo, C, dil);
}

template <class Cfg>
static int wgrad_launch(const void *x, const void *dy, float *dw, float *part, int N, int H, int W, int C, int Ho,
                        int Wo, int dil, int pad, cudaStream_t st) {
  DwTmaParams p{};
  fill_geometry<Cfg>(p, N, C, Ho, Wo, dil, pad);
  p.part = part;
  p.total = (long)N * dil * dil * p.tiles_h * p.tiles_w;
  p.splits = wgrad_splits<Cfg>(N, Ho, Wo, C, dil);
  CUtensorMap tm_x, tm_dy;
  int rc = nhwc_map(&tm_x, x, N, H, W, C, Cfg::CB, Cfg::IH, Cfg::IW, dil);
  if (rc) return rc;
  rc = nhwc_map(&tm_dy, dy, N, Ho, Wo, C, Cfg::CB, Cfg::TH, Cfg::TW, dil);
  if (rc) return rc;
  static int attr_cache[16] = {0};
  if (int e = ensure_dynamic_smem(dw_tma_wgrad_kernel<Cfg>, Cfg::WG_SMEM, attr_cache)) return e;
  dw_tma_wgrad_kernel<Cfg><<<p.ncb * p.splits, Cfg::WG_NT, Cfg::WG_SMEM, st>>>(tm_x, tm_dy, p);
  rc = launch_status();
  if (rc) return rc;
  constexpr int KK = Cfg::K * Cfg::K;
  dw_wgrad_reduce_kernel<<<ceil_div(KK * C, 256), 256, 0, st>>>(part, dw, nullptr, p.splits, C, KK, KK);
  return launch_status();
}

int dw_tma_wgrad(const void *x, const void *dy, float *dw, float *part, int N, int H, int W, int C, int Ho, int Wo,
                 int k, int dil, int pad, cudaStream_t st) {
  if (k == 9) return wgrad_launch<Cfg9>(x, dy, dw, part, N, H, W, C, Ho, Wo, dil, pad, st);
  if (k == 3) return wgrad_launch<Cfg3>(x, dy, dw, part, N, H, W, C, Ho, Wo, dil, pad, st);
  return KDCC_ESHAPE;
}

}  // namespace kdcc
