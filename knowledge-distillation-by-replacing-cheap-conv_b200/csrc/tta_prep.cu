// Test-time window preparation of inference_test, on the device (DESIGN.md 4.3h).
//
// Reference semantics: utils/tta_process.py:52-117 as models/students/depthwise_student.py:187-206 drives it, per image
// and scale: torchvision ToPILImage, PIL Image.resize((int(w * s), int(h * s)), BILINEAR), FLIP_LEFT_RIGHT, ToTensor +
// Normalize, then the overlapping window crops of the plain and of the mirrored image.  The windows written here are
// bit-identical to that host computation:
//   cast      ToPILImage's pic.mul(255).byte(): the product in the input dtype (bf16 rounds it to bf16), then truncate
//             toward zero to int32 and keep the low 8 bits; NaN, +-inf and values outside int32 -> 0
//   resize    Pillow's 8-bit two-pass resampler: horizontal pass into a uint8 image, then the vertical pass; a pass whose
//             size does not change is skipped.  Weights in double (precompute_coeffs, no FMA contraction: Pillow's
//             x86-64 build has none), fixed point with 22 fraction bits, accumulation from 1 << 21, >> 22, clamp to 0..255
//   mirror    pixel (y, x) of the mirrored image is (y, w - 1 - x) of the resized one
//   tensor    u / 255.f, then (. - mean_c) / std_c, each one fp32 IEEE operation: a 3 x 256 table per CTA
//   windows   tta.window_coordinates from the window index: stride given, x outer / y inner, the last window of an axis
//             pulled back inside; (th, tw) = (min(tile, h), min(tile, w))
//
// Up to three launches, no host synchronisation (graph-capturable):
//   1. tta_coeffs_kernel   fixed-point weights of every output column / row of the passes that run (skipped at scale 1)
//   2. tta_hpass_kernel    cast + horizontal pass into a (3, H, w) uint8 intermediate (only when w != W)
//   3. tta_windows_kernel  vertical pass (only when h != H) + mirror + normalise, one thread per window pixel and 3
//                          channels, written straight into the caller's (2n, 3, th, tw) block
#include "kdcc_common.cuh"

namespace kdcc {

constexpr int TTAP_THREADS = 256;
constexpr int TTAP_TW = 64, TTAP_TH = 32;  // window tile of one CTA of the window kernel: 64 columns x 4 row groups
constexpr int PIL_BITS = 22;               // Pillow's PRECISION_BITS for 8-bit images

// Pillow's bilinear_filter((x + xmin - center + 0.5) * ss)
__device__ __forceinline__ double pil_bilinear(int x, double center, double ss) {
  double t = __dmul_rn(__dadd_rn(__dsub_rn((double)x, center), 0.5), ss);
  if (t < 0.0) t = -t;
  return t < 1.0 ? __dsub_rn(1.0, t) : 0.0;
}

// Pillow's precompute_coeffs (BILINEAR, box 0..in) + normalize_coeffs_8bpc for output index xx: (xmin, taps) and the
// fixed-point weights of input pixels xmin .. xmin + taps - 1.  Every double operation is rounded on its own.
__device__ void pil_coeffs(int in, int out, int xx, int2 *bounds, int *k) {
  const double scale = __ddiv_rn((double)__int2float_rn(in), (double)out);  // Pillow's box is float
  const double fs = scale < 1.0 ? 1.0 : scale;                               // filterscale = support of the triangle
  const double ss = __ddiv_rn(1.0, fs);
  const double center = __dmul_rn((double)xx + 0.5, scale);
  int xmin = (int)__dadd_rn(__dsub_rn(center, fs), 0.5);
  if (xmin < 0) xmin = 0;
  int xmax = (int)__dadd_rn(__dadd_rn(center, fs), 0.5);
  if (xmax > in) xmax = in;
  xmax -= xmin;
  double ww = 0.0;
  for (int x = 0; x < xmax; ++x) ww = __dadd_rn(ww, pil_bilinear(x + xmin, center, ss));
  for (int x = 0; x < xmax; ++x) {
    double v = pil_bilinear(x + xmin, center, ss);
    if (ww != 0.0) v = __ddiv_rn(v, ww);
    const double f = __dmul_rn(v, (double)(1 << PIL_BITS));
    k[x] = v < 0.0 ? (int)__dadd_rn(-0.5, f) : (int)__dadd_rn(0.5, f);
  }
  *bounds = make_int2(xmin, xmax);
}

// ToPILImage's byte of one source element; the intermediate is bytes already
__device__ __forceinline__ int pil_byte(float v) { return cast_u8_like_numpy(__fmul_rn(v, 255.f)); }
__device__ __forceinline__ int pil_byte(__nv_bfloat16 v) {
  return cast_u8_like_numpy(__bfloat162float(__float2bfloat16_rn(__fmul_rn(__bfloat162float(v), 255.f))));
}
__device__ __forceinline__ int pil_byte(uint8_t v) { return v; }

__device__ __forceinline__ int pil_clip8(int s) { return min(max(s >> PIL_BITS, 0), 255); }

// one thread per output column of the horizontal pass (first nx threads) or output row of the vertical pass
__global__ void __launch_bounds__(TTAP_THREADS)
tta_coeffs_kernel(int in_x, int nx, int kx, int2 *bx, int *cx, int in_y, int ny, int ky, int2 *by, int *cy) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nx) pil_coeffs(in_x, nx, i, bx + i, cx + (long)i * kx);
  else if (i - nx < ny) pil_coeffs(in_y, ny, i - nx, by + (i - nx), cy + (long)(i - nx) * ky);
}

// tmp[c][y][xx] = horizontal pass of the cast image; 3 * H * w < 2^31
template <typename T>
__global__ void __launch_bounds__(TTAP_THREADS)
tta_hpass_kernel(const T *__restrict__ img, int H, int W, int w, const int2 *__restrict__ bounds,
                 const int *__restrict__ coef, int ksize, uint8_t *__restrict__ tmp) {
  const int total = H * w;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < total; p += gridDim.x * blockDim.x) {
    const int y = p / w, xx = p - y * w;
    const int2 b = __ldg(bounds + xx);
    const int *k = coef + (long)xx * ksize;
    int s[3] = {1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1)};
    for (int i = 0; i < b.y; ++i) {
      const int kv = __ldg(k + i);
#pragma unroll
      for (int c = 0; c < 3; ++c) s[c] += pil_byte(img[((long)c * H + y) * W + b.x + i]) * kv;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) tmp[(long)c * total + p] = (uint8_t)pil_clip8(s[c]);
  }
}

// out[k][c][ty][tx] for window k (the first n plain, the next n mirrored) from the (3, H, w) plane `src`: the cast image
// (S = float / bf16, no horizontal pass) or the horizontal pass's bytes (S = uint8_t); VPASS runs the vertical pass
// H -> h on the fly, else H == h.  One CTA: a 64 x 32 tile of one window.
template <typename S, bool VPASS>
__global__ void __launch_bounds__(TTAP_THREADS)
tta_windows_kernel(const S *__restrict__ src, int H, int h, int w, int tile, int stride, int ny, int n, int th, int tw,
                   int tiles_x, int tiles_y, const int2 *__restrict__ vb, const int *__restrict__ vk, int vksize,
                   float m0, float m1, float m2, float s0, float s1, float s2, float *__restrict__ out) {
  __shared__ float lut[3][256];
  for (int i = threadIdx.x; i < 3 * 256; i += TTAP_THREADS) {
    const int c = i >> 8;
    const float m = c == 0 ? m0 : (c == 1 ? m1 : m2), sd = c == 0 ? s0 : (c == 1 ? s1 : s2);
    lut[c][i & 255] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)(i & 255), 255.f), m), sd);
  }
  const int tiles = tiles_x * tiles_y;
  const int k = blockIdx.x / tiles, t = blockIdx.x - k * tiles;
  const int tx = (t % tiles_x) * TTAP_TW + (threadIdx.x % TTAP_TW), ty0 = (t / tiles_x) * TTAP_TH;
  const bool mirror = k >= n;
  const int j = mirror ? k - n : k, ix = j / ny, iy = j - ix * ny;
  const int x1 = (int)max(min((long)ix * stride + tile, (long)w) - tile, 0L);
  const int y1 = (int)max(min((long)iy * stride + tile, (long)h) - tile, 0L);
  __syncthreads();
  if (tx >= tw) return;
  const int xs = mirror ? w - 1 - (x1 + tx) : x1 + tx;
  const long plane = (long)H * w;
  for (int r = threadIdx.x / TTAP_TW; r < TTAP_TH; r += TTAP_THREADS / TTAP_TW) {
    const int ty = ty0 + r;
    if (ty >= th) break;
    const int y = y1 + ty;
    int u[3];
    if (VPASS) {
      const int2 b = __ldg(vb + y);
      const int *kk = vk + (long)y * vksize;
      int s[3] = {1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1), 1 << (PIL_BITS - 1)};
      for (int i = 0; i < b.y; ++i) {
        const int kv = __ldg(kk + i);
        const long e = (long)(b.x + i) * w + xs;
#pragma unroll
        for (int c = 0; c < 3; ++c) s[c] += pil_byte(src[c * plane + e]) * kv;
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) u[c] = pil_clip8(s[c]);
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) u[c] = pil_byte(src[c * plane + (long)y * w + xs]);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) out[(((long)k * 3 + c) * th + ty) * tw + tx] = lut[c][u[c]];
  }
}

// Pillow's coefficient row length: (int)ceil(support) * 2 + 1, an upper bound of the taps of every output index
static int pil_ksize(int in, int out) {
  const double scale = (double)(float)in / out;
  return (int)ceil(scale < 1.0 ? 1.0 : scale) * 2 + 1;
}

// workspace: [uint8 intermediate (3, H, w)] [horizontal bounds, weights] [vertical bounds, weights], each 256-aligned;
// a part whose pass is skipped has size 0
struct PrepLayout {
  size_t tmp, hb, hk, vb, vk, total;
  int kx, ky;
};

static PrepLayout prep_layout(int H, int W, int h, int w) {
  PrepLayout L = {};
  const bool hpass = w != W, vpass = h != H;
  L.kx = hpass ? pil_ksize(W, w) : 0;
  L.ky = vpass ? pil_ksize(H, h) : 0;
  size_t off = 0;
  auto take = [&off](size_t bytes) {
    const size_t at = off;
    off = (off + bytes + 255) & ~(size_t)255;
    return at;
  };
  L.tmp = take(hpass ? (size_t)3 * H * w : 0);
  L.hb = take(hpass ? (size_t)w * sizeof(int2) : 0);
  L.hk = take(hpass ? (size_t)w * L.kx * sizeof(int) : 0);
  L.vb = take(vpass ? (size_t)h * sizeof(int2) : 0);
  L.vk = take(vpass ? (size_t)h * L.ky * sizeof(int) : 0);
  L.total = off;
  return L;
}

// ceil((size - tile) / stride) + 1 as tta.window_coordinates computes it; <= 0 when the tile overhangs by a stride or more
static long window_count(long size, long tile, long stride) {
  const long d = size - tile;
  return (d >= 0 ? (d + stride - 1) / stride : -(-d / stride)) + 1;
}

template <typename S, bool VPASS>
static void launch_windows(const void *src, int H, int h, int w, int tile, int stride, int ny, int n, int th, int tw,
                           const int2 *vb, const int *vk, int vksize, const float (&ms)[6], float *out, cudaStream_t st) {
  const int tiles_x = ceil_div(tw, TTAP_TW), tiles_y = ceil_div(th, TTAP_TH);
  const long grid = 2L * n * tiles_x * tiles_y;  // <= 2n * th * tw < 2^31
  tta_windows_kernel<S, VPASS><<<(unsigned)grid, TTAP_THREADS, 0, st>>>(
      static_cast<const S *>(src), H, h, w, tile, stride, ny, n, th, tw, tiles_x, tiles_y, vb, vk, vksize, ms[0], ms[1],
      ms[2], ms[3], ms[4], ms[5], out);
}

template <typename T>
static void launch_prep(const void *img, int H, int W, int h, int w, int tile, int stride, int ny, int n, int th, int tw,
                        const float (&ms)[6], float *out, uint8_t *ws, const PrepLayout &L, cudaStream_t st) {
  const bool hpass = w != W, vpass = h != H;
  int2 *hb = reinterpret_cast<int2 *>(ws + L.hb), *vb = reinterpret_cast<int2 *>(ws + L.vb);
  int *hk = reinterpret_cast<int *>(ws + L.hk), *vk = reinterpret_cast<int *>(ws + L.vk);
  if (hpass || vpass) {
    const int nx = hpass ? w : 0, nyc = vpass ? h : 0;
    tta_coeffs_kernel<<<ceil_div(nx + nyc, TTAP_THREADS), TTAP_THREADS, 0, st>>>(W, nx, L.kx, hb, hk, H, nyc, L.ky, vb, vk);
  }
  if (hpass) {
    const int grid = (int)min((long)kNumSMs * 16, ceil_div<long>((long)H * w, TTAP_THREADS));
    tta_hpass_kernel<T><<<grid, TTAP_THREADS, 0, st>>>(static_cast<const T *>(img), H, W, w, hb, hk, L.kx, ws + L.tmp);
    if (vpass) launch_windows<uint8_t, true>(ws + L.tmp, H, h, w, tile, stride, ny, n, th, tw, vb, vk, L.ky, ms, out, st);
    else launch_windows<uint8_t, false>(ws + L.tmp, H, h, w, tile, stride, ny, n, th, tw, vb, vk, 0, ms, out, st);
  } else {
    if (vpass) launch_windows<T, true>(img, H, h, w, tile, stride, ny, n, th, tw, vb, vk, L.ky, ms, out, st);
    else launch_windows<T, false>(img, H, h, w, tile, stride, ny, n, th, tw, vb, vk, 0, ms, out, st);
  }
}

}  // namespace kdcc

using namespace kdcc;

KDCC_API size_t kdcc_tta_windows_workspace_bytes(int H, int W, int h, int w) {
  if (H <= 0 || W <= 0 || h <= 0 || w <= 0) return 0;
  return prep_layout(H, W, h, w).total;
}

KDCC_API int kdcc_tta_windows(const void *img, int H, int W, int dtype, int h, int w, int tile, int stride, float m0,
                              float m1, float m2, float s0, float s1, float s2, float *out, void *workspace,
                              size_t workspace_bytes, kdcc_stream_t stream) {
  if (!img || !out || H <= 0 || W <= 0 || h <= 0 || w <= 0 || tile < 1 || stride < 1) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16) return KDCC_EINVAL;
  const long lim = 1L << 31;
  if (3L * H * W >= lim || 3L * h * w >= lim || 3L * H * w >= lim) return KDCC_ESHAPE;
  const long nx = window_count(w, tile, stride), ny = window_count(h, tile, stride);
  const long n = nx > 0 && ny > 0 ? nx * ny : 0;  // <= w * h
  const int th = min(tile, h), tw = min(tile, w);
  if (2L * n * 3 * th * tw >= lim) return KDCC_ESHAPE;
  const PrepLayout L = prep_layout(H, W, h, w);
  if (L.total > 0 && !workspace) return KDCC_EINVAL;
  if (workspace_bytes < L.total) return KDCC_EWORKSPACE;
  if (n == 0) return KDCC_OK;  // the reference's formula gives no window: nothing to write

  const float ms[6] = {m0, m1, m2, s0, s1, s2};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t *ws = static_cast<uint8_t *>(workspace);
  if (dtype == KDCC_F32)
    launch_prep<float>(img, H, W, h, w, tile, stride, (int)ny, (int)n, th, tw, ms, out, ws, L, st);
  else
    launch_prep<__nv_bfloat16>(img, H, W, h, w, tile, stride, (int)ny, (int)n, th, tw, ms, out, ws, L, st);
  return launch_status();
}
