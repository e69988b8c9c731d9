// Canny edge map of the Gated-SCNN forward, on the device (DESIGN.md 4.3f).
//
// Reference semantics: models/gscnn/gscnn.py:284-288 casts the (N, 3, H, W) image to uint8 the way numpy's astype does,
// runs cv2.Canny(img, low, high) (aperture 3, L1 gradient) per image on the host and copies the 0 / 255 map back.  The
// result here is bit-identical to that map:
//   cast    trunc toward zero to int32, keep the low 8 bits; NaN, +-inf and values whose truncation leaves int32 -> 0
//   Sobel   3x3 per channel in integers, BORDER_REPLICATE; m = |dx| + |dy|; per pixel the channel of largest m wins
//           (first channel on a tie) and gives the direction
//   NMS     cv2's integer tan(22.5) / tan(67.5) sectors; neighbours outside the image have m = 0
//   hyst.   output 255 at every candidate (m > low, NMS passed) whose 8-connected component of candidates contains a
//           strong candidate (m > high)
//
// Four launches whatever the content, no host synchronisation (graph-capturable):
//   1. canny_tile_kernel   one CTA per 16 x 128 output tile: cast, Sobel, NMS, and a union-find of the tile's candidates
//                          in shared memory; writes label = global index of the tile-local root (-1: no candidate) and
//                          flag = 1 at a local root whose tile-local component holds a strong candidate
//   2. canny_merge_kernel  tile-perimeter candidates union with their 8-neighbours in other tiles (lock-free atomicMin
//                          union, the larger root is linked under the smaller: roots end as the component's minimum index)
//   3. canny_root_kernel   every candidate's label is replaced by its final root; flagged local roots flag that root
//   4. canny_output_kernel 255.f where the pixel's root is flagged, else 0.f
// Hysteresis is thus exact for components of any shape and extent: no sweep count bounds how far a weak edge may wind.
#include "kdcc_common.cuh"

namespace kdcc {

constexpr int CANNY_TH = 16, CANNY_TW = 128;  // output tile
constexpr int CANNY_THREADS = 256;
constexpr int CANNY_IH = CANNY_TH + 4, CANNY_IW = CANNY_TW + 4;  // staged uint8 input: tile + 2-pixel halo
constexpr int CANNY_RH = CANNY_TH + 2, CANNY_RW = CANNY_TW + 2;  // magnitudes: tile + 1-pixel ring
constexpr int CANNY_TG22 = 13573;                                // round(tan(22.5 deg) * 2^15), as cv2
constexpr int CANNY_PERIM = CANNY_TW + 2 * (CANNY_TH - 1);       // top row + left and right columns below it

__device__ __forceinline__ float load_f32(const float *p, long i) { return __ldg(p + i); }
__device__ __forceinline__ float load_f32(const __nv_bfloat16 *p, long i) { return __bfloat162float(p[i]); }

// root of x: labels only ever decrease towards an index of the same component, so a stale read just walks further
__device__ __forceinline__ int uf_find(const volatile int *L, int x) {
  int y;
  while ((y = L[x]) != x) x = y;
  return x;
}

// link the larger of the two roots under the smaller; retry while another thread re-linked the root first
__device__ __forceinline__ void uf_union(int *L, int a, int b) {
  const volatile int *V = L;
  while (true) {
    a = uf_find(V, a);
    b = uf_find(V, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(L + b, a);
    if (old == b) return;
    b = old;
  }
}

template <typename T, bool NHWC>
__global__ void __launch_bounds__(CANNY_THREADS)
canny_tile_kernel(const T *__restrict__ img, int *__restrict__ labels, uint8_t *__restrict__ flags, int H, int W, int lo,
                  int hi) {
  __shared__ uint8_t px[3][CANNY_IH][CANNY_IW];
  __shared__ int mag[CANNY_RH][CANNY_RW];
  __shared__ int dxy[CANNY_TH][CANNY_TW];  // (dx << 16) | (dy & 0xffff) of the winning channel
  __shared__ int lab[CANNY_TH * CANNY_TW];
  __shared__ int strong_root[CANNY_TH * CANNY_TW];

  const int tiles_x = (W + CANNY_TW - 1) / CANNY_TW, tiles_y = (H + CANNY_TH - 1) / CANNY_TH;
  const int n = blockIdx.x / (tiles_x * tiles_y);
  const int y0 = (blockIdx.x / tiles_x) % tiles_y * CANNY_TH, x0 = blockIdx.x % tiles_x * CANNY_TW;
  const int tid = threadIdx.x;

  // 1. stage the tile + halo as uint8, rows / columns clamped into the image (BORDER_REPLICATE)
  for (int i = tid; i < 3 * CANNY_IH * CANNY_IW; i += CANNY_THREADS) {
    int c, r, x;
    if (NHWC) {  // channel fastest: a row of the tile is one contiguous run of 3-element pixels
      c = i % 3;
      x = (i / 3) % CANNY_IW;
      r = i / (3 * CANNY_IW);
    } else {
      x = i % CANNY_IW;
      r = (i / CANNY_IW) % CANNY_IH;
      c = i / (CANNY_IW * CANNY_IH);
    }
    const int gy = min(max(y0 + r - 2, 0), H - 1), gx = min(max(x0 + x - 2, 0), W - 1);
    const long e = NHWC ? (((long)n * H + gy) * W + gx) * 3 + c : (((long)n * 3 + c) * H + gy) * W + gx;
    px[c][r][x] = cast_u8_like_numpy(load_f32(img, e));
  }
  __syncthreads();

  // 2. Sobel on the tile + 1-pixel ring; magnitude 0 outside the image
  for (int i = tid; i < CANNY_RH * CANNY_RW; i += CANNY_THREADS) {
    const int r = i / CANNY_RW, x = i % CANNY_RW;  // ring coordinates; image pixel (y0 + r - 1, x0 + x - 1)
    const int gy = y0 + r - 1, gx = x0 + x - 1;
    int best = 0, bdx = 0, bdy = 0;
    if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const uint8_t(*p)[CANNY_IW] = px[c];
        const int a = r, b = r + 1, d = r + 2;      // staged rows above / at / below the pixel
        const int l = x, m = x + 1, rt = x + 2;     // staged columns left / at / right
        const int dx = (p[a][rt] + 2 * p[b][rt] + p[d][rt]) - (p[a][l] + 2 * p[b][l] + p[d][l]);
        const int dy = (p[d][l] + 2 * p[d][m] + p[d][rt]) - (p[a][l] + 2 * p[a][m] + p[a][rt]);
        const int mm = abs(dx) + abs(dy);
        if (c == 0 || mm > best) { best = mm; bdx = dx; bdy = dy; }
      }
    }
    mag[r][x] = best;
    if (r >= 1 && r <= CANNY_TH && x >= 1 && x <= CANNY_TW) dxy[r - 1][x - 1] = (int)((unsigned)bdx << 16) | (bdy & 0xffff);
  }
  __syncthreads();

  // 3. non-maximum suppression (cv2's sectors and comparison senses) -> candidate / strong; local labels start as self
  for (int i = tid; i < CANNY_TH * CANNY_TW; i += CANNY_THREADS) {
    const int r = i / CANNY_TW, x = i % CANNY_TW, R = r + 1, X = x + 1;
    const int m = mag[R][X];
    bool cand = false;
    if (m > lo && y0 + r < H && x0 + x < W) {
      const int v = dxy[r][x], dx = v >> 16, dy = (int)(short)(v & 0xffff);
      const int xs = abs(dx), ys = abs(dy);
      const int yy = ys << 15, tg22x = xs * CANNY_TG22, tg67x = tg22x + (xs << 16);
      if (yy < tg22x) {
        cand = m > mag[R][X - 1] && m >= mag[R][X + 1];
      } else if (yy > tg67x) {
        cand = m > mag[R - 1][X] && m >= mag[R + 1][X];
      } else {
        const int s = (dx ^ dy) < 0 ? -1 : 1;
        cand = m > mag[R - 1][X - s] && m > mag[R + 1][X + s];
      }
    }
    lab[i] = cand ? i : -1;
    strong_root[i] = (cand && m > hi) ? 1 : 0;  // strong marker; turned into a per-root flag below
  }
  __syncthreads();

  // 4. local union-find: every candidate links to its W, NW, N, NE candidate neighbours inside the tile
  for (int i = tid; i < CANNY_TH * CANNY_TW; i += CANNY_THREADS) {
    if (lab[i] < 0) continue;
    const int r = i / CANNY_TW, x = i % CANNY_TW;
    if (x > 0 && lab[i - 1] >= 0) uf_union(lab, i, i - 1);
    if (r > 0) {
      if (x > 0 && lab[i - CANNY_TW - 1] >= 0) uf_union(lab, i, i - CANNY_TW - 1);
      if (lab[i - CANNY_TW] >= 0) uf_union(lab, i, i - CANNY_TW);
      if (x < CANNY_TW - 1 && lab[i - CANNY_TW + 1] >= 0) uf_union(lab, i, i - CANNY_TW + 1);
    }
  }
  __syncthreads();

  // 5. flatten; strong candidates mark their local root
  int root[CANNY_TH * CANNY_TW / CANNY_THREADS];
  bool strong[CANNY_TH * CANNY_TW / CANNY_THREADS];
#pragma unroll
  for (int k = 0; k < CANNY_TH * CANNY_TW / CANNY_THREADS; ++k) {
    const int i = tid + k * CANNY_THREADS;
    root[k] = lab[i] >= 0 ? uf_find(lab, i) : -1;
    strong[k] = strong_root[i] != 0;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < CANNY_TH * CANNY_TW / CANNY_THREADS; ++k) strong_root[tid + k * CANNY_THREADS] = 0;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < CANNY_TH * CANNY_TW / CANNY_THREADS; ++k)
    if (strong[k]) strong_root[root[k]] = 1;  // every writer stores the same value
  __syncthreads();

  // 6. global label = image-wide index of the local root (row-major in the tile is row-major in the image, so the
  //    local minimum is also the global minimum); flag = local root of a component with a strong candidate
#pragma unroll
  for (int k = 0; k < CANNY_TH * CANNY_TW / CANNY_THREADS; ++k) {
    const int i = tid + k * CANNY_THREADS;
    const int r = i / CANNY_TW, x = i % CANNY_TW;
    if (y0 + r >= H || x0 + x >= W) continue;
    const int g = (n * H + y0 + r) * W + x0 + x;
    int gl = -1;
    if (root[k] >= 0) gl = (n * H + y0 + root[k] / CANNY_TW) * W + x0 + root[k] % CANNY_TW;
    labels[g] = gl;
    flags[g] = (root[k] == i && strong_root[i]) ? 1 : 0;
  }
}

// candidates on a tile's top row and side columns union with their W / NW / N / NE neighbours that lie in another
// tile; every cross-tile 8-neighbour pair is visited once, from its later pixel
__global__ void __launch_bounds__(CANNY_THREADS)
canny_merge_kernel(int *labels, int N, int H, int W, int tiles_x, int tiles_y) {
  const long total = (long)N * tiles_y * tiles_x * CANNY_PERIM;
  for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
    const int k = (int)(t % CANNY_PERIM);
    const long tile = t / CANNY_PERIM;
    const int tx = (int)(tile % tiles_x), ty = (int)((tile / tiles_x) % tiles_y), n = (int)(tile / ((long)tiles_x * tiles_y));
    int r, x;
    if (k < CANNY_TW) { r = 0; x = k; }
    else { r = 1 + (k - CANNY_TW) / 2; x = ((k - CANNY_TW) & 1) ? CANNY_TW - 1 : 0; }
    const int y = ty * CANNY_TH + r, gx = tx * CANNY_TW + x;
    if (y >= H || gx >= W) continue;
    const int p = (n * H + y) * W + gx;
    if (__ldcg(labels + p) < 0) continue;
    const int nbr_dy[4] = {0, -1, -1, -1}, nbr_dx[4] = {-1, -1, 0, 1};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int qy = y + nbr_dy[j], qx = gx + nbr_dx[j];
      if (qy < 0 || qx < 0 || qx >= W) continue;
      if (qy / CANNY_TH == ty && qx / CANNY_TW == tx) continue;  // same tile: joined by the tile pass
      const int q = (n * H + qy) * W + qx;
      if (__ldcg(labels + q) >= 0) uf_union(labels, p, q);
    }
  }
}

// after the merge every component has one root: point each candidate straight at it and flag it from the local roots
__global__ void __launch_bounds__(CANNY_THREADS)
canny_root_kernel(int *labels, uint8_t *flags, int P) {
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long)gridDim.x * blockDim.x) {  // P + stride > 2^31
    const int l = labels[p];
    if (l < 0) continue;
    const int r = uf_find(labels, l);
    if (r != l) labels[p] = r;  // concurrent readers see l or r, both ancestors of p
    if (flags[p]) flags[r] = 1;  // a 1 read at a root another thread just flagged only repeats the same store
  }
}

__global__ void __launch_bounds__(CANNY_THREADS)
canny_output_kernel(const int *__restrict__ labels, const uint8_t *__restrict__ flags, float *__restrict__ edges, int P) {
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long)gridDim.x * blockDim.x) {  // P + stride > 2^31
    const int l = labels[p];
    edges[p] = (l >= 0 && flags[l]) ? 255.f : 0.f;
  }
}

static size_t canny_flags_offset(long P) { return ((size_t)P * sizeof(int) + 255) & ~(size_t)255; }

// cv2 swaps reversed thresholds and compares integer magnitudes against their floors; magnitudes lie in [0, 2040]
static int canny_threshold(double t) { return (int)fmin(fmax(floor(t), -1.0), 4096.0); }

template <typename T, bool NHWC>
static void launch_tile(const void *img, int *labels, uint8_t *flags, int N, int H, int W, int lo, int hi, cudaStream_t st) {
  const int tiles = N * ceil_div(W, CANNY_TW) * ceil_div(H, CANNY_TH);  // < P < 2^31
  canny_tile_kernel<T, NHWC><<<tiles, CANNY_THREADS, 0, st>>>(static_cast<const T *>(img), labels, flags, H, W, lo, hi);
}

}  // namespace kdcc

using namespace kdcc;

KDCC_API size_t kdcc_canny_workspace_bytes(int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0) return 0;
  const long P = (long)N * H * W;
  return canny_flags_offset(P) + (size_t)P;
}

KDCC_API int kdcc_canny(const void *img, float *edges, void *workspace, size_t workspace_bytes, int N, int C, int H, int W,
                        int layout, int dtype, double low, double high, kdcc_stream_t stream) {
  if (!img || !edges || !workspace || N <= 0 || C <= 0 || H <= 0 || W <= 0) return KDCC_EINVAL;
  if ((layout != KDCC_LAYOUT_NCHW && layout != KDCC_LAYOUT_NHWC) || (dtype != KDCC_F32 && dtype != KDCC_BF16)) return KDCC_EINVAL;
  if (isnan(low) || isnan(high)) return KDCC_EINVAL;
  const long P = (long)N * H * W;
  if (C != 3 || P >= (1L << 31)) return KDCC_ESHAPE;
  if (workspace_bytes < kdcc_canny_workspace_bytes(N, H, W)) return KDCC_EWORKSPACE;
  if (low > high) { const double t = low; low = high; high = t; }
  const int lo = canny_threshold(low), hi = canny_threshold(high);

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int *labels = static_cast<int *>(workspace);
  uint8_t *flags = static_cast<uint8_t *>(workspace) + canny_flags_offset(P);
  const bool nhwc = layout == KDCC_LAYOUT_NHWC;
  if (dtype == KDCC_F32) {
    if (nhwc) launch_tile<float, true>(img, labels, flags, N, H, W, lo, hi, st);
    else launch_tile<float, false>(img, labels, flags, N, H, W, lo, hi, st);
  } else {
    if (nhwc) launch_tile<__nv_bfloat16, true>(img, labels, flags, N, H, W, lo, hi, st);
    else launch_tile<__nv_bfloat16, false>(img, labels, flags, N, H, W, lo, hi, st);
  }
  const int tiles_x = ceil_div(W, CANNY_TW), tiles_y = ceil_div(H, CANNY_TH);
  const long perim = (long)N * tiles_x * tiles_y * CANNY_PERIM;
  canny_merge_kernel<<<(int)min((long)kNumSMs * 8, ceil_div<long>(perim, CANNY_THREADS)), CANNY_THREADS, 0, st>>>(
      labels, N, H, W, tiles_x, tiles_y);
  const int grid = (int)min((long)kNumSMs * 16, ceil_div<long>(P, CANNY_THREADS));
  canny_root_kernel<<<grid, CANNY_THREADS, 0, st>>>(labels, flags, (int)P);
  canny_output_kernel<<<grid, CANNY_THREADS, 0, st>>>(labels, flags, edges, (int)P);
  return launch_status();
}
