// bf16 activation layout conversion NHWC <-> NCHW (HBM-bound tiled transpose, 16-byte global accesses on both sides).
//
// Why it exists: the depthwise k = 9 kernels that reach tensor-core speed take channel PLANES (NCHW; dw_tc2.cu explains why
// an NHWC-native form is not possible: one 16-byte NHWC vector holds 8 channels, and eight 53 KB plane operands do not
// fit one SM).  A trunk that runs cuDNN in channels_last therefore hands the blocks NHWC tensors; converting at the block
// boundary costs two extra HBM passes per tensor but keeps the 9x9 depthwise on tcgen05 (4x faster than the NHWC
// CUDA-core kernels, DESIGN.md 4.1), and cuDNN's channels_last trunk is faster than its NCHW one by more than that.
// Reference call site this supports: models/students/transform_blocks/depthwise_separable_conv.py:11-14 called from a
// channels_last model.
#include "kdcc_common.cuh"

namespace kdcc {

constexpr int LC_T = 64;          // tile: 64 pixels x 64 channels
constexpr int LC_PITCH = 33;      // words per tile row (32 channel pairs + 1): conflict-free 4-byte row accesses
constexpr int LC_THREADS = 256;

// smem tile: s[pixel][channel pair] as 32-bit words (two bf16 channels of one pixel)
template <bool TO_NCHW>
__global__ void __launch_bounds__(LC_THREADS) layout_convert_kernel(const __nv_bfloat16 *__restrict__ src, __nv_bfloat16 *__restrict__ dst,
                                                                    int C, long HW, int tiles_p, int tiles_c) {
  __shared__ uint32_t s[LC_T * LC_PITCH];
  pdl_prologue_done();
  long t = blockIdx.x;
  const int tc = (int)(t % tiles_c); t /= tiles_c;
  const int tp = (int)(t % tiles_p);
  const long n = t / tiles_p;
  const long p0 = (long)tp * LC_T;
  const int c0 = tc * LC_T;
  const __nv_bfloat16 *img_in = src + n * HW * C;
  __nv_bfloat16 *img_out = dst + n * HW * C;
  const int tid = threadIdx.x;
  if (TO_NCHW) {
    // ---- load NHWC: (pixel, 8-channel chunk) per thread, two rounds ----
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int p = (tid >> 3) + 32 * r, c8 = tid & 7;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (p0 + p < HW && c0 + c8 * 8 < C) v = *reinterpret_cast<const uint4 *>(img_in + (p0 + p) * C + c0 + c8 * 8);
      uint32_t *row = s + p * LC_PITCH + c8 * 4;
      row[0] = v.x; row[1] = v.y; row[2] = v.z; row[3] = v.w;
    }
    __syncthreads();
    // ---- store NCHW: (channel pair, 8-pixel chunk) per thread: 8 words -> two 16-byte rows of 8 pixels ----
#pragma unroll
    for (int r = 0; r < 1; ++r) {
      const int cp = tid >> 3, p8 = tid & 7;    // 32 channel pairs x 8 pixel chunks
      uint32_t w[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) w[e] = s[(p8 * 8 + e) * LC_PITCH + cp];
      uint4 lo, hi;   // lo: channel 2cp, hi: channel 2cp+1; pixels e = 0..7
      lo.x = __byte_perm(w[0], w[1], 0x5410); lo.y = __byte_perm(w[2], w[3], 0x5410);
      lo.z = __byte_perm(w[4], w[5], 0x5410); lo.w = __byte_perm(w[6], w[7], 0x5410);
      hi.x = __byte_perm(w[0], w[1], 0x7632); hi.y = __byte_perm(w[2], w[3], 0x7632);
      hi.z = __byte_perm(w[4], w[5], 0x7632); hi.w = __byte_perm(w[6], w[7], 0x7632);
      const long p = p0 + p8 * 8;
      const int c = c0 + 2 * cp;
      if (p < HW && c < C) {
        *reinterpret_cast<uint4 *>(img_out + (long)c * HW + p) = lo;
        *reinterpret_cast<uint4 *>(img_out + (long)(c + 1) * HW + p) = hi;
      }
    }
  } else {
    // ---- load NCHW: (channel pair, 8-pixel chunk) per thread: two 16-byte rows -> 8 words (pixel e: channels 2cp, 2cp+1) ----
    {
      const int cp = tid >> 3, p8 = tid & 7;
      const long p = p0 + p8 * 8;
      const int c = c0 + 2 * cp;
      uint4 lo = make_uint4(0, 0, 0, 0), hi = make_uint4(0, 0, 0, 0);
      if (p < HW && c < C) {
        lo = *reinterpret_cast<const uint4 *>(img_in + (long)c * HW + p);
        hi = *reinterpret_cast<const uint4 *>(img_in + (long)(c + 1) * HW + p);
      }
      const uint32_t l[4] = {lo.x, lo.y, lo.z, lo.w}, h[4] = {hi.x, hi.y, hi.z, hi.w};
#pragma unroll
      for (int e2 = 0; e2 < 4; ++e2) {
        s[(p8 * 8 + 2 * e2) * LC_PITCH + cp] = __byte_perm(l[e2], h[e2], 0x5410);
        s[(p8 * 8 + 2 * e2 + 1) * LC_PITCH + cp] = __byte_perm(l[e2], h[e2], 0x7632);
      }
    }
    __syncthreads();
    // ---- store NHWC: (pixel, 8-channel chunk) per thread ----
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int p = (tid >> 3) + 32 * r, c8 = tid & 7;
      const uint32_t *row = s + p * LC_PITCH + c8 * 4;
      if (p0 + p < HW && c0 + c8 * 8 < C)
        *reinterpret_cast<uint4 *>(img_out + (p0 + p) * C + c0 + c8 * 8) = make_uint4(row[0], row[1], row[2], row[3]);
    }
  }
}

}  // namespace kdcc

using namespace kdcc;

// dst (NCHW if to_nchw else NHWC) = src (the other layout); bf16; C % 8 == 0 and HW % 8 == 0 (16-byte rows both ways)
KDCC_API int kdcc_layout_convert(const void *src, void *dst, int N, int C, long HW, int to_nchw, int dtype, kdcc_stream_t stream) {
  if (!src || !dst || N < 0 || C <= 0 || HW <= 0) return KDCC_EINVAL;
  if (dtype == KDCC_F32_TF32X3) return KDCC_EINVAL;  // a pointwise-only dtype code
  if (dtype != KDCC_BF16) return KDCC_ESHAPE;
  if (C % 8 != 0 || HW % 8 != 0) return KDCC_ESHAPE;
  if (!aligned16(src) || !aligned16(dst)) return KDCC_EALIGN;
  if (N == 0) return KDCC_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int tiles_p = (int)ceil_div<long>(HW, LC_T), tiles_c = ceil_div(C, LC_T);
  const long blocks = (long)N * tiles_p * tiles_c;
  if (blocks >= (1L << 31)) return KDCC_ESHAPE;
  const __nv_bfloat16 *s = static_cast<const __nv_bfloat16 *>(src);
  __nv_bfloat16 *d = static_cast<__nv_bfloat16 *>(dst);
  if (to_nchw) launch_pdl(layout_convert_kernel<true>, dim3((unsigned)blocks), dim3(LC_THREADS), 0, st, s, d, C, HW, tiles_p, tiles_c);
  else launch_pdl(layout_convert_kernel<false>, dim3((unsigned)blocks), dim3(LC_THREADS), 0, st, s, d, C, HW, tiles_p, tiles_c);
  return launch_status();
}
