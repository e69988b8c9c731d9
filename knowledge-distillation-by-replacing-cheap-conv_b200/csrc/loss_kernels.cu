// Fused distillation losses for sm_100a: one HBM pass reads student+teacher, produces the scalar loss
// and the gradient w.r.t. the student tensor.
//   kd_loss_kernel    losses/KLDiv.py:19-23, losses/EnsembleKLDiv.py:18-22  (reference file:line)
//   hint_loss_kernel  losses/WeightedHintMSELoss.py:12-16, losses/MSELoss.py:14-16
// Both are HBM-bound (algorithmic traffic: 2 reads + 1 write of the tensor, SURVEY.md 8d); they use
// 8/16-byte coalesced streaming accesses, fp32 math in registers, a fixed-order block reduction and a
// one-block finalize so the scalar is bit-reproducible run to run.
#include "loss_common.cuh"

namespace kdcc {

struct KdParams {
  const void *s, *t;
  void *ds;
  float *partials;
  long HW, bs, cs, ps;
  long groups, HWg;
  int C;
  int target_is_prob;
  float k2;     // log2(e) / T : logits -> base-2 exponent
  float gcoef;  // grad_scale * T / (N*HW)
};

// CT = compile-time class capacity (values live in registers), EXACT: C == CT so no predicates.
// PROB: targets are probabilities already (EnsembleKLDiv) -- a template parameter so that each form keeps its own,
// smaller, register footprint (both in one kernel: 170 registers, one block per SM).
template <typename T, int CT, bool EXACT, int PIX, bool PROB>
__global__ void __launch_bounds__(kLossThreads, CT <= 19 ? 2 : 1) kd_loss_kernel(const KdParams p) {
  __shared__ float scratch[32];
  const T *__restrict__ sbase = static_cast<const T *>(p.s);
  const T *__restrict__ tbase = static_cast<const T *>(p.t);
  T *__restrict__ dbase = static_cast<T *>(p.ds);
  const int C = EXACT ? CT : p.C;
  float local = 0.f;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < p.groups; g += (long)gridDim.x * blockDim.x) {
    const long n = g / p.HWg;
    const long q = (g - n * p.HWg) * PIX;
    const long off = n * p.bs + q * p.ps;
    float sv[CT][PIX], tv[CT][PIX];
#pragma unroll
    for (int c = 0; c < CT; ++c) {
      if (EXACT || c < C) {
        load_pix<T, PIX>(sbase + off + c * p.cs, sv[c]);
        load_pix<T, PIX>(tbase + off + c * p.cs, tv[c]);
      }
    }
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      float smax = -INFINITY, tmax = -INFINITY;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) { smax = fmaxf(smax, sv[c][i]); tmax = fmaxf(tmax, tv[c][i]); }
      if (!PROB) {
        // Softmaxed teacher: ONE exponential per logit.  With a = log2-domain student logit, b = teacher logit (both
        // relative to their max), e_s = 2^a, e_t = 2^b:
        //   KL (bits) = sum_c p_t (log2 p_t - log2 p_s) = (sum_c e_t (b - a)) / sum e_t - log2 sum e_t + log2 sum e_s
        //   grad      = gcoef * (e_s / sum e_s - e_t / sum e_t)
        // (the kernel is otherwise limited by the MUFU pipe: 4 exponentials per logit pair cost 72 us of a 164 us pass)
        float ssum = 0.f, tsum = 0.f, cross = 0.f;
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (EXACT || c < C) {
            const float a = (sv[c][i] - smax) * p.k2, b = (tv[c][i] - tmax) * p.k2;
            const float es = exp2f(a), et = exp2f(b);
            ssum += es; tsum += et;
            if (et > 0.f) cross += et * (b - a);   // p_t == 0 contributes 0 (xlogy), whatever the student says
            sv[c][i] = es; tv[c][i] = et;
          }
        const float rs = 1.f / ssum, rt = 1.f / tsum;
        local += cross * rt - log2f(tsum) + log2f(ssum);
        if (dbase != nullptr) {
#pragma unroll
          for (int c = 0; c < CT; ++c)
            if (EXACT || c < C) sv[c][i] = p.gcoef * (sv[c][i] * rs - tv[c][i] * rt);
        }
        continue;
      }
      // targets are probabilities already (losses/EnsembleKLDiv.py): log-softmax of the student only
      float ssum = 0.f, tsum = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          sv[c][i] = (sv[c][i] - smax) * p.k2;  // base-2 exponent relative to the max
          ssum += exp2f(sv[c][i]);
          tsum += tv[c][i];  // probability mass of the (ensemble) target
        }
      const float ls = log2f(ssum);
      float kl2 = 0.f;  // KL in bits; converted to nats at finalize
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          const float lps = sv[c][i] - ls;  // log2 p_s
          const float ps = exp2f(lps);
          const float pt = tv[c][i];
          const float lpt = pt > 0.f ? log2f(pt) : 0.f;
          if (pt > 0.f) kl2 += pt * (lpt - lps);
          // gradient: softmax(s/T) * (target mass) - p_t
          sv[c][i] = p.gcoef * (ps * tsum - pt);
        }
      local += kl2;
    }
    if (dbase != nullptr) {
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) store_pix<T, PIX>(dbase + off + c * p.cs, sv[c]);
    }
  }
  const float tot = block_sum(local, scratch);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = tot;
}

// ------------------------------------------------------------------------------------------------
// Multi-teacher KD (SURVEY.md 8f n3; trainer/ensemble_trainer.py:76-83): the student logits are read ONCE, every
// teacher's softmax is formed in registers, and
//     loss = sum_k w_k * T^2/(N*HW) * sum_pix KL(p_k || p_s)
//          = T^2/(N*HW) * sum_pix [ sum_k w_k sum_c p_kc log p_kc  -  sum_c (sum_k w_k p_kc) log p_sc ]
//     ds   = grad_scale * T/(N*HW) * ( (sum_k w_k) softmax(s/T) - sum_k w_k p_k )
// Traffic K+2 tensors instead of the 3K of K separate kdcc_kd_loss calls.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxTeachers = 8;
struct KdMultiParams {
  const void *s;
  const void *t[kMaxTeachers];
  float w[kMaxTeachers];
  float wsum;
  int K;
  void *ds;
  float *partials;
  long HW, bs, cs, ps;
  long groups, HWg;
  int C;
  float k2, gcoef;
};

template <typename T, int CT, bool EXACT, int PIX>
__global__ void __launch_bounds__(kLossThreads) kd_multi_kernel(const KdMultiParams p) {
  __shared__ float scratch[32];
  const T *__restrict__ sbase = static_cast<const T *>(p.s);
  T *__restrict__ dbase = static_cast<T *>(p.ds);
  const int C = EXACT ? CT : p.C;
  float local = 0.f;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < p.groups; g += (long)gridDim.x * blockDim.x) {
    const long n = g / p.HWg;
    const long q = (g - n * p.HWg) * PIX;
    const long off = n * p.bs + q * p.ps;
    float sv[CT][PIX], pw[CT][PIX];  // student log2-probabilities, weighted teacher probabilities
    float ent[PIX];                  // sum_k w_k sum_c p_kc log2 p_kc
#pragma unroll
    for (int c = 0; c < CT; ++c)
      if (EXACT || c < C) load_pix<T, PIX>(sbase + off + c * p.cs, sv[c]);
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      float smax = -INFINITY;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) smax = fmaxf(smax, sv[c][i]);
      float ssum = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          sv[c][i] = (sv[c][i] - smax) * p.k2;
          ssum += exp2f(sv[c][i]);
          pw[c][i] = 0.f;
        }
      const float ls = log2f(ssum);
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) sv[c][i] -= ls;  // log2 p_s
      ent[i] = 0.f;
    }
    for (int k = 0; k < p.K; ++k) {
      const T *__restrict__ tbase = static_cast<const T *>(p.t[k]);
      const float wk = p.w[k];
      float tv[CT][PIX];
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) load_pix<T, PIX>(tbase + off + c * p.cs, tv[c]);
#pragma unroll
      for (int i = 0; i < PIX; ++i) {
        float tmax = -INFINITY;
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (EXACT || c < C) tmax = fmaxf(tmax, tv[c][i]);
        // one exponential per teacher logit: e = 2^b is kept, sum_c p log2 p = (sum_c e b) / Z - log2 Z, p = e / Z
        float tsum = 0.f, tb = 0.f;
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (EXACT || c < C) {
            const float b = (tv[c][i] - tmax) * p.k2;
            const float et = exp2f(b);
            tsum += et;
            if (et > 0.f) tb += et * b;   // p == 0 contributes 0 (xlogy)
            tv[c][i] = et;
          }
        const float rt = 1.f / tsum;
        ent[i] += wk * (tb * rt - log2f(tsum));
        const float wr = wk * rt;
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (EXACT || c < C) pw[c][i] += wr * tv[c][i];
      }
    }
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      float cross = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          if (pw[c][i] > 0.f) cross += pw[c][i] * sv[c][i];
          sv[c][i] = p.gcoef * (p.wsum * exp2f(sv[c][i]) - pw[c][i]);
        }
      local += ent[i] - cross;
    }
    if (dbase != nullptr) {
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) store_pix<T, PIX>(dbase + off + c * p.cs, sv[c]);
    }
  }
  const float tot = block_sum(local, scratch);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = tot;
}

// Any class count: three passes over the class axis per pixel (re-reads hit L1/L2).
template <typename T>
__global__ void __launch_bounds__(kLossThreads) kd_loss_generic_kernel(const KdParams p) {
  __shared__ float scratch[32];
  const T *__restrict__ sbase = static_cast<const T *>(p.s);
  const T *__restrict__ tbase = static_cast<const T *>(p.t);
  T *__restrict__ dbase = static_cast<T *>(p.ds);
  float local = 0.f;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < p.groups; g += (long)gridDim.x * blockDim.x) {
    const long n = g / p.HWg;
    const long q = g - n * p.HWg;
    const long off = n * p.bs + q * p.ps;
    float smax = -INFINITY, tmax = -INFINITY;
    for (int c = 0; c < p.C; ++c) {
      smax = fmaxf(smax, to_f32(sbase[off + c * p.cs]));
      tmax = fmaxf(tmax, to_f32(tbase[off + c * p.cs]));
    }
    float ssum = 0.f, tsum = 0.f;
    for (int c = 0; c < p.C; ++c) {
      ssum += exp2f((to_f32(sbase[off + c * p.cs]) - smax) * p.k2);
      const float tvv = to_f32(tbase[off + c * p.cs]);
      tsum += p.target_is_prob ? tvv : exp2f((tvv - tmax) * p.k2);
    }
    const float ls = log2f(ssum), lt = p.target_is_prob ? 0.f : log2f(tsum);
    float kl2 = 0.f;
    for (int c = 0; c < p.C; ++c) {
      const float lps = (to_f32(sbase[off + c * p.cs]) - smax) * p.k2 - ls;
      const float ps = exp2f(lps);
      const float tvv = to_f32(tbase[off + c * p.cs]);
      float pt, lpt;
      if (!p.target_is_prob) { lpt = (tvv - tmax) * p.k2 - lt; pt = exp2f(lpt); }
      else { pt = tvv; lpt = pt > 0.f ? log2f(pt) : 0.f; }
      if (pt > 0.f) kl2 += pt * (lpt - lps);
      if (dbase != nullptr)
        dbase[off + c * p.cs] = from_f32<T>(p.gcoef * (p.target_is_prob ? ps * tsum - pt : ps - pt));
    }
    local += kl2;
  }
  const float tot = block_sum(local, scratch);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = tot;
}

// Fixed-order final sum of the per-CTA partials (double), scaled, written as one fp32 scalar.
__global__ void __launch_bounds__(256) loss_finalize_kernel(const float *__restrict__ partials, int count,
                                                            double coef, float *__restrict__ out) {
  __shared__ double sh[256];
  pdl_prologue_done();
  double acc = 0.0;
  for (int i = threadIdx.x; i < count; i += 256) acc += (double)partials[i];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)(sh[0] * coef);
}

// ------------------------------------------------------------------------------------------------
// hint loss
// ------------------------------------------------------------------------------------------------
struct HintParams {
  const void *s, *t;
  void *ds;
  const float *coef;  // [N*C] per-(sample,channel) loss coefficient, or nullptr (uniform)
  float *partials;
  long total;         // elements
  long HW;
  int C;
  int layout;
  float ucoef;        // uniform loss coefficient scale / (N*C*HW)
  float g2;           // 2 * grad_scale
};

// coef[n][c] = scale * w[n,c] / (sum_c w[n,c] * HW * N); one CTA per sample
__global__ void __launch_bounds__(256) hint_coef_kernel(const float *__restrict__ w, int w_per_sample, int C,
                                                        double scale_over_hwn, float *__restrict__ coef) {
  __shared__ float scratch[32];
  const int n = blockIdx.x;
  const float *wr = w + (w_per_sample ? (long)n * C : 0);
  float acc = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) acc += wr[c];
  __shared__ float wsum;
  const float tot = block_sum(acc, scratch);
  if (threadIdx.x == 0) wsum = tot;
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    coef[(long)n * C + c] = (float)(scale_over_hwn * (double)wr[c] / (double)wsum);
}

template <typename T, bool WEIGHTED, int UNROLL>
__global__ void __launch_bounds__(kLossThreads) hint_loss_kernel(const HintParams p) {
  using V = Vec16<T>;
  constexpr int VN = V::N;
  __shared__ float scratch[32];
  pdl_prologue_done();
  const char *__restrict__ sb = static_cast<const char *>(p.s);
  const char *__restrict__ tb = static_cast<const char *>(p.t);
  char *__restrict__ db = static_cast<char *>(p.ds);
  const long nvec = p.total / VN;
  const long stride = (long)gridDim.x * blockDim.x;
  float local = 0.f;
  for (long v0 = (long)blockIdx.x * blockDim.x + threadIdx.x; v0 < nvec; v0 += stride * UNROLL) {
    V sv[UNROLL], tv[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long v = v0 + u * stride;
      if (v < nvec) {
        sv[u] = ld_stream<V>(sb + v * 16);
        tv[u] = ld_stream<V>(tb + v * 16);
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long v = v0 + u * stride;
      if (v < nvec) {
        float a[VN], b[VN], lw[VN];
        sv[u].unpack(a);
        tv[u].unpack(b);
        if (WEIGHTED) {
          const long e = v * VN;
          if (p.layout == KDCC_LAYOUT_NHWC) {
            const long pix = e / p.C;
            const int c0 = (int)(e - pix * p.C);
            const long n = pix / p.HW;
            const float *cf = p.coef + n * p.C + c0;
#pragma unroll
            for (int i = 0; i < VN; ++i) lw[i] = __ldg(cf + i);
          } else {
            const long plane = e / p.HW;  // = n*C + c
            const float cfv = __ldg(p.coef + plane);
#pragma unroll
            for (int i = 0; i < VN; ++i) lw[i] = cfv;
          }
        } else {
#pragma unroll
          for (int i = 0; i < VN; ++i) lw[i] = p.ucoef;
        }
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < VN; ++i) {
          const float d = a[i] - b[i];
          acc = fmaf(lw[i] * d, d, acc);
          a[i] = p.g2 * lw[i] * d;
        }
        local += acc;
        if (db != nullptr) {
          V o;
          o.pack(a);
          st_stream<V>(db + v * 16, o);
        }
      }
    }
  }
  const float tot = block_sum(local, scratch);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = tot;
}

// Element-granular variant for shapes that cannot be vectorised (C or HW not a multiple of the vector).
template <typename T>
__global__ void __launch_bounds__(kLossThreads) hint_loss_scalar_kernel(const HintParams p) {
  __shared__ float scratch[32];
  const T *__restrict__ sb = static_cast<const T *>(p.s);
  const T *__restrict__ tb = static_cast<const T *>(p.t);
  T *__restrict__ db = static_cast<T *>(p.ds);
  float local = 0.f;
  for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < p.total; e += (long)gridDim.x * blockDim.x) {
    float lw = p.ucoef;
    if (p.coef != nullptr) {
      if (p.layout == KDCC_LAYOUT_NHWC) {
        const long pix = e / p.C;
        lw = p.coef[(pix / p.HW) * p.C + (e - pix * p.C)];
      } else {
        lw = p.coef[e / p.HW];
      }
    }
    const float d = to_f32(sb[e]) - to_f32(tb[e]);
    local = fmaf(lw * d, d, local);
    if (db != nullptr) db[e] = from_f32<T>(p.g2 * lw * d);
  }
  const float tot = block_sum(local, scratch);
  if (threadIdx.x == 0) p.partials[blockIdx.x] = tot;
}

// ------------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------------
__global__ void cast_f32_to_bf16_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, long n) {
  pdl_prologue_done();
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i]);
}

template <typename T>
__global__ void scale_inplace_kernel(T *__restrict__ buf, const float *__restrict__ scalar, float expected, long n) {
  // buf *= scalar / expected.  The forward pass already folded `expected` into the emitted gradient; when autograd's
  // upstream value is what was expected (the usual case) every thread leaves without touching memory.
  const float g = __ldg(scalar) / expected;
  if (g == 1.f) return;
  constexpr int V = 16 / sizeof(T);
  const long nv = (reinterpret_cast<uintptr_t>(buf) & 15) == 0 ? n / V : 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long)gridDim.x * blockDim.x) {
    uint4 u = reinterpret_cast<uint4 *>(buf)[i];
    T *e = reinterpret_cast<T *>(&u);
#pragma unroll
    for (int j = 0; j < V; ++j) e[j] = from_f32<T>(to_f32(e[j]) * g);
    reinterpret_cast<uint4 *>(buf)[i] = u;
  }
  for (long i = nv * V + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    buf[i] = from_f32<T>(to_f32(buf[i]) * g);
}

// column sums, stage 1: CTA (bx, by) sums rows [by*rows_per, ...) of 128 columns into part[by][col]
template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const T *__restrict__ a, float *__restrict__ part,
                                                             long M, int Nc, long rows_per) {
  __shared__ float sh[8][32];
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rlane = threadIdx.x >> 5;  // 8 row lanes
  const long r0 = (long)blockIdx.y * rows_per;
  const long r1 = min(M, r0 + rows_per);
  float acc = 0.f;
  if (col < Nc)
    for (long r = r0 + rlane; r < r1; r += 8) acc += to_f32(a[r * Nc + col]);
  sh[rlane][threadIdx.x & 31] = acc;
  __syncthreads();
  if (rlane == 0 && col < Nc) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += sh[i][threadIdx.x];
    part[(long)blockIdx.y * Nc + col] = t;
  }
}
__global__ void colsum_final_kernel(const float *__restrict__ part, float *__restrict__ out, int splits, int Nc) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= Nc) return;
  double t = 0.0;
  for (int s = 0; s < splits; ++s) t += (double)part[(long)s * Nc + col];
  out[col] = (float)t;
}

}  // namespace kdcc

using namespace kdcc;

KDCC_API size_t kdcc_loss_workspace_bytes(void) { return sizeof(float) * kMaxLossBlocks; }

template <typename T>
static int launch_kd(const KdParams &p0, bool vec2, int grid_hint, cudaStream_t st) {
  KdParams p = p0;
  const int C = p.C;
  if (C > 32) {
    p.HWg = p.HW;
    p.groups = p0.groups;  // caller passes N*HW for the scalar path
    const int grid = (int)min((long)kMaxLossBlocks, ceil_div<long>(p.groups, kLossThreads));
    kd_loss_generic_kernel<T><<<grid, kLossThreads, 0, st>>>(p);
    return grid;
  }
  const int grid = grid_hint;
#define KD_LAUNCH(CT, EXACT)                                                             \
  do {                                                                                   \
    if (p.target_is_prob) {                                                              \
      if (vec2) kd_loss_kernel<T, CT, EXACT, 2, true><<<grid, kLossThreads, 0, st>>>(p); \
      else kd_loss_kernel<T, CT, EXACT, 1, true><<<grid, kLossThreads, 0, st>>>(p);      \
    } else {                                                                             \
      if (vec2) kd_loss_kernel<T, CT, EXACT, 2, false><<<grid, kLossThreads, 0, st>>>(p);\
      else kd_loss_kernel<T, CT, EXACT, 1, false><<<grid, kLossThreads, 0, st>>>(p);     \
    }                                                                                    \
  } while (0)
  if (C == 19) KD_LAUNCH(19, true);
  else if (C == 10) KD_LAUNCH(10, true);
  else if (C <= 16) KD_LAUNCH(16, false);
  else KD_LAUNCH(32, false);
#undef KD_LAUNCH
  return grid;
}

KDCC_API int kdcc_kd_loss(const void *s, const void *t, void *ds, float *loss_out, void *workspace,
                          size_t workspace_bytes, int N, int C, long HW, long batch_stride, long class_stride,
                          long pixel_stride, float T, int target_is_prob, int dtype, float grad_scale,
                          kdcc_stream_t stream) {
  if (!s || !t || !loss_out || !workspace) return KDCC_EINVAL;
  if (N <= 0 || C <= 0 || HW <= 0 || !(T > 0.f)) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16) return KDCC_EINVAL;
  if (workspace_bytes < kdcc_loss_workspace_bytes()) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = dtype == KDCC_F32 ? 4 : 2;
  KdParams p;
  p.s = s; p.t = t; p.ds = ds;
  p.partials = static_cast<float *>(workspace);
  p.HW = HW; p.bs = batch_stride; p.cs = class_stride; p.ps = pixel_stride;
  p.C = C; p.target_is_prob = target_is_prob;
  p.k2 = kLog2e / T;
  p.gcoef = (float)((double)grad_scale * (double)T / ((double)N * (double)HW));
  // two pixels per thread when the pixel axis is contiguous and everything stays 2-element aligned
  const size_t valign = 2 * esz;
  const bool vec2 = C <= 32 && pixel_stride == 1 && (HW % 2 == 0) && (batch_stride % 2 == 0) &&
                    (class_stride % 2 == 0) && ((uintptr_t)s % valign == 0) && ((uintptr_t)t % valign == 0) &&
                    (ds == nullptr || (uintptr_t)ds % valign == 0);
  p.HWg = vec2 ? HW / 2 : HW;
  p.groups = (long)N * p.HWg;
  const int grid = (int)min((long)kMaxLossBlocks, ceil_div<long>(p.groups, kLossThreads));
  int used;
  if (dtype == KDCC_F32) used = launch_kd<float>(p, vec2, grid, st);
  else used = launch_kd<__nv_bfloat16>(p, vec2, grid, st);
  int rc = launch_status();
  if (rc) return rc;
  const double coef = (double)kLn2 * (double)T * (double)T / ((double)N * (double)HW);
  launch_pdl(loss_finalize_kernel, dim3(1), dim3(256), 0, st, p.partials, used, coef, loss_out);
  return launch_status();
}

template <typename T>
static void launch_kd_multi(const KdMultiParams &p, bool vec2, int grid, cudaStream_t st) {
#define KDM_LAUNCH(CT, EXACT)                                                             \
  do {                                                                                    \
    if (vec2 && CT <= 10) kd_multi_kernel<T, CT, EXACT, 2><<<grid, kLossThreads, 0, st>>>(p); \
    else kd_multi_kernel<T, CT, EXACT, 1><<<grid, kLossThreads, 0, st>>>(p);              \
  } while (0)
  if (p.C == 19) KDM_LAUNCH(19, true);
  else if (p.C == 10) KDM_LAUNCH(10, true);
  else if (p.C <= 16) KDM_LAUNCH(16, false);
  else KDM_LAUNCH(32, false);
#undef KDM_LAUNCH
}

KDCC_API int kdcc_kd_loss_multi(const void *s, const void *const *teachers, const float *weights, int K, void *ds,
                                float *loss_out, void *workspace, size_t workspace_bytes, int N, int C, long HW,
                                long batch_stride, long class_stride, long pixel_stride, float T, int dtype,
                                float grad_scale, kdcc_stream_t stream) {
  if (!s || !teachers || !weights || !loss_out || !workspace) return KDCC_EINVAL;
  if (N <= 0 || C <= 0 || HW <= 0 || !(T > 0.f) || K <= 0) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16) return KDCC_EINVAL;
  if (K > kMaxTeachers || C > 32) return KDCC_ESHAPE;
  if (workspace_bytes < kdcc_loss_workspace_bytes()) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t esz = dtype == KDCC_F32 ? 4 : 2;
  KdMultiParams p{};
  p.s = s; p.ds = ds; p.K = K;
  p.partials = static_cast<float *>(workspace);
  p.HW = HW; p.bs = batch_stride; p.cs = class_stride; p.ps = pixel_stride; p.C = C;
  p.k2 = kLog2e / T;
  p.gcoef = (float)((double)grad_scale * (double)T / ((double)N * (double)HW));
  const size_t valign = 2 * esz;
  bool vec2 = pixel_stride == 1 && (HW % 2 == 0) && (batch_stride % 2 == 0) && (class_stride % 2 == 0) &&
              ((uintptr_t)s % valign == 0) && (ds == nullptr || (uintptr_t)ds % valign == 0);
  double wsum = 0.0;
  for (int k = 0; k < K; ++k) {
    if (!teachers[k]) return KDCC_EINVAL;
    p.t[k] = teachers[k];
    p.w[k] = weights[k];
    wsum += weights[k];
    vec2 = vec2 && ((uintptr_t)teachers[k] % valign == 0);
  }
  p.wsum = (float)wsum;
  vec2 = vec2 && C == 10;  // three C x PIX register arrays: two pixels per thread only fit for the small class count
  p.HWg = vec2 ? HW / 2 : HW;
  p.groups = (long)N * p.HWg;
  const int grid = (int)min((long)kMaxLossBlocks, ceil_div<long>(p.groups, kLossThreads));
  if (dtype == KDCC_F32) launch_kd_multi<float>(p, vec2, grid, st);
  else launch_kd_multi<__nv_bfloat16>(p, vec2, grid, st);
  int rc = launch_status();
  if (rc) return rc;
  const double coef = (double)kLn2 * (double)T * (double)T / ((double)N * (double)HW);
  launch_pdl(loss_finalize_kernel, dim3(1), dim3(256), 0, st, p.partials, grid, coef, loss_out);
  return launch_status();
}

template <typename T>
static int launch_hint(const HintParams &p, bool vectorised, cudaStream_t st) {
  using V = Vec16<T>;
  if (vectorised) {
    const long nvec = p.total / V::N;
    const int grid = (int)min((long)kMaxLossBlocks, ceil_div<long>(nvec, (long)kLossThreads * 4));
    if (p.coef) launch_pdl(hint_loss_kernel<T, true, 4>, dim3(grid), dim3(kLossThreads), 0, st, p);
    else launch_pdl(hint_loss_kernel<T, false, 4>, dim3(grid), dim3(kLossThreads), 0, st, p);
    return grid;
  }
  const int grid = (int)min((long)kMaxLossBlocks, ceil_div<long>(p.total, kLossThreads));
  hint_loss_scalar_kernel<T><<<grid, kLossThreads, 0, st>>>(p);
  return grid;
}

KDCC_API int kdcc_hint_loss(const void *s, const void *t, const float *w, int w_per_sample, void *ds,
                            float *loss_out, void *workspace, size_t workspace_bytes, int N, int C, long HW,
                            int layout, float scale, int dtype, float grad_scale, kdcc_stream_t stream) {
  if (!s || !t || !loss_out || !workspace) return KDCC_EINVAL;
  if (N <= 0 || C <= 0 || HW <= 0) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16) return KDCC_EINVAL;
  if (layout != KDCC_LAYOUT_NHWC && layout != KDCC_LAYOUT_NCHW) return KDCC_EINVAL;
  const size_t need = kdcc_loss_workspace_bytes() + (w ? sizeof(float) * (size_t)N * C : 0);
  if (workspace_bytes < need) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HintParams p;
  p.s = s; p.t = t; p.ds = ds;
  p.partials = static_cast<float *>(workspace);
  p.coef = nullptr;
  p.total = (long)N * C * HW;
  p.HW = HW; p.C = C; p.layout = layout;
  p.ucoef = (float)((double)scale / ((double)N * (double)C * (double)HW));
  p.g2 = 2.f * grad_scale;
  if (w) {
    float *coef = p.partials + kMaxLossBlocks;
    hint_coef_kernel<<<N, 256, 0, st>>>(w, w_per_sample, C, (double)scale / ((double)HW * (double)N), coef);
    int rc = launch_status();
    if (rc) return rc;
    p.coef = coef;
  }
  const int vn = dtype == KDCC_F32 ? 4 : 8;
  const bool chan_ok = !w || (layout == KDCC_LAYOUT_NHWC ? C % vn == 0 : HW % vn == 0);
  const bool vectorised = chan_ok && (p.total % vn == 0) && aligned16(s) && aligned16(t) && (!ds || aligned16(ds));
  int used;
  if (dtype == KDCC_F32) used = launch_hint<float>(p, vectorised, st);
  else used = launch_hint<__nv_bfloat16>(p, vectorised, st);
  int rc = launch_status();
  if (rc) return rc;
  launch_pdl(loss_finalize_kernel, dim3(1), dim3(256), 0, st, p.partials, used, 1.0, loss_out);
  return launch_status();
}

KDCC_API int kdcc_cast_f32_to_bf16(const float *src, void *dst, long n, kdcc_stream_t stream) {
  if (!src || !dst || n < 0) return KDCC_EINVAL;
  if (n == 0) return KDCC_OK;
  const int grid = (int)min((long)kNumSMs * 8, ceil_div<long>(n, 256));
  launch_pdl(cast_f32_to_bf16_kernel, dim3(grid), dim3(256), 0, static_cast<cudaStream_t>(stream), src, static_cast<__nv_bfloat16 *>(dst), n);
  return launch_status();
}

KDCC_API int kdcc_scale_inplace_expect(void *buf, const float *dev_scalar, float expected, long n, int dtype, kdcc_stream_t stream) {
  if (!buf || !dev_scalar || n < 0 || !(expected != 0.f)) return KDCC_EINVAL;
  if (n == 0) return KDCC_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = (int)min((long)kNumSMs * 8, ceil_div<long>(n, 256 * 8));
  if (dtype == KDCC_F32) scale_inplace_kernel<float><<<grid, 256, 0, st>>>(static_cast<float *>(buf), dev_scalar, expected, n);
  else if (dtype == KDCC_BF16)
    scale_inplace_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<__nv_bfloat16 *>(buf), dev_scalar, expected, n);
  else return KDCC_EINVAL;
  return launch_status();
}

KDCC_API int kdcc_scale_inplace(void *buf, const float *dev_scalar, long n, int dtype, kdcc_stream_t stream) {
  return kdcc_scale_inplace_expect(buf, dev_scalar, 1.f, n, dtype, stream);
}

static int colsum_splits(long M) { return (int)max(1L, min(256L, M / 256)); }

KDCC_API size_t kdcc_colsum_workspace_bytes(long M, int Nc) {
  return sizeof(float) * (size_t)colsum_splits(M) * (size_t)Nc;
}

KDCC_API int kdcc_colsum(const void *a, float *out, void *workspace, size_t workspace_bytes, long M, int Nc,
                         int dtype, kdcc_stream_t stream) {
  if (!a || !out || !workspace || M <= 0 || Nc <= 0) return KDCC_EINVAL;
  if (workspace_bytes < kdcc_colsum_workspace_bytes(M, Nc)) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int splits = colsum_splits(M);
  const long rows_per = ceil_div<long>(M, splits);
  dim3 grid(ceil_div(Nc, 32), splits);
  float *part = static_cast<float *>(workspace);
  if (dtype == KDCC_F32)
    colsum_partial_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float *>(a), part, M, Nc, rows_per);
  else if (dtype == KDCC_BF16)
    colsum_partial_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16 *>(a), part, M, Nc, rows_per);
  else return KDCC_EINVAL;
  int rc = launch_status();
  if (rc) return rc;
  colsum_final_kernel<<<ceil_div(Nc, 128), 128, 0, st>>>(part, out, splits, Nc);
  return launch_status();
}
