// Supervised cross-entropy of the segmentation loops and the logged-only statistics of one layerwise step (sm_100a).
//   ce_loss_kernel       losses/CrossEntropy.py:10-15 (CrossEntropyLoss2d = NLLLoss2d(log_softmax(inputs, 1), weight,
//                        ignore_index)): value and gradient in one pass over the logits
//   logits_stats_kernel  trainer/layerwise_trainer.py:225-227,244-250: CE(student), CE(teacher), the KD term and both
//                        confusion matrices in ONE read of the two logit tensors and the labels, no gradient
//   ensemble_loss_kernel trainer/ensemble_trainer.py:73-90: multi-teacher KD + CE and one gradient of their sum in ONE
//                        pass over the student logits, every teacher and the labels
// All are HBM-bound and follow loss_kernels.cu: logits in registers ([CT][PIX], two pixels per thread on class planes),
// fp32 math with exp2 / log2, a fixed-order block reduction into per-CTA partials and a one-block double finalize, so
// every scalar is bit-reproducible run to run.  Confusion counts are integers (shared-memory atomics, as metrics.cu).
#include "loss_common.cuh"

namespace kdcc {

constexpr int kCeMaxC = 32;
constexpr int kCeWarps = kLossThreads / 32;

// Per-CTA partial sums in the workspace: kCeSlots arrays of `stride` floats (stride = ce_blocks(N, HW) >= the grid),
// then one float: the mean-mode gradient coefficient written by the label pre-pass.
enum { kSlotCeS = 0, kSlotW = 1, kSlotCeT = 2, kSlotKd = 3, kSlotPre = 4, kCeSlots = 5 };

static inline long ce_blocks(int N, long HW) {
  return max(1L, min((long)kMaxLossBlocks, ceil_div<long>((long)max(N, 1) * max(HW, 1L), kLossThreads)));
}

struct CeParams {
  const void *s, *t;           // t: logits_stats only (nullable)
  const long long *labels;     // int64 [N][HW]
  const float *weight;         // fp32 [C] or nullptr (all 1)
  void *ds;                    // ce_loss only (nullable)
  float *part;                 // [kCeSlots][stride]
  long stride;
  const float *gcoef_dev;      // mean-mode gradient coefficient (label pre-pass), or nullptr: use gcoef
  float gcoef;
  unsigned long long *bad;     // nullable: += labels outside [0, C) that are not ignore_index
  unsigned long long *conf_s, *conf_t;  // nullable, [C][C]
  long HW, bs, cs, ps;
  long groups, HWg;
  int C, ignore;
  int kd_mode;                 // 0 none, 1 KL(T), 2 MSE
  int kd_shared;               // kd_mode 1 with T == 1: the CE exponentials are the KD exponentials
  float kd_k2;                 // log2(e) / T
};

template <int PIX>
__device__ __forceinline__ void load_labels(const long long *p, long long (&l)[PIX]) {
  if constexpr (PIX == 2) {
    const longlong2 v = __ldcs(reinterpret_cast<const longlong2 *>(p));
    l[0] = v.x; l[1] = v.y;
  } else {
    l[0] = __ldcs(p);
  }
}

// A label counts when it is a class index and not ignore_index; anything else outside [0, C) is dropped and counted,
// never used as an index.  Returns the class (-1: dropped) and its weight (0 when dropped).
__device__ __forceinline__ int ce_class(long long lab, int C, int ignore, const float *wsh, float &w, int &bad) {
  const bool in = lab >= 0 && lab < C;
  bad += (!in && lab != ignore) ? 1 : 0;
  const int cls = (in && lab != ignore) ? (int)lab : -1;
  w = cls >= 0 ? wsh[cls] : 0.f;
  return cls;
}

__device__ __forceinline__ void ce_load_weights(const float *weight, int C, float *wsh) {
  if (threadIdx.x < kCeMaxC) wsh[threadIdx.x] = (weight != nullptr && (int)threadIdx.x < C) ? __ldg(weight + threadIdx.x) : 1.f;
}

// bad-label count of the CTA -> one global integer atomic; call before a __syncthreads-bearing reduction
__device__ __forceinline__ void ce_count_bad(int bad, unsigned int *bad_sh) {
  if (bad) atomicAdd(bad_sh, (unsigned int)bad);
}

// Label pre-pass of the mean-mode gradient: sum_valid w over the labels only (8 bytes a pixel), so that the main pass
// can write the normalised gradient directly instead of rescaling it afterwards.
__global__ void __launch_bounds__(kLossThreads) ce_weight_sum_kernel(const long long *__restrict__ labels,
                                                                     const float *__restrict__ weight, long total, int C,
                                                                     int ignore, float *__restrict__ part) {
  __shared__ float scratch[32];
  __shared__ float wsh[kCeMaxC];
  ce_load_weights(weight, C, wsh);
  __syncthreads();
  float acc = 0.f;
  int bad = 0;  // counted by the main pass
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    float w;
    ce_class(__ldg(labels + i), C, ignore, wsh, w, bad);
    acc += w;
  }
  const float tot = block_sum(acc, scratch);
  if (threadIdx.x == 0) part[blockIdx.x] = tot;
}

template <typename T, int CT, bool EXACT, int PIX, bool GRAD>
__global__ void __launch_bounds__(kLossThreads, CT <= 19 ? 2 : 1) ce_loss_kernel(const CeParams p) {
  __shared__ float scratch[32];
  __shared__ float wsh[kCeMaxC];
  __shared__ unsigned int bad_sh;
  const T *__restrict__ sbase = static_cast<const T *>(p.s);
  T *__restrict__ dbase = static_cast<T *>(p.ds);
  const int C = EXACT ? CT : p.C;
  ce_load_weights(p.weight, C, wsh);
  if (threadIdx.x == 0) bad_sh = 0u;
  __syncthreads();
  const float gc = GRAD ? (p.gcoef_dev != nullptr ? __ldg(p.gcoef_dev) : p.gcoef) : 0.f;
  float lsum = 0.f, wsum = 0.f;  // loss in bits, sum of the weights of the valid pixels
  int bad = 0;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < p.groups; g += (long)gridDim.x * blockDim.x) {
    const long n = g / p.HWg;
    const long q = (g - n * p.HWg) * PIX;
    const long off = n * p.bs + q * p.ps;
    float sv[CT][PIX];
#pragma unroll
    for (int c = 0; c < CT; ++c)
      if (EXACT || c < C) load_pix<T, PIX>(sbase + off + c * p.cs, sv[c]);
    long long lab[PIX];
    load_labels<PIX>(p.labels + n * p.HW + q, lab);
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      float w;
      const int cls = ce_class(lab[i], C, p.ignore, wsh, w, bad);
      float smax = -INFINITY;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) smax = fmaxf(smax, sv[c][i]);
      // nll = logsumexp_c s - s_label = ln2 * (log2 sum_c 2^a_c - a_label), a = (s - max) * log2(e)
      float ssum = 0.f, alab = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          const float a = (sv[c][i] - smax) * kLog2e;
          const float e = exp2f(a);
          ssum += e;
          if (c == cls) alab = a;
          sv[c][i] = e;
        }
      if (cls >= 0) {
        lsum += w * (log2f(ssum) - alab);
        wsum += w;
      }
      if (GRAD) {
        // ds = gc * w * (softmax - onehot); exactly 0 at dropped pixels (gc is inf in mean mode when nothing is valid)
        const float gw = cls >= 0 ? gc * w : 0.f;
        const float rs = 1.f / ssum;
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (EXACT || c < C) sv[c][i] = gw * (sv[c][i] * rs - (c == cls ? 1.f : 0.f));
      }
    }
    if (GRAD) {
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) store_pix<T, PIX>(dbase + off + c * p.cs, sv[c]);
    }
  }
  ce_count_bad(bad, &bad_sh);
  const float l = block_sum(lsum, scratch);
  const float w = block_sum(wsum, scratch);
  if (threadIdx.x == 0) {
    p.part[kSlotCeS * p.stride + blockIdx.x] = l;
    p.part[kSlotW * p.stride + blockIdx.x] = w;
    if (bad_sh && p.bad != nullptr) atomicAdd(p.bad, (unsigned long long)bad_sh);
  }
}

// first maximum wins; a NaN beats everything (torch.argmax semantics, as confusion_kernel in metrics.cu)
__device__ __forceinline__ void argmax_step(float v, int c, float &best, int &arg) {
  if ((c == 0) || (v > best) || (v != v && best == best)) { best = v; arg = c; }
}

template <typename T, int CT, bool EXACT, int PIX, bool HAS_T>
__global__ void __launch_bounds__(kLossThreads, CT <= 19 ? 2 : 1) logits_stats_kernel(const CeParams p) {
  extern __shared__ unsigned int hist[];  // [2][warps][C*C] per-warp confusion counts (student, teacher)
  __shared__ float scratch[32];
  __shared__ float wsh[kCeMaxC];
  __shared__ unsigned int bad_sh;
  const T *__restrict__ sbase = static_cast<const T *>(p.s);
  const T *__restrict__ tbase = static_cast<const T *>(p.t);
  const int C = EXACT ? CT : p.C;
  const int cells = C * C;
  const bool conf_s = p.conf_s != nullptr, conf_t = HAS_T && p.conf_t != nullptr;
  unsigned int *hs = hist + (threadIdx.x >> 5) * cells;
  unsigned int *ht = hist + (kCeWarps + (threadIdx.x >> 5)) * cells;
  if (conf_s || conf_t)
    for (int i = threadIdx.x; i < 2 * kCeWarps * cells; i += blockDim.x) hist[i] = 0u;
  ce_load_weights(p.weight, C, wsh);
  if (threadIdx.x == 0) bad_sh = 0u;
  __syncthreads();
  float ce_s = 0.f, ce_t = 0.f, wsum = 0.f, kd = 0.f;
  int bad = 0;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < p.groups; g += (long)gridDim.x * blockDim.x) {
    const long n = g / p.HWg;
    const long q = (g - n * p.HWg) * PIX;
    const long off = n * p.bs + q * p.ps;
    float sv[CT][PIX], tv[HAS_T ? CT : 1][PIX];
#pragma unroll
    for (int c = 0; c < CT; ++c)
      if (EXACT || c < C) {
        load_pix<T, PIX>(sbase + off + c * p.cs, sv[c]);
        if (HAS_T) load_pix<T, PIX>(tbase + off + c * p.cs, tv[HAS_T ? c : 0]);
      }
    long long lab[PIX];
    load_labels<PIX>(p.labels + n * p.HW + q, lab);
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      float w;
      const int cls = ce_class(lab[i], C, p.ignore, wsh, w, bad);
      float smax = -INFINITY, tmax = -INFINITY, sbest = 0.f, tbest = 0.f;
      int sarg = 0, targ = 0;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          smax = fmaxf(smax, sv[c][i]);
          argmax_step(sv[c][i], c, sbest, sarg);
          if (HAS_T) {
            const float tvv = tv[HAS_T ? c : 0][i];
            tmax = fmaxf(tmax, tvv);
            argmax_step(tvv, c, tbest, targ);
          }
        }
      // One exponential per logit serves CE(s), CE(t) and -- with T == 1 -- the KL term (kd_loss_kernel's form:
      // KL bits = sum_c e_t (b - a) / sum e_t - log2 sum e_t + log2 sum e_s).
      float ssum = 0.f, tsum = 0.f, alab = 0.f, blab = 0.f, cross = 0.f, sq = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          const float a = (sv[c][i] - smax) * kLog2e;
          ssum += exp2f(a);
          if (c == cls) alab = a;
          if (HAS_T) {
            const float tvv = tv[HAS_T ? c : 0][i];
            const float b = (tvv - tmax) * kLog2e;
            const float et = exp2f(b);
            tsum += et;
            if (c == cls) blab = b;
            if (p.kd_shared && et > 0.f) cross += et * (b - a);
            if (p.kd_mode == 2) {
              const float d = sv[c][i] - tvv;
              sq = fmaf(d, d, sq);
            }
          }
        }
      if (cls >= 0) {
        ce_s += w * (log2f(ssum) - alab);
        if (HAS_T) ce_t += w * (log2f(tsum) - blab);
        wsum += w;
        if (conf_s) atomicAdd(&hs[cls * C + sarg], 1u);
        if (conf_t) atomicAdd(&ht[cls * C + targ], 1u);
      }
      if (HAS_T) {
        if (p.kd_shared) {
          kd += cross * (1.f / tsum) - log2f(tsum) + log2f(ssum);
        } else if (p.kd_mode == 1) {  // T != 1: the softened distributions need their own exponentials
          float s2 = 0.f, t2 = 0.f, x2 = 0.f;
#pragma unroll
          for (int c = 0; c < CT; ++c)
            if (EXACT || c < C) {
              const float a = (sv[c][i] - smax) * p.kd_k2, b = (tv[HAS_T ? c : 0][i] - tmax) * p.kd_k2;
              const float es = exp2f(a), et = exp2f(b);
              s2 += es; t2 += et;
              if (et > 0.f) x2 += et * (b - a);
            }
          kd += x2 * (1.f / t2) - log2f(t2) + log2f(s2);
        } else if (p.kd_mode == 2) {
          kd += sq;
        }
      }
    }
  }
  ce_count_bad(bad, &bad_sh);
  const float r0 = block_sum(ce_s, scratch);
  const float r1 = block_sum(wsum, scratch);
  const float r2 = HAS_T ? block_sum(ce_t, scratch) : 0.f;
  const float r3 = HAS_T ? block_sum(kd, scratch) : 0.f;
  if (threadIdx.x == 0) {
    p.part[kSlotCeS * p.stride + blockIdx.x] = r0;
    p.part[kSlotW * p.stride + blockIdx.x] = r1;
    if (HAS_T) {
      p.part[kSlotCeT * p.stride + blockIdx.x] = r2;
      p.part[kSlotKd * p.stride + blockIdx.x] = r3;
    }
    if (bad_sh && p.bad != nullptr) atomicAdd(p.bad, (unsigned long long)bad_sh);
  }
  // block_sum ended in __syncthreads: every shared-memory count of this CTA is in
  if (conf_s || conf_t) {
    for (int i = threadIdx.x; i < cells; i += blockDim.x) {
      unsigned long long a = 0, b = 0;
      for (int wp = 0; wp < kCeWarps; ++wp) {
        a += hist[(size_t)wp * cells + i];
        b += hist[(size_t)(kCeWarps + wp) * cells + i];
      }
      if (conf_s && a) atomicAdd(p.conf_s + i, a);
      if (conf_t && b) atomicAdd(p.conf_t + i, b);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// The objective of the ensemble loop (trainer/ensemble_trainer.py:73-90, loss = kd + supervised) in ONE pass over the
// student logits: every teacher is read once (kd_multi_kernel's register-resident softmax), the labels once, and
//   kd  = sum_k w_k T^2/(N*HW) sum_pix KL(softmax(t_k/T) || softmax(s/T))      (partials: kSlotKd, in bits)
//   ce  = sum_valid cw * (logsumexp s - s_label)                                 (partials: kSlotCeS / kSlotW)
//   ds  = e_kd T/(N*HW) ((sum_k w_k) softmax(s/T) - sum_k w_k softmax(t_k/T)) + e_ce cw (softmax(s) - onehot) / D
// written once.  With T == 1 the CE exponentials are the KD student exponentials.
// ------------------------------------------------------------------------------------------------
constexpr int kEnsMaxTeachers = 8;
struct EnsParams {
  const void *s;
  const void *t[kEnsMaxTeachers];
  float w[kEnsMaxTeachers];
  float wsum;
  int K;
  const long long *labels;
  const float *weight;         // class weights fp32 [C] or nullptr (all 1)
  void *ds;
  float *part;                 // [kCeSlots][stride]; nullptr on a gradient-only re-launch
  long stride;
  const float *den;            // D on the device (mean-mode label pre-pass, or out3[2]), or nullptr: D = 1
  const float *up2;            // re-launch: the actual upstream pair (g_kd, g_ce) on the device, else nullptr
  float e_kd, e_ce;            // the upstream pair folded into ds (forward) / expected (re-launch)
  unsigned long long *bad;
  long HW, bs, cs, ps;
  long groups, HWg;
  int C, ignore;
  int shared;                  // T == 1
  float k2;                    // log2(e) / T
  float kd_g;                  // T / (N*HW)
};

template <typename T, int CT, bool EXACT, int PIX, bool GRAD>
__global__ void __launch_bounds__(kLossThreads, CT <= 19 ? 2 : 1) ensemble_loss_kernel(const EnsParams p) {
  float e_kd = p.e_kd, e_ce = p.e_ce;
  if (GRAD && p.up2 != nullptr) {
    // gradient-only re-launch: the forward already wrote ds for the expected pair; every CTA leaves when it was right
    e_kd = __ldg(p.up2);
    e_ce = __ldg(p.up2 + 1);
    if (e_kd == p.e_kd && e_ce == p.e_ce) return;
  }
  __shared__ float scratch[32];
  __shared__ float wsh[kCeMaxC];
  __shared__ unsigned int bad_sh;
  const T *__restrict__ sbase = static_cast<const T *>(p.s);
  T *__restrict__ dbase = static_cast<T *>(p.ds);
  const int C = EXACT ? CT : p.C;
  ce_load_weights(p.weight, C, wsh);
  if (threadIdx.x == 0) bad_sh = 0u;
  __syncthreads();
  const float cc = GRAD ? e_ce / (p.den != nullptr ? __ldg(p.den) : 1.f) : 0.f;
  const float kc = GRAD ? e_kd * p.kd_g : 0.f;
  float lsum = 0.f, wsum = 0.f, kd = 0.f;
  int bad = 0;
  for (long g = (long)blockIdx.x * blockDim.x + threadIdx.x; g < p.groups; g += (long)gridDim.x * blockDim.x) {
    const long n = g / p.HWg;
    const long q = (g - n * p.HWg) * PIX;
    const long off = n * p.bs + q * p.ps;
    // sv: log2 softmax(s/T); gd: the gradient, built up teacher by teacher; kl: sum_k w_k KL_k in bits
    float sv[CT][PIX], gd[GRAD ? CT : 1][PIX], kl[PIX];
#pragma unroll
    for (int c = 0; c < CT; ++c)
      if (EXACT || c < C) load_pix<T, PIX>(sbase + off + c * p.cs, sv[c]);
    long long lab[PIX];
    load_labels<PIX>(p.labels + n * p.HW + q, lab);
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      float w;
      const int cls = ce_class(lab[i], C, p.ignore, wsh, w, bad);
      float smax = -INFINITY;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) smax = fmaxf(smax, sv[c][i]);
      // e1 = 2^a (CE, kept in gd), e2 = 2^(a/T) (KD): the same exponential when T == 1
      float e2[CT];
      float s1 = 0.f, s2 = 0.f, alab = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          const float d = sv[c][i] - smax;
          const float a = d * kLog2e;
          const float e1 = exp2f(a);
          s1 += e1;
          if (c == cls) alab = a;
          e2[c] = p.shared ? e1 : exp2f(d * p.k2);
          s2 += e2[c];
          sv[c][i] = d * p.k2;
          if (GRAD) gd[c][i] = e1;
        }
      if (cls >= 0) {
        lsum += w * (log2f(s1) - alab);
        wsum += w;
      }
      const float l2 = log2f(s2), r2 = 1.f / s2, r1 = 1.f / s1;
      const float gw = cls >= 0 ? cc * w : 0.f;   // the CE part is exactly 0 at dropped pixels
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          if (GRAD) gd[c][i] = kc * p.wsum * (e2[c] * r2) + gw * (gd[c][i] * r1 - (c == cls ? 1.f : 0.f));
          sv[c][i] -= l2;
        }
      kl[i] = 0.f;
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
        // one exponential per teacher logit: KL_k bits = (sum_c e b) / Z - log2 Z - (sum_c e log2 p_s) / Z
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
        const float wr = wk * rt, gk = -kc * wr;
        float xs = 0.f;
#pragma unroll
        for (int c = 0; c < CT; ++c)
          if (EXACT || c < C) {
            if (tv[c][i] > 0.f) xs += tv[c][i] * sv[c][i];
            if (GRAD) gd[c][i] = fmaf(gk, tv[c][i], gd[c][i]);
          }
        kl[i] += wk * (tb * rt - log2f(tsum)) - wr * xs;
      }
    }
#pragma unroll
    for (int i = 0; i < PIX; ++i) kd += kl[i];
    if (GRAD) {
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) store_pix<T, PIX>(dbase + off + c * p.cs, gd[c]);
    }
  }
  if (p.part == nullptr) return;   // uniform: a re-launch writes the gradient only
  ce_count_bad(bad, &bad_sh);
  const float r0 = block_sum(lsum, scratch);
  const float r1 = block_sum(wsum, scratch);
  const float r2 = block_sum(kd, scratch);
  if (threadIdx.x == 0) {
    p.part[kSlotCeS * p.stride + blockIdx.x] = r0;
    p.part[kSlotW * p.stride + blockIdx.x] = r1;
    p.part[kSlotKd * p.stride + blockIdx.x] = r2;
    if (bad_sh && p.bad != nullptr) atomicAdd(p.bad, (unsigned long long)bad_sh);
  }
}

// Fixed-order double sums of the per-CTA partials and the scalars made from them.
struct CeFinal {
  const float *part;
  long stride;
  int count;
  int mode;          // 0: gradient coefficient of the pre-pass, 1: CE loss, 2: logits statistics,
                     // 3: normaliser of the pre-pass (sum_valid w), 4: ensemble objective
  unsigned slots;    // bit k: slot k was written
  int mean;
  int den_done;      // mode 4: out[2] already holds the D of the pre-pass
  double gscale;     // mode 0: grad_scale
  double kd_coef;    // mode 2: scale of the KD partial sum
  float *out;
};

__global__ void __launch_bounds__(256) ce_finalize_kernel(const CeFinal f) {
  __shared__ double sh[256];
  __shared__ double tot[kCeSlots];
  pdl_prologue_done();
  for (int k = 0; k < kCeSlots; ++k) {
    if (!(f.slots & (1u << k))) continue;
    const float *pk = f.part + k * f.stride;
    double acc = 0.0;
    for (int i = threadIdx.x; i < f.count; i += 256) acc += (double)pk[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
      if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
      __syncthreads();
    }
    if (threadIdx.x == 0) tot[k] = sh[0];
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const double ln2 = (double)kLn2;
  const double den = f.mean ? tot[kSlotW] : 1.0;  // mean with no valid pixel: 0 / 0 = NaN, as torch
  if (f.mode == 0) {
    f.out[0] = (float)(f.gscale / tot[kSlotPre]);
  } else if (f.mode == 1) {
    f.out[0] = (float)(ln2 * tot[kSlotCeS] / den);
  } else if (f.mode == 3) {
    f.out[0] = (float)tot[kSlotPre];
  } else if (f.mode == 4) {
    f.out[0] = (float)(f.kd_coef * tot[kSlotKd]);
    f.out[1] = (float)(ln2 * tot[kSlotCeS] / den);
    if (!f.den_done) f.out[2] = (float)den;
  } else {
    f.out[1] = (float)(ln2 * tot[kSlotCeS] / den);
    if (f.slots & (1u << kSlotCeT)) f.out[2] = (float)(ln2 * tot[kSlotCeT] / den);
    if (f.slots & (1u << kSlotKd)) f.out[0] = (float)(f.kd_coef * tot[kSlotKd]);
  }
}

}  // namespace kdcc

using namespace kdcc;

KDCC_API size_t kdcc_ce_workspace_bytes(int N, long HW) {
  return sizeof(float) * (size_t)(kCeSlots * ce_blocks(N, HW) + 4);
}

static int ce_args(int N, int C, long HW, int dtype) {
  if (N <= 0 || C <= 0 || HW <= 0) return KDCC_EINVAL;
  if (dtype != KDCC_F32 && dtype != KDCC_BF16) return KDCC_EINVAL;
  if (C > kCeMaxC) return KDCC_ESHAPE;
  return KDCC_OK;
}

// two pixels per thread when the pixel axis is contiguous and every access of a pair stays aligned
static bool ce_vec2(const void *s, const void *t, const void *ds, const long long *labels, long HW, long bs, long cs,
                    long ps, int dtype) {
  const uintptr_t va = dtype == KDCC_F32 ? 8 : 4;
  return ps == 1 && HW % 2 == 0 && bs % 2 == 0 && cs % 2 == 0 && (uintptr_t)s % va == 0 &&
         (t == nullptr || (uintptr_t)t % va == 0) && (ds == nullptr || (uintptr_t)ds % va == 0) && aligned16(labels);
}

template <typename T, bool GRAD>
static void launch_ce(const CeParams &p, bool vec2, int grid, cudaStream_t st) {
#define CE_LAUNCH(CT, EXACT)                                                                  \
  do {                                                                                        \
    if (vec2) ce_loss_kernel<T, CT, EXACT, 2, GRAD><<<grid, kLossThreads, 0, st>>>(p);       \
    else ce_loss_kernel<T, CT, EXACT, 1, GRAD><<<grid, kLossThreads, 0, st>>>(p);            \
  } while (0)
  if (p.C == 19) CE_LAUNCH(19, true);
  else if (p.C <= 16) CE_LAUNCH(16, false);
  else CE_LAUNCH(32, false);
#undef CE_LAUNCH
}

KDCC_API int kdcc_ce_loss(const void *s, const long long *labels, const float *weight, int ignore_index, int mean,
                          void *ds, float *loss_out, long long *bad_labels, void *workspace, size_t workspace_bytes,
                          int N, int C, long HW, long batch_stride, long class_stride, long pixel_stride, int dtype,
                          float grad_scale, kdcc_stream_t stream) {
  int rc = ce_args(N, C, HW, dtype);
  if (rc) return rc;
  if (!s || !labels || !loss_out || !workspace) return KDCC_EINVAL;
  if (workspace_bytes < kdcc_ce_workspace_bytes(N, HW)) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CeParams p{};
  p.s = s; p.labels = labels; p.weight = weight; p.ds = ds;
  p.part = static_cast<float *>(workspace);
  p.stride = ce_blocks(N, HW);
  p.bad = reinterpret_cast<unsigned long long *>(bad_labels);
  p.HW = HW; p.bs = batch_stride; p.cs = class_stride; p.ps = pixel_stride;
  p.C = C; p.ignore = ignore_index;
  p.gcoef = grad_scale;
  const bool vec2 = ce_vec2(s, nullptr, ds, labels, HW, batch_stride, class_stride, pixel_stride, dtype);
  p.HWg = vec2 ? HW / 2 : HW;
  p.groups = (long)N * p.HWg;
  const int grid = (int)min(p.stride, ceil_div<long>(p.groups, kLossThreads));
  if (ds != nullptr && mean) {
    // the gradient is normalised by sum_valid w: one read of the labels first, then the main pass writes ds once
    float *coef = p.part + kCeSlots * p.stride;
    ce_weight_sum_kernel<<<(int)p.stride, kLossThreads, 0, st>>>(labels, weight, (long)N * HW, C, ignore_index,
                                                                 p.part + kSlotPre * p.stride);
    if ((rc = launch_status())) return rc;
    CeFinal f{};
    f.part = p.part; f.stride = p.stride; f.count = (int)p.stride; f.mode = 0; f.slots = 1u << kSlotPre;
    f.gscale = grad_scale; f.out = coef;
    launch_pdl(ce_finalize_kernel, dim3(1), dim3(256), 0, st, f);
    if ((rc = launch_status())) return rc;
    p.gcoef_dev = coef;
  }
  if (ds != nullptr) {
    if (dtype == KDCC_F32) launch_ce<float, true>(p, vec2, grid, st);
    else launch_ce<__nv_bfloat16, true>(p, vec2, grid, st);
  } else {
    if (dtype == KDCC_F32) launch_ce<float, false>(p, vec2, grid, st);
    else launch_ce<__nv_bfloat16, false>(p, vec2, grid, st);
  }
  if ((rc = launch_status())) return rc;
  CeFinal f{};
  f.part = p.part; f.stride = p.stride; f.count = grid; f.mode = 1;
  f.slots = (1u << kSlotCeS) | (1u << kSlotW); f.mean = mean; f.out = loss_out;
  launch_pdl(ce_finalize_kernel, dim3(1), dim3(256), 0, st, f);
  return launch_status();
}

template <typename T, bool GRAD>
static void launch_ensemble(const EnsParams &p, bool vec2, int grid, cudaStream_t st) {
// two pixels per thread only for the 10-class planes: with three C x PIX register arrays the 16 / 19 / 32 forms would spill
#define ENS_LAUNCH(CT, EXACT)                                                                                   \
  do {                                                                                                          \
    if constexpr (CT == 10) {                                                                                   \
      if (vec2) { ensemble_loss_kernel<T, CT, EXACT, 2, GRAD><<<grid, kLossThreads, 0, st>>>(p); break; }       \
    }                                                                                                           \
    ensemble_loss_kernel<T, CT, EXACT, 1, GRAD><<<grid, kLossThreads, 0, st>>>(p);                              \
  } while (0)
  if (p.C == 19) ENS_LAUNCH(19, true);
  else if (p.C == 10) ENS_LAUNCH(10, true);
  else if (p.C <= 16) ENS_LAUNCH(16, false);
  else ENS_LAUNCH(32, false);
#undef ENS_LAUNCH
}

KDCC_API int kdcc_ensemble_loss(const void *s, const void *const *teachers, const float *kd_weights, int K, float T,
                                const long long *labels, const float *class_weight, int ignore_index, int mean,
                                void *ds, float *out3, long long *bad_labels, void *workspace, size_t workspace_bytes,
                                int N, int C, long HW, long batch_stride, long class_stride, long pixel_stride, int dtype,
                                float kd_grad_scale, float ce_grad_scale, const float *upstream2, kdcc_stream_t stream) {
  int rc = ce_args(N, C, HW, dtype);
  if (rc) return rc;
  if (K < 1 || K > kEnsMaxTeachers || !(T > 0.f)) return KDCC_EINVAL;
  if (!s || !teachers || !kd_weights || !labels || !out3 || !workspace || (upstream2 && !ds)) return KDCC_EINVAL;
  for (int k = 0; k < K; ++k)
    if (!teachers[k]) return KDCC_EINVAL;
  if (workspace_bytes < kdcc_ce_workspace_bytes(N, HW)) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  EnsParams p{};
  p.s = s; p.K = K; p.labels = labels; p.weight = class_weight; p.ds = ds;
  double wsum = 0.0;
  bool vec2 = ce_vec2(s, nullptr, ds, labels, HW, batch_stride, class_stride, pixel_stride, dtype) && C == 10;
  const uintptr_t va = dtype == KDCC_F32 ? 8 : 4;
  for (int k = 0; k < K; ++k) {
    p.t[k] = teachers[k];
    p.w[k] = kd_weights[k];
    wsum += kd_weights[k];
    vec2 = vec2 && (uintptr_t)teachers[k] % va == 0;
  }
  p.wsum = (float)wsum;
  p.part = static_cast<float *>(workspace);
  p.stride = ce_blocks(N, HW);
  p.bad = reinterpret_cast<unsigned long long *>(bad_labels);
  p.e_kd = kd_grad_scale; p.e_ce = ce_grad_scale;
  p.HW = HW; p.bs = batch_stride; p.cs = class_stride; p.ps = pixel_stride;
  p.C = C; p.ignore = ignore_index;
  p.shared = T == 1.f;
  p.k2 = kLog2e / T;
  p.kd_g = (float)((double)T / ((double)N * (double)HW));
  p.HWg = vec2 ? HW / 2 : HW;
  p.groups = (long)N * p.HWg;
  const int grid = (int)min(p.stride, ceil_div<long>(p.groups, kLossThreads));
  const bool f32 = dtype == KDCC_F32;
  if (upstream2 != nullptr) {
    // gradient-only re-launch for the upstream pair autograd actually handed over; D is the one the forward used
    p.up2 = upstream2;
    p.den = out3 + 2;
    p.part = nullptr;
    p.bad = nullptr;
    if (f32) launch_ensemble<float, true>(p, vec2, grid, st);
    else launch_ensemble<__nv_bfloat16, true>(p, vec2, grid, st);
    return launch_status();
  }
  const bool pre = ds != nullptr && mean;
  if (pre) {
    // D = sum_valid w from one read of the labels, so that the main pass writes ds once, already normalised
    ce_weight_sum_kernel<<<(int)p.stride, kLossThreads, 0, st>>>(labels, class_weight, (long)N * HW, C, ignore_index,
                                                                 p.part + kSlotPre * p.stride);
    if ((rc = launch_status())) return rc;
    CeFinal f{};
    f.part = p.part; f.stride = p.stride; f.count = (int)p.stride; f.mode = 3; f.slots = 1u << kSlotPre;
    f.out = out3 + 2;
    launch_pdl(ce_finalize_kernel, dim3(1), dim3(256), 0, st, f);
    if ((rc = launch_status())) return rc;
    p.den = out3 + 2;
  }
  if (ds != nullptr) {
    if (f32) launch_ensemble<float, true>(p, vec2, grid, st);
    else launch_ensemble<__nv_bfloat16, true>(p, vec2, grid, st);
  } else {
    if (f32) launch_ensemble<float, false>(p, vec2, grid, st);
    else launch_ensemble<__nv_bfloat16, false>(p, vec2, grid, st);
  }
  if ((rc = launch_status())) return rc;
  CeFinal f{};
  f.part = p.part; f.stride = p.stride; f.count = grid; f.mode = 4; f.mean = mean; f.out = out3;
  f.slots = (1u << kSlotCeS) | (1u << kSlotW) | (1u << kSlotKd);
  f.den_done = pre;   // keep the D the gradient was formed with
  f.kd_coef = (double)kLn2 * (double)T * (double)T / ((double)N * (double)HW);
  launch_pdl(ce_finalize_kernel, dim3(1), dim3(256), 0, st, f);
  return launch_status();
}

template <typename K>
static int launch_stats_kernel(K *kernel, const CeParams &p, int grid, size_t dyn, int (&cache)[16], cudaStream_t st) {
  if (dyn > 48 * 1024) {
    const int rc = ensure_dynamic_smem(kernel, (int)dyn, cache);
    if (rc) return rc;
  }
  kernel<<<grid, kLossThreads, dyn, st>>>(p);
  return launch_status();
}

template <typename T, bool HAS_T>
static int launch_stats(const CeParams &p, bool vec2, int grid, size_t dyn, cudaStream_t st) {
// two pixels per thread with a teacher only for the exact 19 classes: the predicated 16 / 32 forms would spill
#define ST_LAUNCH(CT, EXACT)                                                                                          \
  do {                                                                                                                \
    static int cache2[16], cache1[16];                                                                                \
    if constexpr (EXACT || !HAS_T) {                                                                                  \
      if (vec2) return launch_stats_kernel(logits_stats_kernel<T, CT, EXACT, 2, HAS_T>, p, grid, dyn, cache2, st);    \
    }                                                                                                                 \
    return launch_stats_kernel(logits_stats_kernel<T, CT, EXACT, 1, HAS_T>, p, grid, dyn, cache1, st);                \
  } while (0)
  if (p.C == 19) ST_LAUNCH(19, true);
  else if (p.C <= 16) ST_LAUNCH(16, false);
  else ST_LAUNCH(32, false);
#undef ST_LAUNCH
}

KDCC_API int kdcc_logits_stats(const void *s, const void *t, const long long *labels, const float *weight,
                               int ignore_index, int mean, int kd_mode, float T, float kd_scale, float *out3,
                               long long *conf_s, long long *conf_t, long long *bad_labels, void *workspace,
                               size_t workspace_bytes, int N, int C, long HW, long batch_stride, long class_stride,
                               long pixel_stride, int dtype, kdcc_stream_t stream) {
  int rc = ce_args(N, C, HW, dtype);
  if (rc) return rc;
  if (kd_mode < 0 || kd_mode > 2 || (kd_mode == 1 && !(T > 0.f))) return KDCC_EINVAL;
  if (!s || !labels || !out3 || !workspace) return KDCC_EINVAL;
  if (workspace_bytes < kdcc_ce_workspace_bytes(N, HW)) return KDCC_EWORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool has_t = t != nullptr;
  CeParams p{};
  p.s = s; p.t = t; p.labels = labels; p.weight = weight;
  p.part = static_cast<float *>(workspace);
  p.stride = ce_blocks(N, HW);
  p.bad = reinterpret_cast<unsigned long long *>(bad_labels);
  p.conf_s = reinterpret_cast<unsigned long long *>(conf_s);
  p.conf_t = has_t ? reinterpret_cast<unsigned long long *>(conf_t) : nullptr;
  p.HW = HW; p.bs = batch_stride; p.cs = class_stride; p.ps = pixel_stride;
  p.C = C; p.ignore = ignore_index;
  p.kd_mode = has_t ? kd_mode : 0;
  p.kd_shared = p.kd_mode == 1 && T == 1.f;
  p.kd_k2 = kd_mode == 1 ? kLog2e / T : 0.f;
  const bool vec2 = ce_vec2(s, t, nullptr, labels, HW, batch_stride, class_stride, pixel_stride, dtype) && (!has_t || C == 19);
  p.HWg = vec2 ? HW / 2 : HW;
  p.groups = (long)N * p.HWg;
  const int grid = (int)min(p.stride, ceil_div<long>(p.groups, kLossThreads));
  const size_t dyn = (p.conf_s || p.conf_t) ? sizeof(unsigned int) * 2 * kCeWarps * C * C : 0;
  if (dtype == KDCC_F32) rc = has_t ? launch_stats<float, true>(p, vec2, grid, dyn, st) : launch_stats<float, false>(p, vec2, grid, dyn, st);
  else rc = has_t ? launch_stats<__nv_bfloat16, true>(p, vec2, grid, dyn, st) : launch_stats<__nv_bfloat16, false>(p, vec2, grid, dyn, st);
  if (rc) return rc;
  CeFinal f{};
  f.part = p.part; f.stride = p.stride; f.count = grid; f.mode = 2; f.mean = mean; f.out = out3;
  f.slots = (1u << kSlotCeS) | (1u << kSlotW);
  if (has_t) f.slots |= 1u << kSlotCeT;
  if (p.kd_mode) f.slots |= 1u << kSlotKd;
  if (p.kd_mode == 1) f.kd_coef = (double)kLn2 * (double)T * (double)T / ((double)N * (double)HW);
  if (p.kd_mode == 2) f.kd_coef = (double)kd_scale / ((double)N * (double)C * (double)HW);
  launch_pdl(ce_finalize_kernel, dim3(1), dim3(256), 0, st, f);
  return launch_status();
}
