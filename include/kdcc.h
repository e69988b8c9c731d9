/*
 * kdcc.h -- C ABI of libkdcc.so: the sm_100a (B200) kernels behind the distillation hot path of
 * lehduong/Knowledge-Distillation-by-Replacing-Cheap-Conv.
 *
 * The reference has no FFI of its own (it is pure PyTorch, SURVEY.md F1); each entry point below
 * replaces the torch library call(s) that one reference call site makes, cited as
 * reference-file:line.  INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch caching allocator); the library
 *     allocates nothing persistent apart from cached TMA descriptors / function attributes;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - entry points are re-entrant and hold no thread-affine state (autograd calls backward from its
 *     own worker thread);
 *   - activations are either NHWC-physical (torch.channels_last, x[n][h][w][c]) or NCHW-physical (the
 *     reference's own layout, x[n][c][h][w]); every conv entry point takes a `layout` argument and the two
 *     layouts dispatch to different kernels (NCHW bf16 depthwise runs on the tensor cores); logits carry
 *     explicit strides;
 *   - dtype: KDCC_F32 (parity path, 1e-5 relative) or KDCC_BF16 (production path, fp32 accumulate);
 *   - return 0 on success, a negative KDCC_E* code for bad arguments / unsupported shapes (there is
 *     NO CPU or library fallback), or a positive cudaError_t.  kdcc_strerror() names any of them.
 */
#ifndef KDCC_H_
#define KDCC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KDCC_VERSION 104 /* round 1: layout-aware depthwise/pointwise, confusion matrix, multi-teacher KD, TTA stitch, RAdam */

enum { KDCC_F32 = 0, KDCC_BF16 = 1 };
enum { KDCC_LAYOUT_NHWC = 0, KDCC_LAYOUT_NCHW = 1,
       /* pointwise entry points only: the block-INTERNAL tensor (depthwise output `x`, its gradient `dx`) is channel planes
        * (NCHW), the block-EXTERNAL one (`y`, `dy`) is channels_last -- a block whose depthwise ran on planes inside a
        * channels_last trunk hands its result over without a separate re-layout pass */
       KDCC_LAYOUT_PLANES_TO_NHWC = 2 };

enum {
  KDCC_OK = 0,
  KDCC_EINVAL = -1,      /* null pointer / non-positive dimension / bad enum */
  KDCC_ESHAPE = -2,      /* shape not supported by the sm_100a kernels (e.g. C % 8 != 0 in bf16) */
  KDCC_EWORKSPACE = -3,  /* workspace smaller than kdcc_*_workspace_bytes() says */
  KDCC_EALIGN = -4,      /* pointer not 16-byte aligned */
  KDCC_EDEVICE = -5,     /* not an sm_100 device / driver entry point missing */
};

typedef void *kdcc_stream_t; /* cudaStream_t */

int kdcc_version(void);
const char *kdcc_strerror(int code);
/* CUresult of the calling thread's most recent TMA-descriptor encode (0 = CUDA_SUCCESS); diagnostics only. */
int kdcc_last_driver_status(void);

/* Which implementation a call would dispatch to (for tests / profiles): returns a static string such
 * as "dw_fwd_tma_k9" or "dw_fwd_direct".  op: 0 = dw_fwd, 1 = dw_bwd, 2 = pw_fwd, 3 = pw_bwd_dx,
 * 4 = pw_bwd_dw. */
const char *kdcc_dispatch_name(int op, int N, int H, int W, int C, int Cout, int k, int dil, int pad,
                               int layout, int dtype);

/* ---- depthwise k x k, stride 1, zero padding, dilation `dil` -----------------------------------
 * Replaces self.separable_conv(x)  (models/students/transform_blocks/depthwise_separable_conv.py:7-8,12
 * -> F.conv2d groups=C).  x [N,H,W,C], w fp32 [C,k,k] (the (C,1,k,k) parameter, contiguous),
 * bias fp32 [C] or NULL, y [N,Ho,Wo,C] with Ho = H + 2*pad - dil*(k-1). */
int kdcc_dw_fwd(const void *x, const float *w, const float *bias, void *y, int N, int H, int W, int C,
                int k, int dil, int pad, int layout, int dtype, kdcc_stream_t stream);

/* Autograd backward of the call above (depthwise_separable_conv.py:12 under loss.backward(),
 * trainer/layerwise_trainer.py:235).  dx [N,H,W,C] (NULL: input needs no grad), dw fp32 [C,k,k]
 * (NULL: frozen), dbias fp32 [C] or NULL.  Deterministic two-stage reduction, no atomics. */
size_t kdcc_dw_bwd_workspace_bytes(int N, int H, int W, int C, int k, int dil, int pad, int layout,
                                   int dtype);
int kdcc_dw_bwd(const void *x, const float *w, const void *dy, void *dx, float *dw, float *dbias,
                void *workspace, size_t workspace_bytes, int N, int H, int W, int C, int k, int dil,
                int pad, int layout, int dtype, kdcc_stream_t stream);

/* ---- pointwise 1x1 = GEMM ----------------------------------------------------------------------
 * Replaces self.pointwise_conv(x)  (depthwise_separable_conv.py:9,13).  M = batch*H*W pixels, K = C_in,
 * w [Nc,K] in the activation dtype (the (Co,C,1,1) parameter, cast by kdcc_cast_f32_to_bf16).
 * layout NHWC: x [M,K], out [M,Nc], out[m][n] = sum_k x[m][k] w[n][k]  (batch ignored);
 * layout NCHW: x [batch,K,M/batch], out [batch,Nc,M/batch], out_b = W . x_b  (bf16 tensor-core path only).
 * Optional fused epilogue on the second output:
 *   y_act = relu?( out * scale[n] + shift[n] )   (eval-mode BN fold + ReLU, SURVEY.md F9;
 *   scale NULL -> 1, shift NULL -> 0; shift alone is the conv bias).
 * y_raw (the tensor the hint hook captures) and y_act may each be NULL, not both. */
int kdcc_pw_fwd(const void *x, const void *w, const float *scale, const float *shift, int relu,
                void *y_raw, void *y_act, long M, int K, int Nc, int batch, int layout, int dtype,
                kdcc_stream_t stream);

/* The same with the block's shortcut folded into the epilogue (SURVEY.md 8f n2):
 *   y_act = relu?( out * scale[n] + shift[n] + residual )
 * replaces `out = self.convs(bn1); out.add_(shortcut)` of the teacher's residual blocks when the replaced conv is
 * the last of `convs` (wider_resnet.py:181; 4 of the 9 sites of cfg/cityscapes/51M_deeplab_all.json).  residual has
 * the layout and dtype of y_act, which is required; y_raw (pre-add) stays optional. */
int kdcc_pw_fwd_residual(const void *x, const void *w, const float *scale, const float *shift, const void *residual,
                         int relu, void *y_raw, void *y_act, long M, int K, int Nc, int batch, int layout, int dtype,
                         kdcc_stream_t stream);

/* Autograd backward of the call above.  dx[m][k] = sum_n dy[m][n] w[n][k];
 * dw[n][k] = sum_m dy[m][n] x[m][k] (fp32 out, deterministic split-M reduction). */
size_t kdcc_pw_bwd_workspace_bytes(int which /*0 = dx, 1 = dw*/, long M, int K, int Nc, int dtype);
int kdcc_pw_bwd_dx(const void *dy, const void *w, void *dx, void *workspace, size_t workspace_bytes,
                   long M, int K, int Nc, int batch, int layout, int dtype, kdcc_stream_t stream);
int kdcc_pw_bwd_dw(const void *dy, const void *x, float *dw, void *workspace, size_t workspace_bytes,
                   long M, int K, int Nc, int batch, int layout, int dtype, kdcc_stream_t stream);

/* ---- losses ------------------------------------------------------------------------------------
 * kdcc_kd_loss replaces losses/KLDiv.py:19-23 (target_is_prob = 0) and losses/EnsembleKLDiv.py:18-22
 * (target_is_prob = 1, T = 1): one pass reads s and t, does both softmaxes in registers, writes
 *   *loss_out = T^2/(N*HW) * sum_pix KL(p_t || p_s)          (fp32 device scalar)
 *   ds        = grad_scale * T/(N*HW) * (softmax(s/T) - p_t)  (same dtype/strides as s; NULL: skip)
 * Element (n,c,q) lives at base + n*batch_stride + c*class_stride + q*pixel_stride (elements), so
 * NCHW logits are (C*HW, HW, 1) and channels-last logits are (HW*C, 1, C). */
size_t kdcc_loss_workspace_bytes(void);
int kdcc_kd_loss(const void *s, const void *t, void *ds, float *loss_out, void *workspace,
                 size_t workspace_bytes, int N, int C, long HW, long batch_stride, long class_stride,
                 long pixel_stride, float T, int target_is_prob, int dtype, float grad_scale,
                 kdcc_stream_t stream);

/* kdcc_kd_loss_multi (SURVEY.md 8f n3) replaces the K+1 criterion calls of trainer/ensemble_trainer.py:76-83
 * (kd_loss = sum_k WEIGHT*KL(s, t_k) + KL(s, t_teacher), every term a losses/KLDiv.py KLDivergenceLoss):
 *   *loss_out = sum_k weights[k] * T^2/(N*HW) * sum_pix KL(softmax(t_k/T) || softmax(s/T))
 *   ds        = grad_scale * T/(N*HW) * ( (sum_k weights[k]) softmax(s/T) - sum_k weights[k] softmax(t_k/T) )
 * in ONE pass that reads s once and each teacher once.  `teachers` and `weights` are HOST arrays of K (<= 8) device
 * pointers / floats (copied into the kernel parameters); all tensors share dtype and strides.  C <= 32. */
int kdcc_kd_loss_multi(const void *s, const void *const *teachers, const float *weights, int K, void *ds,
                       float *loss_out, void *workspace, size_t workspace_bytes, int N, int C, long HW,
                       long batch_stride, long class_stride, long pixel_stride, float T, int dtype,
                       float grad_scale, kdcc_stream_t stream);

/* kdcc_hint_loss replaces losses/WeightedHintMSELoss.py:12-16 (w given, scale = 1) and
 * losses/MSELoss.py:14-16 (w NULL, scale = num_classes):
 *   *loss_out = scale/N * sum_n [ sum_c w[n,c] mean_hw (s-t)^2 / sum_c w[n,c] ]
 *   ds        = grad_scale * scale * 2 (s-t) w[n,c] / (sum_c w[n,c] * HW * N)
 * w is fp32 [C] (w_per_sample = 0) or [N,C] (w_per_sample = 1).  layout says how (n,c,q) maps to
 * memory.  Needs workspace of kdcc_loss_workspace_bytes() + N*C*4 bytes when w is given. */
int kdcc_hint_loss(const void *s, const void *t, const float *w, int w_per_sample, void *ds,
                   float *loss_out, void *workspace, size_t workspace_bytes, int N, int C, long HW,
                   int layout, float scale, int dtype, float grad_scale, kdcc_stream_t stream);

/* kdcc_ce_loss replaces losses/CrossEntropy.py:10-15 (CrossEntropyLoss2d = NLLLoss2d(log_softmax(inputs, 1), weight, ignore_index)):
 *   valid pixel: label in [0, C) and != ignore_index;  w = weight[label] (weight NULL -> 1)
 *   *loss_out = sum_valid w * (logsumexp_c s - s_label) / (mean ? sum_valid w : 1)   (mean with no valid pixel -> NaN, as torch)
 *   ds        = grad_scale * w * (softmax(s) - onehot(label)) / (mean ? sum_valid w : 1); 0 at invalid pixels; NULL: skip
 * Logit strides as kdcc_kd_loss (NCHW and channels_last without copies); labels int64 [N][HW]; weight fp32 [C]; C <= 32.
 * In mean mode with ds, a pre-pass over the labels forms the normaliser so that ds is written once, already normalised.
 * bad_labels (nullable, device int64) += number of labels outside [0, C) that are not ignore_index: they are dropped,
 * never used as an index (torch would stop with a device-side assert). */
size_t kdcc_ce_workspace_bytes(int N, long HW);
int kdcc_ce_loss(const void *s, const long long *labels, const float *weight, int ignore_index, int mean,
                 void *ds, float *loss_out, long long *bad_labels, void *workspace, size_t workspace_bytes,
                 int N, int C, long HW, long batch_stride, long class_stride, long pixel_stride,
                 int dtype, float grad_scale, kdcc_stream_t stream);

/* kdcc_logits_stats: the logged-only quantities of one layerwise step (trainer/layerwise_trainer.py:225-227,244-250) in ONE
 * read of s, t and the labels, no gradients:
 *   out3[0] = KD term: kd_mode 0 none (untouched), 1 = kdcc_kd_loss value (temperature T), 2 = MSELoss value x kd_scale
 *   out3[1] = CE(s, labels), out3[2] = CE(t, labels)   (as kdcc_ce_loss, same weight / ignore / mean)
 *   conf_s / conf_t (nullable, int64 [C*C], accumulated) += confusion of argmax(s) / argmax(t), exactly as kdcc_confusion_update.
 * s and t share dtype and strides.  t may be NULL (validation: student only; out3[0], out3[2], conf_t untouched, kd_mode
 * ignored).  With kd_mode 1 and T == 1 the KD term reuses the CE exponentials.  Workspace: kdcc_ce_workspace_bytes. */
int kdcc_logits_stats(const void *s, const void *t, const long long *labels, const float *weight, int ignore_index, int mean,
                      int kd_mode, float T, float kd_scale, float *out3, long long *conf_s, long long *conf_t,
                      long long *bad_labels, void *workspace, size_t workspace_bytes, int N, int C, long HW,
                      long batch_stride, long class_stride, long pixel_stride, int dtype, kdcc_stream_t stream);

/* ---- small utilities used by the host mirror so no torch arithmetic sits on the path ------------ */
/* dst_bf16[i] = bf16(src_f32[i]) */
int kdcc_cast_f32_to_bf16(const float *src, void *dst, long n, kdcc_stream_t stream);
/* buf[i] *= *dev_scalar   (applies autograd's upstream 0-dim grad to an emitted gradient) */
int kdcc_scale_inplace(void *buf, const float *dev_scalar, long n, int dtype, kdcc_stream_t stream);
/* buf[i] *= *dev_scalar / expected: the loss kernels fold the upstream value a caller EXPECTS (grad_scale) into the
 * gradient they emit; backward then only verifies it -- when *dev_scalar == expected the launch touches no memory, otherwise
 * it rescales, so the result is right either way without a host read of the device scalar. */
int kdcc_scale_inplace_expect(void *buf, const float *dev_scalar, float expected, long n, int dtype, kdcc_stream_t stream);
/* Activation layout conversion at a block boundary (layout_convert.cu): dst = src re-laid from NHWC to NCHW (to_nchw = 1) or
 * back (to_nchw = 0); bf16, C % 8 == 0, HW % 8 == 0.  Lets a channels_last trunk feed the NCHW tensor-core depthwise kernels
 * of models/students/transform_blocks/depthwise_separable_conv.py:11-14's replacement. */
int kdcc_layout_convert(const void *src, void *dst, int N, int C, long HW, int to_nchw, int dtype, kdcc_stream_t stream);
/* out[j] = sum_m a[m][j]  (bias gradients), a [M,Nc] in dtype, out fp32 */
int kdcc_colsum(const void *a, float *out, void *workspace, size_t workspace_bytes, long M, int Nc,
                int dtype, kdcc_stream_t stream);
size_t kdcc_colsum_workspace_bytes(long M, int Nc);

/* ---- segmentation metric (SURVEY.md 8f n1) --------------------------------------------------------
 * kdcc_confusion_update replaces utils/util.py:108-128 (CityscapesMetricTracker.update ->
 * confusion_for_batch) and models/metric.py:49-55: pred = argmax_c logits[n][c][q] (first maximum),
 * conf[labels[n][q]][pred] += 1 for labels in [0, C) and != ignore_index.  logits element (n,c,q) at
 * base + n*batch_stride + c*class_stride + q; labels int64 [N][HW]; conf int64 [C][C] on the device,
 * ACCUMULATED (zero it to reset).  One HBM pass, no host copy; C <= 32. */
int kdcc_confusion_update(const void *logits, const long long *labels, long long *conf, int N, int C, long HW,
                          long batch_stride, long class_stride, int ignore_index, int dtype,
                          kdcc_stream_t stream);

/* ---- optimizer step of the layerwise loop -------------------------------------------------------------
 * kdcc_radam_step replaces the per-tensor body of utils/optim/radam.py:41-97 (RAdam, the optimizer of every
 * cfg/cityscapes/*.json) with one pass:  v = beta2 v + (1-beta2) g^2;  m = beta1 m + (1-beta1) g;  then
 *   mode 0 (N_sma >= 5):        p += decay * p;  p += step * m / (sqrt(v) + eps)
 *   mode 1 (degenerated SGD):   p += decay * p;  p += step * m
 *   mode 2 (step_size < 0):     moments only.
 * decay = -weight_decay * lr (0: none), step = -step_size * lr with N_sma / step_size computed by the caller as
 * radam.py:65-84 does (host float64); one_minus_beta* = 1 - beta* evaluated in double by the caller (as the reference
 * does: 1 - 0.999f in float is off by 1.3e-5 relative).  p, g, m, v fp32 [n], 16-byte aligned; p_lp (nullable)
 * receives the bf16 copy of the new parameters, i.e. the pointwise GEMM weights of the next step. */
int kdcc_radam_step(float *p, const float *g, float *m, float *v, void *p_lp, long n, float beta1, float beta2,
                    float one_minus_beta1, float one_minus_beta2, float eps, float decay, float step, int mode,
                    kdcc_stream_t stream);
/* Data-parallel form: g points at n_src copies of the gradient, src_stride floats apart (one per rank, written into this
 * rank's memory by its peers); the step uses their mean, summed in source order (bit-identical on every rank).  The gradient
 * all-reduce of the layerwise loop (SURVEY.md 8e) fused into the optimizer pass. */
int kdcc_radam_step_multi(float *p, const float *g, long src_stride, int n_src, float *m, float *v, void *p_lp, long n,
                          float beta1, float beta2, float one_minus_beta1, float one_minus_beta2, float eps, float decay,
                          float step, int mode, kdcc_stream_t stream);

/* ---- sliding-window test-time inference (SURVEY.md 8f n4) -------------------------------------------
 * kdcc_tta_stitch replaces utils/tta_process.py:39-52 (collect_windows_result) and the np.fliplr of :19-20:
 * out[c][y][x] (+)= alpha * S[c][y][flip ? w-1-x : x],  S = (sum of the windows covering the pixel) / count.
 * windows fp32 [n][C][th][tw] on the device; coords int32 [n][4] = (x1, y1, x2, y2) on the device, 16-byte aligned,
 * x2-x1 <= tw, y2-y1 <= th (a window is cropped to the part inside the image).  count_mode 0 = the reference's
 * counter exactly as written (:46, a (classes, h, w) array sliced [y1:y2, x1:x2]: identical results, including
 * inf/nan where it is 0); 1 = per-pixel coverage.  n <= 512.
 * kdcc_resize_bilinear replaces resize_output (:29-36, cv2.INTER_LINEAR per class plane): dst (+)= alpha * resize. */
int kdcc_tta_stitch(const float *windows, const int *coords, int n, int C, int th, int tw, int h, int w, int flip,
                    int count_mode, float alpha, float *out, int accumulate, kdcc_stream_t stream);
int kdcc_resize_bilinear(const float *src, int C, int h, int w, float *dst, int H, int W, float alpha, int accumulate,
                         kdcc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* KDCC_H_ */
