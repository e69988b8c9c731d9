"""Depthwise and pointwise kernels at the edges of their dispatch predicates, through the C ABI with buffers the test owns.

Each row of DEPTHWISE / POINTWISE names a shape, the epilogue and gradients it asks for, and the kernels that must launch for
it.  Every row runs in two data modes:

* exact: x and dy are integers in +-{1..8}; taps, pointwise weights, bias, scale and shift are eighths in [-1, 1]; the
  residual is integer.  Every product is exact in fp32 and, as long as every partial sum stays below 2^24 units of its value
  grid (test_exact_rows_stay_inside_fp32 checks that for every row from its shapes), so is every sum, whatever the order
  and the split count.  fp32 outputs must then equal the float64 reference and bf16 outputs its round-to-nearest-even:
  a single misplaced, missing or duplicated contribution fails, and the message names the first wrong element.
* bound: Gaussian x and dy, uniform weights, full mantissas.  Per element |dev - ref| <= rho |ref| + gamma S, with S the
  same operation on |inputs| in float64, rho = 2^-8 for a bf16 output (one round-to-nearest-even) and 0 for fp32, and
  gamma = 2 n 2^-24 with n the number of terms of the output's sum, plus one for rounded products and the epilogue's
  operations.  Derivation, the same for every kernel family: any order of summing n terms errs by at most
  (n - 1) 2^-24 sum|terms| (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., eq. 4.4), and the factor 2
  leaves room for an accumulator that truncates instead of rounding.  n per family:
    depthwise forward and input gradient (every kernel):   k^2 + 1   (taps, bias)
    depthwise weight and bias gradients (every kernel):    N Ho Wo + 1   (pixels of the plane, rounded fp32 products)
    pointwise forward (sm100, tf32x3, simt):               K + 4     (reduction, product rounding, scale, shift, residual)
    pointwise input gradient:                              Nc + 1
    pointwise weight gradient:                             M + 1     (all pixels, whatever the split count)
  The tensor-core depthwise kernels hold the taps rounded to bf16 in their Toeplitz operand, so their reference uses the
  rounded taps; the CUDA-core kernels get the fp32 taps.

Every call also checks: the profiled kernel names equal the row's set (split reductions left out); outputs filled with
NaN beforehand hold no NaN afterwards; 4 KB guard bands of 0x5A on both sides of every output and of the workspace, which
is sized at exactly kdcc_*_workspace_bytes, are intact; x, dy and the weights are unchanged; a second call gives
bit-identical outputs.  The reference is torch float64 on the device and does not depend on kdcc."""
import os
import re
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_parity import kdcc  # noqa: F401  (the module fixture)
from test_kernel_routing import DW_NAME, PW_NAME, launched

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "knowledge-distillation-by-replacing-cheap-conv_b200", "csrc")

BF16, F32, TF32X3 = torch.bfloat16, torch.float32, "tf32x3"   # TF32X3: fp32 tensors, products as three tf32 MMAs
GUARD = 4096
FP32_UNITS = 1 << 24

C1, C2 = "dw_tc_conv_kernel", "dw_tc_conv2_kernel"
WG, WG2, WG3 = "dw_tc_wgrad_kernel", "dw_tc_wgrad2_kernel", "dw_tc_wgrad3_kernel"
N3C, N3W = "dw_nhwc3_conv_kernel", "dw_nhwc3_wgrad_kernel"
TC, TW = "dw_tma_conv_kernel", "dw_tma_wgrad_kernel"
DC, DWG = "dw_direct_kernel", "dw_wgrad_direct_kernel"
G64, G128, G256 = "pw_gemm_sm100_kernel<64>", "pw_gemm_sm100_kernel<128>", "pw_gemm_sm100_kernel<256>"
G256P = "pw_gemm_sm100_kernel<256,pair>"   # a CTA pair (cluster of two) per 256 x 256 tile
SIMT, X3 = "pw_simt_kernel", "pw_gemm_tf32x3_kernel"
OTHER_PW_NAME = re.compile(r"\b(pw_simt_kernel|pw_gemm_tf32x3_kernel)\b")

# kernels no row names, each with the reason
NOT_PINNED = {
    "dw_wgrad_reduce_kernel": "sum of the TMA / streaming / direct weight-gradient splits: pinned by the exact dW of those rows",
    "dw_tc_wgrad_reduce_kernel": "sum of the tiled weight-gradient splits: pinned by the exact dW of multi-plane rows",
    "dw_tc_wgrad2_reduce_kernel": "sum of the whole-plane / column-phase weight-gradient splits: pinned by the exact dW of N >= 3 rows",
    "reduce_splits_kernel": "sum of the pointwise weight-gradient splits: pinned by the exact dW of the large-M rows",
}

DwRow = namedtuple("DwRow", "layout dtype N C H W k d p bias grads fwd bwd")
PwRow = namedtuple("PwRow", "layout dtype N K Co H W epi fwd dx dw")


def dw(*a):
    return DwRow(*a)


def pw(*a):
    return PwRow(*a)


DEPTHWISE = [
    # layout, dtype, N, C, H, W, k, d, p, bias, gradients (x, w, b), forward kernels, backward kernels
    # NCHW tensor cores, whole-plane conv2: k in {1,3,5,7,9} x d in {1,2,5} at p = halo/2; H, W in {1,8,120,128};
    # C in {1,3,148,149,300} and N in {1,2,3,5} (tc_unit_splits, odd image pairs); dX only, dW only, both; bias
    dw("nchw", BF16, 1, 16, 8, 8, 1, 1, 0, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 2, 3, 120, 120, 3, 1, 1, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 1, 1, 128, 128, 3, 2, 2, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 3, 16, 8, 128, 3, 5, 5, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 1, 148, 128, 8, 5, 1, 2, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 2, 16, 120, 128, 5, 2, 4, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 1, 8, 128, 120, 5, 5, 10, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 2, 149, 8, 8, 7, 1, 3, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 1, 16, 120, 8, 7, 2, 6, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 1, 3, 128, 128, 7, 5, 15, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 5, 16, 120, 120, 9, 1, 4, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 1, 16, 128, 128, 9, 2, 8, 0, "xw", {C2}, {C2, WG2}),
    dw("nchw", BF16, 2, 148, 128, 128, 9, 5, 20, 0, "xw", {C2}, {C2, WG3}),
    dw("nchw", BF16, 3, 16, 8, 8, 9, 5, 20, 0, "xw", {C2}, {C2, WG3}),
    dw("nchw", BF16, 5, 16, 1, 8, 9, 5, 20, 0, "xw", {C2}, {C2, WG3}),
    dw("nchw", BF16, 1, 300, 40, 40, 9, 5, 20, 0, "x", {C2}, {C2}),
    dw("nchw", BF16, 2, 16, 40, 40, 9, 5, 20, 0, "w", {C2}, {WG3}),
    dw("nchw", BF16, 1, 16, 128, 128, 9, 5, 20, 1, "xw", {C2}, {C2, WG3}),
    # conv2's wide form: 136 .. 256 columns
    dw("nchw", BF16, 1, 16, 128, 136, 9, 5, 20, 0, "xw", {C2}, {C2, WG}),
    dw("nchw", BF16, 2, 3, 64, 248, 9, 5, 20, 0, "xw", {C2}, {C2, WG}),
    dw("nchw", BF16, 1, 16, 128, 256, 9, 5, 20, 1, "xw", {C2}, {C2, WG}),
    # tiled conv: 264 columns and more, 129 rows and more
    dw("nchw", BF16, 1, 16, 120, 264, 9, 5, 20, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 129, 264, 9, 5, 20, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 3, 255, 384, 3, 1, 1, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 1, 256, 520, 5, 2, 4, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 2, 257, 264, 7, 1, 3, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 257, 520, 1, 1, 0, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 2, 16, 129, 128, 9, 5, 20, 0, "x", {C1}, {C1}),
    # dilations conv2 does not instantiate
    dw("nchw", BF16, 3, 16, 64, 64, 3, 3, 3, 0, "xw", {C1}, {C1, WG2}),
    dw("nchw", BF16, 1, 16, 64, 64, 5, 4, 8, 0, "xw", {C1}, {C1, WG2}),
    dw("nchw", BF16, 1, 16, 64, 64, 9, 7, 28, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 149, 40, 48, 3, 7, 7, 0, "xw", {C1}, {C1, WG2}),
    dw("nchw", BF16, 1, 16, 40, 40, 7, 4, 12, 0, "xw", {C1}, {C1, WG2}),
    # padding off halo/2 (Ho < H; halo/2 < p <= halo), pad % 8 != 0 (aligned-window columns), N-tile 16 (reach > 48)
    # against 32, K slices 2 (k1), 3 (k3 d1), 4 (k7 d4), 5 (k9 d5, k3 d28)
    dw("nchw", BF16, 2, 16, 96, 96, 9, 5, 12, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 96, 96, 9, 5, 28, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 64, 64, 9, 5, 40, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 64, 64, 3, 4, 0, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 64, 64, 3, 4, 8, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 64, 264, 5, 1, 2, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 32, 40, 3, 28, 28, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 3, 16, 32, 48, 3, 28, 20, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 32, 264, 1, 1, 0, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 32, 40, 9, 7, 32, 1, "x", {C1}, {C1}),
    # whole-plane weight gradient at pad = W2_GAP = 24 (wgrad2) and one step past it (generic)
    dw("nchw", BF16, 1, 16, 64, 64, 9, 6, 24, 0, "xw", {C1}, {C1, WG2}),
    dw("nchw", BF16, 5, 16, 64, 64, 3, 24, 24, 0, "xw", {C1}, {C1, WG2}),
    dw("nchw", BF16, 1, 16, 64, 64, 3, 25, 25, 0, "xw", {C1}, {C1, WG}),
    dw("nchw", BF16, 1, 16, 48, 48, 5, 12, 24, 0, "w", {C1}, {WG2}),
    dw("nchw", BF16, 1, 16, 64, 64, 7, 8, 24, 0, "xw", {C1}, {C1, WG2}),
    dw("nchw", BF16, 1, 16, 120, 120, 3, 26, 26, 0, "xw", {C1}, {C1, WG}),
    # NHWC streaming 3x3: C/8 in {2,4,8,16,32,64,96}, W narrower than a CTA tile, H not a multiple of 32; bias; every
    # gradient subset (a bias gradient moves dW to the direct kernel)
    dw("nhwc", BF16, 2, 16, 33, 10, 3, 1, 1, 0, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 1, 32, 40, 7, 3, 1, 1, 0, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 3, 64, 17, 3, 3, 1, 1, 0, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 1, 128, 50, 2, 3, 1, 1, 0, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 2, 256, 45, 13, 3, 1, 1, 0, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 1, 512, 9, 9, 3, 1, 1, 1, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 1, 768, 35, 5, 3, 1, 1, 0, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "x", {N3C}, {N3C}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "w", {N3C}, {N3W}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "b", {N3C}, {DWG}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "xw", {N3C}, {N3C, N3W}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "xb", {N3C}, {DWG, N3C}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "wb", {N3C}, {DWG}),
    dw("nhwc", BF16, 2, 64, 33, 20, 3, 1, 1, 1, "xwb", {N3C}, {DWG, N3C}),
    # NHWC TMA k3 / k9: d = 1, 2, 5 and 7 (the largest cfg_fits admits), 8 on the direct kernel; ragged planes; p on both
    # sides of halo/2 and past the halo (dX on the direct kernel); bias; every gradient subset
    dw("nhwc", BF16, 2, 48, 16, 16, 3, 1, 1, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 2, 16, 20, 20, 3, 2, 2, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 32, 37, 45, 3, 5, 5, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 16, 40, 44, 3, 7, 7, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 16, 40, 44, 3, 8, 8, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 2, 16, 33, 29, 9, 1, 4, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 2, 8, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 32, 131, 67, 9, 5, 20, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 16, 60, 60, 9, 7, 28, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 16, 70, 70, 9, 8, 32, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 2, 32, 50, 43, 9, 5, 12, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 32, 30, 27, 9, 5, 30, 0, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 16, 20, 20, 3, 1, 3, 0, "xw", {TC}, {DC, TW}),
    dw("nhwc", BF16, 1, 16, 30, 30, 9, 5, 44, 0, "xw", {TC}, {DC, TW}),
    dw("nhwc", BF16, 2, 48, 16, 16, 3, 1, 1, 1, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "x", {TC}, {TC}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "w", {TC}, {TW}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "b", {TC}, {DWG}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "xw", {TC}, {TC, TW}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "xb", {TC}, {DWG, TC}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "wb", {TC}, {DWG}),
    dw("nhwc", BF16, 1, 32, 40, 44, 9, 5, 20, 1, "xwb", {TC}, {DWG, TC}),
    # NHWC direct: fp32 C in {4, 12}, bf16 C % 16 == 8, k in {1, 2, 4, 5, 7}
    dw("nhwc", F32, 2, 4, 17, 19, 1, 1, 0, 1, "xwb", {DC}, {DC, DWG}),
    dw("nhwc", F32, 1, 12, 20, 23, 2, 1, 1, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", F32, 2, 4, 16, 16, 4, 2, 3, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", F32, 1, 12, 21, 18, 5, 3, 6, 1, "xwb", {DC}, {DC, DWG}),
    dw("nhwc", F32, 1, 4, 30, 30, 7, 1, 3, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 2, 8, 17, 19, 1, 1, 0, 1, "xwb", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 1, 24, 20, 23, 2, 2, 1, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 2, 40, 16, 16, 4, 1, 2, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 1, 24, 21, 18, 5, 2, 4, 1, "xwb", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 1, 8, 30, 30, 7, 1, 3, 0, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 2, 24, 16, 16, 3, 1, 1, 1, "xw", {DC}, {DC, DWG}),
    dw("nhwc", BF16, 1, 16, 20, 20, 5, 1, 2, 0, "xw", {DC}, {DC, DWG}),
]

POINTWISE = [
    # layout ('planes' = PLANES_TO_NHWC), dtype, N, K, Co, H, W (M = N H W, P = H W), epilogue, forward, dX, dW kernels.
    # Epilogues: '' y_raw alone (TMA-store epilogue), 'bias' shift, 'bn' scale + shift + ReLU, 'res' residual,
    # 'resbn' residual + scale + shift + ReLU, 'dual' y_raw and y_act (scale + shift + ReLU) from one GEMM
    # NHWC: M at the 128-row tile edges, K and Nc at the 64 / 128 / 256 BJ edges, CTA pairs on and off, dW splits
    pw("nhwc", BF16, 1, 8, 8, 1, 1, "", {G64}, {G64}, {G64}),
    pw("nhwc", BF16, 1, 56, 64, 1, 8, "", {G64}, {G64}, {G64}),
    pw("nhwc", BF16, 1, 64, 72, 1, 127, "bias", {G128}, {G64}, {G64}),
    pw("nhwc", BF16, 1, 72, 256, 1, 128, "", {G256}, {G128}, {G128}),
    pw("nhwc", BF16, 1, 520, 136, 1, 129, "bn", {G128}, {G128}, {G128}),
    pw("nhwc", BF16, 1, 4096, 264, 1, 255, "", {G128}, {G256P}, {G256}),
    pw("nhwc", BF16, 1, 64, 512, 16, 16, "res", {G256P}, {G64}, {G64}),
    pw("nhwc", BF16, 1, 72, 256, 1, 257, "resbn", {G256}, {G128}, {G128}),
    pw("nhwc", BF16, 1, 4096, 256, 1, 16392, "", {G256}, {G256}, {G256P}),
    pw("nhwc", BF16, 2, 256, 512, 64, 64, "dual", {G256P}, {G256P}, {G256P}),
    pw("nhwc", BF16, 1, 8, 264, 1, 256, "", {G128}, {G64}, {G64}),
    pw("nhwc", BF16, 3, 520, 8, 5, 17, "", {G64}, {G128}, {G128}),
    pw("nhwc", BF16, 2, 64, 136, 16, 16, "dual", {G128}, {G64}, {G64}),
    # NCHW: P = H W at 8, 72, 120, 136, 16384 with batch 1, 2, 3, 5; Nc > 128 so that affine_rows spans row tiles
    pw("nchw", BF16, 5, 64, 136, 2, 4, "", {G64}, {G64}, {G64}),
    pw("nchw", BF16, 3, 72, 264, 8, 9, "bn", {G128}, {G128}, {G128}),
    pw("nchw", BF16, 2, 256, 256, 8, 15, "bias", {G128}, {G128}, {G256P}),
    pw("nchw", BF16, 1, 128, 192, 8, 17, "res", {G128}, {G128}, {G128}),
    pw("nchw", BF16, 1, 64, 256, 128, 128, "resbn", {G256P}, {G256}, {G64}),
    pw("nchw", BF16, 2, 520, 384, 128, 128, "", {G256}, {G256}, {G128}),
    pw("nchw", BF16, 3, 64, 264, 8, 9, "dual", {G128}, {G128}, {G64}),
    pw("nchw", BF16, 2, 8, 136, 8, 9, "", {G128}, {G128}, {G64}),
    # planes in, channels_last out
    pw("planes", BF16, 5, 64, 136, 2, 4, "bias", {G128}, {G64}, {G64}),
    pw("planes", BF16, 2, 64, 264, 8, 9, "", {G128}, {G128}, {G64}),
    pw("planes", BF16, 3, 128, 256, 8, 15, "bn", {G256}, {G128}, {G128}),
    pw("planes", BF16, 1, 256, 512, 128, 128, "res", {G256P}, {G256P}, {G256P}),
    pw("planes", BF16, 2, 72, 136, 8, 17, "resbn", {G128}, {G128}, {G128}),
    pw("planes", BF16, 2, 64, 256, 8, 9, "dual", {G256}, {G128}, {G64}),
    pw("planes", BF16, 1, 4096, 256, 128, 128, "", {G256P}, {G256P}, {G256P}),
    # CUDA-core fallback: bf16 with K or Nc % 8 != 0, fp32 under "highest" (dW splits > 1, Nc K % 4 != 0); tf32x3
    pw("nhwc", BF16, 1, 12, 20, 10, 100, "bn", {SIMT}, {SIMT}, {SIMT}),
    pw("nhwc", BF16, 2, 64, 19, 16, 16, "bias", {SIMT}, {SIMT}, {SIMT}),
    pw("nhwc", BF16, 1, 20, 40, 31, 33, "res", {SIMT}, {SIMT}, {SIMT}),
    pw("nhwc", F32, 1, 3, 5, 32, 32, "", {SIMT}, {SIMT}, {SIMT}),
    pw("nhwc", F32, 1, 64, 32, 16, 64, "resbn", {SIMT}, {SIMT}, {SIMT}),
    pw("nhwc", F32, 1, 64, 32, 16, 16, "dual", {SIMT}, {SIMT}, {SIMT}),
    pw("nhwc", TF32X3, 1, 64, 32, 16, 16, "bn", {X3}, {X3}, {X3}),
]


def out_hw(r):
    return r.H + 2 * r.p - r.d * (r.k - 1), r.W + 2 * r.p - r.d * (r.k - 1)


def dw_id(r):
    return "%s-%s-n%dc%d-%dx%d-k%dd%dp%d%s-%s" % (r.layout, "f32" if r.dtype == F32 else "bf16", r.N, r.C, r.H, r.W, r.k,
                                                 r.d, r.p, "-bias" if r.bias else "", r.grads)


def pw_id(r):
    dt = {BF16: "bf16", F32: "f32", TF32X3: "tf32x3"}[r.dtype]
    return "%s-%s-n%dk%dco%d-%dx%d%s" % (r.layout, dt, r.N, r.K, r.Co, r.H, r.W, "-" + r.epi if r.epi else "")


# ---------------------------------------------------------------------------------------------------------------------
# exactness precondition: the largest partial sum of every output, in units of its value grid
# ---------------------------------------------------------------------------------------------------------------------
def dw_exact_units(r):
    """x, dy <= 8 (unit 1), taps and bias <= 1 (unit 1/8): forward / dX in eighths, dW / dbias in units."""
    Ho, Wo = out_hw(r)
    return max(r.k * r.k * 8 * 8 + 8, r.N * Ho * Wo * 8 * 8)


def pw_exact_units(r):
    """Forward in 64ths once scale applies (GEMM in eighths times an eighth), plus shift (8 / 64ths) and residual (8);
    dX in eighths; dW and the bias column sums in units."""
    M = r.N * r.H * r.W
    fwd = r.K * 8 * 8 * 8 + 8 * 8 + 8 * 64
    return max(fwd, r.Co * 8 * 8, M * 8 * 8)


# ---------------------------------------------------------------------------------------------------------------------
# comparisons
# ---------------------------------------------------------------------------------------------------------------------
def _first_bad(name, bad, dev, want, axes):
    idx = tuple(int(i) for i in torch.nonzero(bad)[0])
    where = ", ".join("%s=%d" % (a, i) for a, i in zip(axes, idx))
    return "%s: %d of %d elements wrong; first at (%s): reference %r, device %r" % (
        name, int(bad.sum()), bad.numel(), where, float(want[idx]), float(dev[idx]))


def assert_exact(name, dev, ref, axes):
    """dev (bf16 or fp32) equals the float64 reference, rounded to nearest even for bf16 (the reference is exact in fp32)."""
    want = ref.float()
    if dev.dtype == torch.bfloat16:
        want = want.to(torch.bfloat16).float()
    got = dev.float()
    bad = got != want
    if bool(bad.any()):
        raise AssertionError(_first_bad(name, bad, got, want, axes))


def assert_bound(name, dev, ref, S, n, axes):
    """|dev - ref| <= rho |ref| + 2 n 2^-24 S per element (rho = 2^-8 for bf16, 0 for fp32); NaN fails."""
    rho = 2.0 ** -8 if dev.dtype == torch.bfloat16 else 0.0
    got = dev.double()
    bad = ~((got - ref).abs() <= rho * ref.abs() + 2.0 * n * 2.0 ** -24 * S)
    if bool(bad.any()):
        raise AssertionError(_first_bad(name, bad, got, ref, axes))


def kernel_set(names):
    out = set()
    for n in names:
        out.update(m.group(1) for m in DW_NAME.finditer(n) if "reduce" not in m.group(1))
        out.update("pw_gemm_sm100_kernel<%s%s>" % (m.group(1), ",pair" if m.group(2) == "true" else "")
                   for m in PW_NAME.finditer(n))
        out.update(m.group(1) for m in OTHER_PW_NAME.finditer(n))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# buffers
# ---------------------------------------------------------------------------------------------------------------------
class Guarded:
    """`nbytes` of device memory between two GUARD-byte bands of 0x5A; the payload starts 16-byte aligned."""

    def __init__(self, nbytes):
        self.n = int(nbytes)
        self.raw = torch.full((2 * GUARD + self.n,), 0x5A, dtype=torch.uint8, device="cuda")
        assert self.ptr % 16 == 0

    @property
    def ptr(self):
        return self.raw.data_ptr() + GUARD

    def payload(self, dtype=torch.uint8):
        return self.raw[GUARD:GUARD + self.n].view(dtype)

    def intact(self):
        return bool((self.raw[:GUARD] == 0x5A).all()) and bool((self.raw[GUARD + self.n:] == 0x5A).all())


class Out(Guarded):
    """A guarded output tensor: logical NCHW shape (or any shape for weights), stored in `layout` order."""

    def __init__(self, shape, dtype, layout="nchw"):
        self.shape, self.dtype, self.layout = tuple(shape), dtype, layout
        super().__init__(int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size())

    def poison(self):
        self.payload(self.dtype).fill_(float("nan"))

    def logical(self):
        flat = self.payload(self.dtype)
        if self.layout == "nhwc":
            N, C, H, W = self.shape
            return flat.view(N, H, W, C).permute(0, 3, 1, 2)
        return flat.view(self.shape)


def physical(t, layout):
    """A logical NCHW tensor laid out contiguously in `layout` order (the tensor the C ABI reads)."""
    return t.permute(0, 2, 3, 1).contiguous() if layout == "nhwc" else t.contiguous()


def draw(gen, shape, kind, exact, dtype=torch.float32):
    """Operands of the two data modes: 'act' (x, dy, residual), 'tap' (weights, bias, scale, shift)."""
    if exact:
        if kind == "act":
            mag = torch.randint(1, 9, shape, generator=gen, device="cuda")
            sign = torch.randint(0, 2, shape, generator=gen, device="cuda") * 2 - 1
            return (mag * sign).to(dtype)
        return (torch.randint(-8, 9, shape, generator=gen, device="cuda").float() / 8).to(dtype)
    if kind == "act":
        return torch.randn(shape, generator=gen, device="cuda").to(dtype)
    return (torch.rand(shape, generator=gen, device="cuda") * 2 - 1).to(dtype)


def run_checked(call, outs, workspace, inputs, expect, what):
    """Two calls under the profiler on NaN-filled outputs and a poisoned workspace: the kernels launched, the first
    call's outputs (logical views), and the checks that need no reference."""
    results = []

    def body():
        for _ in range(2):
            for o in outs.values():
                o.poison()
            if workspace is not None:
                workspace.payload().fill_(0xFF)   # NaN partials, should a reduction read one that was never written
            before = [t.clone() for t in inputs]
            call()
            results.append({k: o.logical().clone() for k, o in outs.items()})
            for t, b in zip(inputs, before):
                assert torch.equal(t.view(torch.uint8), b.view(torch.uint8)), "%s wrote into an input" % what

    names = kernel_set(launched(body))
    assert names == set(expect), "%s launched %s, expected %s" % (what, sorted(names), sorted(expect))
    for k, o in outs.items():
        assert o.intact(), "%s wrote outside %s" % (what, k)
        v = results[0][k]
        assert not bool(torch.isnan(v.float()).any()), "%s left elements of %s unwritten (NaN)" % (what, k)
        a, b = v.contiguous(), results[1][k].contiguous()
        assert torch.equal(a.view(torch.int16 if a.dtype == torch.bfloat16 else torch.int32),
                           b.view(torch.int16 if b.dtype == torch.bfloat16 else torch.int32)), \
            "%s: second call differs in %s" % (what, k)
    if workspace is not None:
        assert workspace.intact(), "%s wrote past the advertised workspace" % what
    return results[0]


def _abi_dtype(kdcc, dtype):
    A = kdcc._abi
    return {BF16: A.BF16, F32: A.F32, TF32X3: A.F32_TF32X3}[dtype]


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------------------------
# depthwise
# ---------------------------------------------------------------------------------------------------------------------
def dw_reference(x, w, b, dy, k, d, p, grads):
    """float64 F.conv2d(groups=C) and its autograd: {y, dx, dw, db} (the requested gradients)."""
    C = x.shape[1]
    x = x.detach().clone().requires_grad_(True)
    w = w.detach().reshape(C, 1, k, k).clone().requires_grad_(True)
    b = b.detach().clone().requires_grad_(True) if b is not None else None
    y = F.conv2d(x, w, b, padding=p, dilation=d, groups=C)
    g = torch.autograd.grad(y, [x, w] + ([b] if b is not None else []), dy)
    gx, gw, gb = g[0], g[1], (g[2] if b is not None else None)
    out = {"y": y.detach()}
    if "x" in grads:
        out["dx"] = gx
    if "w" in grads:
        out["dw"] = gw.reshape(C, k, k)
    if "b" in grads:
        out["db"] = gb
    return out


def dw_case(kdcc, r, seed, exact):
    A, L = kdcc._abi, kdcc._abi.lib()
    N, C, H, W, k, d, p = r.N, r.C, r.H, r.W, r.k, r.d, r.p
    Ho, Wo = out_hw(r)
    gen = torch.Generator("cuda").manual_seed(seed)
    x = draw(gen, (N, C, H, W), "act", exact, r.dtype)
    dy = draw(gen, (N, C, Ho, Wo), "act", exact, r.dtype)
    w = draw(gen, (C, k, k), "tap", exact)
    b = draw(gen, (C,), "tap", exact) if r.bias else None
    lay, code = (A.NCHW if r.layout == "nchw" else A.NHWC), _abi_dtype(kdcc, r.dtype)
    xd, dyd = physical(x, r.layout), physical(dy, r.layout)
    # the tensor-core kernels multiply bf16-rounded taps
    w_ref = w.to(torch.bfloat16) if r.layout == "nchw" else w
    ref = dw_reference(x.double(), w_ref.double(), None if b is None else b.double(), dy.double(), k, d, p, r.grads)
    S = None
    if not exact:
        S = dw_reference(x.double().abs(), w_ref.double().abs(), None if b is None else b.double().abs(), dy.double().abs(),
                         k, d, p, r.grads)

    y = Out((N, C, Ho, Wo), r.dtype, r.layout)
    st = _stream()
    fwd = run_checked(lambda: A.check(L.kdcc_dw_fwd(xd.data_ptr(), w.data_ptr(), None if b is None else b.data_ptr(),
                                                    y.ptr, N, H, W, C, k, d, p, lay, code, st), "kdcc_dw_fwd"),
                      {"y": y}, None, [xd, w] + ([b] if b is not None else []), r.fwd, "forward")

    outs = {}
    if "x" in r.grads:
        outs["dx"] = Out((N, C, H, W), r.dtype, r.layout)
    if "w" in r.grads:
        outs["dw"] = Out((C, k, k), torch.float32)
    if "b" in r.grads:
        outs["db"] = Out((C,), torch.float32)
    ws = Guarded(L.kdcc_dw_bwd_workspace_bytes(N, H, W, C, k, d, p, lay, code))
    ptr = lambda key: outs[key].ptr if key in outs else None  # noqa: E731
    bwd = run_checked(lambda: A.check(L.kdcc_dw_bwd(xd.data_ptr(), w.data_ptr(), dyd.data_ptr(), ptr("dx"), ptr("dw"),
                                                    ptr("db"), ws.ptr, ws.n, N, H, W, C, k, d, p, lay, code, st),
                                      "kdcc_dw_bwd"),
                      outs, ws, [xd, dyd, w], r.bwd, "backward")

    got = dict(fwd, **bwd)
    terms = {"y": k * k + 1, "dx": k * k + 1, "dw": N * Ho * Wo + 1, "db": N * Ho * Wo}
    axes = {"y": "ncij", "dx": "ncij", "dw": "cuv", "db": "c"}
    for key, dev in got.items():
        if exact:
            assert_exact(key, dev, ref[key], axes[key])
        else:
            assert_bound(key, dev, ref[key], S[key], terms[key], axes[key])


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [True, False], ids=["exact", "bound"])
@pytest.mark.parametrize("row", DEPTHWISE, ids=dw_id)
def test_depthwise_edges(kdcc, row, exact):
    dw_case(kdcc, row, DEPTHWISE.index(row), exact)


# ---------------------------------------------------------------------------------------------------------------------
# pointwise
# ---------------------------------------------------------------------------------------------------------------------
EPILOGUES = {  # scale, shift, relu, residual, y_raw, y_act
    "": (False, False, False, False, True, False),
    "bias": (False, True, False, False, False, True),
    "bn": (True, True, True, False, False, True),
    "res": (False, False, False, True, False, True),
    "resbn": (True, True, True, True, False, True),
    "dual": (True, True, True, False, True, True),
}


def pw_case(kdcc, r, seed, exact):
    A, L = kdcc._abi, kdcc._abi.lib()
    N, K, Co, H, W = r.N, r.K, r.Co, r.H, r.W
    M = N * H * W
    tdt = torch.float32 if r.dtype == TF32X3 else r.dtype
    in_l = "nhwc" if r.layout == "nhwc" else "nchw"    # x, dx
    out_l = "nchw" if r.layout == "nchw" else "nhwc"   # y, dy, residual
    lay = {"nhwc": A.NHWC, "nchw": A.NCHW, "planes": A.PLANES_TO_NHWC}[r.layout]
    code = _abi_dtype(kdcc, r.dtype)
    has_scale, has_shift, relu, has_res, raw, act = EPILOGUES[r.epi]
    gen = torch.Generator("cuda").manual_seed(10000 + seed)
    x = draw(gen, (N, K, H, W), "act", exact, tdt)
    dy = draw(gen, (N, Co, H, W), "act", exact, tdt)
    w = draw(gen, (Co, K), "tap", exact, tdt)
    scale = draw(gen, (Co,), "tap", exact) if has_scale else None
    shift = draw(gen, (Co,), "tap", exact) if has_shift else None
    res = draw(gen, (N, Co, H, W), "act", exact, tdt) if has_res else None
    xd, dyd = physical(x, in_l), physical(dy, out_l)
    resd = physical(res, out_l) if res is not None else None

    def reference(x, w, dy, scale, shift, res):
        out = torch.einsum("nkhw,ok->nohw", x, w)
        a = out
        if scale is not None:
            a = a * scale.view(1, -1, 1, 1)
        if shift is not None:
            a = a + shift.view(1, -1, 1, 1)
        if res is not None:
            a = a + res
        if relu:
            a = a.clamp_min(0)
        return {"y_raw": out, "y_act": a, "dx": torch.einsum("nohw,ok->nkhw", dy, w),
                "dw": torch.einsum("nohw,nkhw->ok", dy, x), "db": dy.sum((0, 2, 3))}

    dbl = lambda t: None if t is None else t.double()  # noqa: E731
    ref = reference(x.double(), w.double(), dy.double(), dbl(scale), dbl(shift), dbl(res))
    S = None
    if not exact:
        ab = lambda t: None if t is None else t.double().abs()  # noqa: E731
        S = reference(ab(x), ab(w), ab(dy), ab(scale), ab(shift), ab(res))   # ReLU does not widen a difference

    st = _stream()
    outs = {}
    if raw:
        outs["y_raw"] = Out((N, Co, H, W), tdt, out_l)
    if act:
        outs["y_act"] = Out((N, Co, H, W), tdt, out_l)
    p_ = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    o_ = lambda key: outs[key].ptr if key in outs else None  # noqa: E731

    def fwd():
        if res is not None:
            rc = L.kdcc_pw_fwd_residual(xd.data_ptr(), w.data_ptr(), p_(scale), p_(shift), resd.data_ptr(), int(relu),
                                        o_("y_raw"), o_("y_act"), M, K, Co, N, lay, code, st)
        else:
            rc = L.kdcc_pw_fwd(xd.data_ptr(), w.data_ptr(), p_(scale), p_(shift), int(relu), o_("y_raw"), o_("y_act"),
                               M, K, Co, N, lay, code, st)
        A.check(rc, "kdcc_pw_fwd")

    inputs = [t for t in (xd, w, scale, shift, resd) if t is not None]
    got = run_checked(fwd, outs, None, inputs, r.fwd, "forward")

    dx = Out((N, K, H, W), tdt, in_l)
    got.update(run_checked(lambda: A.check(L.kdcc_pw_bwd_dx(dyd.data_ptr(), w.data_ptr(), dx.ptr, None, 0, M, K, Co, N,
                                                            lay, code, st), "kdcc_pw_bwd_dx"),
                           {"dx": dx}, None, [dyd, w], r.dx, "input gradient"))

    dwo = Out((Co, K), torch.float32)
    ws = Guarded(L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, code))
    got.update(run_checked(lambda: A.check(L.kdcc_pw_bwd_dw(dyd.data_ptr(), xd.data_ptr(), dwo.ptr, ws.ptr, ws.n, M, K,
                                                            Co, N, lay, code, st), "kdcc_pw_bwd_dw"),
                           {"dw": dwo}, ws, [dyd, xd], r.dw, "weight gradient"))

    if r.epi == "bias":   # the conv bias's gradient: column sums of dy over the pixel-major view
        dy_pm = physical(dy, "nhwc")
        db = Out((Co,), torch.float32)
        cws = Guarded(L.kdcc_colsum_workspace_bytes(M, Co))
        got.update(run_checked(lambda: A.check(L.kdcc_colsum(dy_pm.data_ptr(), db.ptr, cws.ptr, cws.n, M, Co,
                                                             A.BF16 if tdt == BF16 else A.F32, st), "kdcc_colsum"),
                               {"db": db}, cws, [dy_pm], set(), "bias gradient"))

    terms = {"y_raw": K + 4, "y_act": K + 4, "dx": Co + 1, "dw": M + 1, "db": M}
    axes = {"y_raw": "ncij", "y_act": "ncij", "dx": "ncij", "dw": "ok", "db": "o"}
    for key, dev in got.items():
        if exact:
            assert_exact(key, dev, ref[key], axes[key])
        else:
            assert_bound(key, dev, ref[key], S[key], terms[key], axes[key])


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [True, False], ids=["exact", "bound"])
@pytest.mark.parametrize("row", POINTWISE, ids=pw_id)
def test_pointwise_edges(kdcc, row, exact):
    if row.dtype == TF32X3 and not exact:
        pytest.skip("tf32x3 bound mode: test_pw_tf32x3.py")
    pw_case(kdcc, row, POINTWISE.index(row), exact)


# ---------------------------------------------------------------------------------------------------------------------
# autograd through kdcc.functional and DepthwiseSeparableBlock (exact mode): the Python-level layout routing
# ---------------------------------------------------------------------------------------------------------------------
FUNCTIONAL = [
    # input ('nchw' plain, 'cl' channels_last), dtype, N, C, H, W, k, d, p, bias, forward kernels, backward kernels
    # NCHW padding past the halo: the transposed padding d(k-1) - p would be negative, so the call runs NHWC
    ("nchw", BF16, 2, 16, 16, 16, 3, 1, 5, False, {TC}, {DC, TW}),
    ("nchw", BF16, 1, 16, 16, 24, 5, 2, 12, False, {DC}, {DC, DWG}),
    ("cl", BF16, 1, 16, 16, 24, 5, 2, 12, False, {DC}, {DC, DWG}),
    ("nchw", BF16, 1, 16, 16, 16, 9, 5, 44, False, {TC}, {DC, TW}),
    # channels_last k > 3 re-laid to planes; fp32 and a bias run NHWC
    ("cl", BF16, 2, 16, 24, 40, 9, 5, 20, False, {C2}, {C2, WG3}),
    ("nchw", F32, 2, 16, 24, 40, 3, 1, 1, False, {DC}, {DC, DWG}),
    ("nchw", BF16, 2, 16, 24, 40, 9, 5, 20, True, {TC}, {TC, DWG}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("row", FUNCTIONAL, ids=lambda r: "%s-%s-c%d-%dx%d-k%dd%dp%d%s" % (
    r[0], "f32" if r[1] == F32 else "bf16", r[3], r[4], r[5], r[6], r[7], r[8], "-bias" if r[9] else ""))
def test_functional_depthwise_routes_and_matches(kdcc, row):
    fmt, dtype, N, C, H, W, k, d, p, bias, exp_fwd, exp_bwd = row
    gen = torch.Generator("cuda").manual_seed(N * C + H + W + k + d + p)
    Ho, Wo = H + 2 * p - d * (k - 1), W + 2 * p - d * (k - 1)
    x = draw(gen, (N, C, H, W), "act", True, dtype)
    if fmt == "cl":
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    w = draw(gen, (C, 1, k, k), "tap", True).requires_grad_(True)
    b = draw(gen, (C,), "tap", True).requires_grad_(True) if bias else None
    dy = draw(gen, (N, C, Ho, Wo), "act", True, dtype)
    out = {}

    def forward():
        out["y"] = kdcc.functional.depthwise_conv(x, w, b, k, d, p)

    ran_fwd = kernel_set(launched(forward))
    y = out["y"]
    ran_bwd = kernel_set(launched(lambda: y.backward(dy)))
    assert (ran_fwd, ran_bwd) == (exp_fwd, exp_bwd)
    if fmt == "cl":
        assert x.grad.is_contiguous(memory_format=torch.channels_last)
    ref = dw_reference(x.detach().double(), w.detach().double(), None if b is None else b.detach().double(), dy.double(),
                       k, d, p, "xwb" if bias else "xw")
    assert_exact("y", y.detach(), ref["y"], "ncij")
    assert_exact("dx", x.grad, ref["dx"], "ncij")
    assert_exact("dw", w.grad.reshape(C, k, k), ref["dw"], "cuv")
    if bias:
        assert_exact("db", b.grad, ref["db"], "c")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["nchw", "cl"])
def test_block_stages_match_in_exact_mode(kdcc, fmt, monkeypatch):
    """DepthwiseSeparableBlock with autograd, each stage against the float64 reference of its own device input: the
    depthwise output and its gradient are the bf16 tensors the pointwise stage produced or read."""
    N, Ci, Co, H, W, k, d, p = 1, 16, 32, 16, 16, 9, 5, 20
    gen = torch.Generator("cuda").manual_seed(7)
    blk = kdcc.DepthwiseSeparableBlock(Ci, Co, k, p, d, Ci, None).cuda()
    with torch.no_grad():
        blk.separable_conv.weight.copy_(draw(gen, (Ci, 1, k, k), "tap", True))
        blk.pointwise_conv.weight.copy_(draw(gen, (Co, Ci, 1, 1), "tap", True))
    x = draw(gen, (N, Ci, H, W), "act", True, BF16)
    if fmt == "cl":
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    dy = draw(gen, (N, Co, H, W), "act", True, BF16)
    mids = []
    real = kdcc.functional.depthwise_conv

    def keep(*a, **kw):
        m = real(*a, **kw)
        m.retain_grad()
        mids.append(m)
        return m

    monkeypatch.setattr(kdcc.functional, "depthwise_conv", keep)
    y = blk(x)
    y.backward(dy)
    mid = mids[0]
    wd, wp = blk.separable_conv.weight.detach().double(), blk.pointwise_conv.weight.detach().double().reshape(Co, Ci)
    m64, dm64 = mid.detach().double(), mid.grad.double()
    # the depthwise stage (on the tensor cores: bf16 taps, which eighths are)
    ref = dw_reference(x.detach().double(), wd, None, dm64, k, d, p, "xw")
    assert_exact("depthwise y", mid.detach(), ref["y"], "ncij")
    assert_exact("depthwise dx", x.grad, ref["dx"], "ncij")
    assert_exact("depthwise dw", blk.separable_conv.weight.grad.reshape(Ci, k, k), ref["dw"], "cuv")
    # the pointwise stage on the depthwise stage's own bf16 output
    assert_exact("pointwise y", y.detach(), torch.einsum("nkhw,ok->nohw", m64, wp), "ncij")
    assert_exact("pointwise dx", mid.grad, torch.einsum("nohw,ok->nkhw", dy.double(), wp), "ncij")
    assert_exact("pointwise dw", blk.pointwise_conv.weight.grad.reshape(Co, Ci),
                 torch.einsum("nohw,nkhw->ok", dy.double(), m64), "ok")


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the table's own guarantees
# ---------------------------------------------------------------------------------------------------------------------
def test_exact_rows_stay_inside_fp32():
    for r in DEPTHWISE:
        assert dw_exact_units(r) < FP32_UNITS, dw_id(r)
    for r in POINTWISE:
        assert pw_exact_units(r) < FP32_UNITS, pw_id(r)
    # the block test: depthwise output <= 8 * 81 in eighths, its gradient <= 8 * 32 in eighths
    assert 8 * 81 * 8 * 8 * 16 * 16 < FP32_UNITS and 8 * 8 * 32 * 8 * 16 * 16 < FP32_UNITS


def test_exact_check_rejects_one_ulp():
    gen = torch.Generator().manual_seed(0)
    ref = torch.randint(-4096, 4096, (2, 3, 5, 7), generator=gen).double() / 8
    dev = ref.float().to(torch.bfloat16)
    assert_exact("y", dev, ref, "ncij")
    bumped = dev.clone()
    bumped.view(torch.int16)[1, 2, 3, 4] += 1   # one bf16 ulp
    with pytest.raises(AssertionError, match=r"1 of 210 elements wrong; first at \(n=1, c=2, i=3, j=4\)"):
        assert_exact("y", bumped, ref, "ncij")
    dw_ref = torch.randint(-1000, 1000, (4, 3, 3), generator=gen).double()
    dw_dev = dw_ref.float().clone()
    dw_dev[2, 0, 1] += 1
    with pytest.raises(AssertionError, match=r"first at \(c=2, u=0, v=1\)"):
        assert_exact("dw", dw_dev, dw_ref, "cuv")


def test_bound_check_rejects_an_edge_pixel_missing_its_smallest_tap():
    gen = torch.Generator().manual_seed(1)
    N, C, H, W, k, d, p = 1, 4, 12, 12, 3, 1, 1
    x = torch.randn(N, C, H, W, generator=gen, dtype=torch.float64)
    x = x.sign() * (x.abs() + 0.25)                     # |x| >= 1/4
    w = torch.rand(C, k, k, generator=gen, dtype=torch.float64) * 0.9 + 0.1
    ref = dw_reference(x, w, None, torch.zeros(N, C, H, W, dtype=torch.float64), k, d, p, "")["y"]
    S = dw_reference(x.abs(), w, None, torch.zeros(N, C, H, W, dtype=torch.float64), k, d, p, "")["y"]
    dev = ref.float()
    assert_bound("y", dev, ref, S, k * k + 1, "ncij")
    # corner (0, 0) of channel 2 without its smallest in-bounds tap term (taps u, v >= 1 reach inside the image)
    terms = {(u, v): w[2, u, v] * x[0, 2, u - 1, v - 1] for u in (1, 2) for v in (1, 2)}
    (u, v), t = min(terms.items(), key=lambda kv: abs(kv[1]))
    dev[0, 2, 0, 0] -= float(t)
    with pytest.raises(AssertionError, match=r"first at \(n=0, c=2, i=0, j=0\)"):
        assert_bound("y", dev, ref, S, k * k + 1, "ncij")
    dev16 = ref.to(torch.bfloat16)                      # the same check of a bf16 output with its RNE allowance
    assert_bound("y", dev16, ref, S, k * k + 1, "ncij")


def _global_kernels():
    names = set()
    for fn in sorted(os.listdir(CSRC)):
        if re.match(r"(dw|pw)_.*\.cu$", fn):
            src = open(os.path.join(CSRC, fn)).read()
            names.update(re.findall(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s+)?(\w+)\s*\(", src))
    return names


def test_every_convolution_kernel_has_a_row():
    kernels = _global_kernels()
    assert {"dw_tc_conv_kernel", "pw_gemm_sm100_kernel", "reduce_splits_kernel"} <= kernels   # the parse works
    pinned = set()
    for r in DEPTHWISE:
        pinned |= r.fwd | r.bwd
    for r in POINTWISE:
        pinned |= r.fwd | r.dx | r.dw
    pinned = {n.split("<")[0] for n in pinned}
    missing = kernels - pinned - set(NOT_PINNED)
    assert not missing, "kernels without a parity row in test_conv_edges.py: %s" % sorted(missing)
    assert set(NOT_PINNED) <= kernels, "exclusions naming no kernel: %s" % sorted(set(NOT_PINNED) - kernels)
    assert not set(NOT_PINNED) & pinned


PAST_HALO = [(3, 1, 5), (5, 2, 12), (9, 5, 44), (1, 1, 4), (3, 4, 12)]


@pytest.mark.parametrize("k,d,p", PAST_HALO)
def test_nchw_padding_past_the_halo_is_not_routed_to_the_tensor_cores(kdcc, k, d, p):
    A = kdcc._abi
    N, C, H, W = 2, 16, 16, 16
    assert (W + 2 * p - d * (k - 1)) % 8 == 0   # every other NCHW condition holds
    for op in (0, 1):
        assert A.dispatch_name(op, N, H, W, C, C, k, d, p, A.NCHW, A.BF16) == "unsupported"
        assert not kdcc.functional._supported(op, N, H, W, C, C, k, d, p, A.NCHW, A.BF16)
    L = A.lib()
    assert L.kdcc_dw_bwd_workspace_bytes(N, H, W, C, k, d, p, A.NCHW, A.BF16) == 0
    rc = L.kdcc_dw_fwd(16, 16, None, 16, N, H, W, C, k, d, p, A.NCHW, A.BF16, None)   # refused before any launch
    assert rc == -2, A.strerror(rc)
    # padding up to the halo still runs there
    assert A.dispatch_name(1, N, H, W, C, C, 9, 5, 40, A.NCHW, A.BF16) == "dw_tc_wgrad"
