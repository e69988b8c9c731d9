"""numpy restatement of the test-time window preparation of utils/tta_process.py:52-117 as kdcc.tta's host mirror runs it
(ToPILImage, PIL resize BILINEAR, FLIP_LEFT_RIGHT, ToTensor + Normalize, window crops), the reference
kdcc.functional.tta_windows is checked against.  It needs numpy only; Pillow 12.2 and torch agree with it bit for bit
(tests/test_tta_prep.py).

It sits beside its tests, like canny_oracle.py: it is pinned on Pillow and torch, not on the reference repository."""
import math

import numpy as np

from canny_oracle import to_uint8_like_numpy

PRECISION_BITS = 22  # Pillow's fixed point for 8-bit resampling: 32 - 8 - 2


def bf16_round(x):
    """float32 -> nearest bfloat16 (ties to even), returned as float32; NaN stays NaN."""
    x = np.asarray(x, np.float32)
    b = x.view(np.uint32).astype(np.uint64)
    r = ((b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000).astype(np.uint32).view(np.float32)
    return np.where(np.isnan(x), x, r)


def to_pil_bytes(x, bf16=False):
    """torchvision ToPILImage's `pic.mul(255).byte()` on the CPU: the product in the input dtype (bf16 rounds it), then
    truncate toward zero to int32 and keep the low 8 bits; NaN, +-inf and values outside int32 give 0."""
    p = np.asarray(x, np.float32) * np.float32(255)
    if bf16:
        p = bf16_round(p)
    return to_uint8_like_numpy(p)


def pil_coeffs(in_size, out_size):
    """Pillow's precompute_coeffs + normalize_coeffs_8bpc for the BILINEAR filter: per output index (xmin, [k]) with k
    the fixed-point weights of input pixels xmin, xmin + 1, ...  Python floats are IEEE doubles without FMA, as the
    C code runs."""
    scale = float(in_size) / out_size
    fs = max(scale, 1.0)
    support = fs
    ss = 1.0 / fs
    out = []
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        ws = []
        for x in range(xmax):
            t = abs((x + xmin - center + 0.5) * ss)
            ws.append(1.0 - t if t < 1.0 else 0.0)
        ww = 0.0
        for v in ws:
            ww += v
        if ww != 0.0:
            ws = [v / ww for v in ws]
        out.append((xmin, [int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
                           for v in ws]))
    return out


def _pass(img, out_size, axis):
    """One 8-bit resampling pass of uint8 `img` along `axis`; a pass whose size is unchanged is skipped."""
    in_size = img.shape[axis]
    if in_size == out_size:
        return img
    src = np.moveaxis(img.astype(np.int64), axis, 0)
    acc = np.empty((out_size,) + src.shape[1:], np.int64)
    for xx, (xmin, k) in enumerate(pil_coeffs(in_size, out_size)):
        s = np.full(src.shape[1:], 1 << (PRECISION_BITS - 1), np.int64)
        for i, kv in enumerate(k):
            s += src[xmin + i] * kv
        acc[xx] = s
    res = np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)
    return np.moveaxis(res, 0, axis)


def pil_resize(img, w, h):
    """`Image.resize((w, h), BILINEAR)` of a uint8 (H, W) or (H, W, C) image: horizontal pass, then vertical."""
    return _pass(_pass(np.asarray(img, np.uint8), w, 1), h, 0)


def normalise(u8_chw, mean, std):
    """ToTensor + Normalize: (u / 255 - mean_c) / std_c, each step one fp32 operation."""
    f = np.asarray(u8_chw).astype(np.float32) / np.float32(255)
    m = np.asarray(mean, np.float32).reshape(-1, 1, 1)
    s = np.asarray(std, np.float32).reshape(-1, 1, 1)
    return (f - m) / s


def window_boxes(w, h, tile, stride):
    """tta.window_coordinates with the stride given: [(x1, y1, x2, y2)], x outer / y inner."""
    nx = int(math.ceil((w - tile) / stride) + 1)
    ny = int(math.ceil((h - tile) / stride) + 1)
    boxes = []
    for ix in range(nx):
        for iy in range(ny):
            x2, y2 = min(ix * stride + tile, w), min(iy * stride + tile, h)
            boxes.append((max(x2 - tile, 0), max(y2 - tile, 0), x2, y2))
    return boxes


def tta_windows(x, h, w, tile, stride, mean, std, bf16=False):
    """One scale of one image: x (3, H, W) float -> (2n, 3, th, tw) float32, the n plain windows of the image resized to
    (w, h), then the n windows of its mirror."""
    u8 = to_pil_bytes(x, bf16).transpose(1, 2, 0)
    scaled = pil_resize(u8, w, h)
    boxes = window_boxes(w, h, tile, stride)
    out = []
    for img in (scaled, scaled[:, ::-1]):
        t = normalise(img.transpose(2, 0, 1), mean, std)
        out += [t[:, y1:y2, x1:x2] for x1, y1, x2, y2 in boxes]
    return np.stack(out)
