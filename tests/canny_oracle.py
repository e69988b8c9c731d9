"""numpy restatement of the Gated-SCNN Canny edge map (models/gscnn/gscnn.py:284-288), the reference kdcc.functional.canny_edges
is checked against.  It needs numpy and scipy only; cv2 4.13 agrees with it bit for bit (tests/test_canny.py).

It sits beside its tests rather than in oracle/: the oracle there is pinned on the reference repository's own modules
(oracle/make_golden.py runs them), while this one is pinned on cv2 alone.  Its golden file, tests/golden/canny.npz, comes
from tools/make_canny_golden.py, which needs only cv2 and numpy."""
import math

import numpy as np

TG22 = 13573  # round(tan(22.5 deg) * 2^15), cv2's integer sector bound


def to_uint8_like_numpy(x):
    """`x.astype(np.uint8)` for float input as numpy does it on x86-64: truncate toward zero to int32 and keep the low 8
    bits; NaN, +-inf and values whose truncation does not fit int32 give 0 (cvttss2si's INT_MIN, low byte 0)."""
    x = np.asarray(x, dtype=np.float64)
    t = np.trunc(x)
    ok = np.isfinite(t) & (t >= -2.0 ** 31) & (t < 2.0 ** 31)
    return (np.where(ok, t, 0).astype(np.int64) & 0xFF).astype(np.uint8)


def canny(img, low, high):
    """cv2.Canny(img, low, high) with aperture 3 and the L1 gradient: img uint8 (H, W) or (H, W, C); returns uint8 0 / 255."""
    img = np.asarray(img)
    if img.ndim == 2:
        img = img[:, :, None]
    if low > high:
        low, high = high, low
    lo, hi = math.floor(low), math.floor(high)
    H, W, _ = img.shape
    p = np.pad(img.astype(np.int32), ((1, 1), (1, 1), (0, 0)), mode="edge")
    col = lambda j: p[:-2, j:j + W] + 2 * p[1:-1, j:j + W] + p[2:, j:j + W]
    row = lambda i: p[i:i + H, :-2] + 2 * p[i:i + H, 1:-1] + p[i:i + H, 2:]
    dx_c, dy_c = col(2) - col(0), row(2) - row(0)
    mag_c = np.abs(dx_c) + np.abs(dy_c)
    ch = np.argmax(mag_c, axis=2)[:, :, None]  # first channel on a tie
    dx = np.take_along_axis(dx_c, ch, 2)[:, :, 0].astype(np.int64)
    dy = np.take_along_axis(dy_c, ch, 2)[:, :, 0].astype(np.int64)
    m = np.take_along_axis(mag_c, ch, 2)[:, :, 0].astype(np.int64)

    M = np.pad(m, 1)  # neighbours outside the image have magnitude 0
    nb = lambda di, dj: M[1 + di:1 + di + H, 1 + dj:1 + dj + W]
    xs, ys = np.abs(dx), np.abs(dy)
    y = ys << 15
    tg22x = xs * TG22
    tg67x = tg22x + (xs << 16)
    horiz = y < tg22x
    vert = ~horiz & (y > tg67x)
    opposite = (dx ^ dy) < 0
    keep = np.where(horiz, (m > nb(0, -1)) & (m >= nb(0, 1)),
           np.where(vert, (m > nb(-1, 0)) & (m >= nb(1, 0)),
           np.where(opposite, (m > nb(-1, 1)) & (m > nb(1, -1)), (m > nb(-1, -1)) & (m > nb(1, 1)))))
    cand = keep & (m > lo)
    strong = cand & (m > hi)

    from scipy import ndimage
    lab, _ = ndimage.label(cand, structure=np.ones((3, 3), dtype=bool))
    hit = np.unique(lab[strong])
    out = np.isin(lab, hit[hit > 0]) & cand
    return np.where(out, 255, 0).astype(np.uint8)


def gscnn_canny(inp, low=10, high=100):
    """The GSCNN forward's edge input with this module in place of cv2: inp (N, 3, H, W) float (numpy or a torch tensor on
    any device) -> (N, 1, H, W) fp32 of 0 / 255."""
    if hasattr(inp, "detach"):
        inp = inp.detach().float().cpu().numpy()
    im = to_uint8_like_numpy(np.asarray(inp).transpose(0, 2, 3, 1))
    N, H, W = im.shape[0], im.shape[1], im.shape[2]
    out = np.zeros((N, 1, H, W), dtype=np.float32)
    for i in range(N):
        out[i, 0] = canny(im[i], low, high)
    return out
