"""Writes tests/golden/canny.npz: a handful of uint8 images with their cv2.Canny output (aperture 3, L1 gradient).

    python tools/make_canny_golden.py [--out tests/golden/canny.npz]

It freezes the output of the call the Gated-SCNN forward makes (models/gscnn/gscnn.py:284-288), so boxes where cv2 is
absent or differs still have it to check against.  Needs numpy and cv2 only.  Case k is stored as img_k (H, W, C) uint8,
thr_k (low, high) float64 and edges_k (H, W) uint8."""
import argparse
import os

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def images(rs):
    yy, xx = np.mgrid[:96, :160]
    noise = rs.randint(0, 256, (96, 160, 3)).astype(np.uint8)
    smooth = np.clip(cv2.GaussianBlur(rs.rand(96, 160, 3).astype(np.float32) * 255, (0, 0), 2.0), 0, 255).astype(np.uint8)
    shapes = np.zeros((96, 160, 3), np.uint8)
    for cy, cx, r, col in ((30, 40, 20, (200, 30, 90)), (60, 110, 28, (40, 180, 240)), (80, 20, 12, (255, 255, 0))):
        shapes[(yy - cy) ** 2 + (xx - cx) ** 2 < r * r] = col
    ramp = ((xx * 3 + yy * 5) % 256).astype(np.uint8)[:, :, None].repeat(3, 2)
    odd = rs.randint(0, 4, (33, 65, 3)).astype(np.uint8) * 60   # few levels: many channel ties
    return [(noise, (10, 100)), (smooth, (10, 100)), (shapes, (50, 150)), (ramp, (100, 10)), (odd, (30.7, 30.2)),
            (smooth, (0, 0))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "canny.npz"))
    a = ap.parse_args()
    rs = np.random.RandomState(2024)
    arrays = {}
    for k, (img, thr) in enumerate(images(rs)):
        arrays["img_%d" % k] = img
        arrays["thr_%d" % k] = np.array(thr, dtype=np.float64)
        arrays["edges_%d" % k] = cv2.Canny(img, thr[0], thr[1])
    np.savez_compressed(a.out, **arrays)
    print("wrote", a.out, os.path.getsize(a.out), "bytes,", len(arrays) // 3, "cases, cv2", cv2.__version__)


if __name__ == "__main__":
    main()
