"""Sliding-window test-time inference on the GPU: window preparation and stitching of utils/tta_process.py.

The reference (models/students/depthwise_student.py:187-206 -> utils/tta_process.py) rescales and mirrors the image
with PIL, cuts overlapping square windows, runs the student on all of them, copies the outputs to the host and
stitches them with numpy + cv2 in float64.  Here `prepare_windows` makes the windows on the device, bit-identical to
the PIL / torchvision preparation (`kdcc_tta_windows`; `scale_and_flip_image` / `get_crops_image` keep the host
formulation as its mirror), the window outputs never leave the device and `reverse_mapping` is two kdcc kernels
(`kdcc_tta_stitch`, `kdcc_resize_bilinear`).

`count_mode="reference"` reproduces the reference's result exactly -- including its window counter, which
utils/tta_process.py:46 indexes `[y1:y2, x1:x2]` on a (classes, h, w) array, so that overlaps are NOT normalised per
pixel (the arg-max over classes is unaffected: every class of a pixel is divided by the same number).
`count_mode="coverage"` divides by the true per-pixel coverage.
"""
import math

import torch

from . import functional as F


def window_coordinates(w, h, tile, overlap=1 / 3):
    """[(x1, y1, x2, y2)] of utils/tta_process.py:81-105: stride ceil(tile * (1 - overlap)), x outer / y inner, the last
    window of an axis pulled back inside the image."""
    stride = math.ceil(tile * (1 - overlap))
    nx = int(math.ceil((w - tile) / stride) + 1)
    ny = int(math.ceil((h - tile) / stride) + 1)
    boxes = []
    for ix in range(nx):
        for iy in range(ny):
            x2, y2 = min(ix * stride + tile, w), min(iy * stride + tile, h)
            boxes.append((max(x2 - tile, 0), max(y2 - tile, 0), x2, y2))
    return boxes


def scale_and_flip_image(image, mean_std, scales=(1.0,)):
    """PIL image -> ((w, h), [[scaled, mirrored] per scale]) as normalised tensors (utils/tta_process.py:55-68)."""
    from PIL import Image
    from torchvision import transforms
    to_tensor = transforms.Compose([transforms.ToTensor(), transforms.Normalize(*mean_std)])
    w, h = image.size
    pairs = []
    for s in scales:
        scaled = image.resize((int(w * s), int(h * s)), Image.BILINEAR)
        pairs.append([to_tensor(scaled), to_tensor(scaled.transpose(Image.FLIP_LEFT_RIGHT))])
    return (w, h), pairs


def get_crops_image(image_data, scales=(1.0,), crop_size=512, overlap=1 / 3):
    """-> (ori_size, mapping, windows): mapping = [[w, h, boxes] per scale]; windows = all crops, per scale the plain
    ones then the mirrored ones (utils/tta_process.py:71-117).  Like the reference this concatenates the crops of all
    scales into one batch, which needs int(scale * crop_size) to be the same for every scale."""
    ori_size, pairs = image_data
    mapping, batches = [], []
    for (plain, mirrored), s in zip(pairs, scales):
        h, w = plain.shape[1:]
        boxes = window_coordinates(w, h, int(s * crop_size), overlap)
        mapping.append([w, h, boxes])
        for img in (plain, mirrored):
            batches.append(torch.stack([img[:, y1:y2, x1:x2] for x1, y1, x2, y2 in boxes]))
    return ori_size, mapping, torch.cat(batches, dim=0)


@torch.no_grad()
def prepare_windows(x, scales, crop_size, mean_std, overlap=1 / 3):
    """get_crops_image(scale_and_flip_image(ToPILImage()(x.cpu()), mean_std, scales), scales, crop_size) on the device:
    the same (ori_size, mapping, windows), bit for bit, with `windows` on x's device.  x (3, H, W) fp32 or bf16 CUDA
    tensor.  Every scale writes its windows straight into one preallocated batch (kdcc_tta_windows); like the
    reference's torch.cat this needs every scale to give the same window size."""
    H, W = x.shape[-2:]
    plan = []
    for s in scales:
        w, h, tile = int(W * s), int(H * s), int(s * crop_size)
        if w < 1 or h < 1:
            raise ValueError("scale %r makes the %dx%d image empty" % (s, W, H))   # as PIL's resize
        stride = math.ceil(tile * (1 - overlap))
        boxes = window_coordinates(w, h, tile, overlap)
        if not boxes:
            raise RuntimeError("scale %r gives no window of %d pixels in the %dx%d image" % (s, tile, w, h))  # torch.stack
        plan.append((w, h, tile, stride, boxes, (min(tile, h), min(tile, w))))
    for p in plan[1:]:
        if p[5] != plan[0][5]:
            raise RuntimeError("Sizes of tensors must match except in dimension 0: scales give %dx%d and %dx%d windows"
                               % (plan[0][5] + p[5]))   # torch.cat's rule
    th, tw = plan[0][5]
    windows = torch.empty((sum(2 * len(p[4]) for p in plan), 3, th, tw), dtype=torch.float32, device=x.device)
    mapping, at = [], 0
    for w, h, tile, stride, boxes, _ in plan:
        F.tta_windows(x, h, w, tile, stride, *mean_std, out=windows[at:at + 2 * len(boxes)])
        mapping.append([w, h, boxes])
        at += 2 * len(boxes)
    return (W, H), mapping, windows


@torch.no_grad()
def reverse_mapping(mapping, results, ori_size, count_mode="reference"):
    """Window outputs -> per-scale class maps at the original size: (n_scales, C, h_ori, w_ori) fp32 on the device
    (utils/tta_process.py:9-26).  results: (total windows, C, th, tw) CUDA tensor in get_crops_image's order."""
    results = results.detach().float().contiguous()
    C = results.shape[1]
    W, H = ori_size
    out = torch.empty((len(mapping), C, H, W), dtype=torch.float32, device=results.device)
    idx = 0
    for k, (w, h, boxes) in enumerate(mapping):
        n = len(boxes)
        coords = torch.tensor(boxes, dtype=torch.int32).reshape(n, 4).to(results.device)
        same = (w, h) == (W, H)   # scale 1.0: cv2.resize to the same size is the identity
        stitched = out[k] if same else torch.empty((C, h, w), dtype=torch.float32, device=results.device)
        F.tta_stitch(results[idx:idx + n], coords, h, w, stitched, flip=False, count_mode=count_mode, alpha=0.5)
        F.tta_stitch(results[idx + n:idx + 2 * n], coords, h, w, stitched, flip=True, count_mode=count_mode, alpha=0.5,
                     accumulate=True)
        if not same:  # resizing is linear: resize(a)/2 + resize(b)/2 == resize((a + b)/2)
            F.resize_bilinear(stitched, out[k])
        idx += 2 * n
    return out


@torch.no_grad()
def inference_test(model, data, args, count_mode="reference"):
    """models/students/depthwise_student.py:187-206 for any callable `model` (windows -> class maps): per image the
    mean over scales of reverse_mapping; returns (N, C, H, W) on the device.  `data` goes through ToPILImage exactly
    as in the reference (which feeds it the already normalised batch), prepared on the device by prepare_windows: the
    same windows as the host preparation, without its round trip."""
    mean_std = ([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
    maps = []
    for x in data:
        ori_size, mapping, windows = prepare_windows(x, args['scales'], args['crop_size'], mean_std)
        maps.append(reverse_mapping(mapping, model(windows), ori_size, count_mode).mean(dim=0))
    return torch.stack(maps)
