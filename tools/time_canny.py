"""Times the Gated-SCNN Canny edge map at (2, 3, 1024, 2048) fp32 (measurement tooling, needs a GPU and cv2).

    python tools/time_canny.py [--iters 20] [--reps 5] [--out profiles/r05_canny.json]

Two images: blurred noise (edges along smooth contours) and pure noise (the most candidates, the most union-find
work).  Two arms, alternated rep by rep in one process:
  a) the host formulation of models/gscnn/gscnn.py:284-288: device->host copy, numpy transpose + uint8 cast, cv2.Canny
     per image, float64 host->device copy and .float(); host clock around `iters` calls ending in a synchronise;
  b) kdcc.functional.canny_edges: CUDA events around `iters` back-to-back calls after a warm-up.  Each call reads a
     different one of 4 input copies (4 x 50 MB, larger than the 126 MB L2).
The outputs of both arms must be equal.  The GPU name, power limit and max SM clock, the host core count and cv2's
thread count are recorded beside the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kdcc  # noqa: E402

N, H, W = 2, 1024, 2048
COPIES = 4


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else "nvidia-smi unavailable"


def make_image(kind, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(N, 3, H, W, device="cuda", generator=g) * 255
    if kind == "blurred_noise":   # 9 x 9 box blur per channel: smooth contours, few candidates
        x = torch.nn.functional.avg_pool2d(x, 9, stride=1, padding=4, count_include_pad=False)
    return x.contiguous()


def host_formulation(inp):
    im_arr = inp.cpu().numpy().transpose((0, 2, 3, 1)).astype(np.uint8)
    canny = np.zeros((inp.shape[0], 1, inp.shape[2], inp.shape[3]))
    for i in range(inp.shape[0]):
        canny[i] = cv2.Canny(im_arr[i], 10, 100)
    return torch.from_numpy(canny).cuda().float()


def time_host(xs, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(iters):
        host_formulation(xs[i % COPIES])
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / iters


def time_device(xs, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        kdcc.functional.canny_edges(xs[i % COPIES], 10, 100)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_canny.py needs a CUDA device")
    info = {"gpu": gpu_info(), "fields": "name, power.limit, clocks.max.sm", "host_cpus": os.cpu_count(),
            "cv2": cv2.__version__, "cv2_threads": cv2.getNumThreads(), "shape": [N, 3, H, W], "dtype": "float32",
            "thresholds": [10, 100], "iters": a.iters, "reps": a.reps,
            # one read of the fp32 image, one write of the map, int32 labels written once and read in ~3 passes
            "alg_bytes_est": N * H * W * (3 * 4 + 4 + 4 * 4), "cases": []}
    print(info["gpu"], "| host cpus", info["host_cpus"], "| cv2 threads", info["cv2_threads"])
    for kind in ("blurred_noise", "pure_noise"):
        xs = [make_image(kind, s) for s in range(COPIES)]
        ref, got = host_formulation(xs[0]), kdcc.functional.canny_edges(xs[0], 10, 100)
        torch.cuda.synchronize()
        equal = bool(torch.equal(ref, got))
        assert equal, "%s: device map differs from the host formulation at %d pixels" % (kind, int((ref != got).sum()))
        time_device(xs, 3)
        ms = {"a_host_cv2": [], "b_kdcc_canny": []}
        for _ in range(a.reps):
            ms["a_host_cv2"].append(time_host(xs, max(2, a.iters // 4)))
            ms["b_kdcc_canny"].append(time_device(xs, a.iters))
        case = {"image": kind, "edge_fraction": float((got > 0).float().mean()), "outputs_equal": equal, "arms": {}}
        for k, v in ms.items():
            med = statistics.median(v)
            case["arms"][k] = {"ms": round(med, 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4)}
            print("%-14s %-13s %9.4f ms  [%0.4f, %0.4f]" % (kind, k, med, min(v), max(v)))
        dev = case["arms"]["b_kdcc_canny"]["ms"]
        case["speedup"] = round(case["arms"]["a_host_cv2"]["ms"] / dev, 1)
        case["b_alg_TBps_est"] = round(info["alg_bytes_est"] / dev / 1e9, 3)
        info["cases"].append(case)
        del xs
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
