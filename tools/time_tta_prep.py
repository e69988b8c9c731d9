"""Times the test-time window preparation of inference_test at 2048 x 1024, crop 1024 (measurement tooling, needs a GPU).

    python tools/time_tta_prep.py [--iters 20] [--reps 7] [--out profiles/r07_tta_prep.json]

One ImageNet-normalised fp32 (3, 1024, 2048) image on the device, as inference_test receives it, at scale 1.0 (a plain
copy: 3 + 3 windows of 1024 x 1024) and at scale 0.75 (both resampling passes: 3 + 3 windows of 768 x 768).  Two arms,
alternated rep by rep in one process, the median of the reps reported:
  a) the host preparation as inference_test ran it before kdcc_tta_windows: ToPILImage(x.cpu()), scale_and_flip_image,
     get_crops_image, windows.to(device); host clock around `iters` calls ending in a synchronise;
  b) kdcc.tta.prepare_windows: CUDA events around `iters` back-to-back calls after a warm-up.  Each call reads a
     different one of 6 input copies (6 x 25 MB, larger than the 126 MB L2).  This includes the Python wrapper's
     enqueue cost where it exceeds the kernels' time;
  c) the kernels alone: the same `iters` kdcc.functional.tta_windows calls captured in one CUDA graph, CUDA events
     around its replay.
The windows of both arms must be equal.  The GPU name, power limit and max SM clock and the host core count are recorded
beside the numbers."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kdcc  # noqa: E402
from kdcc import tta  # noqa: E402

H, W, CROP = 1024, 2048, 1024
COPIES = 6
MEAN_STD = ([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else "nvidia-smi unavailable"


def make_image(seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(3, H, W, device="cuda", generator=g)
    m, s = (torch.tensor(v, device="cuda").view(3, 1, 1) for v in MEAN_STD)
    return ((x - m) / s).contiguous()


def host_formulation(x, scales):
    from torchvision import transforms
    image_data = tta.scale_and_flip_image(transforms.ToPILImage()(x.cpu()), MEAN_STD, scales)
    ori_size, mapping, windows = tta.get_crops_image(image_data, scales, crop_size=CROP)
    return ori_size, mapping, windows.to(x.device)


def time_host(xs, scales, iters):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(iters):
        host_formulation(xs[i % COPIES], scales)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / iters


def time_device(xs, scales, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        tta.prepare_windows(xs[i % COPIES], scales, CROP, MEAN_STD)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def graph_of_calls(xs, s, iters):
    h, w, tile = int(H * s), int(W * s), int(s * CROP)
    stride = math.ceil(tile * (1 - 1 / 3))   # as tta.window_coordinates
    out = torch.empty((2 * len(tta.window_coordinates(w, h, tile)), 3, min(tile, h), min(tile, w)), device="cuda")
    call = lambda i: kdcc.functional.tta_windows(xs[i % COPIES], h, w, tile, stride, *MEAN_STD, out=out)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        call(0)                      # workspace of the capture stream in place
    torch.cuda.current_stream().wait_stream(st)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        for i in range(iters):
            call(i)
    return g


def time_graph(g, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def byte_model(s):
    """Bytes the preparation must move: the fp32 image read once, the uint8 intermediate of the horizontal pass written
    and read once, the fp32 windows written once."""
    h, w, tile = int(H * s), int(W * s), int(s * CROP)
    n = len(tta.window_coordinates(w, h, tile))
    inter = 2 * 3 * H * w if w != W else 0
    return 3 * H * W * 4 + inter + 2 * n * 3 * min(tile, h) * min(tile, w) * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_tta_prep.py needs a CUDA device")
    info = {"gpu": gpu_info(), "fields": "name, power.limit, clocks.max.sm", "host_cpus": os.cpu_count(),
            "image": [3, H, W], "dtype": "float32", "data": "ImageNet-normalised uniform noise", "crop_size": CROP,
            "iters": a.iters, "reps": a.reps, "cases": []}
    print(info["gpu"], "| host cpus", info["host_cpus"])
    xs = [make_image(s) for s in range(COPIES)]
    for s in (1.0, 0.75):
        scales = [s]
        ref, got = host_formulation(xs[0], scales), tta.prepare_windows(xs[0], scales, CROP, MEAN_STD)
        torch.cuda.synchronize()
        equal = ref[:2] == got[:2] and bool(torch.equal(ref[2], got[2]))
        assert equal, "scale %r: device windows differ from the host preparation" % s
        time_device(xs, scales, 3)
        g = graph_of_calls(xs, s, a.iters)
        time_graph(g, a.iters)
        ms = {"a_host_pil": [], "b_prepare_windows": [], "c_kernels_graph": []}
        for _ in range(a.reps):
            ms["a_host_pil"].append(time_host(xs, scales, max(2, a.iters // 4)))
            ms["b_prepare_windows"].append(time_device(xs, scales, a.iters))
            ms["c_kernels_graph"].append(time_graph(g, a.iters))
        del g
        nbytes = byte_model(s)
        case = {"scale": s, "windows": list(got[2].shape), "outputs_equal": equal, "alg_bytes": nbytes,
                "alg_us_at_7.7TBps": round(nbytes / 7.7e12 * 1e6, 2), "arms": {}}
        for k, v in ms.items():
            med = statistics.median(v)
            case["arms"][k] = {"ms": round(med, 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4)}
            print("scale %-5s %-18s %9.4f ms  [%0.4f, %0.4f]" % (s, k, med, min(v), max(v)))
        dev = case["arms"]["b_prepare_windows"]["ms"]
        case["speedup"] = round(case["arms"]["a_host_pil"]["ms"] / dev, 1)
        case["b_alg_TBps"] = round(nbytes / dev / 1e9, 3)
        case["c_alg_TBps"] = round(nbytes / case["arms"]["c_kernels_graph"]["ms"] / 1e9, 3)
        info["cases"].append(case)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
