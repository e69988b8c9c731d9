"""fp32 pointwise GEMMs of the 51M plan's nine sites (batch 4, 128 x 128 maps: M = 65536): fwd, dX and dW, four arms
alternated in one process (DESIGN.md 4.3g):
  simt      kdcc dtype code 0 (the CUDA-core fp32 kernel)
  tf32x3    kdcc dtype code 2 (three tf32 tcgen05 products)
  cudnn     stock fp32 1x1 F.conv2d (and its input / weight gradients), channels_last, TF32 off
  cudnn_tf32  the same with TF32 on (1-pass TF32: fast, not fp32 accurate)
Inputs rotate over copies larger than the 126 MB L2; CUDA events over every timed call; each arm's max error against
float64 on the CPU over sampled rows (fwd, dX) or sampled channel pairs (dW).

    python tools/time_pw_fp32.py [--iters 50] [--warmup 5] [--out profiles/r06_pw_fp32.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import kdcc  # noqa: E402

A = kdcc._abi
SITES = [(512, 512, 5), (1024, 2048, 1), (4096, 256, 3)]   # (C_in, C_out, sites) of the 51M plan
N, H, W = 4, 128, 128
M = N * H * W
L2_BYTES = 126 << 20


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:   # the numbers are still reported, without the limit
        info["power_limit"] = "unknown (%s)" % e
    return info


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def kdcc_call(op, code, x, w, dy, out, ws):
    """x [M][K], w [Co][K], dy [M][Co] as flat row-major views; out is y, dx or dw."""
    L, st = A.lib(), torch.cuda.current_stream().cuda_stream
    K, Co = x.shape[1], w.shape[0]
    if op == "fwd":
        rc = L.kdcc_pw_fwd(x.data_ptr(), w.data_ptr(), None, None, 0, out.data_ptr(), None, M, K, Co, N, A.NHWC, code, st)
    elif op == "dx":
        rc = L.kdcc_pw_bwd_dx(dy.data_ptr(), w.data_ptr(), out.data_ptr(), None, 0, M, K, Co, N, A.NHWC, code, st)
    else:
        rc = L.kdcc_pw_bwd_dw(dy.data_ptr(), x.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), M, K, Co, N, A.NHWC, code, st)
    A.check(rc, "%s code %d" % (op, code))


def nchw(t, C):
    """[M][C] row-major -> the same memory as a channels_last (N, C, H, W) tensor"""
    return t.view(N, H, W, C).permute(0, 3, 1, 2)


def cudnn_call(op, x, w, dy, tf32):
    torch.backends.cudnn.allow_tf32 = tf32
    K, Co = x.shape[1], w.shape[0]
    w4 = w.view(Co, K, 1, 1)
    if op == "fwd":
        return F.conv2d(nchw(x, K), w4)
    if op == "dx":
        return torch.nn.grad.conv2d_input((N, K, H, W), w4, nchw(dy, Co))
    return torch.nn.grad.conv2d_weight(nchw(x, K), w4.shape, nchw(dy, Co))


def flat(t):
    """a channels_last (N, C, H, W) result as [M][C], or a (Co, K, 1, 1) weight gradient as [Co][K]"""
    if t.dim() == 4 and t.shape[2] == 1 and t.shape[3] == 1:
        return t.reshape(t.shape[0], t.shape[1])
    return t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the full result as JSON here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    result = {"card": card(), "M": M, "iters": args.iters, "warmup": args.warmup, "shapes": []}
    L = A.lib()
    arms = ["simt", "tf32x3", "cudnn", "cudnn_tf32"]
    totals = {a: 0.0 for a in arms}
    for K, Co, count in SITES:
        g = torch.Generator().manual_seed(K * 7 + Co)
        set_bytes = 4 * (M * K + M * Co + Co * K)
        copies = max(2, min(4, -(-2 * L2_BYTES // set_bytes)))
        xs = [torch.randn(M, K, generator=g) for _ in range(copies)]
        w_h = torch.randn(Co, K, generator=g) / K ** 0.5
        dys = [torch.randn(M, Co, generator=g) for _ in range(copies)]
        X = [t.cuda() for t in xs]
        Wd = w_h.cuda()
        DY = [t.cuda() for t in dys]
        ws = torch.empty(L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, A.F32_TF32X3), dtype=torch.uint8, device="cuda")
        rows = torch.from_numpy(np.sort(np.random.RandomState(1).choice(M, 256, replace=False)))
        ci = torch.from_numpy(np.sort(np.random.RandomState(2).choice(Co, 32, replace=False)))
        ki = torch.from_numpy(np.sort(np.random.RandomState(3).choice(K, 32, replace=False)))
        x64, w64, dy64 = xs[0].double(), w_h.double(), dys[0].double()
        refs = {"fwd": x64[rows] @ w64.T, "dx": dy64[rows] @ w64, "dw": dy64[:, ci].T @ x64[:, ki]}
        for op in ("fwd", "dx", "dw"):
            outs = {"fwd": (M, Co), "dx": (M, K), "dw": (Co, K)}[op]
            buf = torch.empty(outs, device="cuda")

            def run(arm, i):
                x, dy = X[i % copies], DY[i % copies]
                if arm == "simt":
                    kdcc_call(op, A.F32, x, Wd, dy, buf, ws)
                    return buf
                if arm == "tf32x3":
                    kdcc_call(op, A.F32_TF32X3, x, Wd, dy, buf, ws)
                    return buf
                return flat(cudnn_call(op, x, Wd, dy, arm == "cudnn_tf32"))

            errs = {}
            for arm in arms:
                out = run(arm, 0).cpu()
                mine = out[rows] if op != "dw" else out[ci][:, ki]
                errs[arm] = relerr(mine, refs[op])
            for i in range(args.warmup):
                for arm in arms:
                    run(arm, i)
            times = {a: [] for a in arms}
            for i in range(args.iters):
                for arm in arms:   # alternated: clock and power drift hits every arm alike
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    run(arm, i)
                    e1.record()
                    e1.synchronize()
                    times[arm].append(e0.elapsed_time(e1))
            flop = 2.0 * M * K * Co
            entry = {"K": K, "Co": Co, "sites": count, "op": op, "gflop": flop / 1e9}
            for arm in arms:
                t = float(np.median(times[arm]))
                entry[arm] = {"ms_median": t, "ms_min": float(np.min(times[arm])), "tflops": flop / t / 1e9,
                              "max_rel_err_vs_fp64": errs[arm]}
                totals[arm] += count * t
            result["shapes"].append(entry)
            print(json.dumps(entry), flush=True)
        del X, DY, ws
        torch.cuda.empty_cache()
    result["nine_site_step_ms"] = totals
    result["nine_site_tflop"] = sum(3 * 2.0 * M * K * Co * c for K, Co, c in SITES) / 1e12
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"], "nine_site_step_ms": totals}))


if __name__ == "__main__":
    main()
