"""Times the objective of the ensemble loop on BASELINE-size logits, forward + backward (measurement tooling, needs a GPU).

    python tools/time_ensemble_loss.py [--iters 20] [--reps 5] [--out profiles/r04_ensemble_loss.json]

Student logits (4, 19, 1024, 1024), K = 3 teachers (two ensemble members and the own teacher) and int64 labels (5 %
ignore_index) -- larger than the 126 MB L2 -- in bf16 NCHW, bf16 channels_last and fp32 NCHW, at T = 1 and T = 2.  Two
arms, alternated rep by rep in one process, each timed with CUDA events over `iters` back-to-back iterations after a
warm-up:
  a) today's composition: kdcc CrossEntropyLoss2d + MultiTeacherKLDivergenceLoss, (kd + ce).backward() on a leaf (two
     passes, two gradients, the autograd add and two scale checks);
  b) kdcc.EnsembleDistillationLoss: one pass, one gradient, one re-launch check in backward.
Every arm reports ms (median over reps, with min / max), the algorithmic bytes of the job (the label pre-pass, one read
of the student, of every teacher and of the labels, one write of the gradient) and TB/s on them, and the traffic its own
formulation implies (estimated from shapes).  The GPU name, power limit and max SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kdcc  # noqa: E402

N, C, H, W, K = 4, 19, 1024, 1024, 3


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else "nvidia-smi unavailable"


def make_inputs(dtype, channels_last):
    g = torch.Generator(device="cuda").manual_seed(0)
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    s = torch.randn(N, C, H, W, device="cuda", generator=g).mul_(3).to(dtype).contiguous(memory_format=fmt)
    ts = [torch.randn(N, C, H, W, device="cuda", generator=g).mul_(3).to(dtype).contiguous(memory_format=fmt) for _ in range(K)]
    lab = torch.randint(0, C, (N, H, W), device="cuda", generator=g)
    lab[torch.rand(N, H, W, device="cuda", generator=g) < 0.05] = 255
    return s.requires_grad_(True), ts, lab


def arms(s, ts, lab, T):
    ce = kdcc.CrossEntropyLoss2d()
    kd_multi = kdcc.MultiTeacherKLDivergenceLoss(temperature=T, weight=1)
    obj = kdcc.EnsembleDistillationLoss(temperature=T, weight=1)

    def today():
        s.grad = None
        kd, sup = kd_multi(s, ts[:-1], ts[-1]), ce(s, lab)
        (kd + sup).backward()
        return kd.detach(), sup.detach()

    def fused():
        s.grad = None
        kd, sup = obj(s, ts[:-1], ts[-1], lab)
        (kd + sup).backward()
        return kd.detach(), sup.detach()

    return {"a_ce_plus_kd_multi": today, "b_ensemble_objective": fused}


def traffic(e):
    """Bytes each formulation moves (estimated from shapes).  E logits elements per tensor, P pixels."""
    E, P = N * C * H * W, N * H * W
    lab = 8 * P
    return {
        # CE: pre-pass + read s + write ds_ce; multi-KD: read s + K teachers + write ds_kd; autograd add: 2 reads + 1 write
        "a_ce_plus_kd_multi": (lab + e * E + lab + e * E) + ((K + 1) * e * E + e * E) + 3 * e * E,
        "b_ensemble_objective": lab + (K + 1) * e * E + lab + e * E,
    }


def algorithmic(e):
    E, P = N * C * H * W, N * H * W
    b = 8 * P + (K + 1) * e * E + 8 * P + e * E
    return {"a_ce_plus_kd_multi": b, "b_ensemble_objective": b}


def time_arm(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
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
        sys.exit("time_ensemble_loss.py needs a CUDA device")
    info = {"gpu": gpu_info(), "fields": "name, power.limit, clocks.max.sm", "shape": [N, C, H, W], "teachers": K,
            "iters": a.iters, "reps": a.reps, "cases": []}
    print(info["gpu"])
    for dtype, cl in ((torch.bfloat16, False), (torch.bfloat16, True), (torch.float32, False)):
        s, ts, lab = make_inputs(dtype, cl)
        for T in (1.0, 2.0):
            fns = arms(s, ts, lab, T)
            vals = {k: [float(v) for v in fn()] for k, fn in fns.items()}   # warm-up + the values each arm computes
            for fn in fns.values():
                fn()
            torch.cuda.synchronize()
            ms = {k: [] for k in fns}
            for _ in range(a.reps):
                for k, fn in fns.items():
                    ms[k].append(time_arm(fn, a.iters))
            e = 2 if dtype == torch.bfloat16 else 4
            alg, arm_bytes = algorithmic(e), traffic(e)
            case = {"dtype": str(dtype).replace("torch.", ""), "layout": "channels_last" if cl else "nchw", "T": T, "arms": {}}
            for k in fns:
                med = statistics.median(ms[k])
                case["arms"][k] = {"ms": round(med, 4), "ms_min": round(min(ms[k]), 4), "ms_max": round(max(ms[k]), 4),
                                   "alg_bytes": alg[k], "alg_TBps": round(alg[k] / med / 1e9, 3),
                                   "formulation_bytes_est": arm_bytes[k], "values": vals[k]}
                print("%-9s %-13s T=%g %-21s %8.4f ms  [%0.4f, %0.4f]  alg %7.1f MB  %5.2f TB/s  (formulation ~%7.1f MB)  %s" % (
                    case["dtype"], case["layout"], T, k, med, min(ms[k]), max(ms[k]), alg[k] / 1e6, alg[k] / med / 1e9,
                    arm_bytes[k] / 1e6, ["%.6g" % v for v in vals[k]]))
            info["cases"].append(case)
        del s, ts, lab
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
