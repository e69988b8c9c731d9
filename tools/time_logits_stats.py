"""Times the logged-only work of one layerwise step on BASELINE-size logits (measurement tooling, needs a GPU).

    python tools/time_logits_stats.py [--iters 50] [--reps 5] [--out profiles/r03_logits_stats.json]

Student and teacher logits (4, 19, 1024, 1024) + int64 labels (5 % ignore_index) -- the pair is larger than the 126 MB L2
-- in bf16 NCHW, bf16 channels_last and fp32 NCHW.  Three arms, alternated rep by rep in one process, each timed with CUDA
events over `iters` back-to-back iterations after a warm-up:
  a) as bench.py's whole_step does it today: torch CE(student), torch CE(teacher), kdcc KL value, two .float() copies
     and two kdcc_confusion_update passes;
  b) the same quantities from separate kdcc calls: kdcc_ce_loss x2, kdcc_kd_loss, kdcc_confusion_update x2;
  c) one kdcc_logits_stats pass.
plus, for the ensemble loop, kdcc_ce_loss with its gradient (mean mode: label pre-pass + one pass).
Every arm reports ms (median over reps, with min / max), the algorithmic bytes of the job (one read of both logit tensors
and of the labels; for the gradient arm one read of the logits, one write of the gradient, two reads of the labels) and
TB/s on them, and the traffic its own formulation implies (estimated from shapes).  The GPU name, power limit and max SM
clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kdcc  # noqa: E402
from kdcc import functional as Fk  # noqa: E402

N, C, H, W = 4, 19, 1024, 1024


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else "nvidia-smi unavailable"


def make_inputs(dtype, channels_last):
    g = torch.Generator(device="cuda").manual_seed(0)
    s = torch.randn(N, C, H, W, device="cuda", generator=g).mul_(3).to(dtype)
    t = torch.randn(N, C, H, W, device="cuda", generator=g).mul_(3).to(dtype)
    lab = torch.randint(0, C, (N, H, W), device="cuda", generator=g)
    lab[torch.rand(N, H, W, device="cuda", generator=g) < 0.05] = 255
    if channels_last:
        s, t = s.contiguous(memory_format=torch.channels_last), t.contiguous(memory_format=torch.channels_last)
    return s, t, lab


def arms(s, t, lab):
    torch_ce = torch.nn.CrossEntropyLoss(ignore_index=255)
    kl = kdcc.KLDivergenceLoss(temperature=1)
    cms = [torch.zeros(C * C, dtype=torch.long, device="cuda") for _ in range(2)]
    s_g = s.detach().clone().requires_grad_(True)

    def today():
        with torch.no_grad():
            out = (kl(s, t), torch_ce(s, lab), torch_ce(t, lab))
            Fk.confusion_update(cms[0], s.float(), lab)
            Fk.confusion_update(cms[1], t.float(), lab)
        return out

    def separate():
        with torch.no_grad():
            out = (kl(s, t), Fk.cross_entropy(s, lab), Fk.cross_entropy(t, lab))
            Fk.confusion_update(cms[0], s, lab)
            Fk.confusion_update(cms[1], t, lab)
        return out

    def fused():
        return Fk.logits_stats(s, t, lab, kd_mode=1, temperature=1.0, conf_s=cms[0], conf_t=cms[1])

    def ce_grad():
        return (Fk.cross_entropy(s_g, lab),)

    return {"a_today": today, "b_separate_kdcc": separate, "c_logits_stats": fused, "ce_loss_with_grad": ce_grad}


def traffic(e, channels_last):
    """Bytes each formulation moves (estimated from shapes).  E logits elements per tensor, P pixels."""
    E, P = N * C * H * W, N * H * W
    lab = 8 * P
    conf_copy = 2 * e * E if channels_last else 0        # kdcc_confusion_update reads planes: channels_last is copied first
    f32_copy = (e * E + 4 * E) if e != 4 else 0           # .float() of an fp32 tensor is the tensor itself
    return {
        # CE: log_softmax read + write, NLL gather; .float() copy; confusion on the fp32 copy; KL value: two reads
        "a_today": 2 * (2 * e * E + P * (e + 8)) + 2 * (f32_copy + conf_copy * (e == 4)) + 2 * (4 * E + lab) + 2 * e * E,
        "b_separate_kdcc": 2 * (e * E + lab) + 2 * e * E + 2 * (e * E + lab + conf_copy),
        "c_logits_stats": 2 * e * E + lab,
        "ce_loss_with_grad": 2 * e * E + 2 * lab,
    }


def algorithmic(e):
    E, P = N * C * H * W, N * H * W
    return {"a_today": 2 * e * E + 8 * P, "b_separate_kdcc": 2 * e * E + 8 * P, "c_logits_stats": 2 * e * E + 8 * P,
            "ce_loss_with_grad": 2 * e * E + 16 * P}


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
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_logits_stats.py needs a CUDA device")
    info = {"gpu": gpu_info(), "fields": "name, power.limit, clocks.max.sm", "shape": [N, C, H, W],
            "iters": a.iters, "reps": a.reps, "cases": []}
    print(info["gpu"])
    for dtype, cl in ((torch.bfloat16, False), (torch.bfloat16, True), (torch.float32, False)):
        s, t, lab = make_inputs(dtype, cl)
        fns = arms(s, t, lab)
        vals = {k: [float(v) for v in fn()] for k, fn in fns.items()}   # warm-up + the values each arm logs
        for fn in fns.values():
            fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in fns}
        for _ in range(a.reps):
            for k, fn in fns.items():
                ms[k].append(time_arm(fn, a.iters))
        e = 2 if dtype == torch.bfloat16 else 4
        alg, arm_bytes = algorithmic(e), traffic(e, cl)
        case = {"dtype": str(dtype).replace("torch.", ""), "layout": "channels_last" if cl else "nchw", "arms": {}}
        for k in fns:
            med = statistics.median(ms[k])
            case["arms"][k] = {"ms": round(med, 4), "ms_min": round(min(ms[k]), 4), "ms_max": round(max(ms[k]), 4),
                               "alg_bytes": alg[k], "alg_TBps": round(alg[k] / med / 1e9, 3),
                               "formulation_bytes_est": arm_bytes[k], "values": vals[k]}
            print("%-9s %-13s %-18s %8.4f ms  [%0.4f, %0.4f]  alg %6.1f MB  %5.2f TB/s  (formulation ~%6.1f MB)  %s" % (
                case["dtype"], case["layout"], k, med, min(ms[k]), max(ms[k]), alg[k] / 1e6, alg[k] / med / 1e9,
                arm_bytes[k] / 1e6, ["%.6g" % v for v in vals[k]]))
        info["cases"].append(case)
        del s, t, lab, fns
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
