#!/usr/bin/env python
"""bench.py -- student-KD hot-path throughput (img/s at 1024x1024 crops) on N B200s of one node.

A "step" is one pass of the distillation hot path (SURVEY.md §8) over one synthetic batch: for each of
the replaced sites of cfg/cityscapes/51M_deeplab_all.json the cheap-conv block forward (depthwise 9x9
dil 5 + pointwise GEMM), the hint MSE loss against the teacher feature with its gradient, the block
backward (pointwise dW/dX, depthwise dW/dX), the KD loss on the 19-class logits, the NCCL all-reduce of
the student gradients (N > 1) and the RAdam step.  The frozen DeepLabV3+ trunk that produces the site
inputs is outside the hot path and is not run; inputs have the trunk's shapes.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (libkdcc.so, CUDA)
  python bench.py --impl reference ...                           # the reference's torch-CPU path (oracle port)
  torchrun --nproc-per-node N ... bench.py --gpus N ...          # one rank per GPU
  python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs to DIR/*.npy

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "student KD train img/s @1024^2 crop (cheap-conv hot path)"
PLAN_NAME = "cityscapes/51M_deeplab_all"
# (C_in, C_out) of the nine replaced sites (cfg/cityscapes/51M_deeplab_all.json:123-160), 128x128 maps at a 1024^2 crop
PLAN_51M = [(512, 512)] * 5 + [(1024, 2048)] + [(4096, 256)] * 3


def plan_51m():
    return list(PLAN_51M)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="kdcc", choices=["kdcc", "reference"])
    ap.add_argument("--batch", type=int, default=4, help="images (1024^2 crops) per GPU per step")
    ap.add_argument("--crop", type=int, default=1024)
    ap.add_argument("--dw", default="k9d5p20", help="depthwise geometry kKdDpP (Cityscapes cfgs: k9d5p20; CIFAR: k3d1p1)")
    ap.add_argument("--layout", default="nchw", choices=["nchw", "nhwc", "nhwc_native"],
                    help="activation layout of the block inputs and outputs: nchw = the reference's; nhwc = channels_last I/O, k > 3 re-laid to channel planes at the block boundary (tensor-core depthwise); nhwc_native = NHWC CUDA-core kernels throughout")
    ap.add_argument("--kd-grad", action="store_true", help="also emit d KD / d logits (ClassificationTrainer path)")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip timing the stock-torch CUDA calls of the same path (the bar)")
    ap.add_argument("--no-extras", action="store_true", help="skip the modules-API run and the k3d1p1 sub-runs")
    ap.add_argument("--api-steps", type=int, default=10, help="timed steps of the drop-in modules-API run")
    ap.add_argument("--whole-steps", type=int, default=6, help="timed steps of the whole-step run with the DeepLabV3+ trunk (0 = skip)")
    ap.add_argument("--trunk-format", default="channels_last", choices=["nchw", "channels_last"], help="memory format of the harness trunk")
    ap.add_argument("--grad-exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = gradients pushed into every peer's symmetric buffer by copy engines while the backward runs, "
                         "mean taken inside the fused RAdam pass (kdcc.PeerGradBucket); nccl = one NCCL all-reduce (AVG) after the backward")
    ap.add_argument("--order", default="reference", choices=["reference", "interleaved"],
                    help="reference = forward of every site, hint losses, backward in reverse (the order of model(data) ... loss.backward()); "
                         "interleaved = forward + loss + backward site by site over shared scratch")
    ap.add_argument("--no-timed-events", action="store_true",
                    help="measurement knob: record no CUDA event inside the timed region (the roofline then uses the instrumented pass)")
    ap.add_argument("--torch-optimizer", action="store_true", help="torch.optim.RAdam + a separate weight cast instead of the fused kdcc RAdam step")
    ap.add_argument("--graph", action="store_true",
                    help="replay a CUDA graph of the pass instead of stream launches (measured: 475.8 vs 474.5 img/s, i.e. the "
                         "step is not launch-bound once the CPU runs ahead; stream launches stay the default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (losses, gradients, updated weights, "
                         "input gradient) as DIR/<name>.npy; arrays over %d elements as a fixed seeded sample" % DUMP_MAX_ELEMS)
    return ap.parse_args()


# Per-array cap of --dump-outputs: at most four arrays reach it, so a dump stays under 64 MB of float32.
DUMP_MAX_ELEMS = 3_000_000


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy in float32 (float64 stays float64).  A tensor of more than DUMP_MAX_ELEMS
    elements is flattened and sampled at sorted indices drawn by numpy's default_rng(0), so two runs with the same
    arguments write the same positions."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy() if t.dtype == torch.float64 else t.float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)


def parse_geom(s):
    import re
    m = re.fullmatch(r"k(\d+)d(\d+)p(\d+)", s)
    if not m:
        raise SystemExit("bad --dw %r" % s)
    return tuple(int(v) for v in m.groups())


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons.  Started BEFORE the warm-up (nvidia-smi needs a moment to produce its first
    line); `stop(t0, t1)` keeps the samples whose time stamp falls inside the timed region [t0, t1] (datetime.now())."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t0=None, t1=None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, power, reasons, smax, total = [], [], set(), None, 0
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 8:
                    continue
                total += 1
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f")
                    if t0 is not None and not (t0 <= ts <= t1):
                        continue
                    sm.append(float(f[1])); smax = float(f[2])
                    power.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_min_mhz=sm[0], sm_max_mhz=smax, reasons=sorted(reasons), samples=len(sm),
                       samples_whole_run=total, power_w_max=max(power) if power else None)
        return out


# -------------------------------------------------------------------------------------------------------
# reference / CPU arm: the reference's own calls (torch CPU backend) restated in oracle/torch_port.py
# -------------------------------------------------------------------------------------------------------
# Shared-memory bytes one 128 x 128 plane moves through an SM's 128 B/clk shared-memory / L1 data path in the whole-plane
# tensor-core depthwise kernels (DESIGN.md 4.0/4.1, measured rates: tools/tc_probe2.cu -> profiles/r02_tc_probe2.txt):
#   conv (dw_tc2.cu): 90 SS MMAs x (4 KB image slab + 1 KB Toeplitz chunk) = 450 KB of operand reads, TMA landing 32 KB,
#     regrouping 32 KB read + 40 KB written, epilogue staging 32 KB written + 32 KB read by the TMA store        = 618 KB
#   dW (dw_tc_wgrad3.cu): 130 product MMAs x 1 KB of B + 20 transposing MMAs x 2 KB of B = 170 KB, TMA landing 64 KB,
#     regrouping of x and dy 2 x (32 KB read + 40 KB written)                                                     = 378 KB
#     (dw_tc_wgrad2.cu, which it replaced for this geometry, moved 648 KB and 4.6 kclk of mostly discarded tensor math)
SMEM_BYTES_PER_PLANE = {"conv": 618 * 1024, "wgrad": 378 * 1024}
SMEM_BYTES_PER_CLK = 128


def smem_floor(plan, batch, geom, layout, maps, need_dx, measured_ms, sm_mhz, sms=148):
    """Lower bound of the depthwise backward (dX conv + dW) from the bytes its kernels move through shared memory:
    planes x bytes per plane / (128 B/clk) / 148 SMs at the sampled SM clock.  This -- not HBM, and not tensor-core math
    (90 x 16 clk for the conv) -- is what bounds the k = 9 kernels: tcgen05.mma with both operands in shared memory
    streams them at the same 128 B/clk the rest of the kernel uses (an M=128 N=32 K=16 MMA takes 40 clk = 5 KB / 128).
    Only defined for the geometry the whole-plane kernels cover; returns None otherwise."""
    k, d, p = geom
    if layout != "nchw" or maps > 128 or p % d != 0 or not sm_mhz or not measured_ms or (k, d) != (9, 5):
        return None
    planes_dw = batch * sum(ci for ci, _ in plan)
    planes_dx = batch * sum(ci for (ci, _), nd in zip(plan, need_dx) if nd)
    clk = (planes_dx * SMEM_BYTES_PER_PLANE["conv"] + planes_dw * SMEM_BYTES_PER_PLANE["wgrad"]) / float(SMEM_BYTES_PER_CLK) / sms
    floor_ms = clk / (sm_mhz * 1e3)
    return {"ms": round(floor_ms, 3), "frac": round(floor_ms / measured_ms, 4), "sm_mhz": sm_mhz,
            "model": "(%d dX planes x 618 KB + %d dW planes x 378 KB) / 128 B/clk / %d SMs" % (planes_dx, planes_dw, sms)}


def cpu_reference_image_seconds(plan, maps, geom, budget_s, crop):
    """Seconds the torch-CPU reference path needs for ONE image of the workload, from a bounded sample:
    each distinct site shape is run once (forward, hint MSE, backward) and weighted by its multiplicity,
    plus the KD loss on one image's logits.  If even that exceeds the budget the maps are halved and the
    time scaled by area (both convolutions and losses are linear in the pixel count)."""
    import torch
    from oracle import torch_port as tp
    k, d, p = geom
    torch.set_num_threads(os.cpu_count() or 1)
    shapes = {}
    for s in plan:
        shapes[s] = shapes.get(s, 0) + 1

    def run_site(ci, co, hw):
        x = torch.randn(1, ci, hw, hw)
        site = {"x": x, "w_dw": (torch.rand(ci, 1, k, k) - 0.5).requires_grad_(True),
                "w_pw": (torch.rand(co, ci, 1, 1) - 0.5).requires_grad_(True),
                "teacher": torch.randn(1, co, hw + 2 * p - d * (k - 1), hw + 2 * p - d * (k - 1)), "padding": p, "dilation": d}
        t0 = time.perf_counter()
        y = tp.block_forward(site["x"], site["w_dw"], site["w_pw"], p, d)
        loss = tp.mse_loss(y, site["teacher"], 1000)
        loss.backward()
        return time.perf_counter() - t0

    run_site(16, 16, 16)  # thread-pool / oneDNN warm-up
    scale, hw = 1.0, maps
    probe = run_site(*min(shapes, key=lambda s: s[0] * s[1]), hw)
    flops = lambda s: s[0] * (k * k + s[1])
    projected = probe / flops(min(shapes, key=lambda s: s[0] * s[1])) * sum(flops(s) * 1 for s in shapes)
    while projected > budget_s and hw > 16:
        hw //= 2
        scale *= 4.0
        projected /= 4.0
    total = 0.0
    for (ci, co), count in shapes.items():
        total += count * run_site(ci, co, hw) * scale
    lc = int(crop * (hw / maps))
    s_log, t_log = 3 * torch.randn(1, 19, lc, lc), 3 * torch.randn(1, 19, lc, lc)
    t0 = time.perf_counter()
    with torch.no_grad():
        tp.kl_div_loss(s_log, t_log, 1.0)
    total += (time.perf_counter() - t0) * scale
    sample = ("1 image: each distinct site shape %s once at %dx%d maps%s (fwd + MSE hint + bwd, weighted by multiplicity) "
              "+ KL on (1,19,%d,%d); torch CPU fp32 NCHW" % (sorted(shapes), hw, hw,
                                                           "" if scale == 1.0 else " scaled x%g by area" % scale, lc, lc))
    return total, sample


def gpu_stock_baseline(plan, batch, maps, geom, crop, dev, iters=3):
    """The bar (SURVEY.md 8d, BASELINE.md 3.3): the reference's own calls for this path -- F.conv2d(groups=C)
    (depthwise_separable_conv.py:12), the 1x1 F.conv2d (:13), F.kl_div over log_softmax / softmax (losses/KLDiv.py:20-22),
    nn.MSELoss * num_classes (losses/MSELoss.py:16) and their autograd -- on THIS GPU with stock PyTorch
    (ATen / cuDNN / cuBLAS), in the two forms a user would run them: fp32 NCHW exactly as the reference is written (TF32
    off, its era's default) and bf16 channels_last.  Each distinct site shape is timed once per form (CUDA events, 1
    warm-up + `iters` runs) and weighted by its multiplicity in the plan; plus torch.matmul in bf16 on the plan's GEMM
    shapes.  Returns per-family ms per step, comparable with `kernels[...]["ms_per_step"]`."""
    import torch
    import torch.nn.functional as F
    k, d, p = geom
    shapes = {}
    for s_ in plan:
        shapes[s_] = shapes.get(s_, 0) + 1
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)

    def timed(fn):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / iters

    out = {}
    for form, dtype, fmt in (("fp32_nchw", torch.float32, torch.contiguous_format), ("bf16_channels_last", torch.bfloat16, torch.channels_last)):
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        fam = {"dw_fwd": 0.0, "dw_bwd": 0.0, "pw_fwd": 0.0, "pw_bwd": 0.0, "hint_loss": 0.0}
        for (ci, co), count in shapes.items():
            x = torch.randn(batch, ci, maps, maps, device=dev, dtype=dtype).contiguous(memory_format=fmt).requires_grad_(True)
            w_dw = ((torch.rand(ci, 1, k, k, device=dev) - 0.5).to(dtype)).requires_grad_(True)
            w_pw = ((torch.rand(co, ci, 1, 1, device=dev) - 0.5).to(dtype)).requires_grad_(True)
            teacher = torch.randn(batch, co, maps, maps, device=dev, dtype=dtype).contiguous(memory_format=fmt)
            mid = F.conv2d(x, w_dw, None, 1, p, d, ci)
            g_mid = torch.randn_like(mid)
            fam["dw_fwd"] += count * timed(lambda: F.conv2d(x, w_dw, None, 1, p, d, ci))
            fam["dw_bwd"] += count * timed(lambda: torch.autograd.grad(mid, (x, w_dw), g_mid, retain_graph=True))
            mid_l = mid.detach().requires_grad_(True)
            y = F.conv2d(mid_l, w_pw)
            g_y = torch.randn_like(y)
            fam["pw_fwd"] += count * timed(lambda: F.conv2d(mid_l, w_pw))
            fam["pw_bwd"] += count * timed(lambda: torch.autograd.grad(y, (mid_l, w_pw), g_y, retain_graph=True))
            y_l = y.detach().requires_grad_(True)

            def hint():
                loss = F.mse_loss(y_l, teacher) * 1000
                torch.autograd.grad(loss, y_l)
            fam["hint_loss"] += count * timed(hint)
            del x, w_dw, w_pw, teacher, mid, g_mid, mid_l, y, g_y, y_l
        out[form] = {k_: round(v, 4) for k_, v in fam.items()}
    # KD loss on the logits: fp32 NCHW as written (value only, as the layerwise loop evaluates it under no_grad)
    ls, lt = 3 * torch.randn(batch, 19, crop, crop, device=dev), 3 * torch.randn(batch, 19, crop, crop, device=dev)

    def kl():
        with torch.no_grad():
            return F.kl_div(F.log_softmax(ls / 1.0, dim=1), F.softmax(lt / 1.0, dim=1), reduction="mean") * 19
    out["fp32_nchw"]["kd_loss"] = round(timed(kl), 4)
    del ls, lt
    # cuBLAS bf16 on the plan's GEMMs (forward shape M = pixels, K = C_in, N = C_out)
    mm = []
    M = batch * maps * maps
    for (ci, co), count in shapes.items():
        a = torch.randn(M, ci, device=dev, dtype=torch.bfloat16)
        b = torch.randn(ci, co, device=dev, dtype=torch.bfloat16)
        ms = timed(lambda: torch.matmul(a, b))
        mm.append({"mkn": [M, ci, co], "count": count, "ms": round(ms, 4), "tflops": round(2.0 * M * ci * co / (ms * 1e-3) / 1e12, 1)})
        del a, b
    out["matmul_bf16"] = mm
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.cuda.empty_cache()
    return out


def api_modules_run(plan, batch, maps, geom, crop, dev, world, steps, seed):
    """The same pass through the DROP-IN API a reference user gets (SURVEY.md 8b): kdcc.DepthwiseSeparableBlock modules
    (the class DepthwiseStudent.replace instantiates) + kdcc.MSELoss / kdcc.KLDivergenceLoss + torch autograd +
    kdcc.GradBucket + kdcc.optim.RAdam, i.e. the loop body of trainer/layerwise_trainer.py:223-239 over the nine sites.
    Returns img/s (device-timed, max over ranks) and the launch count of one step."""
    import torch
    import torch.distributed as dist
    import kdcc
    k, d, p = geom
    torch.manual_seed(seed)
    blocks = [kdcc.DepthwiseSeparableBlock(ci, co, k, p, d, ci, None).to(dev) for ci, co in plan]
    params = [prm for b in blocks for prm in b.parameters()]
    opt = kdcc.optim.RAdam(params, lr=5e-3)
    bucket = kdcc.GradBucket(params, peer=world > 1, optimizer=opt)   # N > 1: peer pushes during the backward, mean in the RAdam pass
    hint_crit, kd_crit = kdcc.MSELoss(num_classes=1000), kdcc.KLDivergenceLoss(temperature=1)
    # the first replaced conv's input comes from frozen layers only: no input gradient (SURVEY.md 3.4)
    xs = [torch.randn(batch, ci, maps, maps, device=dev).to(torch.bfloat16).requires_grad_(i > 0) for i, (ci, _) in enumerate(plan)]
    ts = [torch.randn(batch, co, maps, maps, device=dev).to(torch.bfloat16) for _, co in plan]
    ls, lt = 3 * torch.randn(batch, 19, crop, crop, device=dev), 3 * torch.randn(batch, 19, crop, crop, device=dev)

    def one_step():
        hint = 0
        for blk, x, t in zip(blocks, xs, ts):
            hint = hint + hint_crit(blk(x), t)
        with torch.no_grad():
            kd = kd_crit(ls, lt)
        hint.backward()
        for x in xs:
            x.grad = None
        bucket.all_reduce_mean()
        opt.step()
        bucket.zero()
        return hint, kd

    for _ in range(3):
        one_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        hint, kd = one_step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    res = {"value": world * batch * steps / (ms * 1e-3), "unit": "img/s", "ms_per_step": ms / steps, "steps": steps,
           "api": "kdcc.DepthwiseSeparableBlock x%d + kdcc.MSELoss + kdcc.KLDivergenceLoss + autograd + kdcc.GradBucket + kdcc.optim.RAdam" % len(plan),
           "losses": {"hint": float(hint), "kd": float(kd)}}
    del blocks, params, bucket, opt, xs, ts, ls, lt
    torch.cuda.empty_cache()
    return res


def whole_step_run(batch, crop, dev, world, steps, trunk_format, seed):
    """BASELINE.json's metric as named: one layerwise-KD training step at crop x crop with the trunk in the loop --
    frozen DeepLabV3+/WideResNet38 teacher forward, student forward (the frozen trunk with the nine kdcc cheap-conv blocks
    of cfg/cityscapes/51M_deeplab_all.json swapped in by kdcc.prepare_train_epoch), hint MSE over the nine hooked pairs,
    backward (kdcc kernels in the blocks, cuDNN dgrad through the frozen convs between them), gradient all-reduce, fused
    RAdam, plus what the reference loop evaluates for logging every step (supervised CE of both nets, the logits KD term,
    both IoU confusion matrices -- the latter on the device instead of the reference's D2H + numpy, SURVEY.md F13).
    The trunk is harness (stock PyTorch bf16, cuDNN); this is the drop-in API end to end: kdcc.DepthwiseStudent +
    kdcc.LayerwiseStep.  Every step's images and labels are copied from pinned host memory inside the timed region and
    the step's losses are read back, so this is also the end-to-end number."""
    import torch
    import torch.distributed as dist
    import kdcc
    from kdcc.trainer import prepare_train_epoch
    from harness.deeplab_wrn38 import DeepWV3Plus, pruning_section
    torch.backends.cudnn.benchmark = True
    fmt = torch.channels_last if trunk_format == "channels_last" else torch.contiguous_format
    torch.manual_seed(0)                      # the same frozen teacher on every rank
    teacher = DeepWV3Plus(19).to(dev).to(torch.bfloat16).to(memory_format=fmt)
    model = kdcc.DepthwiseStudent(teacher, {"trainer": {"verbosity": 2}})
    del teacher
    opt = prepare_train_epoch(model, pruning_section(), 1, None, lambda ps: kdcc.optim.RAdam(ps, lr=5e-3))
    crit = [torch.nn.CrossEntropyLoss(ignore_index=255), kdcc.KLDivergenceLoss(temperature=1), kdcc.MSELoss(num_classes=1000)]
    step = kdcc.LayerwiseStep(model, crit, opt, accumulation_steps=1)
    cm_s, cm_t = kdcc.ConfusionMatrix(19, 255, device=dev), kdcc.ConfusionMatrix(19, 255, device=dev)
    g = torch.Generator().manual_seed(1000 + seed)
    h_img = torch.randn(batch, 3, crop, crop, generator=g).pin_memory()
    h_lab = torch.randint(0, 19, (batch, crop, crop), generator=g)
    h_lab[torch.rand(batch, crop, crop, generator=g) < 0.05] = 255
    h_lab = h_lab.pin_memory()
    d_img = [torch.empty(batch, 3, crop, crop, device=dev) for _ in range(2)]
    d_lab = [torch.empty(batch, crop, crop, dtype=torch.long, device=dev) for _ in range(2)]
    out_host = torch.empty(4, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    copied, consumed = [torch.cuda.Event(), torch.cuda.Event()], [torch.cuda.Event(), torch.cuda.Event()]
    h2d = h_img.numel() * 4 + h_lab.numel() * 8

    def issue_copy(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i & 1])
            d_img[i & 1].copy_(h_img, non_blocking=True)
            d_lab[i & 1].copy_(h_lab, non_blocking=True)
            copied[i & 1].record(copy_stream)

    def run(n):
        main = torch.cuda.current_stream()
        for c in consumed:
            c.record(main)
        issue_copy(0)
        for i in range(n):
            if i + 1 < n:
                issue_copy(i + 1)
            main.wait_event(copied[i & 1])
            data = d_img[i & 1].to(torch.bfloat16).contiguous(memory_format=fmt)
            out = step(data, d_lab[i & 1], batch_idx=i)
            with torch.no_grad():
                cm_s.update(out["output_st"].float(), d_lab[i & 1])
                cm_t.update(out["output_tc"].float(), d_lab[i & 1])
            consumed[i & 1].record(main)
            out_host.copy_(torch.stack([out["hint_loss"].float(), out["kd_loss"].float(), out["supervised_loss"].float(),
                                        out["teacher_loss"].float()]), non_blocking=True)

    run(3)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(steps)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    res = {"value": world * batch * steps / (ms * 1e-3), "unit": "img/s", "ms_per_step": ms / steps, "steps": steps,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 16, "trunk": "DeepLabV3+ WideResNet38 (harness/deeplab_wrn38.py), bf16 %s, "
           "stock PyTorch / cuDNN; 137.10 M teacher, 85.96 M student, 7.84 M trainable" % trunk_format,
           "api": "kdcc.DepthwiseStudent + kdcc.prepare_train_epoch(cfg 51M_deeplab_all) + kdcc.LayerwiseStep + kdcc.optim.RAdam",
           "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 1),
           "last_losses": {"hint": float(out_host[0]), "kd": float(out_host[1]), "supervised": float(out_host[2]), "teacher": float(out_host[3])}}
    del model, step, opt, d_img, d_lab
    torch.cuda.empty_cache()
    return res


def workload_config(args, world, n_sites, trainable=None):  # noqa: ARG001 (trainable kept for callers; derived below)
    """`config` of the JSON line -- the same dict for both arms (the driver compares them)."""
    maps = args.crop // 8
    cfg = {"workload": "%s hot path: %d cheap-conv sites (dw %s + pw GEMM) fwd+bwd, hint MSE x%d, KD loss on (N,19,%d,%d), "
                       "grad all-reduce, RAdam; frozen trunk not run" % (PLAN_NAME, n_sites, args.dw, n_sites, args.crop, args.crop),
           "global_batch": world * args.batch, "per_gpu_batch": args.batch, "crop": args.crop, "feature_maps": "%dx%d" % (maps, maps),
           "parallelism": "dp%d" % world, "layout": args.layout}
    kk = parse_geom(args.dw)[0] ** 2
    cfg["trainable_params"] = sum(ci * kk + co * ci for ci, co in plan_51m())
    # (both arms print the same dict; these two describe how the CUDA arm launches and why it needs no L2 flush)
    cfg["launch"] = ("CUDA graph of the pass replayed per step; per-kernel times = CUDA events inside the graph, last timed step" if args.graph else
                     "stream launches; the timed region brackets the dominant family with CUDA events (roofline); the other families' "
                     "times come from an instrumented pass of the same number of steps run just before it")
    cfg["cache"] = "inputs larger than L2 (per-step working set of several GB >> 126 MB), no explicit flush"
    return cfg


_CPU_WHOLE = {}


def cpu_whole_step_image_seconds(crop, small=256):
    """Seconds the reference's torch-CPU path needs for one image of a WHOLE layerwise-KD step (teacher forward, student
    forward with the nine replaced blocks, hint MSE, backward, RAdam): run at a `small` x `small` crop and scaled by area
    (BASELINE.md 3.3).  Trunk = harness/deeplab_wrn38.py (bit-identical to the reference class, tests/test_harness_trunk.py),
    blocks and losses = oracle/torch_port.py (the reference's own torch calls)."""
    import torch
    from torch import nn
    import kdcc
    from kdcc.trainer import prepare_train_epoch
    from harness.deeplab_wrn38 import DeepWV3Plus, PRUNING_51M, pruning_section
    from oracle import torch_port as tp
    torch.set_num_threads(os.cpu_count() or 1)
    if "model" not in _CPU_WHOLE:
        class PortBlock(nn.Module):   # depthwise_separable_conv.py:4-14 through the torch port
            def __init__(self, blk):
                super().__init__()
                self.w_dw, self.w_pw = nn.Parameter(blk.separable_conv.weight.detach().clone()), nn.Parameter(blk.pointwise_conv.weight.detach().clone())
                self.p, self.d = blk.separable_conv.padding[0], blk.separable_conv.dilation[0]

            def forward(self, x):
                return tp.block_forward(x, self.w_dw, self.w_pw, self.p, self.d)

        torch.manual_seed(0)
        model = kdcc.DepthwiseStudent(DeepWV3Plus(19), {"trainer": {"verbosity": 2}})
        prepare_train_epoch(model, pruning_section(), 1, None, lambda ps: torch.optim.SGD(ps, lr=0.0))
        for n in PRUNING_51M["names"]:
            model._set_block(n, PortBlock(model.get_block(n, model.student)), model.student)
        model.register_hint_layers(PRUNING_51M["names"])
        _CPU_WHOLE["model"] = model
        _CPU_WHOLE["opt"] = torch.optim.RAdam(model.trainable_parameters(), lr=5e-3)
    model, opt = _CPU_WHOLE["model"], _CPU_WHOLE["opt"]
    x = torch.randn(1, 3, small, small)
    t0 = time.perf_counter()
    out_st, out_tc = model(x)
    hint = sum(tp.mse_loss(a, b, 1000) for a, b in zip(model.student_hidden_outputs, model.teacher_hidden_outputs))
    with torch.no_grad():
        tp.kl_div_loss(out_st, out_tc, 1.0)
    hint.backward()
    opt.step()
    opt.zero_grad()
    sec = time.perf_counter() - t0
    return sec * (crop / float(small)) ** 2, "1 image at %dx%d scaled x%g by area; torch CPU fp32 NCHW, DeepLabV3+ WRN38 teacher + student" % (small, small, (crop / float(small)) ** 2)


def run_reference(args, rank):
    if rank != 0:
        return
    geom = parse_geom(args.dw)
    maps = args.crop // 8
    per_step_budget = max(4.0, 150.0 / max(1, args.steps + args.warmup))
    times, sample = [], ""
    for i in range(args.warmup + args.steps):
        t, sample = cpu_reference_image_seconds(plan_51m(), maps, geom, per_step_budget, args.crop)
        if i >= args.warmup:
            times.append(t)
    sec = sum(times) / len(times)
    cores = os.cpu_count() or 1
    val = 1.0 / sec
    # the whole training step (trunk in the loop) on the CPU, beside our arm's `whole_step`
    whole = None
    if geom == (9, 5, 20) and not args.no_extras:
        try:
            cpu_whole_step_image_seconds(args.crop)                       # builds the model, warms the thread pool
            ws = [cpu_whole_step_image_seconds(args.crop) for _ in range(2)]
            whole = {"value": 1.0 / (sum(w[0] for w in ws) / len(ws)), "unit": "img/s", "cores": cores, "sample": ws[0][1]}
        except Exception as exc:
            whole = {"error": repr(exc)[:200]}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "img/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": args.batch * sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, max(1, args.gpus), len(plan_51m())),
            "note": "reference = its own torch calls on the host CPU (oracle/torch_port.py).  Every image of a batch costs the same, so a "
                    "step times ONE image -- each distinct site shape once, weighted by its multiplicity in the plan -- and the img/s "
                    "is that per-image time extrapolated; ms_per_step is the extrapolated time of a batch of %d" % args.batch,
            "cpu_baseline": {"value": val, "unit": "img/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "whole_step": whole, "gpu_launches": 0}
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------------
# our arm
# -------------------------------------------------------------------------------------------------------
def run_kdcc(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import kdcc
    from kdcc.hotpath import EventLog, HotPathStep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the kdcc path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    kdcc._abi.lib()
    k, d, p = parse_geom(args.dw)
    maps = args.crop // 8
    plan = plan_51m()
    N = args.batch
    logits_shape = (N, 19, args.crop, args.crop)
    # the first replaced conv is fed by frozen layers only, so its input gradient is never needed (SURVEY.md 3.4);
    # every later site's dX continues into the (frozen-weight) student graph towards the earlier trainable blocks
    need_dx = [False] + [True] * (len(plan) - 1)
    hp = HotPathStep(plan, N, maps, maps, k, d, p, dtype=torch.bfloat16, device=dev, logits_shape=logits_shape,
                     kd_temperature=1.0, hint_num_classes=1000.0, accumulation_steps=1, kd_grad=args.kd_grad, need_dx=need_dx,
                     seed=rank, layout=args.layout, order=args.order)
    xs, ts, ls, lt = hp.make_inputs(seed=100 + rank)
    param = torch.nn.Parameter(hp.flat_params)
    param.grad = hp.flat_grads
    # cfg/cityscapes/51M_deeplab_all.json:64-69: the reference's own RAdam (utils/optim/radam.py), here as one fused
    # kdcc kernel that also emits the bf16 weights of the next step's GEMMs (--torch-optimizer: torch.optim.RAdam + cast)
    if args.torch_optimizer:
        opt = torch.optim.RAdam([param], lr=5e-3)
    else:
        opt = kdcc.optim.RAdam([param], lr=5e-3)
        if hp.flat_lp.dtype == torch.bfloat16:
            opt.attach_lp_copy(param, hp.flat_lp)
            hp.refresh_lp()
            hp.lp_maintained = True

    # N > 1: how the student gradients are averaged over the ranks (SURVEY.md 8e)
    peer, exchange = None, "none"
    if world > 1:
        exchange = "nccl all-reduce (AVG) of the flat fp32 bucket after the backward"
        if args.grad_exchange == "peer" and not args.torch_optimizer and not args.graph:
            try:
                peer = kdcc.PeerGradBucket(hp.flat_grads.numel(), dev)
                hp.flat_grads = peer.local()
                param.grad = hp.flat_grads
                opt.attach_grad_sources(param, peer.sources)
                exchange = ("per-site copy-engine pushes into every peer's symmetric buffer during the backward; mean of the %d copies "
                            "taken inside the fused RAdam pass (no collective kernel)" % world)
            except Exception as exc:
                peer = None
                exchange += " [peer exchange unavailable: %s]" % (repr(exc)[:120],)

    # --graph: the 97 libkdcc launches of one pass are captured once into a CUDA graph and replayed; the all-reduce and
    # the optimizer stay ordinary stream work; CUDA events recorded inside the capture give the per-kernel timeline of
    # the last replay.  Default: plain stream launches (the CPU enqueues a step in ~5.5 ms and runs ahead of the GPU).
    use_graph = args.graph
    glog = EventLog(external=True) if use_graph else None
    graph, gout = hp.capture(xs, ts, ls, lt, log=glog) if use_graph else (None, None)

    def one_step(log=None):
        if use_graph:
            graph.replay()
            hint, kd = gout
            if log is not None:
                log.mark("begin")
        else:
            hint, kd = hp.step(xs, ts, ls, lt, log=log, site_done=peer.push if peer is not None else None)
        if peer is not None:
            peer.finish()
            if log is not None:
                log.mark("grad_allreduce")      # here: waiting for the last pushes (own and peers') to land
        elif world > 1:
            dist.all_reduce(hp.flat_grads, op=dist.ReduceOp.AVG)
            if log is not None:
                log.mark("grad_allreduce")
        opt.step()
        if peer is not None:                    # next step writes the other parity of the symmetric buffer
            peer.flip()
            hp.flat_grads = peer.local()
            param.grad = hp.flat_grads
        if log is not None:
            log.mark("optimizer")
        return hint, kd

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    import datetime
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # before the warm-up: nvidia-smi takes a moment to deliver its first line
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    # Instrumented pass (not the timed one): an event after EVERY kernel gives the per-kernel table and says which family
    # dominates.  An event record between two kernels breaks their programmatic-dependent-launch overlap (~4 % of the step),
    # so the timed region below brackets only that dominant family -- whose duration the roofline block needs, measured
    # inside the timed region -- and leaves every other kernel boundary alone.
    full_log = EventLog()
    for _ in range(args.steps):
        one_step(full_log)
    barrier()
    full_durs = full_log.durations_ms()
    alg0 = hp.algorithmic()
    dominant0 = max((n_ for n_ in full_durs if n_ in alg0), key=lambda n_: sum(full_durs[n_]))
    log = EventLog(only={dominant0}) if (dominant0 in ("dw_fwd", "dw_bwd") and not use_graph) else EventLog()
    if args.no_timed_events:
        log = EventLog(only={"none"})
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = datetime.datetime.now()
    torch.cuda.profiler.start()     # ncu --profile-from-start off captures exactly the timed region (tools/gpu_profile_r2.sh)
    e0.record()
    for _ in range(args.steps):
        hint, kd = one_step(log)
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    t_end = datetime.datetime.now()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    elapsed_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * N * args.steps / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # the state the last timed step left, before the e2e and module-API runs below step the weights again
        outs = {"hint_loss": hint, "hint_loss_per_site": hp.hint_losses, "kd_loss": kd, "params": hp.flat_params}
        if world == 1:          # N > 1: the mean gradient exists only inside the fused RAdam pass
            outs["grads"] = hp.flat_grads
        if hp.dx is not None:   # the input gradient of the site whose backward ran last among those that need one
            last = [i for i in (reversed(range(len(plan))) if args.order == "reference" else range(len(plan))) if need_dx[i]][-1]
            dx = hp.dx_cl if hp.relayout else hp.dx
            outs["input_grad_site%d" % last] = dx.reshape(-1)[:N * plan[last][0] * maps * maps]
        if hp.dlogits is not None:
            outs["kd_grad_logits"] = hp.dlogits
        dump_outputs(args.dump_outputs, outs)
    # N > 1: where the step time goes per rank.  A rank's own kernels (everything but the collective) against the time it
    # sits in the all-reduce: under the power cap every GPU runs at its own clock, the collective makes all of them wait
    # for the slowest, so `compute_ms` max - min is the part of the scaling loss no overlap can recover.
    scaling_diag = None
    if world > 1:
        mine = full_durs     # the instrumented pass: every kernel of every step bracketed
        comp = sum(sum(v) for n_, v in mine.items() if n_ != "grad_allreduce") / args.steps
        wait = sum(mine.get("grad_allreduce", [0.0])) / args.steps
        t = torch.tensor([comp, wait], device=dev)
        allv = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allv, t)
        scaling_diag = {"compute_ms_per_rank": [round(float(a[0]), 3) for a in allv],
                        "allreduce_interval_ms_per_rank": [round(float(a[1]), 3) for a in allv],
                        "note": "compute = the rank's own kernels per step (CUDA events); allreduce interval = launch + transfer + waiting "
                                "for the slowest rank.  max(compute) bounds the step from below whatever the collective does"}

    # ---- end to end through the public call: pinned host inputs -> device, step, loss back to the host ----
    e2e = None
    if args.e2e_steps > 0:
        hx, ht, hls, hlt = hp.make_inputs(seed=200 + rank, pinned_host=True)
        h2d = sum(t_.numel() * t_.element_size() for t_ in hx + ht + [hls, hlt])
        out_host = torch.empty(2, dtype=torch.float32).pin_memory()

        # Two device input sets: while step i computes on one, the copy stream lands step i+1's host buffers in
        # the other.  Every step's H2D copy and the D2H of its losses are inside the timed region.
        sets = [(xs, ts, ls, lt), hp.make_inputs(seed=300 + rank)]
        copy_stream = torch.cuda.Stream(device=dev)
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        def issue_copy(i):
            dx, dt, dls, dlt = sets[i & 1]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i & 1])  # the step that last read this set has finished
                for dst, src in zip(dx + dt + [dls, dlt], hx + ht + [hls, hlt]):
                    dst.copy_(src, non_blocking=True)
                copied[i & 1].record(copy_stream)

        def e2e_run(steps):
            main = torch.cuda.current_stream()
            for c in consumed:
                c.record(main)
            issue_copy(0)
            for i in range(steps):
                if i + 1 < steps:
                    issue_copy(i + 1)
                main.wait_event(copied[i & 1])
                dx, dt, dls, dlt = sets[i & 1]
                h_, k_ = hp.step(dx, dt, dls, dlt, site_done=peer.push if peer is not None else None)
                if peer is not None:
                    peer.finish()
                elif world > 1:
                    dist.all_reduce(hp.flat_grads, op=dist.ReduceOp.AVG)
                opt.step()
                if peer is not None:
                    peer.flip()
                    hp.flat_grads = peer.local()
                    param.grad = hp.flat_grads
                consumed[i & 1].record(main)
                out_host.copy_(torch.stack([h_, k_]), non_blocking=True)

        e2e_run(2)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        e2e_run(args.e2e_steps)
        f1.record()
        barrier()
        ems = f0.elapsed_time(f1)
        if world > 1:
            t = torch.tensor([ems], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        e2e = {"value": world * N * args.e2e_steps / (ems * 1e-3), "unit": "img/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 8, "steps": args.e2e_steps,
               "pipeline": "H2D of step i+1 on a copy stream overlaps the kernels of step i (two device input sets)", "last_losses": [float(out_host[0]), float(out_host[1])]}

    # ---- the same pass through the drop-in module API (every rank: it contains the gradient all-reduce) ----
    api = None
    if not args.no_extras and args.api_steps > 0 and args.layout == "nchw":
        xs = ts = ls = lt = None
        if args.e2e_steps > 0:
            del sets, hx, ht, hls, hlt
        torch.cuda.empty_cache()
        api = api_modules_run(plan, N, maps, (k, d, p), args.crop, dev, world, args.api_steps, seed=rank)
        api["vs_hotpath"] = round(api["value"] / value, 4)

    # ---- BASELINE's metric as named: the whole training step with the frozen trunk in the loop (every rank) ----
    whole = None
    if not args.no_extras and args.whole_steps > 0 and (k, d, p) == (9, 5, 20):
        for name in ("mid", "dmid", "dx", "y", "dy", "ws", "mid_s", "y_s", "dy_s", "xp_s", "x_planes", "dx_cl"):
            if hasattr(hp, name):
                delattr(hp, name)
        torch.cuda.empty_cache()
        try:
            whole = whole_step_run(N, args.crop, dev, world, args.whole_steps, args.trunk_format, seed=rank)
            whole["hot_path_share"] = round(ms_per_step / whole["ms_per_step"], 4)
        except Exception as exc:
            if world > 1:
                raise
            whole = {"error": repr(exc)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel roofline from the CUDA events recorded inside the timed region --------------------------
    pk = peaks()
    durs = dict(full_durs)               # every family: the instrumented pass; the dominant one: the timed region itself
    durs.update(log.durations_ms())
    samples = {name: args.steps for name in durs}
    if use_graph:
        for name, lst in glog.durations_ms().items():   # events inside the graph: the last timed step
            durs[name] = lst
            samples[name] = 1
    alg = hp.algorithmic()
    kernels, dominant, dom_ms = {}, None, -1.0
    for name, lst in durs.items():
        per_step_ms = sum(lst) / samples[name]
        entry = {"ms_per_step": round(per_step_ms, 4), "share": round(per_step_ms / ms_per_step, 4), "launches_per_step": len(lst) // samples[name]}
        if name in alg:
            work, unit = alg[name]
            if unit == "B":
                entry.update(bound="hbm", achieved=round(work / (per_step_ms * 1e-3) / 1e9, 1), unit="GB/s",
                             frac=round(work / (per_step_ms * 1e-3) / 1e9 / pk["hbm_gbs"], 4))
            else:
                # the timed region is a fraction of a second at the boost clock: the burst cuBLAS figure is the honest peak
                entry.update(bound="tensor", achieved=round(work / (per_step_ms * 1e-3) / 1e12, 1), unit="TFLOP/s",
                             frac=round(work / (per_step_ms * 1e-3) / 1e12 / pk["bf16_tflops"], 4),
                             frac_of_sustained=round(work / (per_step_ms * 1e-3) / 1e12 / pk["bf16_tflops_sustained"], 4))
            if per_step_ms > dom_ms:
                dominant, dom_ms = name, per_step_ms
        kernels[name] = entry
    # per-site times of every family (instrumented pass, plan order): which site shapes run at which rate
    per_site = {}
    try:
        order_of = list(range(len(plan)))
        for name in ("dw_fwd", "pw_fwd", "hint_loss", "pw_bwd_dw", "pw_bwd_dx", "dw_bwd"):
            lst = full_durs.get(name, [])
            if len(lst) != args.steps * len(plan):
                continue
            backward = name in ("pw_bwd_dw", "pw_bwd_dx", "dw_bwd") and args.order == "reference"   # reverse site order
            ms = [0.0] * len(plan)
            for idx, v in enumerate(lst):
                pos = idx % len(plan)
                ms[len(plan) - 1 - pos if backward else pos] += v / args.steps
            per_site[name] = [round(v, 4) for v in ms]
        per_site["sites"] = ["%d->%d" % s_ for s_ in plan]
        for name, key in (("pw_fwd", "pw_fwd_tflops"), ("pw_bwd_dw", "pw_bwd_dw_tflops"), ("pw_bwd_dx", "pw_bwd_dx_tflops")):
            if name in per_site:
                per_site[key] = [round(2.0 * N * maps * maps * ci * co / (t_ * 1e-3) / 1e12, 1) for (ci, co), t_ in zip(plan, per_site[name])]
    except Exception:
        per_site = None
    dk = kernels[dominant]
    # measured DRAM traffic of the dominant family over one step: ncu dram__bytes_read.sum + dram__bytes_write.sum of
    # every launch of one step of this same default workload (tools/gpu_profile.sh -> profiles/r01_traffic.json)
    traffic = None
    try:
        if (N, args.dw, args.layout, args.crop) == (4, "k9d5p20", "nchw", 1024):
            import glob
            with open(sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))[-1]) as f:
                traffic = json.load(f)["families"][dominant]["dram_bytes_per_step"]
    except Exception:
        traffic = None
    note = ""
    if dominant.startswith("dw") and k >= 7:
        note = ("achieved = algorithmic bytes of all %d launches of one step / their CUDA-event time; traffic = ncu DRAM bytes of the "
                "same launches.  k=9 depthwise is 81 MAC per output element (20 MAC per HBM byte): the kernels run on tcgen05 and are "
                "bound by the 128 B/clk shared-memory data path that feeds the MMAs (618 KB per plane for the conv, 378 KB for dW: "
                "smem_floor; DESIGN.md 4.0/4.1), not by HBM; frac is still reported against the HBM copy peak.  Against the stock "
                "torch CUDA kernels for the same call the family is ~50x faster (gpu_baseline)" % dk["launches_per_step"])
    roofline = {"kernel": dominant, "bound": dk["bound"], "achieved": dk["achieved"],
                "peak": pk["hbm_gbs"] if dk["bound"] == "hbm" else pk["bf16_tflops"], "unit": dk["unit"],
                "frac": dk["frac"], "traffic": traffic, "algorithmic_bytes": alg[dominant][0] if alg[dominant][1] == "B" else None,
                "peak_source": pk["source"] + (" copy bandwidth" if dk["bound"] == "hbm" else " burst cuBLAS bf16"),
                "note": note}
    try:  # the resource that actually binds the dominant family (an annotation: it must never break the line)
        if dominant == "dw_bwd" and k >= 7:
            roofline["smem_floor"] = smem_floor(plan, N, (k, d, p), args.layout, maps, need_dx, dk["ms_per_step"],
                                                (clocks or {}).get("sm_mhz"))
    except Exception:
        pass

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        sec, sample = cpu_reference_image_seconds(plan, maps, (k, d, p), 25.0, args.crop)
        cpu_baseline = {"value": 1.0 / sec, "unit": "img/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": sample}

    # ---- the bar: stock-torch CUDA on the same shapes, and per-site GEMM rates against cuBLAS ----
    gpu_baseline = None
    if not args.no_gpu_baseline and world == 1:
        try:
            torch.cuda.empty_cache()
            gb = gpu_stock_baseline(plan, N, maps, (k, d, p), args.crop, dev)
            ours = {n_: kernels[n_]["ms_per_step"] for n_ in kernels}
            ours["pw_bwd"] = ours.get("pw_bwd_dx", 0) + ours.get("pw_bwd_dw", 0)
            table = {}
            for fam in ("dw_fwd", "dw_bwd", "pw_fwd", "pw_bwd", "hint_loss", "kd_loss"):
                stock = {form: gb[form][fam] for form in ("fp32_nchw", "bf16_channels_last") if fam in gb[form]}
                best = min(stock.values())
                table[fam] = {"kdcc_ms": round(ours[fam], 4), "stock_ms": stock, "speedup_vs_best_stock": round(best / ours[fam], 2)}
            # per-site forward GEMM rate (CUDA events of the timed region, averaged per site) against torch.matmul
            site_ms = {}
            per_call = durs.get("pw_fwd", [])
            for i, site in enumerate(plan):
                vals = per_call[i::len(plan)]
                site_ms.setdefault(site, []).extend(vals)
            for row in gb["matmul_bf16"]:
                site = (row["mkn"][1], row["mkn"][2])
                if site in site_ms and site_ms[site]:
                    ms_ = sum(site_ms[site]) / len(site_ms[site])
                    row["kdcc_pw_fwd_ms"] = round(ms_, 4)
                    row["kdcc_pw_fwd_tflops"] = round(2.0 * row["mkn"][0] * row["mkn"][1] * row["mkn"][2] / (ms_ * 1e-3) / 1e12, 1)
            gpu_baseline = {"note": "cuDNN's bf16 1x1 convolution needs a channels_last input; the kdcc GEMM runs on the reference's own NCHW "
                                    "(and on planes -> channels_last inside a channels_last trunk).  pw_fwd is a tie with cuDNN, box to box 0.99 - 1.17x",
                            "what": "the reference's own torch calls for this path on this GPU (ATen / cuDNN / cuBLAS, TF32 off), ms per step "
                                    "summed over the %d sites: fp32 NCHW as written and bf16 channels_last; pw_bwd = dX + dW; dw_bwd includes dX for every site" % len(plan),
                            "families": table, "matmul_bf16": gb["matmul_bf16"]}
        except Exception as exc:  # an annotation: never break the line
            gpu_baseline = {"error": repr(exc)[:200]}

    kernels_k3 = None
    if not args.no_extras and world == 1 and (k, d, p) != (3, 1, 1):
        try:
            kernels_k3 = {}
            for lay in ("nchw", "nhwc"):
                torch.cuda.empty_cache()
                h3 = HotPathStep(plan, N, maps, maps, 3, 1, 1, dtype=torch.bfloat16, device=dev, logits_shape=None, need_dx=need_dx, seed=7, layout=lay)
                x3, t3, _, _ = h3.make_inputs(seed=11)
                for _ in range(3):
                    h3.step(x3, t3)
                lg = EventLog()
                torch.cuda.synchronize()
                for _ in range(5):
                    h3.step(x3, t3, log=lg)
                torch.cuda.synchronize()
                d3, a3 = lg.durations_ms(), h3.algorithmic()
                kernels_k3[lay] = {n_: {"ms_per_step": round(sum(d3[n_]) / 5, 4), "achieved": round(a3[n_][0] / (sum(d3[n_]) / 5 * 1e-3) / 1e9, 1),
                                        "unit": "GB/s", "frac": round(a3[n_][0] / (sum(d3[n_]) / 5 * 1e-3) / 1e9 / pk["hbm_gbs"], 4)}
                                   for n_ in ("dw_fwd", "dw_bwd")}
                del h3, x3, t3
            kernels_k3["note"] = "the same nine sites with the CIFAR / north-star 3x3 geometry (k3 d1 p1), 5 timed steps per layout"
        except Exception as exc:
            kernels_k3 = {"error": repr(exc)[:200]}

    # ---- BASELINE config 4: the same nine block names in the Gated-SCNN teacher on a 1024 x 2048 input (128 x 256 maps),
    #      KLDiv on the logits + WeightedHintMSE with a per-channel weight vector; per-GPU batch 2 ----
    kernels_gscnn = None
    if not args.no_extras and world == 1 and (k, d, p) == (9, 5, 20) and args.layout == "nchw":
        try:
            torch.cuda.empty_cache()
            hg = HotPathStep(plan, 2, 128, 256, 9, 5, 20, dtype=torch.bfloat16, device=dev, logits_shape=(2, 19, 1024, 2048), need_dx=need_dx,
                             seed=9, layout="nchw", hint_weighted=True)
            xg, tg, lsg, ltg = hg.make_inputs(seed=13)
            for _ in range(3):
                hg.step(xg, tg, lsg, ltg)
            lg = EventLog()
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(5):
                hg.step(xg, tg, lsg, ltg, log=lg)
            g1.record()
            torch.cuda.synchronize()
            dg, ag = lg.durations_ms(), hg.algorithmic()
            kernels_gscnn = {"img_per_s": round(2 * 5 / (g0.elapsed_time(g1) * 1e-3), 1), "ms_per_step": round(g0.elapsed_time(g1) / 5, 3),
                             "note": "cfg/cityscapes/51M_gscnn_all.json shapes: 9 sites on 128x256 maps (1024x2048 input), batch 2, k9 d5 p20, "
                                     "WeightedHintMSELoss with a weight vector, KLDiv on (2,19,1024,2048); the 256-column planes run the whole-plane "
                                     "convolution as two column halves (dw_tc2.cu), the weight gradient on the tiled kernel (dw_tc_wgrad.cu)"}
            for n_ in ("dw_fwd", "dw_bwd", "pw_fwd", "pw_bwd_dx", "pw_bwd_dw", "hint_loss", "kd_loss"):
                ms_ = sum(dg[n_]) / 5
                unit_ = ag[n_][1]
                kernels_gscnn[n_] = {"ms_per_step": round(ms_, 4), "achieved": round(ag[n_][0] / (ms_ * 1e-3) / (1e9 if unit_ == "B" else 1e12), 1),
                                     "unit": "GB/s" if unit_ == "B" else "TFLOP/s"}
            del hg, xg, tg, lsg, ltg
        except Exception as exc:
            kernels_gscnn = {"error": repr(exc)[:200]}

    line = {"metric": METRIC, "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": workload_config(args, world, len(plan), hp.num_trainable),
            "grad_exchange": exchange,
            "clocks": clocks, "e2e": e2e, "gpu_launches": (hp.launches_per_step + (0 if args.torch_optimizer else 1)) * args.steps,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "gpu_baseline": gpu_baseline, "api_modules": api, "whole_step": whole, "scaling_diag": scaling_diag,
            "kernels": kernels, "kernels_per_site": per_site, "kernels_k3": kernels_k3, "kernels_gscnn": kernels_gscnn, "losses": {"hint": float(hint), "kd": float(kd)}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes what the kdcc arm computed; the reference arm times unseeded CPU samples")
        run_reference(args, rank)
    else:
        run_kdcc(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
