"""Freeze step-level golden vectors from the REFERENCE's own student wrapper, teachers and losses (build container only).

    python oracle/make_golden_steps.py          # writes tests/golden/{residual,cifar_step}.npz

Unlike oracle/make_golden.py (which loads single reference files by path) this one imports the reference PACKAGE --
`models.students.DepthwiseStudent`, `models.encoders.wider_resnet.IdentityResidualBlock`, `models.cifar_models.resnet`,
`losses.*` -- with the working directory at the reference root and three `sys.modules` stubs for pip packages the image
lacks (`beautifultable`, `torchsummary`, `tensorboardX`; none of them touches arithmetic).  `nn.Module.cuda` is made the
identity so that `DepthwiseStudent.replace` (depthwise_student.py:119 calls `.cuda()`) runs on the CPU.

residual.npz   SURVEY.md F10: a replaced `convs.conv2` inside the reference's IdentityResidualBlock.  The forward hook
               stores the block's output tensor, the residual unit then does `out.add_(shortcut)` on that very tensor
               (models/encoders/wider_resnet.py:180-182), so the hint that MSELoss sees is output + shortcut.  Frozen:
               input, every teacher / student tensor, the hooked tensors as the loss saw them, the hint loss
               (losses/MSELoss.py, num_classes=1000, summed over the pairs as trainer/layerwise_trainer.py:229-231
               does) and its gradients w.r.t. the trainable block weights.
cifar_step.npz BASELINE config 1 (cfg/cifar10/resnet44/config1.json): the real checkpoints/cifar10/resnet44.th teacher,
               the config's own pruning section (8 cheap-conv blocks in layer3.1-4, those four residual blocks
               unfrozen), student in train mode, one step of trainer/classification_trainer.py:24-39 on a seeded
               batch of 32: logits of both nets, KLDivergenceLoss(T=5), the hint MSE it logs, and d kd / d (every
               trainable parameter).
deepwv3plus_forward.npz  models/deeplabv3/deeplabv3.py:DeepWV3Plus(19) in eval mode, loaded with the state dict of the
               harness trunk (harness/deeplab_wrn38.py) built after torch.manual_seed(0), on torch.randn(1, 3, 64, 96) of
               a generator seeded 3: a seeded sample of 4096 output values, their flat indices, and the per-channel sum
               and absolute sum of the whole (1, 19, 64, 96) output.  The stored file was written with the harness class
               in place of the reference's, which tests/test_harness_trunk.py had held torch.equal to it on this input.
"""
import json
import os
import sys
import types
import warnings
from functools import reduce

import numpy as np
import torch
from torch import nn

REF = os.environ.get("KDCC_REFERENCE", "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def _import_reference():
    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m

    stub("beautifultable", BeautifulTable=type("BeautifulTable", (), {}))
    stub("torchsummary", summary=lambda *a, **k: None)
    stub("tensorboardX", SummaryWriter=object)
    os.chdir(REF)
    sys.path.insert(0, REF)
    nn.Module.cuda = lambda self, device=None: self


class _Config(dict):
    """What DepthwiseStudent touches of a ConfigParser: item access (+ get_logger in reset, unused here)."""


def f32(t):
    return t.detach().to(torch.float32).numpy().copy()


def residual_golden():
    from models.students import DepthwiseStudent
    from models.encoders.wider_resnet import IdentityResidualBlock
    from losses import MSELoss

    class Teacher(nn.Module):  # two pre-activation residual units of the reference, a stem and a head
        def __init__(self):
            super().__init__()
            self.stem = nn.Conv2d(3, 16, 3, padding=1, bias=False)
            self.block1 = IdentityResidualBlock(16, [16, 16], dilation=2)     # identity shortcut: x.clone()
            self.block2 = IdentityResidualBlock(16, [32, 32], dilation=1)     # projected shortcut
            self.head = nn.Conv2d(32, 5, 1, bias=False)

        def forward(self, x):
            return self.head(self.block2(self.block1(self.stem(x))))

    torch.manual_seed(61)
    teacher = Teacher()
    with torch.no_grad():   # BN statistics that are not the identity
        for m in teacher.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.3); m.running_var.uniform_(0.5, 1.5); m.weight.uniform_(0.7, 1.3); m.bias.normal_(0, 0.2)
    model = DepthwiseStudent(teacher, _Config(trainer={"verbosity": 2}))
    names = ["block1.convs.conv2", "block2.convs.conv2"]
    geom = {"kernel_size": 3, "padding": 2, "dilation": 2}
    model.replace([{"name": n, "epoch": 1} for n in names], **geom)
    model.register_hint_layers(names)
    model.unfreeze(names)
    x = torch.randn(2, 3, 12, 16)
    out_st, out_tc = model(x)
    crit = MSELoss(num_classes=1000)
    hint = reduce(lambda acc, e: acc + crit(e[0], e[1]), zip(model.student_hidden_outputs, model.teacher_hidden_outputs), 0)
    hint.backward()
    out = {"x": f32(x), "geom": np.array([geom["kernel_size"], geom["padding"], geom["dilation"]], np.int64),
           "hint_loss": np.array(float(hint), np.float64), "out_st": f32(out_st), "out_tc": f32(out_tc)}
    for k, v in model.state_dict().items():
        out["state/" + k] = f32(v) if v.dtype.is_floating_point else v.numpy().copy()
    for i, (s, t) in enumerate(zip(model.student_hidden_outputs, model.teacher_hidden_outputs)):
        out["hidden_st/%d" % i], out["hidden_tc/%d" % i] = f32(s), f32(t)
    for n, p in model.named_parameters():
        if p.requires_grad:
            out["grad/" + n] = f32(p.grad)
    np.savez_compressed(os.path.join(OUT, "residual.npz"), **out)
    print("residual.npz: hint %.6f, %d trainable tensors" % (float(hint), sum(k.startswith("grad/") for k in out)))


def cifar_step_golden():
    from models.students import DepthwiseStudent
    from models.cifar_models.resnet import resnet44
    from losses import KLDivergenceLoss, MSELoss

    cfg = json.load(open(os.path.join(REF, "cfg/cifar10/resnet44/config1.json")))
    teacher = resnet44()
    ck = torch.load(os.path.join(REF, cfg["teacher"]["snapshot"]), map_location="cpu", weights_only=False)
    teacher.load_state_dict({k.replace("module.", "", 1): v for k, v in ck["state_dict"].items()})
    torch.manual_seed(int(cfg.get("seed", 0)))
    model = DepthwiseStudent(teacher, _Config(trainer=cfg["trainer"]))
    pr = cfg["pruning"]
    # trainer/layerwise_trainer.py:prepare_train_epoch(1): replace, hint, unfreeze of the entries with epoch == 1
    model.replace([b for b in pr["pruning_plan"] if b["epoch"] == 1], **pr["args"])
    model.register_hint_layers([b["name"] for b in pr["hint"] if b["epoch"] == 1])
    model.unfreeze([b["name"] for b in pr["unfreeze"] if b["epoch"] == 1])
    model.train()                                               # classification_trainer.py:21
    x = torch.randn(32, 3, 32, 32)
    before = {k: v.clone() for k, v in model.state_dict().items()}   # BN running statistics move in train mode
    out_st, out_tc = model(x)
    kd = KLDivergenceLoss(**cfg["kd_loss"]["args"])(out_st, out_tc)
    with torch.no_grad():
        mse = MSELoss(**cfg["hint_loss"]["args"])
        hint = reduce(lambda acc, e: acc + mse(e[0], e[1]), zip(model.student_hidden_outputs, model.teacher_hidden_outputs), torch.tensor(0))
    kd.backward()                                               # :38-39 loss = kd_loss
    out = {"x": f32(x), "kd_loss": np.array(float(kd), np.float64), "hint_loss": np.array(float(hint), np.float64),
           "out_st": f32(out_st), "out_tc": f32(out_tc), "T": np.array(float(cfg["kd_loss"]["args"]["temperature"])),
           "plan": np.array([b["name"] for b in pr["pruning_plan"]]), "hint": np.array([b["name"] for b in pr["hint"]]),
           "unfreeze": np.array([b["name"] for b in pr["unfreeze"]]),
           "geom": np.array([pr["args"]["kernel_size"], pr["args"]["padding"], pr["args"]["dilation"]], np.int64)}
    for k, v in before.items():
        if k.startswith("teacher.") and not k.endswith("num_batches_tracked"):
            out["teacher/" + k[len("teacher."):]] = f32(v)
        elif k.startswith("student.") and ("separable_conv" in k or "pointwise_conv" in k):
            out["student/" + k[len("student."):]] = f32(v)       # the only student tensors that differ from the teacher's
    for n, p in model.named_parameters():
        if p.requires_grad:
            out["grad/" + n] = f32(p.grad)
    np.savez_compressed(os.path.join(OUT, "cifar_step.npz"), **out)
    print("cifar_step.npz: kd %.6f hint %.6f, %d trainable tensors, %d bytes" %
          (float(kd), float(hint), sum(k.startswith("grad/") for k in out), os.path.getsize(os.path.join(OUT, "cifar_step.npz"))))


def trunk_forward_golden(ref_cls):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    from harness.deeplab_wrn38 import DeepWV3Plus
    torch.manual_seed(0)
    trunk = DeepWV3Plus(19)
    ref = ref_cls(num_classes=19).eval()
    ref.load_state_dict(trunk.state_dict())
    x = torch.randn(1, 3, 64, 96, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        y = f32(ref(x))
    idx = np.sort(np.random.default_rng(3).choice(y.size, 4096, replace=False))
    y64 = y.astype(np.float64)
    out = {"shape": np.array(y.shape, np.int64), "idx": idx.astype(np.int64), "values": y.reshape(-1)[idx],
           "channel_sum": y64.sum(axis=(0, 2, 3)), "channel_abs_sum": np.abs(y64).sum(axis=(0, 2, 3))}
    np.savez_compressed(os.path.join(OUT, "deepwv3plus_forward.npz"), **out)
    print("deepwv3plus_forward.npz: max |y| %.6f, %d bytes" % (np.abs(y).max(), os.path.getsize(os.path.join(OUT, "deepwv3plus_forward.npz"))))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)
    _import_reference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        residual_golden()
        cifar_step_golden()
        from models.deeplabv3.deeplabv3 import DeepWV3Plus as Ref
        trunk_forward_golden(Ref)


if __name__ == "__main__":
    sys.exit(main())
