"""One-pass objective of the ensemble loop (trainer/ensemble_trainer.py:73-90): multi-teacher KD + supervised cross entropy
and ONE gradient of their sum (kdcc_ensemble_loss, kdcc.EnsembleDistillationLoss, EnsembleStep(objective=...)).

CPU: argument validation of the C ABI, the module interface, and the float64 reference (ce_reference + oracle
kd_loss_multi) against torch's CPU autograd of F.cross_entropy + the reference KD composition.  GPU: the kernel against
that reference, against the separate kdcc calls, the upstream handling of its two outputs, edge cases and the training
step.  Tolerances as test_ce_loss.py: 1e-5 relative in fp32, 2e-2 in bf16, max|a-b| / max|b| per tensor."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import oracle as orc
from oracle import torch_port as tp
from test_ce_loss import ce_reference

TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-2}


@pytest.fixture(scope="module")
def kdcc():
    import __graft_entry__ as entry
    entry.build()
    import kdcc as pkg
    return pkg


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def rel1(a, b):
    a, b = (float(v.detach()) if torch.is_tensor(v) else float(v) for v in (a, b))
    return abs(a - b) / max(abs(b), 1e-30)


def ens_reference(s, teachers, kd_w, y, cw=None, ignore_index=255, mean=True, T=1.0):
    """(kd, ce, d(kd + ce)/ds): oracle.kd_loss_multi for the KD term, ce_reference (float64) for the supervised term."""
    s = torch.as_tensor(s).detach().cpu()
    kd, gkd = orc.kd_loss_multi(s.float().numpy(), [torch.as_tensor(t).detach().float().cpu().numpy() for t in teachers],
                                kd_w, T)
    ce, gce = ce_reference(s.double(), torch.as_tensor(y).cpu(), None if cw is None else torch.as_tensor(cw).cpu(),
                           ignore_index, mean)
    return kd, ce, gkd.astype(np.float64) + gce.numpy()


def _case(seed, shape, K, ignore_frac=0.1, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    C = shape[1]
    x = torch.randn(*shape, generator=g) * scale
    ts = [torch.randn(*shape, generator=g) * scale for _ in range(K)]
    lshape = (shape[0],) + tuple(shape[2:])
    y = torch.randint(0, C, lshape, generator=g)
    y[torch.rand(lshape, generator=g) < ignore_frac] = 255
    cw = torch.rand(C, generator=g) + 0.5
    kd_w = (torch.rand(K, generator=g) + 0.2).tolist()
    total = sum(kd_w)
    return x, ts, y, cw, [w / total for w in kd_w]


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_ensemble_abi_validates_arguments_before_any_cuda_call(kdcc):
    L = kdcc._abi.lib()
    assert "kdcc_ensemble_loss" in kdcc._abi.SIGNATURES and hasattr(L, "kdcc_ensemble_loss")

    def call(K=3, T=1.0, C=19, dtype=0, s=16, teachers=16, out3=16, ws_bytes=1 << 20, ds=None, up2=None, N=1):
        tp_ = (ctypes.c_void_p * max(K, 1))(*([teachers] * max(K, 1)))
        wts = (ctypes.c_float * max(K, 1))(*([1.0] * max(K, 1)))
        return L.kdcc_ensemble_loss(s, tp_, wts, K, T, 16, None, 255, 1, ds, out3, None, 16, ws_bytes,
                                    N, C, 64, C * 64, 64, 1, dtype, 1.0, 1.0, up2, None)

    assert call(K=0) == -1 and call(K=9) == -1                  # K outside [1, 8]
    assert call(T=0.0) == -1 and call(T=-1.0) == -1              # T <= 0
    assert call(dtype=7) == -1                                   # bad dtype
    assert call(N=0) == -1 and call(C=0) == -1
    assert call(s=None) == -1 and call(out3=None) == -1 and call(teachers=None) == -1   # null pointers, N > 0
    assert call(up2=16) == -1                                    # a gradient re-launch without a gradient
    assert call(C=33) == -2 and call(C=33, s=None) == -2         # more classes than the register tile
    assert call(ws_bytes=8) == -3                                # a workspace smaller than kdcc_ce_workspace_bytes says


def test_ensemble_module_interface(kdcc):
    import kdcc.losses as losses
    assert kdcc.EnsembleDistillationLoss is losses.EnsembleDistillationLoss
    mod = kdcc.EnsembleDistillationLoss()
    assert isinstance(mod, nn.Module)
    assert (mod.temperature, mod.weight, mod.class_weight, mod.size_average, mod.ignore_index) == (1, 1, None, True, 255)
    assert mod.expected_upstream == (1.0, 1.0)
    assert "class_weight" in dict(kdcc.EnsembleDistillationLoss(class_weight=torch.ones(19)).named_buffers())
    with pytest.raises(kdcc.KdccError):
        mod(torch.randn(2, 19, 4, 4), [torch.randn(2, 19, 4, 4)], torch.randn(2, 19, 4, 4), torch.zeros(2, 4, 4, dtype=torch.long))


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("T", [1.0, 2.0])
def test_reference_matches_torch_cpu(weighted, mean, T):
    x, ts, y, cw, _ = _case(3, (2, 7, 5, 6), K=3, ignore_frac=0.2)
    wt = cw if weighted else None
    weight = 2.0
    kd_w = [weight / (2 * weight + 1)] * 2 + [1 / (2 * weight + 1)]
    kd, ce, g = ens_reference(x, ts, kd_w, y, wt, 255, mean, T)
    xt = x.double().requires_grad_(True)
    want_kd = tp.ensemble_kd_loss(xt, [t.double() for t in ts[:2]], ts[2].double(), T, weight)
    want_ce = F.cross_entropy(xt, y, weight=None if wt is None else wt.double(), ignore_index=255,
                              reduction="mean" if mean else "sum")
    (want_kd + want_ce).backward()
    assert rel1(kd, want_kd) <= 1e-6 and rel1(ce, want_ce) <= 1e-12
    assert relerr(g, xt.grad.numpy()) <= 1e-6


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _dev(x, dtype, layout):
    t = x.cuda().to(dtype)
    return t.contiguous(memory_format=torch.channels_last) if layout == "nhwc" and t.dim() == 4 else t.contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("T", [1.0, 2.0])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ensemble_seeded_against_reference(kdcc, dtype, layout, T, mean, weighted, K):
    shapes = [(2, 19, 12, 20), (2, 10, 12, 20), (2, 16, 9, 11), (2, 32, 8, 10), (37, 10)]
    for i, shape in enumerate(shapes):
        x, ts, y, cw, kd_w = _case(100 + i + 7 * K + 13 * mean, shape, K)
        s = _dev(x, dtype, layout).requires_grad_(True)
        tdev = [_dev(t, dtype, layout) for t in ts]
        wt = cw.cuda() if weighted else None
        kd, ce = kdcc.functional.ensemble_loss(s, tdev, kd_w, y.cuda(), wt, 255, mean, T)
        (kd + ce).backward()
        rkd, rce, rg = ens_reference(s.detach().float().cpu(), [t.float().cpu() for t in tdev], kd_w, y,
                                     cw if weighted else None, 255, mean, T)
        assert kd.dim() == 0 and kd.dtype == torch.float32 and ce.dim() == 0
        assert rel1(kd, rkd) <= 1e-5, (shape, float(kd), rkd)
        assert rel1(ce, rce) <= 1e-5, (shape, float(ce), rce)
        assert relerr(s.grad.double().cpu().numpy(), rg) < TOL[dtype], shape
        assert s.grad.dtype == dtype and s.grad.stride() == s.stride()


def _big(shape, dtype, K=3, seed=7):
    g = torch.Generator(device="cuda").manual_seed(seed)
    N, C, H, W = shape
    x = (torch.randn(shape, device="cuda", generator=g) * 3).to(dtype)
    ts = [(torch.randn(shape, device="cuda", generator=g) * 3).to(dtype) for _ in range(K)]
    y = torch.randint(0, C, (N, H, W), device="cuda", generator=g)
    y[torch.rand(N, H, W, device="cuda", generator=g) < 0.05] = 255
    return x, ts, y


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 19, 512, 512), (4, 19, 1024, 1024)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ensemble_matches_separate_kdcc_calls(kdcc, shape, dtype):
    x, ts, y = _big(shape, dtype)
    kd_w, T = [0.4, 0.4, 0.2], 1.0
    s = x.detach().requires_grad_(True)
    sep = kdcc.functional.kd_loss_multi(s, ts, kd_w, T)
    ce_sep = kdcc.functional.cross_entropy(s, y)
    (sep + ce_sep).backward()
    gsep = s.grad.clone()
    runs = []
    for _ in range(2):
        s.grad = None
        kd, ce = kdcc.functional.ensemble_loss(s, ts, kd_w, y, temperature=T)
        (kd + ce).backward()
        runs.append((kd.detach().clone(), ce.detach().clone(), s.grad.clone()))
    assert rel1(runs[0][0], sep) <= 1e-5 and rel1(runs[0][1], ce_sep) <= 1e-5
    err = float((runs[0][2].double() - gsep.double()).abs().max()) / float(gsep.double().abs().max())
    assert err < TOL[dtype], err
    assert all(torch.equal(a, b) for a, b in zip(runs[0], runs[1]))   # bit-identical run to run


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ensemble_upstream_handling(kdcc, dtype):
    x, ts, y, cw, kd_w = _case(55, (2, 19, 16, 24), K=3)
    args = ([_dev(t, dtype, "nchw") for t in ts], kd_w, y.cuda(), cw.cuda())
    rkd, rce, _ = ens_reference(x.to(dtype).float(), [t.to(dtype).float() for t in ts], kd_w, y, cw, T=2.0)
    _, g_kd = orc.kd_loss_multi(x.to(dtype).float().numpy(), [t.to(dtype).float().numpy() for t in ts], kd_w, 2.0)
    _, g_ce = ce_reference(x.to(dtype).double(), y, cw)
    g_ce = g_ce.numpy()

    def run(combine, expected=(1.0, 1.0)):
        s = _dev(x, dtype, "nchw").requires_grad_(True)
        kd, ce = kdcc.functional.ensemble_loss(s, *args, temperature=2.0, expected_upstream=expected)
        combine(kd, ce).backward()
        return s.grad.double().cpu().numpy()

    tol = TOL[dtype]
    assert relerr(run(lambda kd, ce: (kd + ce) / 4, (0.25, 0.25)), (g_kd + g_ce) / 4) < tol   # the expected pair
    assert relerr(run(lambda kd, ce: 3 * (kd + ce)), 3 * (g_kd + g_ce)) < tol
    assert relerr(run(lambda kd, ce: kd), g_kd) < tol
    assert relerr(run(lambda kd, ce: ce, (0.5, 2.0)), g_ce) < tol
    assert relerr(run(lambda kd, ce: 2 * kd + 0.5 * ce), 2 * g_kd + 0.5 * g_ce) < tol
    s = _dev(x, dtype, "nchw").requires_grad_(True)
    kd, ce = kdcc.functional.ensemble_loss(s, *args, temperature=2.0)
    assert rel1(kd, rkd) <= 1e-5 and rel1(ce, rce) <= 1e-5
    loss = kd + ce
    loss.backward(retain_graph=True)
    with pytest.raises(kdcc.KdccError):   # the fused gradient buffer is consumed by the first backward
        loss.backward()


@pytest.mark.gpu
def test_ensemble_edge_cases(kdcc):
    x, ts, y, cw, kd_w = _case(77, (2, 19, 16, 16), K=2)
    tdev = [t.cuda() for t in ts]
    _, g_kd = orc.kd_loss_multi(x.numpy(), [t.numpy() for t in ts], kd_w, 1.0)
    # every pixel ignored: CE NaN in mean mode (0 in sum mode), KD finite, gradient = the KD part
    ign = torch.full_like(y, 255).cuda()
    for mean in (True, False):
        s = x.cuda().requires_grad_(True)
        kd, ce = kdcc.functional.ensemble_loss(s, tdev, kd_w, ign, mean=mean)
        (kd + ce).backward()
        assert (math.isnan(float(ce)) if mean else float(ce) == 0.0) and math.isfinite(float(kd))
        assert relerr(s.grad.double().cpu().numpy(), g_kd) < 1e-5
    # labels outside [0, C) that are not ignore_index: dropped and counted
    bad = y.clone()
    bad[0, 0, :5] = torch.tensor([19, 1000, -1, -255, 254])
    clean = bad.clone()
    clean[0, 0, :5] = 255
    cnt = torch.zeros(1, dtype=torch.long, device="cuda")
    for mean in (True, False):
        s = x.cuda().requires_grad_(True)
        kd, ce = kdcc.functional.ensemble_loss(s, tdev, kd_w, bad.cuda(), cw.cuda(), mean=mean, bad_labels=cnt)
        (kd + ce).backward()
        rkd, rce, rg = ens_reference(x, ts, kd_w, clean, cw, 255, mean)
        assert rel1(kd, rkd) <= 1e-5 and rel1(ce, rce) <= 1e-5
        assert relerr(s.grad.double().cpu().numpy(), rg) < 1e-5
    torch.cuda.synchronize()
    assert int(cnt) == 10
    # no gradient wanted: values only, the same as with the gradient
    with torch.no_grad():
        kd0, ce0 = kdcc.functional.ensemble_loss(x.cuda().requires_grad_(True), tdev, kd_w, y.cuda(), cw.cuda())
    assert kd0.grad_fn is None and ce0.grad_fn is None
    kd1, ce1 = kdcc.functional.ensemble_loss(x.cuda(), tdev, kd_w, y.cuda(), cw.cuda())
    s = x.cuda().requires_grad_(True)
    kd2, ce2 = kdcc.functional.ensemble_loss(s, tdev, kd_w, y.cuda(), cw.cuda())
    assert torch.equal(kd0, kd1) and torch.equal(ce0, ce1)
    assert torch.equal(kd0, kd2.detach()) and torch.equal(ce0, ce2.detach())


@pytest.fixture
def deterministic_torch():
    saved = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
             torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32,
     torch.backends.cuda.matmul.allow_tf32) = saved


@pytest.mark.gpu
def test_ensemble_step_with_objective(kdcc, deterministic_torch):
    from test_student_trainer import TinyTeacher, make_student
    torch.manual_seed(5)
    others = [TinyTeacher().cuda().eval() for _ in range(2)]
    data = [torch.randn(2, 3, 24, 32).cuda() for _ in range(2)]
    target = torch.randint(0, 19, (2, 2, 24, 32))
    target[:, :, -3:] = 255
    target = target.cuda()
    runs = {}
    for arm in ("separate", "objective"):
        st = make_student("cuda")
        opt = torch.optim.SGD(st.trainable_parameters(), lr=0.1)
        if arm == "separate":
            step = kdcc.EnsembleStep(st, others, [kdcc.CrossEntropyLoss2d(), kdcc.KLDivergenceLoss(temperature=2)], opt,
                                     accumulation_steps=2, weight=2,
                                     kd_multi=kdcc.MultiTeacherKLDivergenceLoss(temperature=2, weight=2))
        else:
            obj = kdcc.EnsembleDistillationLoss(temperature=2, weight=2)
            step = kdcc.EnsembleStep(st, others, None, opt, accumulation_steps=2, weight=2, objective=obj)
            assert obj.expected_upstream == (0.5, 0.5)
        logs = []
        out = step(data[0], target[0], batch_idx=0)   # (0 + 1) % 2: no optimizer step, the gradients stay in the bucket
        torch.cuda.synchronize()
        grads = step.bucket.dense().clone()
        logs.append({k: out[k].detach().clone() for k in ("loss", "kd_loss", "supervised_loss")})
        out = step(data[1], target[1], batch_idx=1)   # steps
        torch.cuda.synchronize()
        logs.append({k: out[k].detach().clone() for k in ("loss", "kd_loss", "supervised_loss")})
        runs[arm] = (logs, grads, [p.detach().clone() for p in st.trainable_parameters()], set(out))
    (la, ga, pa, ka), (lb, gb, pb, kb) = runs["separate"], runs["objective"]
    assert ka == kb
    for a, b in zip(la, lb):
        for key in a:
            assert rel1(b[key], a[key]) <= 1e-5, (key, float(b[key]), float(a[key]))
    assert relerr(gb.cpu().numpy(), ga.cpu().numpy()) < 1e-5
    for x, y in zip(pa, pb):
        assert float((x - y).abs().max()) <= 1e-5 * max(float(x.abs().max()), 1e-30)
