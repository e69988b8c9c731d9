"""Device cross-entropy (losses/CrossEntropy.py CrossEntropyLoss2d) with its fused gradient, and the one-pass logits
statistics of the layerwise loop (CE of both nets, KD term, both confusion matrices).

CPU: argument validation of the C ABI, the module interface, and the float64 reference below (weighted, sum-mode and
gradient forms of oracle.cross_entropy_2d) against torch's own CPU cross entropy.  GPU: the kernels against that
reference, the golden vectors of tests/golden/ce.npz, the separate kdcc calls, and the training steps that use them.
Tolerances as test_gpu_parity.py: 1e-5 relative in fp32, 2e-2 in bf16, max|a-b| / max|b| per tensor."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from conftest import GOLDEN
from oracle import oracle as orc

TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-2}


@pytest.fixture(scope="module")
def kdcc():
    import __graft_entry__ as entry
    entry.build()
    import kdcc as pkg
    return pkg


def ce_reference(logits, target, weight=None, ignore_index=255, mean=True):
    """float64 restatement of losses/CrossEntropy.py:10-15 (NLLLoss2d(log_softmax(x, 1), weight, size_average,
    ignore_index)) with its gradient.  A pixel counts when its label is in [0, C) and != ignore_index (other labels are
    dropped here; torch refuses them); loss = sum w*nll / (mean ? sum w : 1), NaN for a mean over no pixel;
    grad = w * (softmax - onehot) / (mean ? sum w : 1), 0 at pixels that do not count.  Runs on the tensors' device."""
    x = torch.as_tensor(logits).double()
    t = torch.as_tensor(target).to(x.device).long()
    C = x.shape[1]
    valid = (t >= 0) & (t < C) & (t != ignore_index)
    tc = torch.where(valid, t, torch.zeros_like(t))
    wt = torch.ones(C, dtype=torch.float64, device=x.device) if weight is None else torch.as_tensor(weight).double().to(x.device)
    w = wt[tc] * valid
    lsm = torch.log_softmax(x, 1)
    nll = -lsm.gather(1, tc.unsqueeze(1)).squeeze(1)
    den = w.sum() if mean else torch.tensor(1.0, dtype=torch.float64, device=x.device)
    loss = (w * nll).sum() / den
    g = lsm.exp_()
    g.scatter_add_(1, tc.unsqueeze(1), -torch.ones_like(tc.unsqueeze(1), dtype=torch.float64))
    g = torch.where(valid.unsqueeze(1), g * (w / torch.where(den == 0, 1.0, den)).unsqueeze(1), 0.0)
    return float(loss), g


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def host(t):
    return t.detach().double().cpu().numpy()


def _case(seed, N=2, C=19, H=24, W=40, ignore_frac=0.1, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, C, H, W, generator=g) * scale
    y = torch.randint(0, C, (N, H, W), generator=g)
    y[torch.rand(N, H, W, generator=g) < ignore_frac] = 255
    w = torch.rand(C, generator=g) + 0.5
    return x, y, w


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_ce_abi_validates_arguments_before_any_cuda_call(kdcc):
    L = kdcc._abi.lib()
    assert L.kdcc_ce_workspace_bytes(4, 1 << 20) > 0
    args = lambda N, C, dtype, ptr: (ptr, ptr, None, 255, 1, None, ptr, None, ptr, 1 << 20, N, C, 64, C * 64, 64, 1, dtype, 1.0, None)
    assert L.kdcc_ce_loss(*args(1, 0, 0, 16)) == -1                  # C = 0
    assert L.kdcc_ce_loss(*args(1, 19, 7, 16)) == -1                 # bad dtype
    assert L.kdcc_ce_loss(*args(1, 19, 0, None)) == -1               # null pointers, N > 0
    assert L.kdcc_ce_loss(*args(1, 33, 0, 16)) == -2                 # more classes than the register tile
    assert L.kdcc_ce_loss(*args(1, 33, 1, None)) == -2
    st = lambda N, C, dtype, ptr, mode=1, T=1.0: (ptr, ptr, ptr, None, 255, 1, mode, T, 1.0, ptr, None, None, None, ptr, 1 << 20,
                                                 N, C, 64, C * 64, 64, 1, dtype, None)
    assert L.kdcc_logits_stats(*st(1, 0, 0, 16)) == -1
    assert L.kdcc_logits_stats(*st(1, 19, 7, 16)) == -1
    assert L.kdcc_logits_stats(*st(1, 19, 0, None)) == -1
    assert L.kdcc_logits_stats(*st(1, 19, 0, 16, mode=3)) == -1      # unknown KD mode
    assert L.kdcc_logits_stats(*st(1, 19, 0, 16, T=0.0)) == -1       # KL needs T > 0
    assert L.kdcc_logits_stats(*st(1, 33, 0, 16)) == -2
    # a workspace smaller than kdcc_ce_workspace_bytes says
    small = (16, 16, None, 255, 1, None, 16, None, 16, 8, 1, 19, 64, 19 * 64, 64, 1, 0, 1.0, None)
    assert L.kdcc_ce_loss(*small) == -3


def test_cross_entropy_module_keeps_reference_interface(kdcc):
    import kdcc.losses as losses
    assert kdcc.CrossEntropyLoss2d is losses.CrossEntropyLoss2d
    for kwargs in ({}, {"weight": None, "size_average": True, "ignore_index": 255}, {"weight": torch.ones(19)},
                   {"size_average": False, "ignore_index": 0}):
        mod = losses.CrossEntropyLoss2d(**kwargs)
        assert isinstance(mod, nn.Module) and mod.expected_upstream == 1.0
    assert "weight" in dict(losses.CrossEntropyLoss2d(torch.ones(19)).named_buffers())   # moves with .cuda() as NLLLoss2d's
    with pytest.raises(kdcc.KdccError):
        losses.CrossEntropyLoss2d()(torch.randn(2, 19, 4, 4), torch.zeros(2, 4, 4, dtype=torch.long))
    with pytest.raises(kdcc.KdccError):
        kdcc.functional.logits_stats(torch.randn(2, 19, 4, 4), None, torch.zeros(2, 4, 4, dtype=torch.long))


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("mean", [True, False])
def test_reference_matches_torch_cpu_fp64(weighted, mean):
    x, y, w = _case(11, N=2, C=7, H=5, W=6, ignore_frac=0.2)
    wt = w[:7] if weighted else None
    loss, grad = ce_reference(x, y, wt, 255, mean)
    xt = x.double().requires_grad_(True)
    want = F.cross_entropy(xt, y, weight=None if wt is None else wt.double(), ignore_index=255,
                           reduction="mean" if mean else "sum")
    want.backward()
    want = float(want.detach())
    assert abs(loss - want) <= 1e-12 * abs(want)
    assert float((grad - xt.grad).abs().max()) <= 1e-12
    if not weighted and mean:   # the existing oracle, unchanged
        assert abs(orc.cross_entropy_2d(x.numpy(), y.numpy()) - loss) <= 1e-12 * abs(loss)


def test_reference_all_ignored_and_out_of_range_labels():
    x = torch.randn(1, 3, 2, 2, dtype=torch.float64)
    y = torch.full((1, 2, 2), 255)
    loss, grad = ce_reference(x, y)
    xt = x.clone().requires_grad_(True)
    want = F.cross_entropy(xt, y, ignore_index=255)
    want.backward()
    assert math.isnan(loss) and math.isnan(float(want.detach()))
    assert float(grad.abs().max()) == 0.0 and float(xt.grad.abs().max()) == 0.0
    # labels outside [0, C): dropped, i.e. the same as the labels rewritten to ignore_index (torch on the CPU)
    x, y, w = _case(5, N=1, C=5, H=4, W=4, ignore_frac=0.0)
    y = y % 5
    y[0, 0, :2] = torch.tensor([7, -3])
    clean = y.clone()
    clean[0, 0, :2] = 255
    for mean in (True, False):
        loss, grad = ce_reference(x, y, w[:5], 255, mean)
        want, wgrad = ce_reference(x, clean, w[:5], 255, mean)
        t = F.cross_entropy(x.double(), clean, weight=w[:5].double(), ignore_index=255, reduction="mean" if mean else "sum")
        assert loss == want and torch.equal(grad, wgrad) and abs(loss - float(t)) <= 1e-12 * abs(float(t))


# ---- GPU: kdcc_ce_loss ------------------------------------------------------------------------------------------------
def _dev(x, dtype, layout):
    t = x.cuda().to(dtype)
    return t.contiguous(memory_format=torch.channels_last) if layout == "nhwc" else t.contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_ce_golden(kdcc, layout):
    g = np.load(os.path.join(GOLDEN, "ce.npz"))
    for i in range(3):
        s = _dev(torch.from_numpy(g["c%d/logits" % i]), torch.float32, layout).requires_grad_(True)
        lab = torch.from_numpy(g["c%d/labels" % i]).cuda()
        loss = kdcc.CrossEntropyLoss2d()(s, lab)
        loss.backward()
        want = float(g["c%d/loss" % i])
        assert abs(float(loss) - want) <= 1e-5 * abs(want), (i, float(loss), want)
        _, rg = ce_reference(g["c%d/logits" % i], g["c%d/labels" % i])
        assert relerr(host(s.grad), rg.numpy()) < 1e-5, i


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("mean", [True, False])
@pytest.mark.parametrize("weighted", [False, True])
def test_ce_seeded_against_reference(kdcc, dtype, layout, mean, weighted):
    x, y, w = _case(21 + 2 * mean + weighted, W=40 if mean else 41)   # odd HW: one pixel per thread on planes too
    s = _dev(x, dtype, layout).requires_grad_(True)
    lab = y.cuda()
    wt = w.cuda() if weighted else None
    loss = kdcc.CrossEntropyLoss2d(weight=wt, size_average=mean)(s, lab)
    acc = 4
    (loss / acc).backward()
    rl, rg = ce_reference(s.detach().double().cpu(), y, w if weighted else None, 255, mean)   # the rounded inputs
    assert abs(float(loss) - rl) <= 1e-5 * abs(rl), (float(loss), rl)
    assert relerr(host(s.grad), rg.numpy() / acc) < TOL[dtype]
    assert s.grad.dtype == dtype and s.grad.is_contiguous(memory_format=torch.channels_last if layout == "nhwc" else torch.contiguous_format)
    # an expected upstream that turns out wrong only costs a rescale in backward
    s2 = s.detach().clone().requires_grad_(True)
    crit = kdcc.CrossEntropyLoss2d(weight=wt, size_average=mean)
    crit.expected_upstream = 0.5
    (crit(s2, lab) * 3.0).backward()
    assert relerr(host(s2.grad), rg.numpy() * 3.0) < TOL[dtype]
    with pytest.raises(kdcc.KdccError):   # the fused gradient buffer is consumed by the first backward
        l3 = kdcc.CrossEntropyLoss2d()(s2, lab)
        l3.backward(retain_graph=True)
        l3.backward()


@pytest.mark.gpu
def test_ce_edge_cases(kdcc):
    x, y, w = _case(31, C=19, H=16, W=16)
    s = x.cuda().requires_grad_(True)
    # every pixel ignored: NaN loss, zero gradient (mean); 0 and zero gradient (sum)
    ign = torch.full_like(y, 255).cuda()
    loss = kdcc.functional.cross_entropy(s, ign)
    loss.backward()
    assert math.isnan(float(loss)) and float(s.grad.abs().max()) == 0.0
    s.grad = None
    loss = kdcc.functional.cross_entropy(s, ign, mean=False)
    loss.backward()
    assert float(loss) == 0.0 and float(s.grad.abs().max()) == 0.0
    # labels outside [0, C) that are not ignore_index: dropped and counted, never used as an index
    bad = y.clone()
    bad[0, 0, :5] = torch.tensor([19, 1000, -1, -255, 254])
    clean = bad.clone()
    clean[0, 0, :5] = 255
    cnt = torch.zeros(1, dtype=torch.long, device="cuda")
    for mean in (True, False):
        s.grad = None
        loss = kdcc.functional.cross_entropy(s, bad.cuda(), w.cuda(), mean=mean, bad_labels=cnt)
        loss.backward()
        rl, rg = ce_reference(x, clean, w, 255, mean)
        assert abs(float(loss) - rl) <= 1e-5 * abs(rl)
        assert relerr(host(s.grad), rg.numpy()) < 1e-5
    out3 = kdcc.functional.logits_stats(s, None, bad.cuda(), w.cuda(), bad_labels=cnt)
    torch.cuda.synchronize()
    assert int(cnt) == 15 and abs(float(out3[1]) - ce_reference(x, clean, w)[0]) <= 1e-5 * abs(ce_reference(x, clean, w)[0])
    # bit-identical from run to run, value and gradient
    runs = []
    for _ in range(2):
        t = x.cuda().to(torch.bfloat16).requires_grad_(True)
        l = kdcc.functional.cross_entropy(t, y.cuda(), w.cuda())
        l.backward()
        runs.append((l.detach().clone(), t.grad.clone()))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    # a second call without a gradient gives the same value as the one that wrote it
    with torch.no_grad():
        assert torch.equal(kdcc.functional.cross_entropy(x.cuda().to(torch.bfloat16), y.cuda(), w.cuda()), runs[0][0])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ce_full_size(kdcc, dtype):
    """BASELINE shapes: (4, 19, 1024, 1024) logits, 5 % ignored labels, both layouts, against the float64 reference."""
    g = torch.Generator(device="cuda").manual_seed(7)
    x = (torch.randn(4, 19, 1024, 1024, device="cuda", generator=g) * 3).to(dtype)
    y = torch.randint(0, 19, (4, 1024, 1024), device="cuda", generator=g)
    y[torch.rand(4, 1024, 1024, device="cuda", generator=g) < 0.05] = 255
    rl, rg = ce_reference(x, y)
    gmax = float(rg.abs().max())
    for layout in ("nchw", "nhwc"):
        s = (x.contiguous(memory_format=torch.channels_last) if layout == "nhwc" else x).detach().requires_grad_(True)
        loss = kdcc.CrossEntropyLoss2d()(s, y)
        loss.backward()
        assert abs(float(loss) - rl) <= 1e-5 * abs(rl), (layout, float(loss), rl)
        err = float((s.grad.double() - rg).abs().max()) / gmax
        assert err < TOL[dtype], (layout, err)
        del s, loss


# ---- GPU: kdcc_logits_stats -------------------------------------------------------------------------------------------
def _rel1(a, b):
    a, b = float(a), float(b)
    return abs(a - b) / max(abs(b), 1e-30)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("kd", ["kl1", "kl2", "mse", "none"])
def test_logits_stats_matches_separate_calls(kdcc, dtype, layout, kd):
    x, y, w = _case(41, N=2, C=19, H=64, W=96)
    tx = torch.randn(x.shape, generator=torch.Generator().manual_seed(42)) * 3
    x[:, 4, :8] = x[:, 9, :8] = x.max(1).values[:, :8] + 1    # ties: the first maximum wins
    tx[:, 2, 8:16] = tx[:, 0, 8:16] = tx.max(1).values[:, 8:16] + 1
    s, t, lab = _dev(x, dtype, layout), _dev(tx, dtype, layout), y.cuda()
    wt = w.cuda() if kd in ("kl2", "none") else None
    mode, T, scale = {"kl1": (1, 1.0, 1.0), "kl2": (1, 2.0, 1.0), "mse": (2, 1.0, 19.0), "none": (0, 1.0, 1.0)}[kd]
    cs, ct = (torch.zeros(19 * 19, dtype=torch.long, device="cuda") for _ in range(2))
    kdv, ce_s, ce_t = kdcc.functional.logits_stats(s, t, lab, wt, 255, True, mode, T, scale, conf_s=cs, conf_t=ct)
    rs, rt = (torch.zeros(19 * 19, dtype=torch.long, device="cuda") for _ in range(2))
    kdcc.functional.confusion_update(rs, s.float(), lab)
    kdcc.functional.confusion_update(rt, t.float(), lab)
    assert torch.equal(cs, rs) and torch.equal(ct, rt)
    assert int(cs.sum()) == int(((y >= 0) & (y < 19)).sum())
    assert _rel1(ce_s, kdcc.functional.cross_entropy(s, lab, wt)) <= 1e-6
    assert _rel1(ce_t, kdcc.functional.cross_entropy(t, lab, wt)) <= 1e-6
    if kd.startswith("kl"):
        assert _rel1(kdv, kdcc.KLDivergenceLoss(temperature=T)(s, t)) <= 1e-6
    elif kd == "mse":
        assert _rel1(kdv, kdcc.MSELoss(num_classes=19)(s, t)) <= 1e-6
    else:
        assert kdv is None
    assert kdv is None or kdv.dim() == 0 and kdv.dtype == torch.float32 and kdv.is_cuda
    # validation form: the student only
    cs2 = torch.zeros_like(cs)
    k2, ce_s2, ct2 = kdcc.functional.logits_stats(s, None, lab, wt, conf_s=cs2)
    assert k2 is None and ct2 is None and torch.equal(cs2, rs) and _rel1(ce_s2, ce_s) <= 1e-6


# ---- GPU: the training steps ------------------------------------------------------------------------------------------
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
@pytest.mark.parametrize("kd", ["kl", "mse"])
def test_layerwise_step_fused_statistics(kdcc, deterministic_torch, kd):
    from test_student_trainer import make_student
    torch.manual_seed(3)
    data = torch.randn(2, 3, 24, 32).cuda()
    target = torch.randint(0, 19, (2, 24, 32))
    target[:, :2] = 255
    target = target.cuda()
    kd_crit = (lambda: kdcc.KLDivergenceLoss(temperature=2)) if kd == "kl" else (lambda: kdcc.MSELoss(num_classes=1))
    runs = {}
    for arm in ("torch", "kdcc"):
        st = make_student("cuda")
        ce = nn.CrossEntropyLoss(ignore_index=255) if arm == "torch" else kdcc.CrossEntropyLoss2d()
        crit = [ce, kd_crit(), kdcc.MSELoss(num_classes=1000)]
        opt = torch.optim.SGD(st.trainable_parameters(), lr=0.1)
        cms = (kdcc.ConfusionMatrix(19, 255, device="cuda"), kdcc.CityscapesMetricTracker(device="cuda"))
        if arm == "torch":
            step = kdcc.LayerwiseStep(st, crit, opt, accumulation_steps=2)
            out = step(data, target, batch_idx=0)
            cms[0].update(out["output_st"], target)
            cms[1].update(out["output_tc"], target)
        else:
            step = kdcc.LayerwiseStep(st, crit, opt, accumulation_steps=2, metrics=cms)
            out = step(data, target, batch_idx=0)
        torch.cuda.synchronize()
        runs[arm] = (out, [p.detach().clone() for p in st.trainable_parameters()], cms)
    (a, pa, ca), (b, pb, cb) = runs["torch"], runs["kdcc"]
    assert set(a) == set(b)
    assert torch.equal(a["hint_loss"], b["hint_loss"])
    assert all(torch.equal(x, y) for x, y in zip(pa, pb))
    for key in ("kd_loss", "supervised_loss", "teacher_loss"):
        assert _rel1(b[key], a[key]) <= 1e-5, (key, float(b[key]), float(a[key]))
    assert torch.equal(ca[0].mat, cb[0].mat) and torch.equal(ca[1]._cm.mat, cb[1]._cm.mat)
    assert int(cb[0].mat.sum()) == int((target != 255).sum())


@pytest.mark.gpu
def test_layerwise_step_metrics_with_torch_criterions(kdcc, deterministic_torch):
    """Stock torch criterions: the step runs as before and only adds the metric updates."""
    from test_student_trainer import make_student
    st = make_student("cuda")
    data, target = torch.randn(2, 3, 24, 32).cuda(), torch.randint(0, 19, (2, 24, 32)).cuda()
    cms = (kdcc.ConfusionMatrix(19, 255, device="cuda"), kdcc.ConfusionMatrix(19, 255, device="cuda"))
    crit = [nn.CrossEntropyLoss(ignore_index=255), kdcc.KLDivergenceLoss(2), kdcc.MSELoss(num_classes=1000)]
    out = kdcc.LayerwiseStep(st, crit, torch.optim.SGD(st.trainable_parameters(), lr=0.0), metrics=cms)(data, target, 0)
    ref = kdcc.ConfusionMatrix(19, 255, device="cuda")
    ref.update(out["output_st"], target)
    assert torch.equal(cms[0].mat, ref.mat) and int(cms[1].mat.sum()) == target.numel()
    assert _rel1(out["supervised_loss"], F.cross_entropy(out["output_st"], target)) <= 1e-6


@pytest.mark.gpu
def test_ensemble_step_backpropagates_kdcc_cross_entropy(kdcc, deterministic_torch):
    from test_student_trainer import TinyTeacher, make_student
    torch.manual_seed(5)
    others = [TinyTeacher().cuda().eval() for _ in range(2)]
    data = torch.randn(2, 3, 24, 32).cuda()
    target = torch.randint(0, 19, (2, 24, 32))
    target[:, -3:] = 255
    target = target.cuda()
    grads, losses = {}, {}
    for arm in ("torch", "kdcc"):
        st = make_student("cuda")
        ce = nn.CrossEntropyLoss(ignore_index=255) if arm == "torch" else kdcc.CrossEntropyLoss2d()
        step = kdcc.EnsembleStep(st, others, [ce, kdcc.KLDivergenceLoss(temperature=2)],
                                 torch.optim.SGD(st.trainable_parameters(), lr=0.1), accumulation_steps=2, weight=2)
        if arm == "kdcc":
            assert ce.expected_upstream == 0.5
        out = step(data, target, batch_idx=0)    # (0 + 1) % 2: no optimizer step, the gradients stay in the bucket
        torch.cuda.synchronize()
        grads[arm], losses[arm] = step.bucket.dense().clone(), out["supervised_loss"].detach().clone()
    assert _rel1(losses["kdcc"], losses["torch"]) <= 1e-5
    assert relerr(grads["kdcc"].cpu().numpy(), grads["torch"].cpu().numpy()) < 1e-5
