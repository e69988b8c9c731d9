"""fp32 pointwise convolution as three tf32 tensor-core products (dtype code KDCC_F32_TF32X3; DESIGN.md 4.3g).

`functional.pointwise_conv` selects it for fp32 input when torch's float32 matmul precision is not "highest".  The
tolerance is the project's fp32 one: max|a-b| / max|b| per tensor below 1e-5, against float64 torch on the CPU.  CPU:
the C ABI's validation of the new code, dispatch names, the workspace bound and the selection rule.  GPU: the three
GEMMs at the plan's shapes, ragged tails and small channel counts; a sensitivity check against 1-pass TF32; inf / NaN;
repeatability and CUDA-graph replay; the block and a layerwise step under "high" against "highest"."""
import copy
import ctypes

import numpy as np
import pytest
import torch

import kdcc
from kdcc import functional as F_kdcc

A = kdcc._abi
TOL = 1e-5
X3 = A.F32_TF32X3


@pytest.fixture(autouse=True)
def restore_precision():
    """Every test leaves torch's float32 precision settings as it found them."""
    prec = torch.get_float32_matmul_precision()
    cudnn_tf32, mm_tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    yield
    torch.set_float32_matmul_precision(prec)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = cudnn_tf32, mm_tf32


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_abi_rejects_code2_outside_the_pointwise_entry_points():
    L = A.lib()
    p = ctypes.c_void_p(256)   # never dereferenced: validation returns before any CUDA call
    big = 1 << 30
    NHWC, NCHW = A.NHWC, A.NCHW
    assert L.kdcc_dw_fwd(p, p, None, p, 2, 8, 8, 16, 3, 1, 1, NHWC, X3, None) == -1
    assert L.kdcc_dw_bwd_workspace_bytes(2, 8, 8, 16, 3, 1, 1, NHWC, X3) == 0
    assert L.kdcc_dw_bwd(p, p, p, p, p, None, p, big, 2, 8, 8, 16, 3, 1, 1, NHWC, X3, None) == -1
    lw = L.kdcc_loss_workspace_bytes()
    assert L.kdcc_kd_loss(p, p, p, p, p, lw, 2, 19, 64, 19 * 64, 64, 1, 1.0, 0, X3, 1.0, None) == -1
    teachers = (ctypes.c_void_p * 1)(256)
    weights = (ctypes.c_float * 1)(1.0)
    assert L.kdcc_kd_loss_multi(p, teachers, weights, 1, p, p, p, lw, 2, 19, 64, 19 * 64, 64, 1, 1.0, X3, 1.0, None) == -1
    assert L.kdcc_hint_loss(p, p, None, 0, p, p, p, big, 2, 16, 64, NCHW, 1.0, X3, 1.0, None) == -1
    cw = L.kdcc_ce_workspace_bytes(2, 64)
    assert L.kdcc_ce_loss(p, p, None, 255, 1, p, p, None, p, cw, 2, 19, 64, 19 * 64, 64, 1, X3, 1.0, None) == -1
    out3 = p
    assert L.kdcc_logits_stats(p, p, p, None, 255, 1, 1, 1.0, 1.0, out3, None, None, None, p, cw, 2, 19, 64, 19 * 64, 64, 1,
                               X3, None) == -1
    assert L.kdcc_ensemble_loss(p, teachers, weights, 1, 1.0, p, None, 255, 1, p, out3, None, p, cw, 2, 19, 64, 19 * 64, 64, 1,
                                X3, 1.0, 1.0, None, None) == -1
    assert L.kdcc_scale_inplace(p, p, 64, X3, None) == -1
    assert L.kdcc_scale_inplace(p, p, 0, X3, None) == -1
    assert L.kdcc_scale_inplace_expect(p, p, 2.0, 64, X3, None) == -1
    assert L.kdcc_layout_convert(p, p, 2, 16, 64, 1, X3, None) == -1
    assert L.kdcc_colsum(p, p, p, L.kdcc_colsum_workspace_bytes(64, 16), 64, 16, X3, None) == -1
    assert L.kdcc_confusion_update(p, p, p, 2, 19, 64, 19 * 64, 64, 255, X3, None) == -1
    assert L.kdcc_canny(p, p, p, L.kdcc_canny_workspace_bytes(2, 64, 64), 2, 3, 64, 64, NCHW, X3, 10.0, 100.0, None) == -1
    # the depthwise ops have no tf32x3 kernel
    for op in (0, 1):
        assert A.dispatch_name(op, 2, 8, 8, 16, 16, 3, 1, 1, NHWC, X3) == "unsupported"


def test_abi_pointwise_code2_is_nhwc_only():
    L = A.lib()
    p = ctypes.c_void_p(256)
    ws = L.kdcc_pw_bwd_workspace_bytes(1, 4096, 64, 64, X3)
    for layout in (A.NCHW, A.PLANES_TO_NHWC):
        assert L.kdcc_pw_fwd(p, p, None, None, 0, p, None, 4096, 64, 64, 4, layout, X3, None) == -2
        assert L.kdcc_pw_fwd_residual(p, p, None, None, p, 0, None, p, 4096, 64, 64, 4, layout, X3, None) == -2
        assert L.kdcc_pw_bwd_dx(p, p, p, None, 0, 4096, 64, 64, 4, layout, X3, None) == -2
        assert L.kdcc_pw_bwd_dw(p, p, p, p, ws, 4096, 64, 64, 4, layout, X3, None) == -2
        for op in (2, 3, 4):
            assert A.dispatch_name(op, 4, 32, 32, 64, 64, 1, 1, 0, layout, X3) == "unsupported"
    # an unknown code is still a bad enum, and bad dimensions still come first
    assert L.kdcc_pw_fwd(p, p, None, None, 0, p, None, 4096, 64, 64, 4, A.NHWC, 3, None) == -1
    assert L.kdcc_pw_fwd(p, p, None, None, 0, p, None, 4096, 0, 64, 4, A.NCHW, X3, None) == -1
    # M >= 2^31 is refused as for the other codes
    assert L.kdcc_pw_fwd(p, p, None, None, 0, p, None, 1 << 31, 64, 64, 1, A.NHWC, X3, None) == -2


@pytest.mark.parametrize("K,Co", [(4, 4), (12, 36), (64, 64), (260, 12), (512, 512), (4096, 256), (6, 8), (8, 6), (3, 5), (258, 260)])
def test_dispatch_names(K, Co):
    ok = K % 4 == 0 and Co % 4 == 0
    names = ["pw_tf32x3_fwd", "pw_tf32x3_dx", "pw_tf32x3_dw"] if ok else ["pw_simt"] * 3
    for op, name in zip((2, 3, 4), names):
        assert A.dispatch_name(op, 4, 16, 16, K, Co, 1, 1, 0, A.NHWC, X3) == name
        assert A.dispatch_name(op, 4, 16, 16, K, Co, 1, 1, 0, A.NHWC, A.F32) == "pw_simt"   # code 0 is unchanged


@pytest.mark.parametrize("M,K,Co", [(1, 4, 4), (129, 12, 36), (100003, 260, 4), (65536, 512, 512), (65536, 1024, 2048),
                                    (65536, 4096, 256), (1 << 24, 64, 64), (4000, 6, 8)])
def test_workspace_covers_fp32(M, K, Co):
    L = A.lib()
    f32 = L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, A.F32)
    x3 = L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, X3)
    assert x3 >= f32 > 0
    assert L.kdcc_pw_bwd_workspace_bytes(0, M, K, Co, X3) == 0


def test_selection_follows_torch_precision():
    x32, x16 = torch.zeros(1, 4, 2, 2), torch.zeros(1, 4, 2, 2, dtype=torch.bfloat16)
    for prec, want in (("highest", A.F32), ("high", X3), ("medium", X3)):
        torch.set_float32_matmul_precision(prec)
        assert F_kdcc._pw_code(x32) == want, prec
        assert F_kdcc._pw_code(x16) == A.BF16, prec


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _st():
    return torch.cuda.current_stream().cuda_stream


def pw_fwd(x, w, code, scale=None, shift=None, residual=None, relu=False, act=False):
    """[M][K] x [Co][K] -> (raw, act) through the C ABI"""
    M, K = x.shape
    Co = w.shape[0]
    raw = torch.empty((M, Co), device=x.device)
    y = torch.empty((M, Co), device=x.device) if (act or residual is not None) else None
    ptr = lambda t: t.data_ptr() if t is not None else None
    L = A.lib()
    if residual is not None:
        rc = L.kdcc_pw_fwd_residual(ptr(x), ptr(w), ptr(scale), ptr(shift), ptr(residual), int(relu), ptr(raw), ptr(y),
                                    M, K, Co, 1, A.NHWC, code, _st())
    else:
        rc = L.kdcc_pw_fwd(ptr(x), ptr(w), ptr(scale), ptr(shift), int(relu), ptr(raw), ptr(y), M, K, Co, 1, A.NHWC, code, _st())
    A.check(rc, "kdcc_pw_fwd")
    return raw, y


def pw_dx(dy, w, code):
    M, Co = dy.shape
    K = w.shape[1]
    dx = torch.empty((M, K), device=dy.device)
    A.check(A.lib().kdcc_pw_bwd_dx(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), None, 0, M, K, Co, 1, A.NHWC, code, _st()), "dx")
    return dx


def pw_dw(dy, x, code):
    M, Co = dy.shape
    K = x.shape[1]
    L = A.lib()
    ws = torch.empty(max(16, L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, code)), dtype=torch.uint8, device=dy.device)
    dw = torch.empty((Co, K), device=dy.device)
    A.check(L.kdcc_pw_bwd_dw(dy.data_ptr(), x.data_ptr(), dw.data_ptr(), ws.data_ptr(), ws.numel(), M, K, Co, 1, A.NHWC, code,
                             _st()), "dw")
    return dw


def _rows(M, n=512, seed=0):
    if M <= n:
        return np.arange(M)
    return np.sort(np.random.RandomState(seed).choice(M, n, replace=False))


def _data(M, K, Co, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(Co, K, generator=g) / K ** 0.5
    dy = torch.randn(M, Co, generator=g)
    return x, w, dy


def _check_three(M, K, Co, seed=0):
    """fwd / dX on sampled rows, dW on sampled (out, in) channels, all against float64 on the CPU."""
    x, w, dy = _data(M, K, Co, seed)
    xc, wc, dyc = x.cuda(), w.cuda(), dy.cuda()
    y, _ = pw_fwd(xc, wc, X3)
    dx = pw_dx(dyc, wc, X3)
    dw = pw_dw(dyc, xc, X3)
    torch.cuda.synchronize()
    r = torch.from_numpy(_rows(M))
    x64, w64, dy64 = x.double(), w.double(), dy.double()
    errs = {"fwd": relerr(y.cpu()[r], x64[r] @ w64.T), "dx": relerr(dx.cpu()[r], dy64[r] @ w64)}
    ci = torch.from_numpy(_rows(Co, 64, seed + 1))
    ki = torch.from_numpy(_rows(K, 64, seed + 2))
    errs["dw"] = relerr(dw.cpu()[ci][:, ki], dy64[:, ci].T @ x64[:, ki])
    return errs


PLAN = [(65536, 512, 512), (65536, 1024, 2048), (65536, 4096, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("M,K,Co", PLAN)
def test_plan_shapes_within_fp32_tolerance(M, K, Co):
    errs = _check_three(M, K, Co)
    assert all(e < TOL for e in errs.values()), errs


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 127, 129, 100003])
@pytest.mark.parametrize("K,Co", [(4, 4), (12, 36), (36, 260), (260, 12)])
def test_tails(M, K, Co):
    errs = _check_three(M, K, Co, seed=M)
    assert all(e < TOL for e in errs.values()), errs


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 12, 36, 260])
@pytest.mark.parametrize("Co", [4, 12, 36, 260])
def test_small_channel_counts(K, Co):
    assert A.dispatch_name(2, 1, 1, 1000, K, Co, 1, 1, 0, A.NHWC, X3) == "pw_tf32x3_fwd"
    errs = _check_three(1000, K, Co, seed=K * 1000 + Co)
    assert all(e < TOL for e in errs.values()), errs


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["affine_relu", "shift_only", "residual", "residual_relu"])
def test_fused_epilogue(mode):
    M, K, Co = 4099, 36, 260
    x, w, _ = _data(M, K, Co, 5)
    g = torch.Generator().manual_seed(6)
    scale = torch.rand(Co, generator=g) + 0.5
    shift = torch.randn(Co, generator=g)
    res = torch.randn(M, Co, generator=g)
    s = scale.cuda() if mode == "affine_relu" else None
    b = shift.cuda() if mode in ("affine_relu", "shift_only") else None
    r = res.cuda() if mode.startswith("residual") else None
    relu = mode.endswith("relu")
    raw, y = pw_fwd(x.cuda(), w.cuda(), X3, scale=s, shift=b, residual=r, relu=relu, act=True)
    ref = x.double() @ w.double().T
    assert relerr(raw.cpu(), ref) < TOL
    if s is not None:
        ref = ref * scale.double()
    if b is not None:
        ref = ref + shift.double()
    if r is not None:
        ref = ref + res.double()
    if relu:
        ref = ref.clamp_min(0)
    assert relerr(y.cpu(), ref) < TOL


@pytest.mark.gpu
def test_one_pass_tf32_misses_the_tolerance_tf32x3_does_not():
    """The check tells the two apart: 1-pass TF32 (torch's own matmul with TF32 on) misses 1e-5 on the same data, and
    the 3-product form is at least 50x closer to float64."""
    M, K, Co = 65536, 512, 512
    x, w, _ = _data(M, K, Co, 11)
    xc, wc = x.cuda(), w.cuda()
    torch.backends.cuda.matmul.allow_tf32 = True
    one = (xc @ wc.T)
    y, _ = pw_fwd(xc, wc, X3)
    torch.cuda.synchronize()
    r = torch.from_numpy(_rows(M, 2048))
    ref = x.double()[r] @ w.double().T
    e1, e3 = relerr(one.cpu()[r], ref), relerr(y.cpu()[r], ref)
    assert e1 > TOL, e1
    assert e3 < TOL and e3 * 50 <= e1, (e3, e1)


@pytest.mark.gpu
def test_inf_nan_positions_match_the_cuda_core_kernel():
    """Every output the fp32 CUDA-core kernel makes non-finite is non-finite here, and only those; every NaN of the
    fp32 kernel is NaN here (an inf of the fp32 kernel may read NaN: the split product adds inf * 0 cross terms)."""
    M, K, Co = 1000, 36, 44
    x, w, dy = _data(M, K, Co, 13)
    x[3, 5], x[10, 0], x[500, 35], x[777, 7] = float("inf"), float("-inf"), float("nan"), 3e38
    w[2, 5], w[9, 9] = float("nan"), float("inf")
    dy[4, 1], dy[999, 43] = float("inf"), float("nan")
    xc, wc, dyc = x.cuda(), w.cuda(), dy.cuda()
    pairs = [(pw_fwd(xc, wc, A.F32)[0], pw_fwd(xc, wc, X3)[0]), (pw_dx(dyc, wc, A.F32), pw_dx(dyc, wc, X3)),
             (pw_dw(dyc, xc, A.F32), pw_dw(dyc, xc, X3))]
    for ref, mine in pairs:
        ref, mine = ref.cpu().numpy(), mine.cpu().numpy()
        assert (~np.isfinite(ref)).any()
        assert np.array_equal(np.isfinite(ref), np.isfinite(mine))
        assert not (np.isnan(ref) & ~np.isnan(mine)).any()


@pytest.mark.gpu
def test_repeatable_and_graph_replay_bit_identical():
    M, K, Co = 65536, 512, 512
    x, w, dy = [t.cuda() for t in _data(M, K, Co, 17)]
    first = [pw_fwd(x, w, X3)[0], pw_dx(dy, w, X3), pw_dw(dy, x, X3)]
    second = [pw_fwd(x, w, X3)[0], pw_dx(dy, w, X3), pw_dw(dy, x, X3)]
    for a, b in zip(first, second):
        assert torch.equal(a, b)
    L = A.lib()
    y, dx, dw = torch.empty(M, Co, device="cuda"), torch.empty(M, K, device="cuda"), torch.empty(Co, K, device="cuda")
    ws = torch.empty(L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, X3), dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            st = s.cuda_stream
            A.check(L.kdcc_pw_fwd(x.data_ptr(), w.data_ptr(), None, None, 0, y.data_ptr(), None, M, K, Co, 1, A.NHWC, X3, st), "fwd")
            A.check(L.kdcc_pw_bwd_dx(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), None, 0, M, K, Co, 1, A.NHWC, X3, st), "dx")
            A.check(L.kdcc_pw_bwd_dw(dy.data_ptr(), x.data_ptr(), dw.data_ptr(), ws.data_ptr(), ws.numel(), M, K, Co, 1, A.NHWC,
                                     X3, st), "dw")
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        y.zero_(); dx.zero_(); dw.zero_()
        graph.replay()
        torch.cuda.synchronize()
        for a, b in zip(first, (y, dx, dw)):
            assert torch.equal(a, b)


# ---- the block and a training step --------------------------------------------------------------------------------
def _block_run(x, w_dw, w_pw, dy, k, d, p, prec, layout, switch_to=None):
    """One fp32 block forward under `prec`, backward under `switch_to` (default: the same); input NCHW or channels_last.
    Returns y and the three gradients as numpy arrays."""
    torch.set_float32_matmul_precision(prec)
    Ci, Co = w_dw.shape[0], w_pw.shape[0]
    blk = kdcc.DepthwiseSeparableBlock(Ci, Co, k, p, d, Ci, None).cuda()
    with torch.no_grad():
        blk.separable_conv.weight.copy_(torch.from_numpy(np.ascontiguousarray(w_dw)))
        blk.pointwise_conv.weight.copy_(torch.from_numpy(np.ascontiguousarray(w_pw)))
    xt = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    if layout == "nhwc":
        xt = xt.contiguous(memory_format=torch.channels_last)
    xt.requires_grad_(True)
    y = blk(xt)
    torch.set_float32_matmul_precision(switch_to or prec)
    dyt = torch.from_numpy(np.ascontiguousarray(dy)).cuda()
    y.backward(dyt.contiguous(memory_format=torch.channels_last) if layout == "nhwc" else dyt)
    torch.cuda.synchronize()
    return [t.detach().cpu().numpy() for t in (y, xt.grad, blk.separable_conv.weight.grad, blk.pointwise_conv.weight.grad)]


def _block_data(N, Ci, Co, H, W, seed):
    rs = np.random.RandomState(seed)
    x = rs.standard_normal((N, Ci, H, W)).astype(np.float32)
    w_dw = (rs.standard_normal((Ci, 1, 3, 3)) / 3).astype(np.float32)
    w_pw = (rs.standard_normal((Co, Ci, 1, 1)) / Ci ** 0.5).astype(np.float32)
    dy = rs.standard_normal((N, Co, H, W)).astype(np.float32)
    return x, w_dw, w_pw, dy


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_block_high_matches_highest(layout):
    x, w_dw, w_pw, dy = _block_data(2, 64, 128, 33, 47, 21)
    assert A.dispatch_name(2, 2, 33, 47, 64, 128, 1, 1, 0, A.NHWC, X3) == "pw_tf32x3_fwd"
    hi = _block_run(x, w_dw, w_pw, dy, 3, 1, 1, "high", layout)
    ref = _block_run(x, w_dw, w_pw, dy, 3, 1, 1, "highest", layout)
    for name, a, b in zip(("y", "dx", "dw_dw", "dw_pw"), hi, ref):
        assert relerr(a, b) < TOL, name
        assert not np.array_equal(a, b) or name == "dw_dw", name   # the products did run differently


@pytest.mark.gpu
def test_block_backward_keeps_the_forward_choice():
    """Switching the precision between forward and backward changes nothing: backward runs what forward chose."""
    x, w_dw, w_pw, dy = _block_data(2, 64, 128, 20, 24, 23)
    mixed = _block_run(x, w_dw, w_pw, dy, 3, 1, 1, "high", "nhwc", switch_to="highest")
    high = _block_run(x, w_dw, w_pw, dy, 3, 1, 1, "high", "nhwc", switch_to="high")
    for a, b in zip(mixed, high):
        assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("tag", ["cifar_k3", "city_k9d5", "ragged_k3d2", "k5", "shrink_k3p0", "onepix_k1"])
def test_block_golden_fp32_under_high(golden_block, tag, layout):
    g = golden_block
    N, Ci, Co, H, W, k, d, p = [int(v) for v in g[f"{tag}/geom"]]
    out = _block_run(g[f"{tag}/x"], g[f"{tag}/w_dw"], g[f"{tag}/w_pw"], g[f"{tag}/dy"], k, d, p, "high", layout)
    for name, mine in zip(("y", "dx", "dw_dw", "dw_pw"), out):
        assert relerr(mine, g[f"{tag}/{name}"]) < TOL, name


@pytest.mark.gpu
def test_layerwise_step_high_matches_highest():
    from harness_models import ResidualTeacher
    torch.backends.cudnn.allow_tf32 = False   # the frozen teacher convolutions stay fp32 in both runs
    torch.manual_seed(0)
    teacher = ResidualTeacher().cuda()
    names = ["block1.convs.conv2", "block2.convs.conv2"]
    data = torch.randn(2, 3, 24, 32, generator=torch.Generator().manual_seed(1)).cuda()
    target = torch.randint(0, 5, (2, 24, 32), generator=torch.Generator().manual_seed(2)).cuda()

    def run(prec):
        torch.set_float32_matmul_precision(prec)
        st = kdcc.DepthwiseStudent(copy.deepcopy(teacher), {"trainer": {"verbosity": 2}})
        torch.manual_seed(3)
        st.replace([{"name": n, "epoch": 1} for n in names], kernel_size=3, padding=1, dilation=1)
        st.register_hint_layers(names)
        st.unfreeze(names)
        crit = [torch.nn.CrossEntropyLoss(ignore_index=255), kdcc.KLDivergenceLoss(temperature=2), kdcc.MSELoss(num_classes=1000)]
        opt = torch.optim.SGD(st.trainable_parameters(), lr=0.0)
        step = kdcc.LayerwiseStep(st, crit, opt, accumulation_steps=2)
        out = step(data, target, batch_idx=1)
        torch.cuda.synchronize()
        losses = {k: float(v.detach()) for k, v in out.items() if k.endswith("loss")}
        grads = {n: p.grad.detach().cpu().numpy().copy() for n, p in st.named_parameters() if p.requires_grad and p.grad is not None}
        return losses, grads

    l_hi, g_hi = run("highest")
    l_x3, g_x3 = run("high")
    assert l_hi.keys() == l_x3.keys() and len(l_hi) >= 2
    for k in l_hi:
        assert abs(l_x3[k] - l_hi[k]) <= TOL * abs(l_hi[k]), (k, l_x3[k], l_hi[k])
    assert g_hi.keys() == g_x3.keys() and len(g_hi) >= 4
    for n in g_hi:
        assert relerr(g_x3[n], g_hi[n]) < TOL, n
