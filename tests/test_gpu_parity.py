"""GPU parity tests: the CUDA path (through the C ABI, libkdcc.so) against the CPU oracle and the
fixtures frozen from the reference modules.  Tolerances are BASELINE.json's: 1e-5 relative in fp32,
2e-2 in bf16, measured as max|a-b| / max|b| per tensor."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-2}
BLOCK_CASES = ["cifar_k3", "city_k9d5", "ragged_k3d2", "k5", "shrink_k3p0", "onepix_k1"]


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def to_dev(a, dtype, grad=False, layout="nhwc"):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda().to(dtype)
    if t.dim() == 4 and layout == "nhwc":
        t = t.contiguous(memory_format=torch.channels_last)
    return t.requires_grad_(grad)


def host(t):
    return t.detach().float().cpu().numpy()


def q(a, dtype):
    """Quantise a float32 array the way the device tensor will be (so the oracle sees the same inputs)."""
    return host(torch.from_numpy(np.ascontiguousarray(a)).to(dtype))


def run_block(kdcc, x, w_dw, w_pw, dy, k, d, p, dtype, layout="nhwc"):
    Ci, Co = w_dw.shape[0], w_pw.shape[0]
    blk = kdcc.DepthwiseSeparableBlock(Ci, Co, k, p, d, Ci, None).cuda()
    with torch.no_grad():
        blk.separable_conv.weight.copy_(torch.from_numpy(w_dw))
        blk.pointwise_conv.weight.copy_(torch.from_numpy(w_pw))
    xt = to_dev(x, dtype, grad=True, layout=layout)
    y = blk(xt)
    if layout == "nchw":  # the tensor-core path keeps the reference's layout end to end
        assert y.is_contiguous() and not (y.dim() == 4 and y.shape[1] > 1 and y.shape[2] * y.shape[3] > 1 and
                                          y.is_contiguous(memory_format=torch.channels_last))
    y.backward(to_dev(dy, dtype, layout=layout))
    torch.cuda.synchronize()
    return host(y), host(xt.grad), host(blk.separable_conv.weight.grad), host(blk.pointwise_conv.weight.grad)


@pytest.fixture(scope="module")
def kdcc():
    import kdcc as pkg
    pkg._abi.lib()  # fails loudly when libkdcc.so is missing
    return pkg


@pytest.mark.parametrize("tag", BLOCK_CASES)
def test_block_fp32_matches_reference_golden(kdcc, golden_block, tag):
    g = golden_block
    N, Ci, Co, H, W, k, d, p = [int(v) for v in g[f"{tag}/geom"]]
    y, dx, dwd, dwp = run_block(kdcc, g[f"{tag}/x"], g[f"{tag}/w_dw"], g[f"{tag}/w_pw"], g[f"{tag}/dy"], k, d, p,
                                torch.float32)
    assert y.shape == g[f"{tag}/y"].shape
    for name, mine in (("y", y), ("dx", dx), ("dw_dw", dwd), ("dw_pw", dwp)):
        assert relerr(mine, g[f"{tag}/{name}"]) < TOL[torch.float32], name


@pytest.mark.parametrize("tag", BLOCK_CASES)
def test_block_bf16_matches_reference_golden(kdcc, golden_block, tag):
    # every golden shape has W % 8 != 0, C % 16 != 0 or k <= 3: the channels_last input stays on the NHWC kernels
    g = golden_block
    N, Ci, Co, H, W, k, d, p = [int(v) for v in g[f"{tag}/geom"]]
    y, dx, dwd, dwp = run_block(kdcc, g[f"{tag}/x"], g[f"{tag}/w_dw"], g[f"{tag}/w_pw"], g[f"{tag}/dy"], k, d, p,
                                torch.bfloat16)
    for name, mine in (("y", y), ("dx", dx), ("dw_dw", dwd), ("dw_pw", dwp)):
        assert relerr(mine, g[f"{tag}/{name}"]) < TOL[torch.bfloat16], name


def oracle_block(x, w_dw, w_pw, dy, k, d, p, dtype):
    """Oracle on inputs quantised like the device tensors; the intermediate is re-quantised too (bf16 path)."""
    from oracle import oracle as orc
    xq, dyq = q(x, dtype), q(dy, dtype)
    wpq = q(w_pw, dtype)
    mid = q(orc.dw_fwd(xq, w_dw, k, d, p), dtype)
    y = orc.pw_fwd(mid, wpq)
    dmid, dwp, _ = orc.pw_bwd(mid, wpq, dyq)
    dx, dwd, _ = orc.dw_bwd(xq, w_dw, q(dmid, dtype), k, d, p)
    return y, dx, dwd, dwp


SEEDED = [
    # N, Ci, Co,  H,  W, k, d,  p      (channels_last; bf16 kernel in brackets, fp32 always runs the direct kernels;
    #                                    k9 widths are not multiples of 8, so the input is not re-laid to planes)
    (2, 64, 128, 40, 44, 9, 5, 20),    # Cityscapes geometry, several 26x26 sub-image tiles         [TMA k9]
    (1, 32, 64, 131, 67, 9, 5, 20),    # ragged: residues with unequal sub-image sizes, partial tiles [TMA k9]
    (2, 32, 64, 33, 47, 3, 1, 1),      # 3x3, ragged edges                                          [streaming 3x3]
    (3, 16, 8, 20, 20, 3, 2, 2),       # dilated 3x3                                                [TMA k3]
    (32, 64, 64, 8, 8, 3, 1, 1),       # CIFAR ResNet44 layer3 block shape                          [streaming 3x3]
    (1, 384, 384, 32, 36, 9, 5, 20),   # HRNet-OCR site channels                                    [TMA k9]
    (2, 24, 32, 30, 37, 9, 5, 20),     # C % 16 == 8                                                [direct]
    (2, 24, 48, 20, 20, 3, 1, 1),      # C % 16 == 8                                                [direct]
    (2, 48, 64, 24, 30, 3, 1, 1),      # six channel vectors: not streamed                          [TMA k3]
]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("geom", SEEDED)
def test_block_matches_oracle_seeded(kdcc, geom, dtype):
    N, Ci, Co, H, W, k, d, p = geom
    rs = np.random.RandomState(1234 + Ci + H)
    x = rs.standard_normal((N, Ci, H, W)).astype(np.float32)
    w_dw = (rs.uniform(-1, 1, (Ci, 1, k, k)) / k).astype(np.float32)
    w_pw = (rs.uniform(-1, 1, (Co, Ci, 1, 1)) / np.sqrt(Ci)).astype(np.float32)
    Ho, Wo = H + 2 * p - d * (k - 1), W + 2 * p - d * (k - 1)
    dy = rs.standard_normal((N, Co, Ho, Wo)).astype(np.float32)
    y, dx, dwd, dwp = run_block(kdcc, x, w_dw, w_pw, dy, k, d, p, dtype)
    ry, rdx, rdwd, rdwp = oracle_block(x, w_dw, w_pw, dy, k, d, p, dtype)
    for name, mine, ref in (("y", y, ry), ("dx", dx, rdx), ("dw_dw", dwd, rdwd), ("dw_pw", dwp, rdwp)):
        assert relerr(mine, ref) < TOL[dtype], name


SEEDED_NHWC3 = [
    # N,  C,   H,   W      (k=3, d=1, p=1, channels_last bf16 -> dw_nhwc3.cu)
    (3, 64, 8, 8),          # CIFAR ResNet44 layer3 shape: 8 vectors per pixel, 4 columns per warp
    (2, 16, 5, 7),          # two vectors per pixel: a warp spans 16 columns, ragged
    (2, 8, 5, 7),           # one vector per pixel: not streamed (falls to the TMA-staged / direct kernels)
    (1, 256, 33, 19),       # exactly one warp of vectors, rows not a multiple of the 32-row tile
    (2, 512, 40, 24),       # two channel groups
    (1, 128, 70, 130),      # 16 vectors per pixel, more than one tile in both directions
]


@pytest.mark.parametrize("geom", SEEDED_NHWC3)
def test_depthwise_nhwc3_streaming_matches_oracle(kdcc, geom):
    from oracle import oracle as orc
    N, C, H, W = geom
    rs = np.random.RandomState(77 + C + W)
    x = q(rs.standard_normal((N, C, H, W)).astype(np.float32), torch.bfloat16)
    w = (rs.uniform(-1, 1, (C, 1, 3, 3)) / 3).astype(np.float32)
    dy = q(rs.standard_normal((N, C, H, W)).astype(np.float32), torch.bfloat16)
    xt = torch.from_numpy(x).cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    wt = torch.from_numpy(w).cuda().requires_grad_(True)
    y = kdcc.functional.depthwise_conv(xt, wt, None, 3, 1, 1)
    y.backward(torch.from_numpy(dy).cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
    ry = orc.dw_fwd(x, w, 3, 1, 1)
    rdx, rdw, _ = orc.dw_bwd(x, w, dy, 3, 1, 1)
    assert relerr(y.detach().float().cpu().numpy(), ry) < TOL[torch.bfloat16]
    assert relerr(xt.grad.float().cpu().numpy(), rdx) < TOL[torch.bfloat16]
    assert relerr(wt.grad.cpu().numpy(), rdw) < 1e-4   # fp32 accumulation of exact bf16 products


SEEDED_NCHW = [
    # N, Ci, Co,   H,   W, k, d,  p      (W % 8 == 0: rows are 16-byte multiples for TMA)
    (2, 64, 128, 40, 40, 9, 5, 20),     # Cityscapes geometry, one partial 128x128 tile per plane
    (1, 16, 32, 136, 200, 9, 5, 20),    # 2 x 2 tiles with real halos between them, ragged edges
    (32, 64, 64, 8, 8, 3, 1, 1),        # CIFAR ResNet44 layer3 block shape (N-tile 32 path)
    (1, 384, 384, 32, 32, 9, 5, 20),    # HRNet-OCR site shape
    (2, 8, 8, 24, 16, 5, 2, 4),         # 5x5 dilated
    (1, 16, 16, 16, 24, 7, 1, 3),       # 7x7
    (2, 8, 16, 20, 24, 5, 2, 0),        # no padding: output (12 x 16) smaller than input
    (1, 512, 512, 128, 128, 9, 5, 20),  # one full-size 51M-plan site
    (3, 24, 8, 37, 40, 9, 5, 20),       # odd batch (weight-gradient image pairs: 2 + 1), ragged rows
    (5, 8, 8, 16, 32, 5, 1, 2),         # undilated 5x5: a single phase exactly 32 columns wide
    (1, 8, 8, 128, 128, 3, 1, 1),       # 3x3 on a full plane: tiled Toeplitz conv + whole-plane weight gradient
    (2, 16, 8, 64, 64, 3, 2, 2),        # dilation 2, two phases of 32 columns
    (1, 16, 8, 128, 256, 9, 5, 20),     # Gated-SCNN site shape (1024 x 2048 input): two 128-column tiles per plane
]


@pytest.mark.parametrize("geom", SEEDED_NCHW)
def test_block_nchw_tensor_core_matches_oracle(kdcc, geom):
    N, Ci, Co, H, W, k, d, p = geom
    dtype = torch.bfloat16
    rs = np.random.RandomState(4321 + Ci + H)
    x = rs.standard_normal((N, Ci, H, W)).astype(np.float32)
    w_dw = (rs.uniform(-1, 1, (Ci, 1, k, k)) / k).astype(np.float32)
    w_pw = (rs.uniform(-1, 1, (Co, Ci, 1, 1)) / np.sqrt(Ci)).astype(np.float32)
    Ho, Wo = H + 2 * p - d * (k - 1), W + 2 * p - d * (k - 1)
    dy = rs.standard_normal((N, Co, Ho, Wo)).astype(np.float32)
    assert kdcc._abi.dispatch_name(0, N, H, W, Ci, Co, k, d, p, kdcc._abi.NCHW, kdcc._abi.BF16) == "dw_tc_conv"
    y, dx, dwd, dwp = run_block(kdcc, x, w_dw, w_pw, dy, k, d, p, dtype, layout="nchw")
    # the tensor-core depthwise multiplies bf16-rounded taps (the Toeplitz operand), so the oracle gets them too
    ry, rdx, rdwd, rdwp = oracle_block(x, q(w_dw, dtype), w_pw, dy, k, d, p, dtype)
    for name, mine, ref in (("y", y, ry), ("dx", dx, rdx), ("dw_dw", dwd, rdwd), ("dw_pw", dwp, rdwp)):
        assert relerr(mine, ref) < TOL[dtype], name


def test_block_nchw_golden_cifar(kdcc, golden_block):
    g, tag = golden_block, "cifar_k3"
    N, Ci, Co, H, W, k, d, p = [int(v) for v in g[f"{tag}/geom"]]
    y, dx, dwd, dwp = run_block(kdcc, g[f"{tag}/x"], g[f"{tag}/w_dw"], g[f"{tag}/w_pw"], g[f"{tag}/dy"], k, d, p,
                                torch.bfloat16, layout="nchw")
    for name, mine in (("y", y), ("dx", dx), ("dw_dw", dwd), ("dw_pw", dwp)):
        assert relerr(mine, g[f"{tag}/{name}"]) < TOL[torch.bfloat16], name


def test_full_size_nchw_impulse_adjoint(kdcc):
    """NCHW tensor-core depthwise at the 51M-plan size: impulse response = mirrored taps; forward, input-gradient
    and weight-gradient kernels satisfy the adjoint identities."""
    torch.manual_seed(5)
    C, H, W, k, d, p = 512, 128, 128, 9, 5, 20
    w = (torch.randn(C, 1, k, k, device="cuda") / k).to(torch.bfloat16).float().requires_grad_(True)
    x = torch.zeros(1, C, H, W, device="cuda", dtype=torch.bfloat16)
    x[0, :, 64, 70] = 1.0
    y = kdcc.functional.depthwise_conv(x, w, None, k, d, p)
    assert y.is_contiguous()
    expect = torch.zeros(1, C, H, W, device="cuda")
    for u in range(k):
        for v in range(k):
            i, j = 64 - u * d + p, 70 - v * d + p
            if 0 <= i < H and 0 <= j < W:
                expect[0, :, i, j] = w.detach()[:, 0, u, v]
    assert torch.equal(y.float(), expect.to(torch.bfloat16).float())
    a = torch.randn(2, C, H, W, device="cuda", dtype=torch.bfloat16).requires_grad_(True)
    g = torch.randn(2, C, H, W, device="cuda", dtype=torch.bfloat16)
    ya = kdcc.functional.depthwise_conv(a, w, None, k, d, p)
    ya.backward(g)
    lhs = (ya.double() * g.double()).sum()
    mid = (a.detach().double() * a.grad.double()).sum()
    rhs = (w.detach().double() * w.grad.double()).sum()
    assert abs(lhs - mid) / abs(lhs) < 1e-2
    assert abs(lhs - rhs) / abs(lhs) < 1e-2


GEMMS = [(4096, 512, 512), (2048, 1024, 2048), (1024, 4096, 256), (2000, 72, 24), (128 * 5 + 8, 64, 64), (300, 384, 384)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mkn", GEMMS)
def test_pointwise_gemm_matches_oracle(kdcc, mkn, dtype):
    from oracle import oracle as orc
    M, K, Nc = mkn
    rs = np.random.RandomState(M + K)
    x = q(rs.standard_normal((1, K, M, 1)).astype(np.float32), dtype)
    w = q((rs.uniform(-1, 1, (Nc, K, 1, 1)) / np.sqrt(K)).astype(np.float32), dtype)
    dy = q(rs.standard_normal((1, Nc, M, 1)).astype(np.float32), dtype)
    xt = to_dev(x, dtype, grad=True)
    wt = torch.from_numpy(w).cuda().requires_grad_(True)
    y = kdcc.functional.pointwise_conv(xt, wt)
    y.backward(to_dev(dy, dtype))
    torch.cuda.synchronize()
    ry = orc.pw_fwd(x, w)
    rdx, rdw, _ = orc.pw_bwd(x, w, dy)
    assert relerr(host(y), ry) < TOL[dtype]
    assert relerr(host(xt.grad), rdx) < TOL[dtype]
    assert relerr(host(wt.grad), rdw) < TOL[dtype]


def test_pointwise_fused_bn_relu_epilogue(kdcc):
    from oracle import oracle as orc
    rs = np.random.RandomState(5)
    M, K, Nc = 1024, 256, 512
    x = q(rs.standard_normal((1, K, M, 1)).astype(np.float32), torch.bfloat16)
    w = q((rs.uniform(-1, 1, (Nc, K, 1, 1)) / np.sqrt(K)).astype(np.float32), torch.bfloat16)
    scale = rs.uniform(0.5, 1.5, Nc).astype(np.float32)
    shift = rs.uniform(-0.5, 0.5, Nc).astype(np.float32)
    with torch.no_grad():
        y = kdcc.functional.pointwise_conv(to_dev(x, torch.bfloat16), torch.from_numpy(w).cuda(), None,
                                           torch.from_numpy(scale).cuda(), torch.from_numpy(shift).cuda(), True)
    ref = np.maximum(orc.pw_fwd(x, w) * scale[None, :, None, None] + shift[None, :, None, None], 0)
    assert relerr(host(y), ref) < TOL[torch.bfloat16]


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pointwise_residual_epilogue(kdcc, layout, dtype):
    """`out = conv(x); out.add_(shortcut)` (wider_resnet.py:181) in one kernel: forward, and the gradients of x, w
    and the shortcut, against the oracle GEMM plus a host add; with BN fold + ReLU on top (inference form)."""
    if dtype == torch.float32 and layout == "nchw":
        pytest.skip("the NCHW pointwise form exists on the bf16 tensor-core path only")
    from oracle import oracle as orc
    rs = np.random.RandomState(11)
    N, K, Nc, H, W = 2, 64, 128, 16, 24
    x = q(rs.standard_normal((N, K, H, W)).astype(np.float32), dtype)
    w = q((rs.uniform(-1, 1, (Nc, K, 1, 1)) / np.sqrt(K)).astype(np.float32), dtype)
    r = q(rs.standard_normal((N, Nc, H, W)).astype(np.float32), dtype)
    dy = q(rs.standard_normal((N, Nc, H, W)).astype(np.float32), dtype)
    fmt = torch.contiguous_format if layout == "nchw" else torch.channels_last
    xt = to_dev(x, dtype).contiguous(memory_format=fmt).requires_grad_(True)
    rt = to_dev(r, dtype).contiguous(memory_format=fmt).requires_grad_(True)
    wt = torch.from_numpy(w).cuda().requires_grad_(True)
    y = kdcc.functional.pointwise_conv(xt, wt, residual=rt)
    y.backward(to_dev(dy, dtype).contiguous(memory_format=fmt))
    ry = orc.pw_fwd(x, w) + r
    rdx, rdw, _ = orc.pw_bwd(x, w, dy)
    assert relerr(host(y), ry) < TOL[dtype]
    assert relerr(host(xt.grad), rdx) < TOL[dtype]
    assert relerr(host(wt.grad), rdw) < TOL[dtype]
    assert relerr(host(rt.grad), dy) < 1e-6
    scale = rs.uniform(0.5, 1.5, Nc).astype(np.float32)
    shift = rs.uniform(-0.5, 0.5, Nc).astype(np.float32)
    with torch.no_grad():
        ya = kdcc.functional.pointwise_conv(xt.detach(), wt.detach(), None, torch.from_numpy(scale).cuda(),
                                            torch.from_numpy(shift).cuda(), True, residual=rt.detach())
    ref = np.maximum(orc.pw_fwd(x, w) * scale[None, :, None, None] + shift[None, :, None, None] + r, 0)
    assert relerr(host(ya), ref) < TOL[dtype]


# ---- losses ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("tag", ["kl_T1", "kl_T2", "kl_T5", "kl_big", "kl_cifar_T5"])
def test_kd_loss_golden(kdcc, golden_losses, tag, dtype):
    from oracle import oracle as orc
    g = golden_losses
    T = float(g[f"{tag}/T"])
    s = to_dev(g[f"{tag}/arg0"], dtype, grad=True)
    t = to_dev(g[f"{tag}/arg1"], dtype)
    loss = kdcc.KLDivergenceLoss(temperature=T)(s, t)
    loss.backward()
    if dtype == torch.float32:
        ref_loss, ref_grad = float(g[f"{tag}/loss"]), g[f"{tag}/grad"]
    else:  # oracle on the bf16-rounded logits
        ref_loss, ref_grad = orc.kd_loss(q(g[f"{tag}/arg0"], dtype), q(g[f"{tag}/arg1"], dtype), T=T)
    assert abs(float(loss) - ref_loss) <= TOL[dtype] * abs(ref_loss)
    assert relerr(host(s.grad), ref_grad) < TOL[dtype]


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_kd_loss_layouts_and_no_grad(kdcc, golden_losses, layout):
    g, tag = golden_losses, "kl_T2"
    s = torch.from_numpy(g[f"{tag}/arg0"]).cuda()
    t = torch.from_numpy(g[f"{tag}/arg1"]).cuda()
    if layout == "nhwc":
        s, t = s.contiguous(memory_format=torch.channels_last), t.contiguous(memory_format=torch.channels_last)
    s.requires_grad_(True)
    loss = kdcc.KLDivergenceLoss(temperature=2)(s, t)
    (loss * 0.25).backward()  # upstream scalar is applied by kdcc_scale_inplace
    assert abs(float(loss) - float(g[f"{tag}/loss"])) <= 1e-5 * abs(float(g[f"{tag}/loss"]))
    assert relerr(host(s.grad), 0.25 * g[f"{tag}/grad"]) < 1e-5
    with torch.no_grad():
        l2 = kdcc.KLDivergenceLoss(temperature=2)(s, t)
    assert not l2.requires_grad and float(l2) == float(loss)


@pytest.mark.parametrize("tag", ["ekl", "ekl_onehot"])
def test_ensemble_kd_loss_golden(kdcc, golden_losses, tag):
    g = golden_losses
    s = to_dev(g[f"{tag}/arg0"], torch.float32, grad=True)
    loss = kdcc.EnsembleKLDivergenceLoss()(s, to_dev(g[f"{tag}/arg1"], torch.float32))
    loss.backward()
    assert abs(float(loss) - float(g[f"{tag}/loss"])) <= 1e-5 * abs(float(g[f"{tag}/loss"]))
    assert relerr(host(s.grad), g[f"{tag}/grad"]) < 1e-5


def test_kd_loss_many_classes_generic_kernel(kdcc):
    from oracle import oracle as orc
    rs = np.random.RandomState(3)
    s = rs.standard_normal((16, 100)).astype(np.float32) * 3   # CIFAR-100 sized class axis
    t = rs.standard_normal((16, 100)).astype(np.float32) * 3
    st = torch.from_numpy(s).cuda().requires_grad_(True)
    loss = kdcc.KLDivergenceLoss(temperature=4)(st, torch.from_numpy(t).cuda())
    loss.backward()
    rl, rg = orc.kd_loss(s, t, T=4.0)
    assert abs(float(loss) - rl) <= 1e-5 * abs(rl)
    assert relerr(host(st.grad), rg) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("tag", ["whint_vec", "whint_tab", "mse_nc1000", "mse_nc1", "mse_1x1"])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_hint_losses_golden(kdcc, golden_losses, tag, dtype, layout):
    from oracle import oracle as orc
    g = golden_losses
    s_np, t_np = g[f"{tag}/arg0"], g[f"{tag}/arg1"]
    s = torch.from_numpy(s_np).cuda().to(dtype)
    t = torch.from_numpy(t_np).cuda().to(dtype)
    if layout == "nhwc":
        s, t = s.contiguous(memory_format=torch.channels_last), t.contiguous(memory_format=torch.channels_last)
    s.requires_grad_(True)
    if tag.startswith("whint"):
        w_np = g[f"{tag}/arg2"]
        loss = kdcc.WeightedHintMSELoss()(s, t, torch.from_numpy(w_np).cuda())
        ref_loss, ref_grad = orc.hint_loss(q(s_np, dtype), q(t_np, dtype), w=w_np, scale=1.0)
    else:
        nc = float(g[f"{tag}/nc"])
        loss = kdcc.MSELoss(num_classes=nc)(s, t)
        ref_loss, ref_grad = orc.hint_loss(q(s_np, dtype), q(t_np, dtype), w=None, scale=nc)
    loss.backward()
    if dtype == torch.float32:
        ref_loss, ref_grad = float(g[f"{tag}/loss"]), g[f"{tag}/grad"]
    assert abs(float(loss) - ref_loss) <= TOL[dtype] * abs(ref_loss)
    assert relerr(host(s.grad), ref_grad) < TOL[dtype]


# ---- BASELINE-size properties (no oracle: size-independent identities) -------------------------------
def test_full_size_depthwise_impulse_and_linearity(kdcc):
    """1024^2 crop -> 128x128 maps, C=512, k=9 d=5 p=20: an impulse reproduces the (mirrored) taps, and the
    conv is linear in x."""
    torch.manual_seed(0)
    C, H, W, k, d, p = 512, 128, 128, 9, 5, 20
    w = torch.randn(C, 1, k, k, device="cuda")
    x = torch.zeros(1, C, H, W, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    x[0, :, 64, 70] = 1.0
    y = kdcc.functional.depthwise_conv(x, w, None, k, d, p).float()
    # y[i,j] = w[u,v] where (64,70) = (i + u*d - p, j + v*d - p)
    expect = torch.zeros(1, C, H, W, device="cuda")
    for u in range(k):
        for v in range(k):
            i, j = 64 - u * d + p, 70 - v * d + p
            if 0 <= i < H and 0 <= j < W:
                expect[0, :, i, j] = w[:, 0, u, v]
    assert torch.allclose(y, expect.to(torch.bfloat16).float(), atol=0, rtol=0)
    a = torch.randn(1, C, H, W, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    y1 = kdcc.functional.depthwise_conv(a, w, None, k, d, p).float()
    y2 = kdcc.functional.depthwise_conv(a * 2, w, None, k, d, p).float()
    assert torch.equal(y2, 2 * y1)  # exact: scaling by 2 commutes with every rounding


def test_full_size_depthwise_backward_adjoint(kdcc):
    """<dw(x), g> == <x, dw^T(g)> and == sum(w * dW): the three kernels are mutually consistent at full size."""
    torch.manual_seed(1)
    C, H, W, k, d, p = 512, 128, 128, 9, 5, 20
    w = (torch.randn(C, 1, k, k, device="cuda") / k).requires_grad_(True)
    x = torch.randn(2, C, H, W, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    g = torch.randn(2, C, H, W, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    y = kdcc.functional.depthwise_conv(x, w, None, k, d, p)
    y.backward(g)
    lhs = (y.double() * g.double()).sum()
    mid = (x.detach().double() * x.grad.double()).sum()
    rhs = (w.detach().double() * w.grad.double()).sum()
    assert abs(lhs - mid) / abs(lhs) < 1e-2
    assert abs(lhs - rhs) / abs(lhs) < 1e-2


def test_full_size_gemm_identity_and_colsum(kdcc):
    """M = 16384 pixels, 512 -> 512: identity weights reproduce x bit-exactly; dW against dy = 1 is the column sum."""
    torch.manual_seed(2)
    M, K = 16384, 512
    x = torch.randn(1, K, 128, 128, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    w = torch.eye(K, device="cuda").reshape(K, K, 1, 1).requires_grad_(True)
    y = kdcc.functional.pointwise_conv(x, w)
    assert torch.equal(y, x.detach())
    y.backward(torch.ones_like(y))
    colsum = x.detach().float().sum(dim=(0, 2, 3))
    assert torch.allclose(w.grad.reshape(K, K), colsum[None, :].expand(K, K), rtol=1e-3, atol=1e-2)
    assert torch.equal(x.grad.float(), torch.ones_like(x.grad).float())


def test_full_size_losses_zero_at_equality_and_deterministic(kdcc):
    torch.manual_seed(3)
    s = (3 * torch.randn(1, 19, 1024, 1024, device="cuda")).requires_grad_(True)
    l0 = kdcc.KLDivergenceLoss(temperature=5)(s, s.detach().clone())
    l0.backward()
    assert abs(float(l0)) < 1e-6 and float(s.grad.abs().max()) < 1e-9
    t = 3 * torch.randn(1, 19, 1024, 1024, device="cuda")
    a = kdcc.KLDivergenceLoss(temperature=5)(s, t)
    b = kdcc.KLDivergenceLoss(temperature=5)(s, t)
    assert float(a) == float(b) and float(a) > 0      # fixed-order reduction: bit-reproducible
    # gradient of each pixel sums to zero over classes
    s.grad = None
    a.backward()
    assert float(s.grad.sum(dim=1).abs().max()) < 1e-9
    f = torch.randn(1, 512, 128, 128, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    h0 = kdcc.MSELoss(num_classes=1000)(f, f.detach().clone())
    assert float(h0) == 0.0
    tt = torch.randn_like(f)
    h1 = kdcc.MSELoss(num_classes=1000)(f, tt)
    ref = torch.nn.functional.mse_loss(f.detach().float(), tt.float()) * 1000
    assert abs(float(h1) - float(ref)) / float(ref) < 1e-4


def test_errors_are_loud(kdcc):
    with pytest.raises(kdcc.KdccError):
        kdcc.functional.depthwise_conv(torch.randn(1, 8, 4, 4), torch.randn(8, 1, 3, 3), None, 3, 1, 1)  # CPU tensor
    with pytest.raises(kdcc.KdccError):  # 6 channels: not a 16-byte vector -> KDCC_ESHAPE, no fallback
        kdcc.functional.depthwise_conv(torch.randn(1, 6, 4, 4, device="cuda"), torch.randn(6, 1, 3, 3, device="cuda"), None, 3, 1, 1)
    with pytest.raises(RuntimeError):    # reference behaviour: a Tensor bias is rejected by nn.Conv2d (SURVEY F5)
        kdcc.DepthwiseSeparableBlock(8, 8, 3, 1, 1, 8, torch.zeros(8))
