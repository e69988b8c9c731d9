"""GPU parity, second batch (VERDICT round 1): the tensor-core NCHW path against reference goldens with UN-rounded taps,
full-size sites of both Cityscapes plans against the oracle, the pointwise weight-gradient workspace bound, and the
host-glue guarantees (double backward raises, gradients aligned in the bucket).  Tolerances as in test_gpu_parity.py."""
import ctypes
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from test_gpu_parity import TOL, host, kdcc, q, relerr, run_block  # noqa: F401  (kdcc is the module fixture)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden_extra():
    return np.load(os.path.join(GOLDEN, "block_extra.npz"))


@pytest.mark.parametrize("tag", ["city_k9d5_w32", "city_k9d5_plane"])
def test_block_nchw_tensor_core_matches_reference_golden_unrounded_taps(kdcc, golden_extra, tag):
    """The Cityscapes geometry (k9 d5 p20) on the NCHW tensor-core kernels against the reference's own fp32 block.
    Documented deviation: the Toeplitz operand holds the taps rounded to bf16 (as every bf16 conv holds its weights);
    the golden was computed with the fp32 taps and nothing is pre-rounded here -- the result stays inside 2e-2."""
    g = golden_extra
    N, Ci, Co, H, W, k, d, p = [int(v) for v in g[f"{tag}/geom"]]
    assert kdcc._abi.dispatch_name(0, N, H, W, Ci, Co, k, d, p, kdcc._abi.NCHW, kdcc._abi.BF16) == "dw_tc_conv"
    y, dx, dwd, dwp = run_block(kdcc, g[f"{tag}/x"], g[f"{tag}/w_dw"], g[f"{tag}/w_pw"], g[f"{tag}/dy"], k, d, p,
                                torch.bfloat16, layout="nchw")
    for name, mine in (("y", y), ("dx", dx), ("dw_dw", dwd), ("dw_pw", dwp)):
        assert relerr(mine, g[f"{tag}/{name}"]) < TOL[torch.bfloat16], name
    # the depthwise stage alone (what the bench times), forward / dX / dW
    x = torch.from_numpy(g[f"{tag}/x"]).cuda().to(torch.bfloat16).requires_grad_(True)
    w = torch.from_numpy(g[f"{tag}/w_dw"]).cuda().requires_grad_(True)
    from oracle import oracle as orc
    mid = kdcc.functional.depthwise_conv(x, w, None, k, d, p)
    gm = torch.randn(mid.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(3)).to(torch.bfloat16)
    mid.backward(gm)
    xq, gq = host(x), host(gm)
    assert relerr(host(mid), orc.dw_fwd(xq, g[f"{tag}/w_dw"], k, d, p)) < TOL[torch.bfloat16]
    rdx, rdw, _ = orc.dw_bwd(xq, g[f"{tag}/w_dw"], gq, k, d, p)
    assert relerr(host(x.grad), rdx) < TOL[torch.bfloat16]
    assert relerr(host(w.grad), rdw) < TOL[torch.bfloat16]


FULL_SITES = [(4096, 256), (1024, 2048), (512, 1024)]   # 51M plan ASPP / mod7 sites, 58M plan mod5.block2 (SURVEY 8a a2)


@pytest.mark.parametrize("site", FULL_SITES)
def test_full_size_site_matches_oracle_on_subsets(kdcc, site):
    """A whole site at the BASELINE size (image pair, 128 x 128 maps, k9 d5 p20, NCHW bf16) against the C oracle.  The
    oracle is evaluated exactly on subsets it finishes in seconds: depthwise on a spread of channels (channels are
    independent), pointwise forward / dX on a spread of pixels, pointwise dW on a spread of output channels (each row
    of dW is an independent reduction over all pixels).  fp32 taps are NOT pre-rounded for the oracle."""
    from oracle import oracle as orc
    Ci, Co = site
    N, H, W, k, d, p = 2, 128, 128, 9, 5, 20
    gen = torch.Generator("cuda").manual_seed(Ci + Co)
    x = torch.randn(N, Ci, H, W, device="cuda", generator=gen).to(torch.bfloat16).requires_grad_(True)
    w_dw = ((torch.rand(Ci, 1, k, k, device="cuda", generator=gen) * 2 - 1) / k).requires_grad_(True)
    w_pw = ((torch.rand(Co, Ci, 1, 1, device="cuda", generator=gen) * 2 - 1) / Ci ** 0.5).requires_grad_(True)
    dy = torch.randn(N, Co, H, W, device="cuda", generator=gen).to(torch.bfloat16)
    mid = kdcc.functional.depthwise_conv(x, w_dw, None, k, d, p)
    mid.retain_grad()
    y = kdcc.functional.pointwise_conv(mid, w_pw)
    y.backward(dy)
    torch.cuda.synchronize()
    tol = TOL[torch.bfloat16]

    # ---- depthwise: 48 channels spread over the range (first, last, both sides of CTA-unit boundaries) ----
    ch = np.unique(np.concatenate([np.arange(0, 8), np.arange(Ci - 8, Ci), np.linspace(8, Ci - 9, 32).astype(int)]))
    chs = torch.from_numpy(ch).cuda()
    xs, ws, dmids = host(x[:, chs]), host(w_dw[chs]), host(mid.grad[:, chs])
    assert relerr(host(mid[:, chs]), orc.dw_fwd(xs, ws, k, d, p)) < tol
    rdx, rdw, _ = orc.dw_bwd(xs, ws, dmids, k, d, p)
    assert relerr(host(x.grad[:, chs]), rdx) < tol
    assert relerr(host(w_dw.grad[chs]), rdw) < tol

    # ---- pointwise forward / dX: 1536 pixels spread over both images (as a (N, C, P', 1) problem) ----
    pix = torch.from_numpy(np.unique(np.concatenate([np.arange(0, 64), np.arange(H * W - 64, H * W),
                                                     np.linspace(64, H * W - 65, 640).astype(int)]))).cuda()
    mid_q = host(mid.detach().reshape(N, Ci, H * W)[:, :, pix])[..., None]
    dy_q = host(dy.reshape(N, Co, H * W)[:, :, pix])[..., None]
    w_q = q(host(w_pw), torch.bfloat16)                     # the GEMM reads the bf16 copy of the fp32 master weights
    assert relerr(host(y.detach().reshape(N, Co, H * W)[:, :, pix])[..., None], orc.pw_fwd(mid_q, w_q)) < tol
    rdmid, _, _ = orc.pw_bwd(mid_q, w_q, dy_q)
    assert relerr(host(mid.grad.reshape(N, Ci, H * W)[:, :, pix])[..., None], rdmid) < tol

    # ---- pointwise dW: 24 output channels, reduction over ALL pixels of both images ----
    co = torch.from_numpy(np.unique(np.concatenate([np.arange(0, 8), np.arange(Co - 8, Co), [Co // 2, Co // 3]]))).cuda()
    _, rdw_pw, _ = orc.pw_bwd(host(mid.detach()), w_q[host(co).astype(int)], host(dy[:, co]), need_dx=False)
    assert relerr(host(w_pw.grad[co]), rdw_pw) < tol


@pytest.mark.parametrize("geom", [(2, 30, 40, 64, 128), (3, 28, 28, 256, 64), (2, 45, 80, 32, 512), (5, 8, 8, 128, 256)])
def test_pointwise_dw_nchw_splits_stay_inside_the_workspace(kdcc, geom):
    """ADVICE round 1: with batch > 1 and P = H*W not a multiple of 64 the NCHW weight-gradient launch used more splits
    than kdcc_pw_bwd_workspace_bytes had sized.  The C ABI is called with EXACTLY the advertised workspace in front of a
    guard region; the guard must stay untouched and dW must match the oracle."""
    from oracle import oracle as orc
    N, H, W, K, Co = geom
    L = kdcc._abi.lib()
    M = N * H * W
    rs = np.random.RandomState(M + K)
    x = q(rs.standard_normal((N, K, H, W)).astype(np.float32), torch.bfloat16)
    dy = q(rs.standard_normal((N, Co, H, W)).astype(np.float32), torch.bfloat16)
    xt, dyt = torch.from_numpy(x).cuda().to(torch.bfloat16), torch.from_numpy(dy).cuda().to(torch.bfloat16)
    need = int(L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, kdcc._abi.BF16))
    guard = 1 << 20
    buf = torch.full((need + guard,), 0x5A, dtype=torch.uint8, device="cuda")
    dw = torch.empty(Co, K, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    kdcc._abi.check(L.kdcc_pw_bwd_dw(dyt.data_ptr(), xt.data_ptr(), dw.data_ptr(), buf.data_ptr(), need, M, K, Co, N,
                                     kdcc._abi.NCHW, kdcc._abi.BF16, st), "kdcc_pw_bwd_dw")
    torch.cuda.synchronize()
    assert bool((buf[need:] == 0x5A).all()), "weight-gradient partials were written past the advertised workspace"
    _, rdw, _ = orc.pw_bwd(x, np.zeros((Co, K, 1, 1), np.float32), dy, need_dx=False)
    assert relerr(host(dw), rdw.reshape(Co, K)) < TOL[torch.bfloat16]
    # one byte less is refused, not overrun
    rc = L.kdcc_pw_bwd_dw(dyt.data_ptr(), xt.data_ptr(), dw.data_ptr(), buf.data_ptr(), need - 1, M, K, Co, N,
                          kdcc._abi.NCHW, kdcc._abi.BF16, st)
    assert rc != 0 and "workspace" in kdcc._abi.strerror(rc).lower()


def test_loss_backward_twice_raises_instead_of_dropping_the_gradient(kdcc):
    s = torch.randn(2, 19, 8, 8, device="cuda", requires_grad=True)
    t = torch.randn(2, 19, 8, 8, device="cuda")
    for crit in (kdcc.KLDivergenceLoss(temperature=2), kdcc.MSELoss(num_classes=19)):
        loss = crit(s, t)
        loss.backward(retain_graph=True)
        assert s.grad is not None and float(s.grad.abs().sum()) > 0
        with pytest.raises(kdcc._abi.KdccError, match="already back-propagated"):
            loss.backward()
        s.grad = None


def test_radam_steps_through_a_bucket_with_odd_sized_parameters(kdcc):
    """ADVICE round 1: a 19-element classifier bias in front of other parameters used to misalign every gradient view
    after it, and kdcc_radam_step refuses unaligned pointers."""
    torch.manual_seed(0)
    params = [torch.nn.Parameter(torch.randn(n, device="cuda")) for n in (19, 64 * 9, 7, 33, 512)]
    bucket = kdcc.GradBucket(params)
    opt = kdcc.optim.RAdam(params, lr=1e-2)
    expect = []
    for p in params:
        gcpu = torch.randn(p.shape)
        p.grad.copy_(gcpu)
        # step 1 of the reference's RAdam (utils/optim/radam.py:65-97, N_sma < 5, degenerated_to_sgd): p -= lr * g
        expect.append(p.detach().cpu() - 1e-2 * gcpu)
    assert all(p.grad.data_ptr() % 16 == 0 for p in params)
    opt.step()
    torch.cuda.synchronize()
    for p, e in zip(params, expect):
        assert torch.allclose(p.detach().cpu(), e, rtol=1e-5, atol=1e-6)
    bucket.zero()
    assert all(float(p.grad.abs().sum()) == 0 for p in params)


def test_expected_upstream_is_a_hint_not_an_assumption(kdcc):
    """The loss kernels fold the upstream gradient a caller expects into the gradient they emit; backward verifies it on
    the device.  Whether the hint is right (no memory traffic in backward) or wrong (rescaled), ds is the same."""
    torch.manual_seed(1)
    t = torch.randn(2, 16, 8, 8, device="cuda")
    grads = []
    for expected, divide in ((1.0, 4.0), (0.25, 4.0), (0.25, 1.0), (3.0, 7.0)):
        s = torch.randn(2, 16, 8, 8, device="cuda", generator=torch.Generator("cuda").manual_seed(5)).requires_grad_(True)
        crit = kdcc.MSELoss(num_classes=1000)
        crit.expected_upstream = expected
        (crit(s, t) / divide).backward()
        grads.append(s.grad * divide)
    for g in grads[1:]:
        assert torch.allclose(g, grads[0], rtol=1e-6, atol=0)
    s = torch.randn(2, 19, 8, 8, device="cuda", requires_grad=True)
    tt = torch.randn(2, 19, 8, 8, device="cuda")
    a = kdcc.functional.kd_loss(s, tt, 2.0, expected_upstream=1.0)
    a.backward()
    ga, s.grad = s.grad.clone(), None
    (kdcc.functional.kd_loss(s, tt, 2.0, expected_upstream=0.5) * 1.0).backward()
    assert torch.allclose(s.grad, ga, rtol=1e-6, atol=0)


def test_cached_bf16_weight_copy_follows_the_master_weight(kdcc):
    """pointwise_conv caches the bf16 copy of its fp32 master weight by the parameter's version counter: an in-place torch
    update invalidates it, and kdcc.optim.RAdam refreshes it inside its fused step (no cast launch afterwards)."""
    torch.manual_seed(2)
    x = torch.randn(2, 64, 8, 8, device="cuda").to(torch.bfloat16)
    w = torch.nn.Parameter(torch.randn(32, 64, 1, 1, device="cuda") / 8)
    ref = lambda: torch.nn.functional.conv2d(x.float(), w.detach().to(torch.bfloat16).float())
    y0 = kdcc.functional.pointwise_conv(x, w)
    assert relerr(host(y0), host(ref())) < TOL[torch.bfloat16]
    lp0 = kdcc.functional.lp_copy_of(w)
    assert lp0 is not None and kdcc.functional.lp_weight(w, torch.bfloat16) is lp0          # reused while w is unchanged
    with torch.no_grad():
        w.mul_(-2.0)                                                                         # torch in-place op: version moves
    y1 = kdcc.functional.pointwise_conv(x, w)
    assert relerr(host(y1), host(ref())) < TOL[torch.bfloat16] and relerr(host(y1), -2 * host(y0)) < 2e-2
    opt = kdcc.optim.RAdam([w], lr=0.1)
    w.grad = torch.ones_like(w)
    lp1 = kdcc.functional.lp_copy_of(w)
    opt.step()                                                                               # rewrites w AND its cached copy
    assert kdcc.functional.lp_weight(w, torch.bfloat16) is lp1
    torch.cuda.synchronize()
    assert torch.equal(lp1.float(), w.detach().to(torch.bfloat16).float())
    y2 = kdcc.functional.pointwise_conv(x, w)
    assert relerr(host(y2), host(ref())) < TOL[torch.bfloat16]


@pytest.mark.parametrize("shape", [(2, 64, 16, 24), (1, 72, 5, 8), (3, 8, 128, 128), (2, 4096, 8, 16), (1, 200, 9, 40)])
def test_layout_convert_is_a_bit_exact_transpose(kdcc, shape):
    """kdcc_layout_convert (the channels_last <-> NCHW re-layout at a block boundary): exact, both directions, ragged tiles."""
    N, C, H, W = shape
    L = kdcc._abi.lib()
    st = torch.cuda.current_stream().cuda_stream
    x = torch.randn(N, C, H, W, device="cuda").to(torch.bfloat16)                        # NCHW-physical
    cl = torch.empty_like(x, memory_format=torch.channels_last)
    kdcc._abi.check(L.kdcc_layout_convert(x.data_ptr(), cl.data_ptr(), N, C, H * W, 0, kdcc._abi.BF16, st), "to nhwc")
    assert torch.equal(cl, x) and cl.is_contiguous(memory_format=torch.channels_last)
    back = torch.empty(N, C, H, W, device="cuda", dtype=torch.bfloat16)
    kdcc._abi.check(L.kdcc_layout_convert(cl.data_ptr(), back.data_ptr(), N, C, H * W, 1, kdcc._abi.BF16, st), "to nchw")
    assert torch.equal(back, x) and back.is_contiguous()
    assert L.kdcc_layout_convert(x.data_ptr(), cl.data_ptr(), N, C + 1, H * W, 0, kdcc._abi.BF16, st) != 0   # C % 8 != 0: refused


@pytest.mark.parametrize("geom", [(2, 64, 128, 40, 40, 9, 5, 20), (1, 512, 512, 128, 128, 9, 5, 20), (3, 24, 8, 37, 40, 9, 5, 20)])
def test_channels_last_block_runs_on_the_tensor_core_path_and_returns_channels_last(kdcc, geom):
    """A channels_last (cuDNN-style) trunk around the block: the k = 9 depthwise is re-laid to channel planes at the block
    boundary, runs on the NCHW tensor-core kernels, and output / input gradient come back channels_last."""
    from test_gpu_parity import oracle_block
    N, Ci, Co, H, W, k, d, p = geom
    dtype = torch.bfloat16
    rs = np.random.RandomState(99 + Ci + H)
    x = rs.standard_normal((N, Ci, H, W)).astype(np.float32)
    w_dw = (rs.uniform(-1, 1, (Ci, 1, k, k)) / k).astype(np.float32)
    w_pw = (rs.uniform(-1, 1, (Co, Ci, 1, 1)) / np.sqrt(Ci)).astype(np.float32)
    dy = rs.standard_normal((N, Co, H, W)).astype(np.float32)
    blk = kdcc.DepthwiseSeparableBlock(Ci, Co, k, p, d, Ci, None).cuda()
    with torch.no_grad():
        blk.separable_conv.weight.copy_(torch.from_numpy(w_dw))
        blk.pointwise_conv.weight.copy_(torch.from_numpy(w_pw))
    xt = torch.from_numpy(x).cuda().to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = blk(xt)
    assert y.is_contiguous(memory_format=torch.channels_last) and not y.is_contiguous()
    y.backward(torch.from_numpy(dy).cuda().to(dtype).contiguous(memory_format=torch.channels_last))
    assert xt.grad.is_contiguous(memory_format=torch.channels_last)
    ry, rdx, rdwd, rdwp = oracle_block(x, w_dw, w_pw, dy, k, d, p, dtype)
    for name, mine, ref in (("y", host(y), ry), ("dx", host(xt.grad), rdx), ("dw_dw", host(blk.separable_conv.weight.grad), rdwd),
                            ("dw_pw", host(blk.pointwise_conv.weight.grad), rdwp)):
        assert relerr(mine, ref) < TOL[dtype], name


@pytest.mark.parametrize("geom", [(2, 64, 128, 16, 24), (1, 512, 512, 128, 128), (3, 256, 72, 12, 20), (2, 4096, 256, 16, 16)])
def test_pointwise_planes_in_channels_last_out(kdcc, geom):
    """KDCC_LAYOUT_PLANES_TO_NHWC: the pointwise GEMMs take the block-internal tensor as channel planes and read / write the
    block-external one channels_last (forward, dX, dW) -- no re-layout pass for y and dy inside a channels_last trunk."""
    from oracle import oracle as orc
    N, K, Co, H, W = geom
    dtype = torch.bfloat16
    rs = np.random.RandomState(K + Co + H)
    x = q(rs.standard_normal((N, K, H, W)).astype(np.float32), dtype)
    w = q((rs.uniform(-1, 1, (Co, K, 1, 1)) / np.sqrt(K)).astype(np.float32), dtype)
    dy = q(rs.standard_normal((N, Co, H, W)).astype(np.float32), dtype)
    xt = torch.from_numpy(x).cuda().to(dtype).requires_grad_(True)                       # plain NCHW: planes
    wt = torch.from_numpy(w).cuda().requires_grad_(True)
    assert kdcc._abi.dispatch_name(2, N, H, W, K, Co, 1, 1, 0, kdcc._abi.PLANES_TO_NHWC, kdcc._abi.BF16) == "pw_gemm_sm100_fwd"
    y = kdcc.functional.pointwise_conv(xt, wt, out_channels_last=True)
    assert y.is_contiguous(memory_format=torch.channels_last) and not y.is_contiguous()
    y.backward(torch.from_numpy(dy).cuda().to(dtype).contiguous(memory_format=torch.channels_last))
    assert xt.grad.is_contiguous()
    ry = orc.pw_fwd(x, w)
    rdx, rdw, _ = orc.pw_bwd(x, w, dy)
    assert relerr(host(y), ry) < TOL[dtype]
    assert relerr(host(xt.grad), rdx) < TOL[dtype]
    assert relerr(host(wt.grad), rdw) < TOL[dtype]


def test_hot_path_step_orders_and_layouts_agree(kdcc):
    """kdcc.hotpath.HotPathStep (what bench.py times): the reference loop's order (all forwards, losses, backward in reverse)
    and the site-by-site order produce bit-identical losses and gradients (every kernel is deterministic), and the
    channels_last form (inputs re-laid to planes, mixed-layout GEMMs) agrees with the NCHW form to bf16 accuracy.  Each
    site is also checked against the oracle through its hint loss and pointwise weight gradient."""
    from kdcc.hotpath import HotPathStep
    from oracle import oracle as orc
    plan = [(32, 64), (64, 32), (16, 48)]
    N, H, W = 2, 40, 48
    kw = dict(kernel_size=9, dilation=5, padding=20, dtype=torch.bfloat16, device="cuda", logits_shape=(N, 19, 32, 32),
              need_dx=[False, True, True], seed=3)
    steps = {name: HotPathStep(plan, N, H, W, order=order, layout=layout, **kw)
             for name, order, layout in (("ref", "reference", "nchw"), ("inter", "interleaved", "nchw"), ("cl", "reference", "nhwc"))}
    xs, ts, ls, lt = steps["ref"].make_inputs(seed=5)
    out = {}
    for name, hp in steps.items():
        a, b = (xs, ts) if name != "cl" else ([x.permute(0, 2, 3, 1).contiguous() for x in xs], [t.permute(0, 2, 3, 1).contiguous() for t in ts])
        hint, kd = hp.step(a, b, ls, lt)
        torch.cuda.synchronize()
        out[name] = (float(hint), float(kd), hp.flat_grads.clone(), hp.hint_losses.clone())
    assert out["ref"][0] == out["inter"][0] and out["ref"][1] == out["inter"][1]
    assert torch.equal(out["ref"][2], out["inter"][2])
    assert abs(out["cl"][0] - out["ref"][0]) <= 2e-2 * abs(out["ref"][0])
    assert relerr(host(out["cl"][2]), host(out["ref"][2])) < TOL[torch.bfloat16]
    assert steps["cl"].relayout and steps["cl"].layout == kdcc._abi.NCHW
    # site 0 against the oracle: hint loss value and the pointwise weight gradient
    hp = steps["ref"]
    a0, b0, c0 = hp._views[0]
    ci, co = plan[0]
    w_dw = host(hp.flat_params[a0:b0]).reshape(ci, 1, 9, 9)
    w_pw = q(host(hp.flat_params[b0:c0]).reshape(co, ci, 1, 1), torch.bfloat16)
    mid = q(orc.dw_fwd(host(xs[0]), w_dw, 9, 5, 20), torch.bfloat16)
    y = q(orc.pw_fwd(mid, w_pw), torch.bfloat16)
    loss, ds = orc.hint_loss(y, host(ts[0]), None, scale=1000.0)
    assert abs(float(out["ref"][3][0]) - loss) <= 2e-2 * abs(loss)
    _, rdw, _ = orc.pw_bwd(mid, w_pw, q(ds, torch.bfloat16), need_dx=False)
    assert relerr(host(hp.flat_grads[b0:c0]).reshape(co, ci, 1, 1), rdw) < TOL[torch.bfloat16]


@pytest.mark.parametrize("geom", [(2, 8, 8, 128, 256), (3, 24, 16, 100, 200), (1, 8, 16, 64, 136), (1, 40, 8, 128, 248)])
def test_wide_planes_run_as_two_column_halves(kdcc, geom):
    """Planes of 129 .. 256 columns (Gated-SCNN sites on a 1024 x 2048 input, BASELINE config 4) on the whole-plane
    tensor-core convolution: two column halves with their own landing window and Toeplitz offset; forward, dX and dW against
    the oracle (fp32 taps un-rounded), and bit-identical to the tiled kernel's result semantics at the seam columns."""
    from test_gpu_parity import oracle_block
    N, Ci, Co, H, W = geom
    k, d, p = 9, 5, 20
    dtype = torch.bfloat16
    rs = np.random.RandomState(7 + W + Ci)
    x = rs.standard_normal((N, Ci, H, W)).astype(np.float32)
    w_dw = (rs.uniform(-1, 1, (Ci, 1, k, k)) / k).astype(np.float32)
    w_pw = (rs.uniform(-1, 1, (Co, Ci, 1, 1)) / np.sqrt(Ci)).astype(np.float32)
    dy = rs.standard_normal((N, Co, H, W)).astype(np.float32)
    y, dx, dwd, dwp = run_block(kdcc, x, w_dw, w_pw, dy, k, d, p, dtype, layout="nchw")
    ry, rdx, rdwd, rdwp = oracle_block(x, w_dw, w_pw, dy, k, d, p, dtype)
    for name, mine, ref in (("y", y, ry), ("dx", dx, rdx), ("dw_dw", dwd, rdwd), ("dw_pw", dwp, rdwp)):
        assert relerr(mine, ref) < TOL[dtype], name
    # the depthwise alone, column by column around the seam (columns 100 .. 160 are touched by both halves' windows)
    from oracle import oracle as orc
    xt = torch.from_numpy(x).cuda().to(dtype)
    mid = kdcc.functional.depthwise_conv(xt, torch.from_numpy(w_dw).cuda(), None, k, d, p)
    ref_mid = orc.dw_fwd(host(xt), w_dw, k, d, p)
    err_cols = np.abs(host(mid) - ref_mid).max(axis=(0, 1, 2)) / np.abs(ref_mid).max()
    assert err_cols.max() < TOL[dtype], int(err_cols.argmax())


@pytest.mark.parametrize("geom", [(1, 8, 128, 128), (3, 37, 128, 128), (2, 16, 96, 104), (5, 300, 128, 128), (2, 40, 65, 128),
                                  (1, 3, 128, 8), (4, 512, 128, 128)])
def test_depthwise_weight_gradient_column_phase_kernel(kdcc, geom):
    """9 x 9, dilation 5 weight gradient on the column-phase tensor-core kernel (dw_tc_wgrad3.cu: four tap rows per MMA, dy
    transposed by the tensor core) over ragged planes, odd batch sizes and channel counts that split units across CTAs:
    against torch's fp64 autograd of the reference's depthwise conv (depthwise_separable_conv.py:12).  Both operands are
    exact bf16 and the sums are fp32: 2e-5."""
    n, c, h, w_ = geom
    gen = torch.Generator("cuda").manual_seed(11)
    x = torch.randn(n, c, h, w_, device="cuda", generator=gen).to(torch.bfloat16)
    dy = torch.randn(n, c, h, w_, device="cuda", generator=gen).to(torch.bfloat16)
    w = torch.randn(c, 1, 9, 9, device="cuda", generator=gen) * 0.1

    def grad():
        wt = w.detach().clone().requires_grad_(True)
        kdcc.functional.depthwise_conv(x, wt, None, 9, 5, 20).backward(dy)
        return wt.grad.detach().clone()

    mine = grad()
    wd = w.double().requires_grad_(True)
    torch.nn.functional.conv2d(x.double(), wd, None, 1, 20, 5, c).backward(dy.double())
    ref = wd.grad
    assert ((mine.double() - ref).abs().max() / ref.abs().max()).item() < 2e-5
    assert torch.equal(mine, grad())  # deterministic: fixed-order sums, no atomics
