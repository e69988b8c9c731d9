"""Which kernel runs for which arguments: forward + backward under torch.profiler, launched kernel names against the
table below.  The library picks its kernels from the call's arguments alone, so the parity tests prove a kernel by
the shapes that reach it; this table keeps those shapes reaching it.  It and test_conv_edges.py, whose parity rows pin
the kernels of every shape they run, are the only places a test names a kernel."""
import re

import pytest
import torch

from test_gpu_parity import kdcc  # noqa: F401  (the module fixture)

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32

DEPTHWISE = [
    # layout, dtype, N,  C,   H,   W, k, d,  p   depthwise kernels of forward + backward (split sums left out)
    ("nhwc", BF16, 2, 64, 16, 16, 3, 1, 1, {"dw_nhwc3_conv_kernel", "dw_nhwc3_wgrad_kernel"}),
    ("nhwc", BF16, 2, 48, 16, 16, 3, 1, 1, {"dw_tma_conv_kernel", "dw_tma_wgrad_kernel"}),
    ("nhwc", BF16, 2, 16, 20, 20, 3, 2, 2, {"dw_tma_conv_kernel", "dw_tma_wgrad_kernel"}),
    ("nhwc", BF16, 1, 32, 40, 67, 9, 5, 20, {"dw_tma_conv_kernel", "dw_tma_wgrad_kernel"}),
    ("nhwc", BF16, 2, 24, 16, 16, 3, 1, 1, {"dw_direct_kernel", "dw_wgrad_direct_kernel"}),
    ("nhwc", F32, 1, 16, 40, 40, 9, 5, 20, {"dw_direct_kernel", "dw_wgrad_direct_kernel"}),
    ("nchw", BF16, 1, 16, 128, 128, 9, 5, 20, {"dw_tc_conv2_kernel", "dw_tc_wgrad3_kernel"}),
    ("nchw", BF16, 1, 16, 128, 256, 9, 5, 20, {"dw_tc_conv2_kernel", "dw_tc_wgrad_kernel"}),
    ("nchw", BF16, 1, 16, 128, 128, 3, 1, 1, {"dw_tc_conv2_kernel", "dw_tc_wgrad2_kernel"}),
    ("nchw", BF16, 1, 16, 40, 264, 9, 5, 20, {"dw_tc_conv_kernel", "dw_tc_wgrad_kernel"}),
]

POINTWISE = [
    # N,  K,  H,  W,  Co   CTA pairs: 256-column tiles over an even number of 128-pixel tiles
    ((1, 64, 16, 16, 256), True),
    ((3, 64, 8, 16, 256), False),
]

DW_NAME = re.compile(r"\b(dw_[a-z0-9_]+_kernel)\b")
PW_NAME = re.compile(r"\bpw_gemm_sm100_kernel<(\d+), (?:true|false), (?:true|false), (true|false)>")


def launched(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                            torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("row", DEPTHWISE, ids=lambda r: "%s-%s-c%d-%dx%d-k%dd%dp%d" % (r[0], str(r[1])[6:], *r[3:9]))
def test_depthwise_kernel_follows_arguments(kdcc, row):
    layout, dtype, N, C, H, W, k, d, p, expect = row
    gen = torch.Generator("cuda").manual_seed(0)
    x = torch.randn(N, C, H, W, device="cuda", generator=gen).to(dtype)
    if layout == "nhwc":
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    w = (torch.randn(C, 1, k, k, device="cuda", generator=gen) / k).requires_grad_(True)

    def step():
        y = kdcc.functional.depthwise_conv(x, w, None, k, d, p)
        y.backward(torch.ones_like(y))

    names = {m.group(1) for n in launched(step) for m in DW_NAME.finditer(n) if "reduce" not in m.group(1)}
    assert names == expect


@pytest.mark.parametrize("row", POINTWISE, ids=lambda r: "pair" if r[1] else "single")
def test_pointwise_cta_pairs_follow_arguments(kdcc, row):
    (N, K, H, W, Co), pair = row
    gen = torch.Generator("cuda").manual_seed(0)
    x = torch.randn(N, K, H, W, device="cuda", generator=gen).to(BF16).contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    w = (torch.randn(Co, K, 1, 1, device="cuda", generator=gen) / K ** 0.5).requires_grad_(True)

    def step():
        y = kdcc.functional.pointwise_conv(x, w)
        y.backward(torch.ones_like(y))

    gemms = {(int(m.group(1)), m.group(2) == "true") for n in launched(step) for m in PW_NAME.finditer(n)}
    assert (256, pair) in gemms
    assert any(p for _, p in gemms) == pair
