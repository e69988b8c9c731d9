"""Column-phase depthwise weight gradient (dw_tc_wgrad3.cu) against an fp64 torch reference, over ragged shapes; then
its timing on the 4096-channel site.  Run on the GPU box."""
import importlib
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
kdcc = importlib.import_module("knowledge-distillation-by-replacing-cheap-conv_b200")
F = kdcc.functional


def dw_grad(x, w, dy):
    x = x.detach().requires_grad_(False)
    w = w.detach().clone().requires_grad_(True)
    y = F.depthwise_conv(x, w, None, 9, 5, 20)
    y.backward(dy)
    return w.grad.detach().clone()


def ref_grad(x, w, dy):
    xd, wd = x.double(), w.double().detach().clone().requires_grad_(True)
    y = torch.nn.functional.conv2d(xd, wd, None, 1, 20, 5, x.shape[1])
    y.backward(dy.double())
    return wd.grad


def main():
    torch.manual_seed(0)
    dev = "cuda"
    shapes = [(1, 8, 128, 128), (4, 64, 128, 128), (3, 37, 128, 128), (2, 16, 96, 104), (5, 300, 128, 128), (2, 40, 65, 128), (1, 3, 128, 8), (4, 512, 128, 128)]
    for (n, c, h, w_) in shapes:
        x = torch.randn(n, c, h, w_, device=dev).to(torch.bfloat16)
        dy = torch.randn(n, c, h, w_, device=dev).to(torch.bfloat16)
        w = torch.randn(c, 1, 9, 9, device=dev) * 0.1
        g = dw_grad(x, w, dy).cpu()
        r = ref_grad(x, w, dy).float().cpu()
        err = (g - r).abs().max().item() / max(r.abs().max().item(), 1e-9)
        print("shape", (n, c, h, w_), "rel err vs fp64 %.3e" % err, flush=True)
        assert err < 2e-5, err   # both operands are exact bf16, fp32 accumulation
    # timing
    n, c = 4, 4096
    x = torch.randn(n, c, 128, 128, device=dev).to(torch.bfloat16)
    dy = torch.randn(n, c, 128, 128, device=dev).to(torch.bfloat16)
    w = torch.randn(c, 1, 9, 9, device=dev) * 0.1
    from importlib import import_module
    abi = import_module("knowledge-distillation-by-replacing-cheap-conv_b200._abi")
    lib = abi.lib()
    dwg = torch.empty(c, 81, device=dev)
    ws_bytes = lib.kdcc_dw_bwd_workspace_bytes(n, 128, 128, c, 9, 5, 20, abi.NCHW, abi.BF16)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def run():
        rc = lib.kdcc_dw_bwd(x.data_ptr(), None, dy.data_ptr(), None, dwg.data_ptr(), None, ws.data_ptr(), ws_bytes, n, 128, 128, c, 9, 5, 20,
                             abi.NCHW, abi.BF16, st)
        assert rc == 0, rc
    for _ in range(5):
        run()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(20):
        run()
    e1.record()
    torch.cuda.synchronize()
    print("dW 4096 ch x 4 images: %.4f ms" % (e0.elapsed_time(e1) / 20))


if __name__ == "__main__":
    main()
