"""Data-parallel gradient exchange (SURVEY.md 8e): kdcc_radam_step_multi (the mean of the ranks' gradient copies taken inside
the optimizer pass) on one GPU, and -- when the box has two -- kdcc.PeerGradBucket end to end: symmetric buffers, per-region
peer pushes on a side stream, the finishing signal exchange, bit-identical parameters on both ranks, against the NCCL
all-reduce it replaces.  (The gloo / CPU form of the exchange is test_student_trainer.py's two-rank test.)"""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import kdcc

pytestmark = pytest.mark.gpu


def test_multi_source_radam_equals_a_step_on_the_mean():
    torch.manual_seed(0)
    n, nsrc, stride = 1000 + 37, 3, 1088
    srcs = torch.randn(nsrc, stride, device="cuda")
    for steps in (1, 7):        # 7: past the degenerated-to-SGD phase of RAdam (N_sma >= 5 from step 6)
        a = torch.nn.Parameter(torch.randn(n, device="cuda"))
        b = torch.nn.Parameter(a.detach().clone())
        oa, ob = kdcc.optim.RAdam([a], lr=1e-2), kdcc.optim.RAdam([b], lr=1e-2)
        a.grad = torch.empty(n, device="cuda")
        ob.attach_grad_sources(b, lambda: (srcs[0, :n], stride, nsrc))
        b.grad = srcs[1, :n]    # only its presence matters: the step reads the sources
        for _ in range(steps):
            a.grad.copy_(((srcs[0, :n] + srcs[1, :n]) + srcs[2, :n]) * (1.0 / 3.0))   # the kernel's own summation order
            oa.step()
            ob.step()
        torch.cuda.synchronize()
        assert torch.equal(a.detach(), b.detach()), steps


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        n = 3 * 4096 + 19
        bucket = kdcc.PeerGradBucket(n, dev)
        p = torch.nn.Parameter(torch.linspace(-1, 1, n, device=dev))
        ref = torch.nn.Parameter(p.detach().clone())
        opt, ropt = kdcc.optim.RAdam([p], lr=1e-2), kdcc.optim.RAdam([ref], lr=1e-2)
        opt.attach_grad_sources(p, bucket.sources)
        for step in range(4):                                   # both parities, twice
            g = torch.randn(n, device=dev, generator=torch.Generator(dev).manual_seed(100 * step + rank))
            p.grad = bucket.local()
            p.grad.copy_(g)
            for lo, hi in ((0, 4096), (4096, 8000), (8000, n)):   # regions become final one after the other
                bucket.push(lo, hi)
            bucket.finish()
            opt.step()
            bucket.flip()
            ref.grad = g.clone()
            dist.all_reduce(ref.grad, op=dist.ReduceOp.AVG)
            ropt.step()
        torch.cuda.synchronize()
        err = float((p.detach() - ref.detach()).abs().max())
        both = [torch.empty_like(p.detach()) for _ in range(world)]
        dist.all_gather(both, p.detach().contiguous())
        if rank == 0:
            out.put((err, bool(torch.equal(both[0], both[1]))))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs of one box")
def test_peer_grad_bucket_matches_nccl_allreduce_on_two_gpus():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29700 + os.getpid() % 200
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for pr in procs:
        pr.start()
    for pr in procs:
        pr.join(180)
        assert pr.exitcode == 0
    err, identical = out.get(timeout=5)
    assert identical, "ranks ended with different parameters"
    assert err < 1e-6     # NCCL's AVG sums in another order than the fixed rank order: equal to rounding
