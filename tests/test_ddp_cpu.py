"""world_size-2 gloo test of the bucketed reducer: averaged per-rank grads == single-process grad on the
concatenated batch (the DDP equivalence SURVEY.md §4 asks for), including a parameter that gets no grad."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class Net(nn.Module):
    def __init__(self):
        super().__init__()
        self.a = nn.Linear(16, 32, bias=False)
        self.b = nn.Linear(32, 8, bias=False)
        self.unused = nn.Linear(4, 4, bias=False)

    def forward(self, x):
        return self.b(torch.tanh(self.a(x)))


def _worker(rank, world, port, q, done):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from dreamllm_b200.ddp import BucketedGradReducer
    torch.manual_seed(0)
    net = Net()
    red = BucketedGradReducer(net.parameters(), bucket_cap_mb=0.001)   # tiny cap -> several buckets
    g = torch.Generator().manual_seed(1)
    x = torch.randn(8, 16, generator=g)
    for step in range(2):                     # second step exercises grad-as-bucket-view reuse
        red.zero_grad()
        net(x[rank * 4:(rank + 1) * 4]).pow(2).mean().backward()
        red.finalize()
    q.put((rank, {k: v.grad.clone() for k, v in net.named_parameters()}, red.launched))
    done.wait(240)                    # the queued tensors live in this process's shared memory until the parent has received them
    dist.destroy_process_group()


def _run_two_ranks():
    ctx = mp.get_context("spawn")
    q, done = ctx.Queue(), ctx.Event()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, done)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=240) for _ in range(2)]
    finally:
        done.set()
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    assert all(p.exitcode == 0 for p in procs)
    return res


def test_bucketed_reducer_matches_single_process():
    try:
        res = _run_two_ranks()
    except Exception:            # rendezvous port race / a loaded build box: one retry on a fresh port
        res = _run_two_ranks()
    torch.manual_seed(0)
    net = Net()
    g = torch.Generator().manual_seed(1)
    x = torch.randn(8, 16, generator=g)
    # mean over the two half-batches of per-half mean losses == loss on the full batch
    (0.5 * (net(x[:4]).pow(2).mean() + net(x[4:]).pow(2).mean())).backward()
    for rank, grads, launched in res:
        assert launched >= 4            # >1 bucket per step, 2 steps
        for k, v in net.named_parameters():
            want = v.grad if v.grad is not None else torch.zeros_like(v)
            torch.testing.assert_close(grads[k], want, rtol=1e-5, atol=1e-7)
