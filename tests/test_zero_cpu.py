"""CPU tests of the sharded data-parallel optimizer (dreamllm_b200/zero.py, SURVEY.md §8f row 4).

* the AdamW oracle (oracle/adamw_oracle.py) is pinned bit-for-bit to `torch.optim.AdamW` — the reference's optimizer
  (`optim="adamw_torch"`, projects/dreamllm/configs/stage1/base.py:85) — in bf16 (the reference's dtype) and fp32;
* the LR schedule equals transformers' `get_cosine_schedule_with_warmup`;
* host logic (bucket layout, shard ownership, reduce-scatter / all-gather, missing grads, checkpoint round trip) is driven on CPU
  tensors with the oracle's arithmetic injected, single process and world_size 2 over gloo.
The CUDA arithmetic itself is checked in tests/test_zero_gpu.py.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from oracle import adamw_oracle as AO

BF = torch.bfloat16
HP = dict(lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


# ------------------------------------------------------------------------------------------------ oracle pin
@pytest.mark.parametrize("dtype", [BF, torch.float32])
def test_adamw_oracle_is_torch_adamw_bit_for_bit(dtype):
    g = torch.Generator().manual_seed(0)
    shapes = [(37, 16), (16,), (5, 8, 3)]
    ps = [nn.Parameter((torch.randn(s, generator=g) * 0.05).to(dtype)) for s in shapes]
    opt = torch.optim.AdamW(ps, foreach=False, fused=False, **HP)
    flat_p = torch.cat([p.detach().reshape(-1) for p in ps]).clone()
    m, v = torch.zeros_like(flat_p), torch.zeros_like(flat_p)
    for step in range(1, 4):
        grads = [(torch.randn(s, generator=g) * 0.1).to(dtype) for s in shapes]
        for p, gr in zip(ps, grads):
            p.grad = gr.clone()
        opt.step()
        AO.adamw_flat_(torch.cat([x.reshape(-1) for x in grads]), flat_p, m, v, None, lr=HP["lr"], beta1=0.9, beta2=0.999, eps=HP["eps"],
                       weight_decay=HP["weight_decay"], step=step)
        want = torch.cat([p.detach().reshape(-1) for p in ps])
        assert torch.equal(flat_p, want), f"step {step}: oracle differs from torch.optim.AdamW ({dtype})"
        st = opt.state[ps[0]]
        assert torch.equal(m[: ps[0].numel()], st["exp_avg"].reshape(-1)) and torch.equal(v[: ps[0].numel()], st["exp_avg_sq"].reshape(-1))


def test_clip_coef_is_clip_grad_norm():
    g = torch.Generator().manual_seed(1)
    ps = [nn.Parameter(torch.randn(9, 7, generator=g)), nn.Parameter(torch.randn(11, generator=g))]
    for p in ps:
        p.grad = torch.randn(p.shape, generator=g) * 3
    before = [p.grad.clone() for p in ps]
    ss = sum(b.pow(2).sum() for b in before)
    total = torch.nn.utils.clip_grad_norm_(ps, 1.0)
    torch.testing.assert_close(total, ss.sqrt(), rtol=1e-6, atol=0)
    coef = AO.clip_coef(ss, 1.0)
    for p, b in zip(ps, before):
        torch.testing.assert_close(p.grad, b * coef, rtol=1e-6, atol=0)


def test_cosine_schedule_matches_transformers():
    from transformers.optimization import get_cosine_schedule_with_warmup

    from dreamllm_b200.zero import cosine_schedule_with_warmup
    p = nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=1.0)
    total, warm = 200, 7
    sched = get_cosine_schedule_with_warmup(opt, warm, total)
    for step in range(total + 5):
        assert abs(sched.get_last_lr()[0] - cosine_schedule_with_warmup(step, warm, total)) < 1e-12, step
        opt.step()
        sched.step()


# ------------------------------------------------------------------------------------------------ host logic, single process
class Net(nn.Module):
    """q/k/v-like same-shaped neighbours + odd sizes (padding) + a parameter that never gets a gradient."""

    def __init__(self):
        super().__init__()
        self.q = nn.Linear(24, 24, bias=False)
        self.k = nn.Linear(24, 24, bias=False)
        self.v = nn.Linear(24, 24, bias=False)
        self.out = nn.Linear(24, 7, bias=True)
        self.norm = nn.Parameter(torch.ones(24))
        self.unused = nn.Linear(5, 3, bias=False)

    def forward(self, x):
        h = x * self.norm
        return self.out(torch.tanh(self.q(h)) + self.k(h) * 0.5 + self.v(h))


def _net(seed=0):
    torch.manual_seed(seed)
    return Net().to(BF)


def _data():
    g = torch.Generator().manual_seed(5)
    return torch.randn(8, 24, generator=g).to(BF)


def _make(net, **kw):
    from dreamllm_b200.zero import ShardedAdamW
    kw.setdefault("update_fn", AO.adamw_flat_)
    kw.setdefault("sumsq_fn", AO.sumsq_flat)
    return ShardedAdamW(net.parameters(), bucket_cap_mb=0.001, **HP, **kw)


def test_layout_keeps_fused_rows_adjacent_and_pads():
    from dreamllm_b200.modeling_dreamllm import _fuse_rows
    from dreamllm_b200.zero import ALIGN
    net = _net()
    before = {k: v.detach().clone() for k, v in net.named_parameters()}
    opt = _make(net, max_grad_norm=0.0)
    assert len(opt.buckets) >= 2
    for k, v in net.named_parameters():
        assert torch.equal(v.detach(), before[k])                       # re-seating keeps the values ...
    for b in opt.buckets:
        assert b.padded % ALIGN == 0 and b.padded >= b.n and b.chunk == b.padded
        off = 0
        for p in b.params:                                                 # ... and puts them back to back in forward order
            assert p.data_ptr() == b.flat_param.data_ptr() + 2 * off
            off += p.numel()
    w = _fuse_rows([net.q.weight, net.k.weight, net.v.weight])             # q|k|v stayed adjacent: a view, not a re-allocation
    assert w.data_ptr() == net.q.weight.data_ptr() and w.shape == (72, 24)
    assert net.k.weight.data_ptr() == opt._bucket_of[net.k.weight].pviews[net.k.weight].data_ptr()
    opt.zero_grad()
    net(_data()).float().pow(2).mean().backward()
    opt.step()                                                             # integrity check passes
    net.k.weight.data = net.k.weight.data.clone()
    opt.zero_grad()
    net(_data()).float().pow(2).mean().backward()
    with pytest.raises(RuntimeError, match="moved out of its optimizer bucket"):
        opt.step()
    opt.reseat()
    opt.step()


@pytest.mark.parametrize("state_dtype", [BF, torch.float32])
def test_single_process_equals_torch_adamw(state_dtype):
    """world 1, no clipping: bf16 state == torch.optim.AdamW on the bf16 model bit for bit; fp32 state == AdamW on an fp32 master copy."""
    net, ref = _net(), _net()
    opt = _make(net, max_grad_norm=0.0, state_dtype=state_dtype)
    x = _data()
    if state_dtype == BF:
        ropt = torch.optim.AdamW([p for p in ref.parameters()], foreach=False, **HP)
        masters = None
    else:
        masters = [nn.Parameter(p.detach().float()) for p in ref.parameters()]
        ropt = torch.optim.AdamW(masters, foreach=False, **HP)
    for _ in range(3):
        opt.zero_grad()
        net(x).float().pow(2).mean().backward()
        opt.step()
        for p in ref.parameters():
            p.grad = None
        ref(x).float().pow(2).mean().backward()
        if masters is not None:
            for mp_, p in zip(masters, ref.parameters()):
                mp_.grad = None if p.grad is None else p.grad.float()
        ropt.step()
        if masters is not None:
            with torch.no_grad():
                for mp_, p in zip(masters, ref.parameters()):
                    p.copy_(mp_)
        for (k, a), (_, b) in zip(net.named_parameters(), ref.named_parameters()):
            assert torch.equal(a.detach(), b.detach()), k
    assert torch.equal(net.unused.weight.detach(), _net().unused.weight.detach())     # never got a gradient -> untouched (torch skips None grads)


def test_clipping_and_state_dict_round_trip():
    net, ref = _net(), _net()
    opt = _make(net, max_grad_norm=0.05, state_dtype=torch.float32)
    masters = [nn.Parameter(p.detach().float()) for p in ref.parameters()]
    ropt = torch.optim.AdamW(masters, foreach=False, **HP)
    x = _data()
    for it in range(2):
        opt.zero_grad()
        net(x).float().pow(2).mean().backward()
        norm = opt.step()
        for p in ref.parameters():
            p.grad = None
        ref(x).float().pow(2).mean().backward()
        live = []
        for mp_, p in zip(masters, ref.parameters()):
            mp_.grad = None if p.grad is None else p.grad.float()
            if mp_.grad is not None:
                live.append(mp_)
        want_norm = torch.nn.utils.clip_grad_norm_(live, 0.05)
        assert float(want_norm) > 0.05                                   # the clip is active
        torch.testing.assert_close(norm, want_norm, rtol=1e-5, atol=0)
        ropt.step()
        with torch.no_grad():
            for mp_, p in zip(masters, ref.parameters()):
                p.copy_(mp_)
        for (k, a), (_, b) in zip(net.named_parameters(), ref.named_parameters()):
            torch.testing.assert_close(a.detach().float(), b.detach().float(), rtol=2 ** -7, atol=1e-6, msg=k)   # <= 1 bf16 ulp
    sd = opt.state_dict()
    net2 = _net()
    with torch.no_grad():
        for a, b in zip(net2.parameters(), net.parameters()):
            a.copy_(b)
    opt2 = _make(net2, max_grad_norm=0.05, state_dtype=torch.float32)
    opt2.load_state_dict(sd)
    for o, n in ((opt, net), (opt2, net2)):
        o.zero_grad()
        n(x).float().pow(2).mean().backward()
        o.step()
    for a, b in zip(net.parameters(), net2.parameters()):
        assert torch.equal(a.detach(), b.detach())


# ------------------------------------------------------------------------------------------------ world_size 2 over gloo
def _worker(rank, world, port, q, done, state_dtype_name, defer=False):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    state_dtype = getattr(torch, state_dtype_name)
    net = _net()
    opt = _make(net, max_grad_norm=0.0, state_dtype=state_dtype)
    if defer:
        opt.attach(net)
    x = _data()
    norms = []
    for _ in range(3):
        opt.zero_grad()
        per = 8 // world if world in (2, 4) else 2
        net(x[rank * per:(rank + 1) * per]).float().pow(2).mean().backward()
        norms.append(float(opt.step(defer_gather=defer)))
    opt.wait_gathers()
    q.put((rank, {k: v.detach().clone() for k, v in net.named_parameters()}, opt.launched, opt.state_bytes_per_rank(), norms))
    done.wait(240)                    # the queued tensors live in this process's shared memory until the parent has received them
    dist.destroy_process_group()


def _run_two(state_dtype_name, world=2, defer=False):
    ctx = mp.get_context("spawn")
    q, done = ctx.Queue(), ctx.Event()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, done, state_dtype_name, defer)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=240) for _ in range(world)]
    finally:
        done.set()
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    assert all(p.exitcode == 0 for p in procs)
    return sorted(res, key=lambda r: r[0])


@pytest.mark.parametrize("state_dtype_name", ["bfloat16", "float32"])
def test_two_ranks_sharded_equals_single_process_on_averaged_grads(state_dtype_name):
    try:
        res = _run_two(state_dtype_name)
    except Exception:                # rendezvous port race on a loaded build box: one retry on a fresh port
        res = _run_two(state_dtype_name)
    (_, p0, launched0, bytes0, norms0), (_, p1, launched1, bytes1, norms1) = res
    for k in p0:
        assert torch.equal(p0[k], p1[k]), f"ranks diverged on {k}"          # all-gather left every rank with the same parameters
    assert norms0 == norms1
    # single-process expectation: the same class at world 1, fed the average of the two ranks' bf16 gradients
    state_dtype = getattr(torch, state_dtype_name)
    net = _net()
    opt = _make(net, max_grad_norm=0.0, state_dtype=state_dtype)
    halves = [_net(), _net()]
    x = _data()
    for _ in range(3):
        grads = []
        for r, h in enumerate(halves):
            with torch.no_grad():
                for a, b in zip(h.parameters(), net.parameters()):
                    a.copy_(b)
                    a.grad = None
            h(x[r * 4:(r + 1) * 4]).float().pow(2).mean().backward()
            grads.append([p.grad for p in h.parameters()])
        opt.zero_grad()
        for p, g0, g1 in zip(net.parameters(), *grads):
            if g0 is None and g1 is None:
                g0 = g1 = torch.zeros_like(p)                                # multi-rank buckets treat a missing grad as zero
            p.grad = (g0 / 2 + g1 / 2)
            opt._on_grad(p)
        opt.step()
    for k, v in net.named_parameters():
        assert torch.equal(v.detach(), p0[k]), k
    assert launched0 == launched1 and launched0 >= 3 * 2 * len(opt.buckets)
    full = _make(_net(), max_grad_norm=0.0, state_dtype=state_dtype).state_bytes_per_rank()
    assert bytes0 <= full // 2 + 3 * 4 * 128 * len(opt.buckets)             # each rank holds half the state (+ padding)


def test_three_ranks_uneven_padding_stay_in_lockstep():
    """world 3: bucket sizes are not multiples of the world size -> padded shards; every rank must end with identical parameters that
    moved away from the initial ones, and own a third of the optimizer state."""
    try:
        res = _run_two("float32", world=3)
    except Exception:
        res = _run_two("float32", world=3)
    ref = _net()
    base = {k: v.detach().clone() for k, v in ref.named_parameters()}
    p0 = res[0][1]
    for _, pr, launched, nbytes, norms in res[1:]:
        for k in p0:
            assert torch.equal(p0[k], pr[k]), k
        assert norms == res[0][4] and launched == res[0][2]
    assert any(not torch.equal(p0[k], base[k]) for k in p0 if k != "unused.weight")
    full = _make(_net(), max_grad_norm=0.0, state_dtype=torch.float32).state_bytes_per_rank()
    assert res[0][3] <= full // 3 + 3 * 4 * 128 * 8


def test_no_sync_accumulates_micro_batches():
    """Two micro-batches under no_sync() + one synced backward == one backward over the summed loss (world 1; the wire path is the same
    reduce-scatter as every other step)."""
    net, ref = _net(), _net()
    opt, ropt = _make(net, max_grad_norm=0.0, state_dtype=BF), _make(ref, max_grad_norm=0.0, state_dtype=BF)
    x = _data()
    for _ in range(2):
        opt.zero_grad()
        with opt.no_sync():
            net(x[:3]).float().pow(2).mean().backward()
            net(x[3:5]).float().pow(2).mean().backward()
        net(x[5:]).float().pow(2).mean().backward()
        acc = {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}
        opt.step()
        # expectation: autograd's own accumulation of the three micro-batch gradients (bf16 adds in the same order)
        ropt.zero_grad()
        for p in ref.parameters():
            p.grad = None
        for sl in (slice(0, 3), slice(3, 5), slice(5, 8)):
            ref(x[sl]).float().pow(2).mean().backward()
        for k, p in ref.named_parameters():
            if p.grad is not None:
                assert torch.equal(acc[k], p.grad), k
        ropt.step()
        for (k, a), (_, b) in zip(net.named_parameters(), ref.named_parameters()):
            assert torch.equal(a.detach(), b.detach()), k


def test_deferred_all_gather_gives_the_same_parameters():
    """step(defer_gather=True): all-gathers are waited for by forward pre-hooks (attach) instead of at the end of step() — same result."""
    try:
        plain, deferred = _run_two("float32"), _run_two("float32", defer=True)
    except Exception:
        plain, deferred = _run_two("float32"), _run_two("float32", defer=True)
    for (_, pa, *_), (_, pb, *_) in zip(plain, deferred):
        for k in pa:
            assert torch.equal(pa[k], pb[k]), k
    net = _net()
    opt = _make(net, max_grad_norm=0.0)
    with pytest.raises(RuntimeError, match="attach"):
        opt.zero_grad()
        net(_data()).float().pow(2).mean().backward()
        opt.step(defer_gather=True)


def test_decay_groups_match_transformers_get_parameter_names():
    """`decay_parameter_names` == transformers' `get_parameter_names(model, ALL_LAYERNORM_LAYERS)` minus "bias" (what the reference's
    Trainer.create_optimizer does, omni/train/trainer.py:381-446), on a model mixing nn.LayerNorm, DreamLLMRMSNorm, biases and a bare Parameter."""
    from transformers.trainer_pt_utils import get_parameter_names

    from dreamllm_b200.modeling_dreamllm import DreamLLMConfig, DreamLLMForCausalMLM, DreamLLMRMSNorm
    from dreamllm_b200.modeling_plugins import DreamEmbedding
    from dreamllm_b200.zero import decay_parameter_names, optimizer_param_groups
    m = DreamLLMForCausalMLM(DreamLLMConfig(vocab_size=64, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2))
    m.model.dream_embedding = DreamEmbedding(num_dream_queries=4, embed_hidden_size=128)
    m.extra = nn.Sequential(nn.Linear(8, 8, bias=True), nn.LayerNorm(8))
    want = [n for n in get_parameter_names(m, [nn.LayerNorm, DreamLLMRMSNorm]) if "bias" not in n]
    got = decay_parameter_names(m)
    assert sorted(got) == sorted(want)
    assert "model.layers.0.input_layernorm.weight" not in got and "model.norm.weight" not in got and "extra.0.bias" not in got
    assert "model.dream_embedding.dream_queries" in got and "model.layers.1.mlp.down_proj.weight" in got
    m.lm_head.weight.requires_grad_(False)
    groups = optimizer_param_groups(m, 0.1)
    assert groups[0]["weight_decay"] == 0.1 and groups[1]["weight_decay"] == 0.0
    n_train = sum(p.requires_grad for p in m.parameters())
    assert len(groups[0]["params"]) + len(groups[1]["params"]) == n_train
    assert all(p is not m.lm_head.weight for g in groups for p in g["params"])


def test_training_step_glue_with_groups_and_accumulation():
    from dreamllm_b200.zero import ShardedAdamW, optimizer_param_groups, training_step

    class Wrapped(nn.Module):
        def __init__(self):
            super().__init__()
            self.net = _net()

        def forward(self, x):
            from types import SimpleNamespace
            return SimpleNamespace(loss=self.net(x).float().pow(2).mean())
    torch.manual_seed(0)
    m = Wrapped()
    opt = ShardedAdamW(optimizer_param_groups(m, 0.05), lr=1e-2, max_grad_norm=1.0, bucket_cap_mb=0.001, update_fn=AO.adamw_flat_,
                       sumsq_fn=AO.sumsq_flat)
    assert {g["weight_decay"] for g in opt.param_groups} == {0.05, 0.0}
    x = _data()
    before = m.net.q.weight.detach().clone()
    l0, n0 = training_step(m, opt, dict(x=x[:4]), accumulate=True)
    assert n0 is None and torch.equal(m.net.q.weight.detach(), before)           # micro-step: no update yet
    l1, n1 = training_step(m, opt, dict(x=x[4:]))
    assert float(n1) > 0 and not torch.equal(m.net.q.weight.detach(), before)
    assert all(p.grad is None for p in m.parameters())                            # zero_grad after the step
    losses = [float(training_step(m, opt, dict(x=x))[0]) for _ in range(25)]
    assert losses[-1] < 0.5 * losses[0]


# ------------------------------------------------------------------------------------------------ ADVICE r1: ranks with different unused parameters
class BranchNet(nn.Module):
    """`proj` is only used when the batch carries "images" (stage-2 interleaved data: a text-only rank produces no gradient for the CLIP /
    SD projectors and the dream queries, modeling_plugins.py:242)."""

    def __init__(self):
        super().__init__()
        self.body = nn.Linear(24, 24, bias=False)
        self.head = nn.Linear(24, 7, bias=False)
        self.proj = nn.Linear(24, 24, bias=False)

    def forward(self, x, use_proj):
        h = torch.tanh(self.body(x))
        if use_proj:
            h = h + self.proj(x)
        return self.head(h)


def _branch_net():
    torch.manual_seed(3)
    return BranchNet().to(BF)


def _uneven_worker(rank, world, port, q, done, kind):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    net = _branch_net()
    x = _data()
    if kind == "zero":
        opt = _make(net, max_grad_norm=0.0, state_dtype=torch.float32)
        for _ in range(2):
            opt.zero_grad()
            net(x[rank * 4:(rank + 1) * 4], use_proj=(rank == 0)).float().pow(2).mean().backward()
            opt.step()
        q.put((rank, {k: v.detach().clone() for k, v in net.named_parameters()}))
    else:
        from dreamllm_b200.ddp import BucketedGradReducer
        red = BucketedGradReducer(net.parameters(), bucket_cap_mb=0.001)
        assert len(red.buckets) >= 3
        for _ in range(2):
            red.zero_grad()
            net(x[rank * 4:(rank + 1) * 4], use_proj=(rank == 0)).float().pow(2).mean().backward()
            red.finalize()
        q.put((rank, {k: v.grad.detach().clone() for k, v in net.named_parameters()}))
    done.wait(240)                    # see _worker
    dist.destroy_process_group()


def _run_uneven(kind):
    ctx = mp.get_context("spawn")
    q, done = ctx.Queue(), ctx.Event()
    port = _free_port()
    procs = [ctx.Process(target=_uneven_worker, args=(r, 2, port, q, done, kind)) for r in range(2)]
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
    return sorted(res, key=lambda r: r[0])


@pytest.mark.parametrize("kind", ["ddp", "zero"])
def test_ranks_with_different_unused_parameters_issue_matching_collectives(kind):
    """Only rank 0's batch touches `proj`.  Collectives must still pair up (bucket-order launch rule): before the fix rank 1 flushed the
    proj bucket at the end while rank 0 launched it mid-backward -> gloo 'Received data size doesn't match', NCCL hang."""
    try:
        res = _run_uneven(kind)
    except Exception:
        res = _run_uneven(kind)
    (_, a), (_, b) = res
    for k in a:
        assert torch.equal(a[k], b[k]), f"ranks diverged on {k}"
    if kind == "ddp":                         # proj's averaged gradient = rank 0's half; rank 1 contributed zeros
        net = _branch_net()
        x = _data()
        net(x[:4], use_proj=True).float().pow(2).mean().backward()
        torch.testing.assert_close(a["proj.weight"].float(), net.proj.weight.grad.float() / 2, rtol=2 ** -7, atol=1e-6)
        assert float(a["proj.weight"].float().abs().sum()) > 0
    else:
        assert not torch.equal(a["proj.weight"], _branch_net().proj.weight.detach())      # the weight moved on both ranks


def test_accumulated_gradient_survives_a_micro_batch_that_skips_the_parameter():
    """ADVICE r1 (zero.py:277): micro-step 1 (no_sync) uses `proj`, micro-step 2 (synced) is 'text-only'.  The accumulated proj gradient
    must reach the optimizer, and the bucket must be reduced exactly once."""
    net = _branch_net()
    opt = _make(net, max_grad_norm=0.0, state_dtype=torch.float32)
    x = _data()
    before = net.proj.weight.detach().clone()
    opt.zero_grad()
    with opt.no_sync():
        net(x[:4], use_proj=True).float().pow(2).mean().backward()
    g1 = net.proj.weight.grad.detach().clone()
    assert float(g1.float().abs().sum()) > 0
    net(x[4:], use_proj=False).float().pow(2).mean().backward()
    assert torch.equal(net.proj.weight.grad, g1)                       # untouched by the second micro-batch ...
    launched_before = sum(b.launched for b in opt.buckets)
    opt.step()
    assert launched_before < len(opt.buckets)                           # ... its bucket was flushed by step(), once
    assert not torch.equal(net.proj.weight.detach(), before)            # ... and it stepped the weight


def test_training_step_scales_the_loss_by_grad_accum_steps():
    """accelerate.backward / Trainer.training_step (omni/train/trainer.py:1043-1047): each micro-batch back-propagates loss / GA, so the
    accumulated gradient (hence grad_norm and the clip threshold) is the mean over micro-batches."""
    from types import SimpleNamespace

    from dreamllm_b200.zero import ShardedAdamW, training_step

    class Wrapped(nn.Module):
        def __init__(self):
            super().__init__()
            self.net = _net()

        def forward(self, x):
            return SimpleNamespace(loss=self.net(x).float().pow(2).mean())
    x = _data()
    norms, losses = {}, {}
    for ga in (1, 2):
        m = Wrapped()
        opt = ShardedAdamW(m.parameters(), lr=0.0, max_grad_norm=1e9, bucket_cap_mb=0.001, update_fn=AO.adamw_flat_, sumsq_fn=AO.sumsq_flat)
        if ga == 1:
            losses[ga], norms[ga] = training_step(m, opt, dict(x=x[:4]))
        else:
            l0, _ = training_step(m, opt, dict(x=x[:4]), accumulate=True, grad_accum_steps=2)
            l1, norms[ga] = training_step(m, opt, dict(x=x[:4]), grad_accum_steps=2)
            losses[ga] = l0 + l1
    torch.testing.assert_close(losses[2], losses[1], rtol=1e-6, atol=0)         # two half-weighted copies of the same micro-batch
    torch.testing.assert_close(norms[2], norms[1], rtol=2e-2, atol=0)           # not 2x: bf16 accumulation of two halves
