"""Attention at the shapes the diffusion side and the C2 decoder run, against the eager core of test_attn_gpu.py::_ref_core restated on
the GPU in float64 (softmax(q k^T / sqrt(d)) v, causal positions masked out), checked per (batch, head) at the worst element.

* UNet self-attention (d = 64, non-causal) at the four UNet planes and at the C4 size (32 images of 64^2: many items per persistent CTA);
* cross-attention on the dream queries / prompt (Skv = 1, 7, 64, 77: all shorter than one 128-key tile) through attn_fwd_cross_lse /
  attn_bwd_cross, every (batch, head);
* the d = 128 causal backward at the C2 shape (B = 8, S = 2048, 32 heads; about 14 items per persistent CTA).

Bounds: lse (natural log of sum exp(scale * q.k), the kernel's convention) within 1e-4 * (1 + |lse|) (fp32 softmax statistics);
out, dq, dk, dv within 2x the worst error of the same eager core run in bf16 (the reference's own bf16 path), + 1e-4 absolute.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
F64 = torch.float64
DEV = "cuda"


def _core(q, k, v, causal):
    """q [Sq, d], k / v [Skv, d] in one dtype -> (out, lse).  Eager math as _ref_core: scores in the input dtype, fp32 softmax (float64
    when the inputs are float64) cast back, P V in the input dtype."""
    dt = q.dtype
    s = (q @ k.t()) / math.sqrt(q.shape[-1])
    if causal:
        s = s.masked_fill(torch.ones(s.shape, dtype=torch.bool, device=s.device).triu(1), float("-inf"))
    lse = torch.logsumexp(s.to(F64), dim=-1)
    p = torch.softmax(s, dim=-1, dtype=F64 if dt == F64 else torch.float32).to(dt)
    return p @ v, lse


def _grads(q, k, v, dout, causal, dt):
    qq, kk, vv = (t.to(dt, copy=True).requires_grad_(True) for t in (q, k, v))
    o, lse = _core(qq, kk, vv, causal)
    o.backward(dout.to(dt))
    return o.detach(), lse, qq.grad, kk.grad, vv.grad


def _worst(got, ref, yard, what):
    e_o = float((got.to(F64) - ref).abs().max())
    e_r = float((yard.to(F64) - ref).abs().max())
    # + 1e-4: where the exact answer is 0 (dk with a single key) the bf16 eager path is exact too, while any fp32 kernel is not
    assert e_o <= 2.0 * e_r + 1e-4, f"{what}: worst error ours {e_o:.4g} vs eager bf16 {e_r:.4g}"


def _check_head(what, q, k, v, dout, out, lse, dq, dk, dv, causal, c2_bound=False):
    """one (b, h): q [Sq, d] ... as bf16 device tensors; out / lse / dq / dk / dv the kernel's slices for that head"""
    o64, l64, dq64, dk64, dv64 = _grads(q, k, v, dout, causal, F64)
    ob, _, dqb, dkb, dvb = _grads(q, k, v, dout, causal, BF)
    err = (lse.to(F64) - l64).abs()
    assert bool((err <= 1e-4 * (1 + l64.abs())).all()), f"{what} lse: worst {float(err.max()):.3g}"
    _worst(out, o64, ob, f"{what} out")
    for name, g, r, y in (("dq", dq, dq64, dqb), ("dk", dk, dk64, dkb), ("dv", dv, dv64, dvb)):
        _worst(g, r, y, f"{what} {name}")
        if c2_bound:      # test_attn_gpu.py's bound, per head
            e = (g.to(F64) - r).abs()
            scale = float(r.abs().max())
            assert float(e.max()) < 3e-2 * scale + 1e-3, f"{what} {name}: max err {float(e.max())} vs scale {scale}"
            e_r = float((y.to(F64) - r).abs().mean())
            assert float(e.mean()) <= 1.5 * e_r + 1e-5 * scale, f"{what} {name}: ours {float(e.mean()):.3e} vs eager bf16 {e_r:.3e}"


def _self_attn(N, S, nh, d, causal, pairs, seed, c2_bound=False):
    from dreamllm_b200 import ops
    g = torch.Generator(device=DEV).manual_seed(seed)
    qkv = torch.randn((N, S, 3, nh, d), generator=g, device=DEV).to(BF)
    dout = (torch.randn((N, S, nh * d), generator=g, device=DEV) * 0.5).to(BF)
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    out, lse = ops.attn_fwd(q, k, v, causal=causal)
    dqkv = torch.zeros_like(qkv)
    ops.attn_bwd(dout, q, k, v, out, lse, dqkv[:, :, 0], dqkv[:, :, 1], dqkv[:, :, 2], causal=causal)
    torch.cuda.synchronize()
    for b, h in pairs:
        sl = slice(h * d, (h + 1) * d)
        _check_head(f"self N={N} S={S} nh={nh} d={d} (b={b}, h={h})", q[b, :, h], k[b, :, h], v[b, :, h], dout[b, :, sl],
                    out[b, :, sl], lse[b, h], dqkv[b, :, 0, h], dqkv[b, :, 1, h], dqkv[b, :, 2, h], causal, c2_bound)


@pytest.mark.parametrize("N,S,nh", [(4, 4096, 5), (4, 1024, 10), (4, 256, 20), (4, 64, 20), (32, 4096, 5)])
def test_unet_self_attention_d64_vs_fp64(N, S, nh):
    _self_attn(N, S, nh, 64, False, [(0, 0), (N // 2, nh // 2), (N - 1, nh - 1)], seed=S + nh + N)


def test_c2_causal_d128_backward_vs_fp64():
    _self_attn(8, 2048, 32, 128, True, [(0, 0), (3, 17), (7, 31)], seed=2048, c2_bound=True)


@pytest.mark.parametrize("Skv", [1, 7, 64, 77])
@pytest.mark.parametrize("B,Sq,nh", [(2, 1024, 10), (2, 4096, 5)])
def test_cross_attention_vs_fp64(B, Sq, nh, Skv):
    """every (b, h): the keys are fewer than one 128-key tile, so the tail masking decides everything"""
    from dreamllm_b200 import ops
    d = 64
    g = torch.Generator(device=DEV).manual_seed(Sq + Skv)
    q = torch.randn((B, Sq, nh, d), generator=g, device=DEV).to(BF)
    kv = torch.randn((B, Skv, 2, nh, d), generator=g, device=DEV).to(BF)
    dout = (torch.randn((B, Sq, nh * d), generator=g, device=DEV) * 0.5).to(BF)
    out, lse = ops.attn_fwd_cross_lse(q, kv[:, :, 0], kv[:, :, 1])
    assert torch.equal(ops.attn_fwd_cross(q, kv[:, :, 0], kv[:, :, 1]), out)
    dq = torch.empty_like(q)
    dkv = torch.zeros_like(kv)
    ops.attn_bwd_cross(dout, q, kv[:, :, 0], kv[:, :, 1], out, lse, dq, dkv[:, :, 0], dkv[:, :, 1])
    torch.cuda.synchronize()
    for b in range(B):
        for h in range(nh):
            sl = slice(h * d, (h + 1) * d)
            _check_head(f"cross Sq={Sq} Skv={Skv} (b={b}, h={h})", q[b, :, h], kv[b, :, 0, h], kv[b, :, 1, h], dout[b, :, sl],
                        out[b, :, sl], lse[b, h], dq[b, :, h], dkv[b, :, 0, h], dkv[b, :, 1, h], False)
