"""B200-native SD-2.1 `UNet2DConditionModel` (forward / denoising) and the CUDA-graph sampler loop.

Reference call sites: `StableDiffusionHead.pipeline`, modeling_plugins.py:672-850 — per step
`cat([latents]*2) -> scale_model_input -> unet(latent_model_input, t, encoder_hidden_states=prompt_embeds).sample -> chunk ->
eps_u + g (eps_c - eps_u) -> scheduler.step` (:809-833).  The UNet / scheduler arithmetic lives in diffusers 0.24 (not vendored);
module tree and parameter names below are diffusers' (state-dict compatible: 686 keys, 865 910 724 parameters), the restated
oracle is oracle/unet_oracle.py (SURVEY.md Appendix A.1 / A.2).

B200 design (SURVEY §8 rows U1-U6, a15, a16):
  * activations NHWC bf16; every 3x3 conv is an implicit GEMM on tcgen05 (4-D TMA im2col with zero-fill padding), 1x1 convs and all
    Linear layers are the same GEMM kernel with fused bias / time-embedding row-bias / residual epilogues;
  * self-attention (seq 4096/1024/256/64, d = 64) and cross-attention on the dream-query conditioning (kv len 64 / 77) use the tcgen05
    flash-attention kernel; the cross-attention K/V projections are timestep-invariant and computed ONCE per prompt, outside the loop;
  * GroupNorm(+SiLU), LayerNorm, GEGLU, upsample, concat are single-pass HBM-bound kernels;
  * the step (time embedding -> UNet -> fused CFG + DDIM/DDPM update) is captured once in a CUDA graph and replayed; the timestep and
    scheduler coefficients come from device tables indexed by a device-side step counter, so the host is not in the loop.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import ops
from .modeling_dreamllm import _fuse_rows

BF16 = torch.bfloat16

SD21 = dict(in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280), layers_per_block=2,
            attention_head_dim=(5, 10, 20, 20), cross_attention_dim=1024, norm_num_groups=32, norm_eps=1e-5,
            down_attn=(True, True, True, False), up_attn=(False, True, True, True))


# ------------------------------------------------------------------------------------------------ parameter containers
class TimestepEmbedding(nn.Module):
    def __init__(self, cin, cout):
        super().__init__()
        self.linear_1 = nn.Linear(cin, cout)
        self.linear_2 = nn.Linear(cout, cout)


class ResnetBlock2D(nn.Module):
    def __init__(self, cin, cout, temb, groups, eps):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=eps)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.time_emb_proj = nn.Linear(temb, cout)
        self.norm2 = nn.GroupNorm(groups, cout, eps=eps)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None


class Attention(nn.Module):
    def __init__(self, dim, heads, kv_dim=None):
        super().__init__()
        self.heads = heads
        kv_dim = dim if kv_dim is None else kv_dim
        self.to_q = nn.Linear(dim, dim, bias=False)
        self.to_k = nn.Linear(kv_dim, dim, bias=False)
        self.to_v = nn.Linear(kv_dim, dim, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(dim, dim), nn.Dropout(0.0)])


class GEGLU(nn.Module):
    def __init__(self, dim, inner):
        super().__init__()
        self.proj = nn.Linear(dim, inner * 2)


class FeedForward(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.net = nn.ModuleList([GEGLU(dim, dim * 4), nn.Dropout(0.0), nn.Linear(dim * 4, dim)])


class BasicTransformerBlock(nn.Module):
    def __init__(self, dim, heads, ctx_dim):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn1 = Attention(dim, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.attn2 = Attention(dim, heads, ctx_dim)
        self.norm3 = nn.LayerNorm(dim)
        self.ff = FeedForward(dim)


class Transformer2DModel(nn.Module):
    def __init__(self, dim, heads, ctx_dim, groups):
        super().__init__()
        self.norm = nn.GroupNorm(groups, dim, eps=1e-6)
        self.proj_in = nn.Linear(dim, dim)
        self.transformer_blocks = nn.ModuleList([BasicTransformerBlock(dim, heads, ctx_dim)])
        self.proj_out = nn.Linear(dim, dim)


class Downsample2D(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=2, padding=1)


class Upsample2D(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, padding=1)


class _Block(nn.Module):
    pass


class UNet2DConditionModel(nn.Module):
    def __init__(self, cfg=None):
        super().__init__()
        c = dict(SD21)
        c.update(cfg or {})
        self.cfg = c
        ch, heads, ctx, G, L, eps = (c["block_out_channels"], c["attention_head_dim"], c["cross_attention_dim"], c["norm_num_groups"],
                                    c["layers_per_block"], c["norm_eps"])
        for co, h in zip(ch, heads):
            if co // h != 64:
                raise ValueError("UNet attention head_dim must be 64 (SD-2.x)")
        temb = ch[0] * 4
        self.conv_in = nn.Conv2d(c["in_channels"], ch[0], 3, padding=1)
        self.time_embedding = TimestepEmbedding(ch[0], temb)
        self.down_blocks = nn.ModuleList()
        out = ch[0]
        for i, co in enumerate(ch):
            b = _Block()
            cin, out = out, co
            b.resnets = nn.ModuleList([ResnetBlock2D(cin if j == 0 else out, out, temb, G, eps) for j in range(L)])
            if c["down_attn"][i]:
                b.attentions = nn.ModuleList([Transformer2DModel(out, heads[i], ctx, G) for _ in range(L)])
            if i < len(ch) - 1:
                b.downsamplers = nn.ModuleList([Downsample2D(out)])
            self.down_blocks.append(b)
        self.mid_block = _Block()
        self.mid_block.resnets = nn.ModuleList([ResnetBlock2D(ch[-1], ch[-1], temb, G, eps), ResnetBlock2D(ch[-1], ch[-1], temb, G, eps)])
        self.mid_block.attentions = nn.ModuleList([Transformer2DModel(ch[-1], heads[-1], ctx, G)])
        self.up_blocks = nn.ModuleList()
        rev, rheads = list(reversed(ch)), list(reversed(heads))
        prev = rev[0]
        for i, co in enumerate(rev):
            b = _Block()
            skip_in = rev[min(i + 1, len(ch) - 1)]
            b.resnets = nn.ModuleList([ResnetBlock2D((prev if j == 0 else co) + (skip_in if j == L else co), co, temb, G, eps)
                                       for j in range(L + 1)])
            if c["up_attn"][i]:
                b.attentions = nn.ModuleList([Transformer2DModel(co, rheads[i], ctx, G) for _ in range(L + 1)])
            if i < len(ch) - 1:
                b.upsamplers = nn.ModuleList([Upsample2D(co)])
            prev = co
            self.up_blocks.append(b)
        self.conv_norm_out = nn.GroupNorm(G, ch[0], eps=eps)
        self.conv_out = nn.Conv2d(ch[0], c["out_channels"], 3, padding=1)
        self._wcache = {}

    # ---- weight layout caches (frozen tower: built once) ----
    def _conv_w(self, conv: nn.Conv2d):
        """[Cout, Cin, 3, 3] -> [Cout, 9*Cin] with k = (r, s, c): the implicit-GEMM / im2col K order."""
        key = id(conv)
        w = conv.weight
        ent = self._wcache.get(key)
        if ent is None or ent[0] != (w.data_ptr(), w._version):
            wk = w.detach().permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()
            ent = ((w.data_ptr(), w._version), wk)
            self._wcache[key] = ent
        return ent[1]

    def transformers(self):
        for b in list(self.down_blocks) + [self.mid_block] + list(self.up_blocks):
            if hasattr(b, "attentions"):
                for t in b.attentions:
                    yield t

    # ---- building blocks (x: NHWC bf16) ----
    def _resnet(self, r: ResnetBlock2D, x, temb_act):
        N, H, W, Cin = x.shape
        G = self.cfg["norm_num_groups"]
        h = ops.groupnorm(x, r.norm1.weight, r.norm1.bias, G, r.norm1.eps, silu=True)
        rowb = ops.linear(temb_act, r.time_emb_proj.weight, bias=r.time_emb_proj.bias)            # [N, Cout]
        h = ops.conv3x3(h, self._conv_w(r.conv1), bias=r.conv1.bias, rowbias=rowb)
        h = ops.groupnorm(h, r.norm2.weight, r.norm2.bias, G, r.norm2.eps, silu=True)
        if r.conv_shortcut is None:
            sc = x
        else:
            wsc = r.conv_shortcut.weight.view(r.conv_shortcut.weight.shape[0], Cin)
            sc = ops.linear(x.view(-1, Cin), wsc, bias=r.conv_shortcut.bias).view(N, H, W, -1)
        return ops.conv3x3(h, self._conv_w(r.conv2), bias=r.conv2.bias, residual=sc)

    def _transformer(self, t: Transformer2DModel, x, ctx_kv):
        N, H, W, C = x.shape
        T, S = N * H * W, H * W
        blk = t.transformer_blocks[0]
        nh = blk.attn1.heads
        x2 = x.view(T, C)
        h = ops.groupnorm(x, t.norm.weight, t.norm.bias, self.cfg["norm_num_groups"], t.norm.eps, silu=False).view(T, C)
        h = ops.linear(h, t.proj_in.weight, bias=t.proj_in.bias)
        # self-attention
        y = ops.layernorm_fwd(h, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps)
        wqkv = _fuse_rows([blk.attn1.to_q.weight, blk.attn1.to_k.weight, blk.attn1.to_v.weight])
        qkv = ops.linear(y, wqkv).view(N, S, 3, nh, 64)
        ao, _ = ops.attn_fwd(qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2], causal=False)
        h = ops.linear(ao.view(T, C), blk.attn1.to_out[0].weight, bias=blk.attn1.to_out[0].bias, residual=h)
        # cross-attention on the dream-query conditioning (K/V precomputed per prompt)
        y = ops.layernorm_fwd(h, blk.norm2.weight, blk.norm2.bias, blk.norm2.eps)
        q = ops.linear(y, blk.attn2.to_q.weight).view(N, S, nh, 64)
        Q = ctx_kv.shape[1]
        kv = ctx_kv.view(N, Q, 2, nh, 64)
        ao = ops.attn_fwd_cross(q, kv[:, :, 0], kv[:, :, 1])
        h = ops.linear(ao.view(T, C), blk.attn2.to_out[0].weight, bias=blk.attn2.to_out[0].bias, residual=h)
        # GEGLU feed-forward
        y = ops.layernorm_fwd(h, blk.norm3.weight, blk.norm3.bias, blk.norm3.eps)
        g = ops.linear_geglu(y, *self._geglu_w(blk.ff.net[0].proj))       # FF-in GEMM with h * gelu(gate) in its epilogue
        h = ops.linear(g, blk.ff.net[2].weight, bias=blk.ff.net[2].bias, residual=h)
        return ops.linear(h, t.proj_out.weight, bias=t.proj_out.bias, residual=x2).view(N, H, W, C)

    def _geglu_w(self, proj: nn.Linear):
        """Row-permuted copy of `GEGLU.proj` ([64 value | 64 gate] per 128 rows) for the fused epilogue; the parameter itself keeps the
        diffusers layout (state-dict compatible).  Frozen tower: built once."""
        key = ("geglu", id(proj))
        w = proj.weight
        ent = self._wcache.get(key)
        if ent is None or ent[0] != (w.data_ptr(), w._version):
            ent = ((w.data_ptr(), w._version), ops.geglu_permute(w.detach(), proj.bias.detach()))
            self._wcache[key] = ent
        return ent[1]

    @torch.no_grad()
    def precompute_cross_kv(self, encoder_hidden_states):
        """[N, Q, ctx] -> one [N, Q, 2C] K|V tensor per transformer block (timestep-invariant, SURVEY §8 row U5)."""
        N, Q, D = encoder_hidden_states.shape
        e2 = encoder_hidden_states.to(BF16).reshape(N * Q, D).contiguous()
        out = []
        for t in self.transformers():
            a = t.transformer_blocks[0].attn2
            wkv = _fuse_rows([a.to_k.weight, a.to_v.weight])
            out.append(ops.linear(e2, wkv).view(N, Q, -1))
        return out

    @torch.no_grad()
    def forward_nhwc(self, latents_nchw_f32, temb_sin, cross_kv, batch, eps_out=None):
        """latents [Bl,4,H,W] fp32 (Bl divides batch: CFG duplication); temb_sin [batch, 320] bf16 sinusoidal embedding;
        cross_kv from `precompute_cross_kv` -> eps [batch,4,H,W] fp32."""
        te = self.time_embedding
        t1 = ops.linear(temb_sin, te.linear_1.weight, bias=te.linear_1.bias, act=ops.ACT_SILU)
        temb_act = ops.linear(t1, te.linear_2.weight, bias=te.linear_2.bias, act=ops.ACT_SILU)    # silu(temb): all the resnets read
        x = ops.conv_in(latents_nchw_f32, self.conv_in.weight, self.conv_in.bias, batch)
        skips = [x]
        kv = iter(cross_kv)
        for b in self.down_blocks:
            for j, r in enumerate(b.resnets):
                x = self._resnet(r, x, temb_act)
                if hasattr(b, "attentions"):
                    x = self._transformer(b.attentions[j], x, next(kv))
                skips.append(x)
            if hasattr(b, "downsamplers"):
                conv = b.downsamplers[0].conv
                N, H, W, C = x.shape
                cols = ops.im2col_s2(x)
                x = ops.linear(cols, self._conv_w(conv), bias=conv.bias).view(N, H // 2, W // 2, -1)
                skips.append(x)
        x = self._resnet(self.mid_block.resnets[0], x, temb_act)
        x = self._transformer(self.mid_block.attentions[0], x, next(kv))
        x = self._resnet(self.mid_block.resnets[1], x, temb_act)
        for b in self.up_blocks:
            for j, r in enumerate(b.resnets):
                x = self._resnet(r, ops.concat_channels(x, skips.pop()), temb_act)
                if hasattr(b, "attentions"):
                    x = self._transformer(b.attentions[j], x, next(kv))
            if hasattr(b, "upsamplers"):
                conv = b.upsamplers[0].conv
                x = ops.conv3x3(ops.upsample2x(x), self._conv_w(conv), bias=conv.bias)
        x = ops.groupnorm(x, self.conv_norm_out.weight, self.conv_norm_out.bias, self.cfg["norm_num_groups"], self.conv_norm_out.eps, silu=True)
        return ops.conv_out(x, self.conv_out.weight, self.conv_out.bias, out=eps_out)


    # ================================================================================================ training path
    # StableDiffusionHead.forward (modeling_plugins.py:493-577) back-propagates through the FROZEN UNet into the dream-query
    # conditioning.  `forward_train` is the same forward with a tape; `backward_cond` walks it in reverse computing input
    # gradients only (conv dgrad = implicit-GEMM conv with the flipped/transposed filter, Linear dgrad = NN GEMM, GroupNorm /
    # LayerNorm / GEGLU / attention backward kernels) and returns d(loss)/d(encoder_hidden_states).
    def _conv_w_dgrad(self, conv: nn.Conv2d):
        """w2[ci, r', s', co] = w[co, ci, 2-r', 2-s'] as [Cin, 9*Cout]: dgrad(x) = conv3x3(dy, w2)."""
        key = ("dg", id(conv))
        w = conv.weight
        ent = self._wcache.get(key)
        if ent is None or ent[0] != (w.data_ptr(), w._version):
            wk = w.detach().flip(2, 3).permute(1, 2, 3, 0).reshape(w.shape[1], -1).contiguous()
            ent = ((w.data_ptr(), w._version), wk)
            self._wcache[key] = ent
        return ent[1]

    def _resnet_fwd(self, r, x, temb_act, tape):
        N, H, W, Cin = x.shape
        G = self.cfg["norm_num_groups"]
        h, st1 = ops.groupnorm(x, r.norm1.weight, r.norm1.bias, G, r.norm1.eps, silu=True, return_stats=True)
        rowb = ops.linear(temb_act, r.time_emb_proj.weight, bias=r.time_emb_proj.bias)
        c1 = ops.conv3x3(h, self._conv_w(r.conv1), bias=r.conv1.bias, rowbias=rowb)
        h, st2 = ops.groupnorm(c1, r.norm2.weight, r.norm2.bias, G, r.norm2.eps, silu=True, return_stats=True)
        if r.conv_shortcut is None:
            sc = x
        else:
            sc = ops.linear(x.view(-1, Cin), r.conv_shortcut.weight.view(-1, Cin), bias=r.conv_shortcut.bias).view(N, H, W, -1)
        out = ops.conv3x3(h, self._conv_w(r.conv2), bias=r.conv2.bias, residual=sc)
        tape.append(("res", r, x, st1, c1, st2))
        return out

    def _resnet_bwd(self, ent, dout):
        _, r, x, st1, c1, st2 = ent
        N, H, W, Cin = x.shape
        G = self.cfg["norm_num_groups"]
        dh2 = ops.conv3x3(dout, self._conv_w_dgrad(r.conv2))
        dc1 = ops.groupnorm_bwd(dh2, c1, r.norm2.weight, r.norm2.bias, st2, G, True)
        dh1 = ops.conv3x3(dc1, self._conv_w_dgrad(r.conv1))
        if r.conv_shortcut is None:
            dsc = dout
        else:
            Cout = dout.shape[-1]
            dsc = ops.linear_dgrad(dout.view(-1, Cout), r.conv_shortcut.weight.view(Cout, Cin)).view(N, H, W, Cin)
        return ops.groupnorm_bwd(dh1, x, r.norm1.weight, r.norm1.bias, st1, G, True, dres=dsc)

    def _transformer_fwd(self, t, x, ctx_kv, tape):
        N, H, W, C = x.shape
        T, S = N * H * W, H * W
        blk = t.transformer_blocks[0]
        nh = blk.attn1.heads
        x2 = x.view(T, C)
        g, st = ops.groupnorm(x, t.norm.weight, t.norm.bias, self.cfg["norm_num_groups"], t.norm.eps, silu=False, return_stats=True)
        h0 = ops.linear(g.view(T, C), t.proj_in.weight, bias=t.proj_in.bias)
        y = ops.layernorm_fwd(h0, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps)
        wqkv = _fuse_rows([blk.attn1.to_q.weight, blk.attn1.to_k.weight, blk.attn1.to_v.weight])
        qkv = ops.linear(y, wqkv).view(N, S, 3, nh, 64)
        ao1, lse1 = ops.attn_fwd(qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2], causal=False)
        h1 = ops.linear(ao1.view(T, C), blk.attn1.to_out[0].weight, bias=blk.attn1.to_out[0].bias, residual=h0)
        y = ops.layernorm_fwd(h1, blk.norm2.weight, blk.norm2.bias, blk.norm2.eps)
        q2 = ops.linear(y, blk.attn2.to_q.weight).view(N, S, nh, 64)
        Q = ctx_kv.shape[1]
        kv = ctx_kv.view(N, Q, 2, nh, 64)
        ao2, lse2 = ops.attn_fwd_cross_lse(q2, kv[:, :, 0], kv[:, :, 1])
        h2 = ops.linear(ao2.view(T, C), blk.attn2.to_out[0].weight, bias=blk.attn2.to_out[0].bias, residual=h1)
        y = ops.layernorm_fwd(h2, blk.norm3.weight, blk.norm3.bias, blk.norm3.eps)
        f = ops.linear(y, blk.ff.net[0].proj.weight, bias=blk.ff.net[0].proj.bias)
        gg = ops.geglu(f)
        h3 = ops.linear(gg, blk.ff.net[2].weight, bias=blk.ff.net[2].bias, residual=h2)
        out = ops.linear(h3, t.proj_out.weight, bias=t.proj_out.bias, residual=x2).view(N, H, W, C)
        tape.append(("tr", t, x, st, h0, qkv, ao1, lse1, h1, q2, ctx_kv, ao2, lse2, h2, f))
        return out

    def _transformer_bwd(self, ent, dout, dkv_list):
        _, t, x, st, h0, qkv, ao1, lse1, h1, q2, ctx_kv, ao2, lse2, h2, f = ent
        N, H, W, C = x.shape
        T, S = N * H * W, H * W
        blk = t.transformer_blocks[0]
        nh = blk.attn1.heads
        d2 = dout.view(T, C)
        dh3 = ops.linear_dgrad(d2, t.proj_out.weight)
        # feed-forward
        dgg = ops.linear_dgrad(dh3, blk.ff.net[2].weight)
        df = ops.geglu_bwd(dgg, f)
        dy = ops.linear_dgrad(df, blk.ff.net[0].proj.weight)
        dh2 = ops.layernorm_bwd(dy, h2, blk.norm3.weight, blk.norm3.eps, dres=dh3)
        # cross-attention
        dao2 = ops.linear_dgrad(dh2, blk.attn2.to_out[0].weight)
        Q = ctx_kv.shape[1]
        kv = ctx_kv.view(N, Q, 2, nh, 64)
        dq2 = torch.empty_like(q2)
        dkv = torch.empty_like(ctx_kv)
        dkv5 = dkv.view(N, Q, 2, nh, 64)
        ops.attn_bwd_cross(dao2.view(N, S, C), q2, kv[:, :, 0], kv[:, :, 1], ao2, lse2, dq2, dkv5[:, :, 0], dkv5[:, :, 1])
        dkv_list.append((t, dkv))
        dy = ops.linear_dgrad(dq2.view(T, C), blk.attn2.to_q.weight)
        dh1 = ops.layernorm_bwd(dy, h1, blk.norm2.weight, blk.norm2.eps, dres=dh2)
        # self-attention
        dao1 = ops.linear_dgrad(dh1, blk.attn1.to_out[0].weight)
        dqkv = torch.empty_like(qkv)
        ops.attn_bwd(dao1.view(N, S, C), qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2], ao1, lse1, dqkv[:, :, 0], dqkv[:, :, 1], dqkv[:, :, 2],
                     causal=False)
        wqkv = _fuse_rows([blk.attn1.to_q.weight, blk.attn1.to_k.weight, blk.attn1.to_v.weight])
        dy = ops.linear_dgrad(dqkv.view(T, 3 * C), wqkv)
        dh0 = ops.layernorm_bwd(dy, h0, blk.norm1.weight, blk.norm1.eps, dres=dh1)
        dg = ops.linear_dgrad(dh0, t.proj_in.weight).view(N, H, W, C)
        return ops.groupnorm_bwd(dg, x, t.norm.weight, t.norm.bias, st, self.cfg["norm_num_groups"], False, dres=dout)

    def forward_train(self, latents_nchw_f32, t_i32, encoder_hidden_states):
        """noisy latents [B,4,H,W] fp32, per-sample timesteps int32 [B], cond [B,Q,ctx] -> (eps [B,4,H,W] fp32, tape)."""
        B = latents_nchw_f32.shape[0]
        tape = []
        cond2 = encoder_hidden_states.to(BF16).reshape(-1, encoder_hidden_states.shape[-1]).contiguous()
        Q = encoder_hidden_states.shape[1]
        kvs = []
        for t in self.transformers():
            a = t.transformer_blocks[0].attn2
            kvs.append(ops.linear(cond2, _fuse_rows([a.to_k.weight, a.to_v.weight])).view(B, Q, -1))
        te = self.time_embedding
        temb_sin = ops.timestep_embedding_batch(t_i32, self.cfg["block_out_channels"][0])
        t1 = ops.linear(temb_sin, te.linear_1.weight, bias=te.linear_1.bias, act=ops.ACT_SILU)
        temb_act = ops.linear(t1, te.linear_2.weight, bias=te.linear_2.bias, act=ops.ACT_SILU)
        x = ops.conv_in(latents_nchw_f32, self.conv_in.weight, self.conv_in.bias, B)
        skips = [x]
        kv = iter(kvs)
        for b in self.down_blocks:
            for j, r in enumerate(b.resnets):
                x = self._resnet_fwd(r, x, temb_act, tape)
                if hasattr(b, "attentions"):
                    x = self._transformer_fwd(b.attentions[j], x, next(kv), tape)
                skips.append(x)
                tape.append(("skip_push",))
            if hasattr(b, "downsamplers"):
                conv = b.downsamplers[0].conv
                N, H, W, C = x.shape
                x = ops.linear(ops.im2col_s2(x), self._conv_w(conv), bias=conv.bias).view(N, H // 2, W // 2, -1)
                tape.append(("down", conv, (N, H, W, C)))
                skips.append(x)
                tape.append(("skip_push",))
        x = self._resnet_fwd(self.mid_block.resnets[0], x, temb_act, tape)
        x = self._transformer_fwd(self.mid_block.attentions[0], x, next(kv), tape)
        x = self._resnet_fwd(self.mid_block.resnets[1], x, temb_act, tape)
        for b in self.up_blocks:
            for j, r in enumerate(b.resnets):
                sk = skips.pop()
                tape.append(("cat", x.shape[-1]))
                x = self._resnet_fwd(r, ops.concat_channels(x, sk), temb_act, tape)
                if hasattr(b, "attentions"):
                    x = self._transformer_fwd(b.attentions[j], x, next(kv), tape)
            if hasattr(b, "upsamplers"):
                conv = b.upsamplers[0].conv
                x = ops.conv3x3(ops.upsample2x(x), self._conv_w(conv), bias=conv.bias)
                tape.append(("up", conv))
        xn, stn = ops.groupnorm(x, self.conv_norm_out.weight, self.conv_norm_out.bias, self.cfg["norm_num_groups"], self.conv_norm_out.eps,
                               silu=True, return_stats=True)
        tape.append(("out", x, stn))
        eps = ops.conv_out(xn, self.conv_out.weight, self.conv_out.bias)
        return eps, (tape, B, Q)

    def backward_cond(self, deps_nchw_f32, tape_pack):
        """d(loss)/d(eps) [B,4,H,W] fp32 -> d(loss)/d(encoder_hidden_states) [B,Q,ctx] bf16."""
        tape, B, Q = tape_pack
        dkv_list = []
        skip_grads = []          # gradients flowing into skip connections, LIFO mirror of the forward's stack
        ent = tape[-1]
        _, x_last, stn = ent
        C0 = x_last.shape[-1]
        dxn = ops.conv_out_bwd(deps_nchw_f32.contiguous(), self.conv_out.weight, C0)
        dx = ops.groupnorm_bwd(dxn, x_last, self.conv_norm_out.weight, self.conv_norm_out.bias, stn, self.cfg["norm_num_groups"], True)
        for ent in reversed(tape[:-1]):
            kind = ent[0]
            if kind == "res":
                dx = self._resnet_bwd(ent, dx)
            elif kind == "tr":
                dx = self._transformer_bwd(ent, dx, dkv_list)
            elif kind == "up":
                dx = ops.upsample2x_bwd(ops.conv3x3(dx, self._conv_w_dgrad(ent[1])))
            elif kind == "cat":
                dx, dsk = ops.split_channels(dx, ent[1])
                skip_grads.append(dsk)
            elif kind == "skip_push":
                # this activation was also pushed on the skip stack: add the gradient that came back through the up path
                dx = ops.add(dx, skip_grads.pop())     # LIFO: the last activation pushed was the first one popped by the up path
            elif kind == "down":
                conv, (N, H, W, C) = ent[1], ent[2]
                Cout = dx.shape[-1]
                dcols = ops.linear_dgrad(dx.reshape(-1, Cout), self._conv_w(conv))
                dx = ops.col2im_s2(dcols, N, H, W, C)
            else:
                raise RuntimeError(kind)
        # conv_in's skip (the first push) has no upstream consumer of dx: the latents need no gradient
        # cond gradient: sum over the 16 cross-attention blocks of dkv @ [Wk; Wv]
        dcond = None
        for t, dkv in dkv_list:
            a = t.transformer_blocks[0].attn2
            g = ops.linear_dgrad(dkv.view(B * Q, -1), _fuse_rows([a.to_k.weight, a.to_v.weight]))
            dcond = g if dcond is None else ops.add(dcond, g)
        return dcond.view(B, Q, -1)

    @torch.no_grad()
    def forward(self, sample, timestep, encoder_hidden_states):
        """diffusers-style entry: sample [B,4,H,W], timestep int / tensor, encoder_hidden_states [B,Q,ctx] -> eps [B,4,H,W] fp32."""
        if not sample.is_cuda:
            raise RuntimeError("dreamllm_b200 UNet requires CUDA tensors; there is no CPU fallback")
        B = sample.shape[0]
        dev = sample.device
        ts = torch.as_tensor(timestep, device=dev).reshape(-1)[:1].to(torch.int32)
        step0 = torch.zeros(1, device=dev, dtype=torch.int32)
        temb_sin = ops.timestep_embedding(ts, step0, B, self.cfg["block_out_channels"][0])
        return self.forward_nhwc(sample.float().contiguous(), temb_sin, self.precompute_cross_kv(encoder_hidden_states), B)


# ------------------------------------------------------------------------------------------------ supported image sizes
def check_planes(h: int, w: int, levels: int, what: str) -> None:
    """Raise ValueError unless every plane h / 2^i x w / 2^i (i < levels) of a UNet or VAE runs on the implicit-GEMM conv.

    The reference accepts any size divisible by 8; here every 3x3 conv is a tcgen05 implicit GEMM over 128-pixel tiles, so each plane's
    width must divide 128 or be a multiple of it and its height must fill whole tiles (`ops.conv3x3_plane_supported`).  Checked before
    anything is launched, so an unsupported size fails here and not inside a captured CUDA graph."""
    for i in range(levels):
        f = 1 << i
        if h % f or w % f or not ops.conv3x3_plane_supported(h // f, w // f):
            raise ValueError(f"{what} are not supported: the level-{i} plane is {h / f:g}x{w / f:g}, and every plane's "
                             f"width must divide 128 or be a multiple of 128, and its height a multiple of 128 / width (or divide it). "
                             f"Image sides of 256, 512 and 1024 satisfy this.")


# ------------------------------------------------------------------------------------------------ sampler
def scheduler_tables(num_inference_steps, kind="ddim", num_train=1000, beta_start=0.00085, beta_end=0.012, steps_offset=1):
    """SD-2.1-base scheduler_config (SURVEY Appendix A.2): scaled_linear betas, leading spacing, steps_offset 1, epsilon prediction.
    Returns (timesteps int32 [N], coef fp32 [N,5]) with coef = {sqrt(a_t), sqrt(1-a_t), c_x0, c_eps|c_xt, sigma}."""
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train, dtype=torch.float64) ** 2
    ac = torch.cumprod(1.0 - betas, dim=0)
    ratio = num_train // num_inference_steps
    ts = (torch.arange(num_inference_steps) * ratio).flip(0) + steps_offset
    if num_inference_steps < 1 or int(ts.max()) >= num_train:
        raise ValueError(f"num_inference_steps={num_inference_steps} with steps_offset={steps_offset} reaches timestep {int(ts.max())} "
                         f">= num_train_timesteps={num_train} (diffusers' leading spacing has the same limit)")
    coef = torch.zeros(num_inference_steps, 5, dtype=torch.float64)
    for i, t in enumerate(ts.tolist()):
        a_t = ac[t]
        tp = t - ratio
        if kind == "ddim":                      # eta = 0, set_alpha_to_one = False
            a_p = ac[tp] if tp >= 0 else ac[0]
            coef[i] = torch.tensor([a_t.sqrt(), (1 - a_t).sqrt(), a_p.sqrt(), (1 - a_p).sqrt(), 0.0])
        else:                                   # DDPM fixed_small — what the reference's sampler runs (plugins:379, :833)
            a_p = ac[tp] if tp >= 0 else torch.tensor(1.0, dtype=torch.float64)
            a_cur = a_t / a_p
            b_cur = 1 - a_cur
            var = torch.clamp((1 - a_p) / (1 - a_t) * b_cur, min=1e-20)
            coef[i] = torch.tensor([a_t.sqrt(), (1 - a_t).sqrt(), a_p.sqrt() * b_cur / (1 - a_t), a_cur.sqrt() * (1 - a_p) / (1 - a_t),
                                    var.sqrt() if t > 0 else 0.0])
    return ts.to(torch.int32), coef.to(torch.float32)


def rescale_noise_cfg(noise_cfg, noise_pred_text, guidance_rescale: float):
    """`StableDiffusionHead._rescale_noise_cfg` (modeling_plugins.py:658-669; "Common Diffusion Noise Schedules and Sample Steps are
    Flawed" §3.4): match the per-sample std of the guided prediction to the text-conditioned one, then blend by `guidance_rescale`.
    [B, 4, h, w] fp32 — a few hundred KB per step, plain torch ops inside the captured step."""
    dims = list(range(1, noise_pred_text.ndim))
    std_text = noise_pred_text.std(dim=dims, keepdim=True)
    std_cfg = noise_cfg.std(dim=dims, keepdim=True)
    return guidance_rescale * (noise_cfg * (std_text / std_cfg)) + (1 - guidance_rescale) * noise_cfg


class DenoiseLoop:
    """N-step sampler.  The step {time embedding -> UNet -> fused CFG + scheduler update -> step counter += 1} reads its timestep and
    scheduler coefficients from device tables indexed by a device-side step counter, so it is position-independent:
      * `whole_loop_graph=True` (default): ALL N steps are captured into ONE CUDA graph and `run()` is a single `graph.replay()` — the host
        is out of the loop entirely (the "CUDA-graph-captured persistent loop" of the north star; reference: the Python `for t in
        timesteps` loop of modeling_plugins.py:809-833);
      * with a `callback` (which must observe the latents between steps, :836-839) one single-step graph is replayed N times."""

    def __init__(self, unet: UNet2DConditionModel, cond, num_inference_steps=50, guidance_scale=7.5, scheduler="ddim",
                 latents=None, noise=None, height=512, width=512, use_cuda_graph=True, generator=None, guidance_rescale: float = 0.0,
                 whole_loop_graph: bool = True):
        """cond: [B, Q, ctx] projected prompt embeddings, or [2B, Q, ctx] = cat([negative, positive]) when guidance_scale > 1
        (reference order, modeling_plugins.py:774-784)."""
        check_planes(height // 8, width // 8, len(unet.cfg["block_out_channels"]), f"UNet latents of a {height}x{width} image")
        self.unet = unet
        dev = cond.device
        self.use_cfg = guidance_scale > 1.0
        self.guidance = float(guidance_scale)
        self.guidance_rescale = float(guidance_rescale)
        self.nb = cond.shape[0]
        self.B = self.nb // 2 if self.use_cfg else self.nb
        self.N = num_inference_steps
        self.mode = 0 if scheduler == "ddim" else 1
        h, w = height // 8, width // 8
        ts, coef = scheduler_tables(num_inference_steps, scheduler)
        self.timesteps, self.coef = ts.to(dev), coef.to(dev)
        self.timesteps_host = ts.tolist()
        self.step = torch.zeros(1, device=dev, dtype=torch.int32)
        if latents is None:
            latents = torch.randn((self.B, 4, h, w), generator=generator, device=dev, dtype=torch.float32)
        self.latents = latents.to(device=dev, dtype=torch.float32).clone().contiguous()        # init_noise_sigma = 1
        self.noise = None
        if self.mode == 1:
            self.noise = (torch.randn((self.N,) + tuple(self.latents.shape), generator=generator, device=dev) if noise is None
                          else noise.to(dev)).float().contiguous()
        self.cross_kv = unet.precompute_cross_kv(cond)
        self.eps = torch.empty((self.nb, 4, h, w), device=dev, dtype=torch.float32)
        self.graph = None              # single-step graph (callback path)
        self.loop_graph = None         # all N steps in one graph
        self.use_cuda_graph = use_cuda_graph
        self.whole_loop_graph = whole_loop_graph
        self._latents0 = self.latents.clone()

    def reset(self, latents=None):
        """Rewind to step 0 with the initial (or the given) latents — the captured graphs stay valid (static buffers)."""
        self.step.zero_()
        self.latents.copy_(self._latents0 if latents is None else latents.to(self.latents.dtype))

    def _capture(self, n_steps):
        lat0, st0 = self.latents.clone(), self.step.clone()
        s = torch.cuda.Stream()                      # warm up on a side stream (allocator + lazy attribute setup), then restore state
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._one_step()
        torch.cuda.current_stream().wait_stream(s)
        self.latents.copy_(lat0)
        self.step.copy_(st0)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(n_steps):
                self._one_step()
        self.latents.copy_(lat0)
        self.step.copy_(st0)
        return graph

    def _one_step(self):
        temb_sin = ops.timestep_embedding(self.timesteps, self.step, self.nb, self.unet.cfg["block_out_channels"][0])
        self.unet.forward_nhwc(self.latents, temb_sin, self.cross_kv, self.nb, eps_out=self.eps)
        if self.use_cfg and self.guidance_rescale > 0.0:          # (:826-831) guided prediction rescaled before the scheduler update
            eu, ec = self.eps[: self.B], self.eps[self.B:]
            self.eps[: self.B].copy_(rescale_noise_cfg(eu + self.guidance * (ec - eu), ec, self.guidance_rescale))
            ops.sampler_step_(self.eps, self.latents, self.coef, self.step, 1.0, False, self.mode, self.noise)
            return
        ops.sampler_step_(self.eps, self.latents, self.coef, self.step, self.guidance, self.use_cfg, self.mode, self.noise)

    @torch.no_grad()
    def run(self, callback=None, callback_steps: int = 1):
        """`callback(i, t, latents)` every `callback_steps` steps, between graph replays (reference :836-839)."""
        def report(i):
            if callback is not None and i % callback_steps == 0:
                callback(i, self.timesteps_host[i], self.latents)

        if not self.use_cuda_graph:
            for i in range(self.N):
                self._one_step()
                report(i)
            return self.latents
        if self.whole_loop_graph and callback is None:
            if self.loop_graph is None:
                self.loop_graph = self._capture(self.N)
            self.loop_graph.replay()
            return self.latents
        if self.graph is None:
            self.graph = self._capture(1)
        for i in range(self.N):
            self.graph.replay()
            report(i)
        return self.latents
