"""B200-native SD `AutoencoderKL` ENCODER (forward only; frozen tower: freeze_vae=True) for the diffusion-loss path.

Reference call site: `latents = self.vae.encode(images).latent_dist.sample() * scaling_factor`, modeling_plugins.py:511-512
(arithmetic: diffusers 0.24 AutoencoderKL, SURVEY.md Appendix A.3 / §8(f) row 1; oracle: oracle/vae_oracle.py, diffusers key names:
`encoder.*`, `quant_conv.*`).  1 116.7 GFLOP per 512x512 image — more than one UNet forward — on the same kernels as the UNet:
implicit-GEMM 3x3 convs (planes up to 512x512: the 128-pixel M tile is a row segment), GroupNorm+SiLU, GEMM epilogues; the single
512-wide attention head of the mid block runs as GEMM -> row softmax -> GEMM.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .modeling_dreamllm import _fuse_rows
from .unet import check_planes

BF16 = torch.bfloat16
SDVAE = dict(in_channels=3, latent_channels=4, block_out_channels=(128, 256, 512, 512), layers_per_block=2, norm_num_groups=32,
             scaling_factor=0.18215)


class ResnetBlock2D(nn.Module):
    def __init__(self, cin, cout, groups, eps=1e-6):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=eps)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.norm2 = nn.GroupNorm(groups, cout, eps=eps)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None


class Downsample2D(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=2, padding=0)


class Attention(nn.Module):
    def __init__(self, c, groups, eps=1e-6):
        super().__init__()
        self.group_norm = nn.GroupNorm(groups, c, eps=eps)
        self.to_q = nn.Linear(c, c)
        self.to_k = nn.Linear(c, c)
        self.to_v = nn.Linear(c, c)
        self.to_out = nn.ModuleList([nn.Linear(c, c), nn.Dropout(0.0)])


class _B(nn.Module):
    pass


class Encoder(nn.Module):
    def __init__(self, c):
        super().__init__()
        ch, G, L = c["block_out_channels"], c["norm_num_groups"], c["layers_per_block"]
        self.conv_in = nn.Conv2d(c["in_channels"], ch[0], 3, padding=1)
        self.down_blocks = nn.ModuleList()
        out = ch[0]
        for i, co in enumerate(ch):
            b = _B()
            cin, out = out, co
            b.resnets = nn.ModuleList([ResnetBlock2D(cin if j == 0 else out, out, G) for j in range(L)])
            if i < len(ch) - 1:
                b.downsamplers = nn.ModuleList([Downsample2D(out)])
            self.down_blocks.append(b)
        self.mid_block = _B()
        self.mid_block.resnets = nn.ModuleList([ResnetBlock2D(ch[-1], ch[-1], G), ResnetBlock2D(ch[-1], ch[-1], G)])
        self.mid_block.attentions = nn.ModuleList([Attention(ch[-1], G)])
        self.conv_norm_out = nn.GroupNorm(G, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], 2 * c["latent_channels"], 3, padding=1)


class AutoencoderKLEncoder(nn.Module):
    def __init__(self, cfg=None):
        super().__init__()
        c = dict(SDVAE)
        c.update(cfg or {})
        self.cfg = c
        self.encoder = Encoder(c)
        self.quant_conv = nn.Conv2d(2 * c["latent_channels"], 2 * c["latent_channels"], 1)
        self._wcache = {}

    def _conv_w(self, conv):
        key = id(conv)
        w = conv.weight
        ent = self._wcache.get(key)
        if ent is None or ent[0] != (w.data_ptr(), w._version):
            ent = ((w.data_ptr(), w._version), w.detach().permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous())
            self._wcache[key] = ent
        return ent[1]

    def _resnet(self, r, x):
        N, H, W, Cin = x.shape
        G = self.cfg["norm_num_groups"]
        h = ops.groupnorm(x, r.norm1.weight, r.norm1.bias, G, r.norm1.eps, silu=True)
        h = ops.conv3x3(h, self._conv_w(r.conv1), bias=r.conv1.bias)
        h = ops.groupnorm(h, r.norm2.weight, r.norm2.bias, G, r.norm2.eps, silu=True)
        sc = x if r.conv_shortcut is None else ops.linear(x.view(-1, Cin), r.conv_shortcut.weight.view(-1, Cin),
                                                         bias=r.conv_shortcut.bias).view(N, H, W, -1)
        return ops.conv3x3(h, self._conv_w(r.conv2), bias=r.conv2.bias, residual=sc)

    def _attention(self, a, x):
        N, H, W, C = x.shape
        S = H * W
        h = ops.groupnorm(x, a.group_norm.weight, a.group_norm.bias, self.cfg["norm_num_groups"], a.group_norm.eps, silu=False).view(N * S, C)
        wqkv = _fuse_rows([a.to_q.weight, a.to_k.weight, a.to_v.weight])
        bqkv = _fuse_rows([a.to_q.bias, a.to_k.bias, a.to_v.bias])
        qkv = ops.linear(h, wqkv, bias=bqkv).view(N, S, 3 * C)
        o = torch.empty((N, S, C), device=x.device, dtype=BF16)
        for n in range(N):                                   # one 512-wide head per image: GEMM -> row softmax -> GEMM
            q, k, v = qkv[n, :, :C], qkv[n, :, C:2 * C], qkv[n, :, 2 * C:]
            p = ops.softmax_rows_(ops.gemm(q, k), float(C) ** -0.5)       # [S, S]
            ops.gemm(p, v, b_mn=True, out=o[n])
        return ops.linear(o.view(N * S, C), a.to_out[0].weight, bias=a.to_out[0].bias, residual=x.view(N * S, C)).view(N, H, W, C)

    @torch.no_grad()
    def encode_sample(self, images, z=None, generator=None):
        """images [B,3,H,W] (any float dtype, NCHW) -> latents [B,4,H/8,W/8] fp32 = latent_dist.sample() * scaling_factor."""
        if not images.is_cuda:
            raise RuntimeError("dreamllm_b200 VAE encoder requires CUDA tensors; there is no CPU fallback")
        e = self.encoder
        B, _, H, W = images.shape
        check_planes(H, W, len(self.cfg["block_out_channels"]), f"VAE encoder planes of a {H}x{W} image")
        x = ops.conv_in(images.float().contiguous(), e.conv_in.weight, e.conv_in.bias, B)
        for b in e.down_blocks:
            for r in b.resnets:
                x = self._resnet(r, x)
            if hasattr(b, "downsamplers"):
                conv = b.downsamplers[0].conv
                N, Hh, Ww, C = x.shape
                x = ops.linear(ops.im2col_s2(x, pad=0), self._conv_w(conv), bias=conv.bias).view(N, Hh // 2, Ww // 2, -1)
        x = self._resnet(e.mid_block.resnets[0], x)
        x = self._attention(e.mid_block.attentions[0], x)
        x = self._resnet(e.mid_block.resnets[1], x)
        x = ops.groupnorm(x, e.conv_norm_out.weight, e.conv_norm_out.bias, self.cfg["norm_num_groups"], e.conv_norm_out.eps, silu=True)
        h = ops.conv_out(x, e.conv_out.weight, e.conv_out.bias)                      # [B, 8, h, w] fp32
        L = self.cfg["latent_channels"]
        if z is None:
            z = torch.randn((B, L, h.shape[2], h.shape[3]), device=h.device, dtype=torch.float32, generator=generator)
        wq = self.quant_conv.weight.view(2 * L, 2 * L)
        return ops.vae_sample(h, wq, self.quant_conv.bias, z.float().contiguous(), self.cfg["scaling_factor"])


class Upsample2D(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, padding=1)


class Decoder(nn.Module):
    def __init__(self, c):
        super().__init__()
        ch, G, L = c["block_out_channels"], c["norm_num_groups"], c["layers_per_block"]
        rev = list(reversed(ch))
        self.conv_in = nn.Conv2d(c["latent_channels"], rev[0], 3, padding=1)
        self.mid_block = _B()
        self.mid_block.resnets = nn.ModuleList([ResnetBlock2D(rev[0], rev[0], G), ResnetBlock2D(rev[0], rev[0], G)])
        self.mid_block.attentions = nn.ModuleList([Attention(rev[0], G)])
        self.up_blocks = nn.ModuleList()
        out = rev[0]
        for i, co in enumerate(rev):
            b = _B()
            cin, out = out, co
            b.resnets = nn.ModuleList([ResnetBlock2D(cin if j == 0 else out, out, G) for j in range(L + 1)])
            if i < len(ch) - 1:
                b.upsamplers = nn.ModuleList([Upsample2D(out)])
            self.up_blocks.append(b)
        self.conv_norm_out = nn.GroupNorm(G, ch[0], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[0], c["in_channels"], 3, padding=1)


class AutoencoderKLDecoder(AutoencoderKLEncoder):
    """`vae.decode(latents / scaling_factor)` (modeling_plugins.py:842; 2 514.5 GFLOP per 512x512 image, SURVEY 8(f) row 1) on the same
    kernels as the encoder.  Keys: `decoder.*`, `post_quant_conv.*` (diffusers)."""

    def __init__(self, cfg=None):
        nn.Module.__init__(self)
        c = dict(SDVAE)
        c.update(cfg or {})
        self.cfg = c
        self.decoder = Decoder(c)
        self.post_quant_conv = nn.Conv2d(c["latent_channels"], c["latent_channels"], 1)
        self._wcache = {}

    @torch.no_grad()
    def decode(self, latents):
        """latents [B,4,h,w] fp32 (scaled) -> images [B,3,8h,8w] fp32 in roughly [-1, 1]."""
        if not latents.is_cuda:
            raise RuntimeError("dreamllm_b200 VAE decoder requires CUDA tensors; there is no CPU fallback")
        d = self.decoder
        L = self.cfg["latent_channels"]
        nlev = len(self.cfg["block_out_channels"])
        check_planes(latents.shape[2] << (nlev - 1), latents.shape[3] << (nlev - 1), nlev,
                     f"VAE decoder planes of {tuple(latents.shape[2:])} latents")
        z = latents.float() / self.cfg["scaling_factor"]
        B = z.shape[0]
        # post_quant_conv (1x1, 4 -> 4) folded into conv_in's input: tiny, done as a per-pixel 4x4 matmul on the fp32 latents
        wq = self.post_quant_conv.weight.view(L, L).float()
        z = torch.einsum("oc,bchw->bohw", wq, z) + self.post_quant_conv.bias.float().view(1, L, 1, 1)
        x = ops.conv_in(z.contiguous(), d.conv_in.weight, d.conv_in.bias, B)
        x = self._resnet(d.mid_block.resnets[0], x)
        x = self._attention(d.mid_block.attentions[0], x)
        x = self._resnet(d.mid_block.resnets[1], x)
        for b in d.up_blocks:
            for r in b.resnets:
                x = self._resnet(r, x)
            if hasattr(b, "upsamplers"):
                conv = b.upsamplers[0].conv
                x = ops.conv3x3(ops.upsample2x(x), self._conv_w(conv), bias=conv.bias)
        x = ops.groupnorm(x, d.conv_norm_out.weight, d.conv_norm_out.bias, self.cfg["norm_num_groups"], d.conv_norm_out.eps, silu=True)
        return ops.conv_out(x, d.conv_out.weight, d.conv_out.bias)
