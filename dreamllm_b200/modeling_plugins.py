"""B200-native mirror of `omni/models/dreamllm/modeling_plugins.py` (plugin ABCs :32-112, DreamEmbedding :116-181,
CLIPVisionEmbedding :184-331) plus the index plumbing of the embedding splice / conditioning gather
(modeling_dreamllm.py:1082-1141, :1401-1418).

Plugin contract kept: `plugin_type`, `processor`, `config`, `embed_len`, `embed_dim`, `save_model(dir)`, `load_model(dir)`,
`forward`, `fsdp_ignored_modules()`; attribute names `clip_vision_model`, `projector`, `dream_queries`; save files
`clip_vision_embedding.bin`, `dream_embedding.bin`.  `StableDiffusionHead` (UNet/VAE) is the next row (DESIGN.md §1).
"""
from __future__ import annotations

import os
from abc import ABC, abstractmethod
from dataclasses import dataclass

import torch
import torch.nn as nn

from . import ops
from .clip_vision import CLIPVisionConfigLite, CLIPVisionModel
from .projector import build_projector

BF16 = torch.bfloat16


class PluginBase(ABC, nn.Module):
    initializer_range: float = 0.02
    plugin_type: str | None = None

    def _init_weights(self, module):
        std = self.initializer_range
        if isinstance(module, nn.Linear):
            module.weight.data.normal_(mean=0.0, std=std)
            if module.bias is not None:
                module.bias.data.zero_()
        elif isinstance(module, nn.Embedding):
            module.weight.data.normal_(mean=0.0, std=std)
        elif isinstance(module, nn.Parameter):
            module.data.normal_(mean=0.0, std=std)
        elif isinstance(module, nn.Module):
            for m in module.modules():
                if isinstance(m, nn.Linear):
                    self._init_weights(m)

    @property
    def device(self):
        return next(self.parameters()).device

    @property
    def dtype(self):
        return next(self.parameters()).dtype

    def fsdp_ignored_modules(self) -> list:
        return []

    @property
    @abstractmethod
    def processor(self):
        pass

    @property
    @abstractmethod
    def config(self):
        pass

    @abstractmethod
    def save_model(self, output_dir: str):
        pass

    @abstractmethod
    def load_model(self, output_dir: str):
        pass

    @abstractmethod
    def forward(self):
        pass


class MultimodalEmbedding(PluginBase):
    plugin_type = "embedding"

    @property
    @abstractmethod
    def embed_len(self):
        pass

    @property
    @abstractmethod
    def embed_dim(self):
        pass


class MultimodalHead(PluginBase):
    plugin_type = "head"

    @abstractmethod
    @torch.no_grad()
    def pipeline(self):
        pass


class DreamEmbedding(MultimodalEmbedding):
    def __init__(self, pretrained_model_name_or_path: str | None = None, num_dream_queries: int = 64,
                 embed_hidden_size: int = 4096, freeze_dream_queries: bool = False):
        super().__init__()
        self.save_model_name = "dream_embedding"
        self.pretrained_model_name_or_path = pretrained_model_name_or_path
        self.num_dream_queries = num_dream_queries
        self.embed_hidden_size = embed_hidden_size
        self.freeze_dream_queries = freeze_dream_queries
        self.dream_queries = nn.Parameter(torch.zeros(1, num_dream_queries, embed_hidden_size))
        self._init_weights(self.dream_queries)
        if pretrained_model_name_or_path is not None:
            self.load_model(pretrained_model_name_or_path)
        self.dream_queries.requires_grad_(not freeze_dream_queries)

    def fsdp_ignored_modules(self) -> list:
        return [self] if self.freeze_dream_queries else []

    @property
    def processor(self):
        return None

    @property
    def embed_len(self):
        return self.num_dream_queries

    @property
    def embed_dim(self):
        return self.embed_hidden_size

    @property
    def config(self):
        return dict(pretrained_model_name_or_path=self.pretrained_model_name_or_path, num_dream_queries=self.num_dream_queries,
                    embed_len=self.embed_len, embed_dim=self.embed_dim, freeze_dream_queries=self.freeze_dream_queries)

    def save_model(self, output_dir: str):
        torch.save(self.state_dict(), os.path.join(output_dir, f"{self.save_model_name}.bin"))

    def load_model(self, output_dir: str):
        f = os.path.join(output_dir, f"{self.save_model_name}.bin")
        if os.path.isfile(f):
            self.load_state_dict(torch.load(f, map_location="cpu", weights_only=True))

    def forward(self, batch_size: int = 1):
        return self.dream_queries.repeat(batch_size, 1, 1)


class CLIPVisionEmbedding(MultimodalEmbedding):
    """`clip_vision_model_name_or_path` may be a checkpoint directory (weights are read through transformers and loaded
    into the native tower — identical state-dict keys) or a dict / CLIPVisionConfig with the architecture for random init
    (no checkpoints exist in the build sandbox)."""

    def __init__(self, clip_vision_model_name_or_path, projector_type: str = "linear", projector_depth: int = 1,
                 projector_name_or_path: str = None, pretrained_model_name_or_path: str | None = None,
                 use_additional_post_layernorm: bool = False, select_layer: int = -2, embed_hidden_size: int = 4096,
                 freeze_clip_vision_model: bool = True, freeze_embedding_layers: bool = True, freeze_projector: bool = False,
                 local_files_only: bool = False):
        super().__init__()
        self.save_model_name = "clip_vision_embedding"
        self.clip_vision_model_name_or_path = clip_vision_model_name_or_path
        self.projector_type = projector_type
        self.projector_depth = projector_depth
        self.projector_name_or_path = projector_name_or_path
        self.pretrained_model_name_or_path = pretrained_model_name_or_path
        self.use_additional_post_layernorm = use_additional_post_layernorm
        self.select_layer = select_layer
        self.embed_hidden_size = embed_hidden_size
        self.freeze_clip_vision_model = freeze_clip_vision_model
        self.freeze_embedding_layers = freeze_embedding_layers
        self.freeze_projector = freeze_projector
        if use_additional_post_layernorm:
            raise ValueError("use_additional_post_layernorm=True is not used by any shipped config and is not built")
        if not freeze_clip_vision_model:
            raise ValueError("the native CLIP tower is forward-only: freeze_clip_vision_model must be True "
                             "(projects/dreamllm/configs/common.py:35)")

        src = clip_vision_model_name_or_path
        if isinstance(src, str):
            from transformers import CLIPVisionModel as HFCLIP
            hf = HFCLIP.from_pretrained(src, local_files_only=local_files_only)
            cfg = CLIPVisionConfigLite(**{k: getattr(hf.config, k) for k in
                                          ("hidden_size", "intermediate_size", "num_hidden_layers", "num_attention_heads", "image_size",
                                           "patch_size", "layer_norm_eps", "hidden_act", "num_channels")})
            self.clip_vision_model = CLIPVisionModel(cfg)
            self.clip_vision_model.load_state_dict(hf.state_dict())
        else:
            cfg = src if isinstance(src, CLIPVisionConfigLite) else CLIPVisionConfigLite(**(src if isinstance(src, dict) else src.to_dict()))
            self.clip_vision_model = CLIPVisionModel(cfg)
        self._processor = None

        projector_cfg = dict(projector=projector_type, freeze_projector=freeze_projector, depth=projector_depth,
                             save_model_name=self.save_model_name, model_name_or_path=None)
        self.projector = build_projector(projector_cfg, in_hidden_size=cfg.hidden_size, out_hidden_size=embed_hidden_size, bias=True)
        self._init_weights(self.projector)
        self.post_layernorm = nn.Identity()
        self.image_embed_len = (cfg.image_size // cfg.patch_size) ** 2
        if pretrained_model_name_or_path is not None:
            self.load_model(pretrained_model_name_or_path)
        self.projector.load_model(projector_name_or_path)
        self.clip_vision_model.requires_grad_(False)
        self.projector.requires_grad_(not freeze_projector)

    @property
    def processor(self):
        if self._processor is None:
            from transformers import CLIPImageProcessor
            r = self.clip_vision_model.config.image_size
            self._processor = CLIPImageProcessor(size={"shortest_edge": r}, crop_size={"height": r, "width": r})
        return self._processor

    @property
    def embed_len(self):
        return self.image_embed_len

    @property
    def embed_dim(self):
        return self.embed_hidden_size

    @property
    def config(self) -> dict:
        return dict(clip_vision_model_name_or_path=self.clip_vision_model_name_or_path,
                    clip_vision_model_config=self.clip_vision_model.config.to_dict(),
                    pretrained_model_name_or_path=self.pretrained_model_name_or_path, select_layer=self.select_layer,
                    embed_len=self.embed_len, embed_dim=self.embed_dim, freeze_clip_vision_model=self.freeze_clip_vision_model,
                    freeze_embedding_layers=self.freeze_embedding_layers, freeze_projector=self.freeze_projector)

    def fsdp_ignored_modules(self) -> list:
        out = [self.clip_vision_model]
        if self.freeze_projector:
            out.append(self.projector)
        return out

    def save_model(self, output_dir: str):
        torch.save(self.state_dict(), os.path.join(output_dir, f"{self.save_model_name}.bin"))

    def load_model(self, output_dir: str):
        f = os.path.join(output_dir, f"{self.save_model_name}.bin")
        if os.path.isfile(f):
            self.load_state_dict(torch.load(f, map_location="cpu", weights_only=True))

    def forward(self, images: torch.Tensor | None = None):
        """[Ni,3,R,R] -> [Ni,P,H].  `images=None` returns None: the reference's dummy CLIP pass on a zero image (:316-319,
        :328-329) only exists to satisfy DDP's unused-parameter check, which our reducer does not need."""
        if images is None:
            return None
        hidden_state = self.clip_vision_model.hidden_state(images, self.select_layer)
        image_features = hidden_state[:, 1:]
        image_embeds = self.projector(image_features)[-1]
        return self.post_layernorm(image_embeds)


# ------------------------------------------------------------------------------------------------ splice plumbing
@dataclass
class SplicePlan:
    """Host-built index maps for one batch (all int32, on device).  Built once per batch from input_ids — this is what
    SURVEY §8(f) row 3 moves into the collator; it replaces the per-sample torch.where / torch.cat loops and their host
    syncs (modeling_dreamllm.py:1082-1141)."""
    img_dst: torch.Tensor      # rows of [B*S] that receive image features
    img_src: torch.Tensor      # rows of [Ni*P]
    dq_dst: torch.Tensor       # rows of [B*S] that receive dream queries
    dq_src: torch.Tensor       # rows of [Q]
    dq_seg: torch.Tensor       # CSR over query index -> positions in dq_rows  (gradient of the broadcast)
    dq_rows: torch.Tensor
    cond_rows: torch.Tensor    # rows of [B*S] gathered as SD conditioning, [Nd*Q]
    n_images_used: int
    n_dreams: int

    _FIELDS = ("img_dst", "img_src", "dq_dst", "dq_src", "dq_seg", "dq_rows", "cond_rows")

    def to(self, device, non_blocking: bool = True) -> "SplicePlan":
        """Host plan (built by the collator in a dataloader worker, ideally pinned) -> device plan; async H2D, no sync."""
        return SplicePlan(*[getattr(self, f).to(device, non_blocking=non_blocking) for f in self._FIELDS], self.n_images_used, self.n_dreams)

    def pin_memory(self) -> "SplicePlan":
        return SplicePlan(*[getattr(self, f).pin_memory() for f in self._FIELDS], self.n_images_used, self.n_dreams)

    @property
    def device(self):
        return self.img_dst.device


def build_splice_plan(input_ids_cpu: torch.Tensor, image_start_id: int, dream_start_id: int, P: int, Q: int, n_images: int,
                      n_dream_images: int | None, device) -> SplicePlan:
    """Pure host integer bookkeeping, semantics of the reference loops:
      * dream queries: for every <dream_start> at (b, p): rows [p+1, p+1+Q) <- dream_queries        (:1082-1099)
      * images: the j-th <im_start> counted globally in batch-major order, while j < n_images: rows [p+1, p+1+P)
        <- image_features[j]                                                                         (:1104-1141)
      * conditioning gather: for every <dream_start> in batch-major order until n_dream_images: rows [p+1, p+1+Q)  (:1401-1418)
    """
    ids = input_ids_cpu
    assert ids.device.type == "cpu" and ids.dim() == 2
    B, S = ids.shape
    flat = ids.reshape(-1)
    ar = torch.arange(B * S)
    img_pos = ar[flat == image_start_id][:max(n_images, 0)] if n_images else ar[:0]
    dq_pos = ar[flat == dream_start_id]
    for pos, L in ((img_pos, P), (dq_pos, Q)):
        if pos.numel():
            assert int(((pos % S) + L + 1).max()) <= S, "span runs past the end of the sequence (reference assert :1126)"
    img_dst = (img_pos[:, None] + 1 + torch.arange(P)[None]).reshape(-1)
    img_src = torch.arange(img_pos.numel() * P)
    dq_dst = (dq_pos[:, None] + 1 + torch.arange(Q)[None]).reshape(-1)
    dq_src = torch.arange(Q).repeat(dq_pos.numel())
    K = dq_pos.numel()
    dq_seg = torch.arange(Q + 1) * K
    dq_rows = (dq_pos[None, :] + 1 + torch.arange(Q)[:, None]).reshape(-1)          # query-major
    nd = K if n_dream_images is None else min(K, n_dream_images)
    cond_rows = (dq_pos[:nd, None] + 1 + torch.arange(Q)[None]).reshape(-1)
    to = lambda t: t.to(torch.int32).to(device, non_blocking=True)
    return SplicePlan(to(img_dst), to(img_src), to(dq_dst), to(dq_src), to(dq_seg), to(dq_rows), to(cond_rows),
                      int(img_pos.numel()), int(nd))


class _SpliceFn(torch.autograd.Function):
    """inputs_embeds with image-feature / dream-query rows written in (bit-exact row copies); backward routes row
    gradients back (token-embedding grads are zero at replaced positions, exactly as torch.cat drops them)."""

    @staticmethod
    def forward(ctx, embeds, image_features, dream_queries, plan: SplicePlan):
        B, S, H = embeds.shape
        out = embeds.reshape(B * S, H).clone()
        if image_features is not None and plan.img_dst.numel():
            ops.copy_rows_(out, plan.img_dst, image_features.reshape(-1, H).contiguous(), plan.img_src)
        if dream_queries is not None and plan.dq_dst.numel():
            ops.copy_rows_(out, plan.dq_dst, dream_queries.reshape(-1, H).contiguous(), plan.dq_src)
        ctx.plan = plan
        ctx.shapes = (None if image_features is None else image_features.shape, None if dream_queries is None else dream_queries.shape)
        return out.view(B, S, H)

    @staticmethod
    def backward(ctx, dy):
        plan = ctx.plan
        B, S, H = dy.shape
        dy2 = dy.reshape(B * S, H).contiguous()
        d_img = d_dq = None
        img_shape, dq_shape = ctx.shapes
        if img_shape is not None and ctx.needs_input_grad[1]:
            d_img = torch.zeros(img_shape, device=dy.device, dtype=dy.dtype)
            if plan.img_dst.numel():
                ops.copy_rows_(d_img.view(-1, H), plan.img_src, dy2, plan.img_dst)
        if dq_shape is not None and ctx.needs_input_grad[2]:
            if plan.dq_dst.numel():
                d_dq = ops.segment_sum_rows(dy2, plan.dq_seg, plan.dq_rows, dq_shape[-2]).view(dq_shape)
            else:
                d_dq = torch.zeros(dq_shape, device=dy.device, dtype=dy.dtype)
        d_emb = None
        if ctx.needs_input_grad[0]:
            d_emb = dy2.clone()
            if plan.img_dst.numel():
                ops.zero_rows_(d_emb, plan.img_dst)
            if plan.dq_dst.numel():
                ops.zero_rows_(d_emb, plan.dq_dst)
            d_emb = d_emb.view(B, S, H)
        return d_emb, d_img, d_dq, None


class _GatherRowsFn(torch.autograd.Function):
    """out[r] = x2d[rows[r]] (unique rows) — the dream-query conditioning gather (:1401-1418)."""

    @staticmethod
    def forward(ctx, x, rows):
        H = x.shape[-1]
        x2 = x.reshape(-1, H).contiguous()
        out = torch.empty((rows.numel(), H), device=x.device, dtype=x.dtype)
        ident = torch.arange(rows.numel(), device=x.device, dtype=torch.int32)
        ops.copy_rows_(out, ident, x2, rows)
        ctx.save_for_backward(rows, ident)
        ctx.shape = x.shape
        return out

    @staticmethod
    def backward(ctx, dy):
        rows, ident = ctx.saved_tensors
        H = dy.shape[-1]
        dx = torch.zeros(ctx.shape, device=dy.device, dtype=dy.dtype)
        ops.copy_rows_(dx.view(-1, H), rows, dy.contiguous(), ident)
        return dx, None


def splice_embeddings(embeds, image_features, dream_queries, plan):
    return _SpliceFn.apply(embeds, image_features, dream_queries, plan)


def gather_rows(x, rows):
    return _GatherRowsFn.apply(x, rows)


# ------------------------------------------------------------------------------------------------ StableDiffusionHead
class _DiffusionLossFn(torch.autograd.Function):
    """loss = mse(unet(noisy, t, cond), target) — plain mean (:559) or min-SNR weighted (:561-572) when `snr` = (alphas_cumprod, gamma).
    The UNet is frozen, so the only gradient is d(loss)/d(cond); it is computed eagerly (forward tape -> dgrad-only backward) so the
    UNet activations are freed before the LLM backward starts."""

    @staticmethod
    def forward(ctx, cond, unet, noisy, t32, target, snr=None):
        need = ctx.needs_input_grad[0]          # (grad mode is off inside Function.forward; ask autograd instead)

        def mse(eps):
            if snr is None:
                return ops.mse_fwd_bwd(eps, target)
            return ops.mse_minsnr_fwd_bwd(eps, target, t32, snr[0], snr[1])

        with torch.no_grad():
            if need:
                eps, tape = unet.forward_train(noisy, t32, cond)
                loss, deps = mse(eps)
                dcond = unet.backward_cond(deps, tape).to(cond.dtype)
                del tape
                ctx.save_for_backward(dcond)
            else:
                eps, _ = unet.forward_train(noisy, t32, cond)
                loss, _ = mse(eps)
        ctx.has_grad = need
        return loss

    @staticmethod
    def backward(ctx, g):
        if not ctx.has_grad:
            return None, None, None, None, None, None
        (dcond,) = ctx.saved_tensors
        return dcond * g.to(dcond.dtype), None, None, None, None, None


class _CfgDropFn(torch.autograd.Function):
    """Classifier-free-guidance dropout of the conditioning (reference :539-543): sample b takes `u[b]` where mask[b] == 1, else
    `enc[b]`.  The reference writes it as (1 - mask) * enc + mask * u with a {0,1} mask, which is exactly a per-sample row select, so
    it is done with bit-exact row copies; `u` may be [1, Q, H] (the null-prompt pass before its `.repeat`, :1438-1439) or [B, Q, H].
    Backward: enc gets dy on kept samples / 0 on dropped ones; u gets dy of the dropped samples (summed when u is broadcast)."""

    @staticmethod
    def forward(ctx, enc, u, drop_mask_cpu):
        B, Q, H = enc.shape
        assert u.shape[1:] == (Q, H) and u.shape[0] in (1, B), (u.shape, enc.shape)
        dropped = [b for b in range(B) if bool(drop_mask_cpu[b])]
        out = enc.reshape(B * Q, H).clone()
        ctx.meta = (B, Q, H, u.shape[0], len(dropped))
        if dropped:
            dev = enc.device
            q = torch.arange(Q)
            dst = torch.cat([b * Q + q for b in dropped])
            src = torch.cat([(b if u.shape[0] == B else 0) * Q + q for b in dropped])
            K = len(dropped)
            seg = torch.arange(Q + 1) * K                                                   # query-major CSR for the broadcast sum
            rows = (torch.tensor(dropped)[None, :] * Q + q[:, None]).reshape(-1)
            to = lambda t: t.to(torch.int32).to(dev)
            dst, src, seg, rows = to(dst), to(src), to(seg), to(rows)
            ops.copy_rows_(out, dst, u.reshape(-1, H).contiguous(), src)
            ctx.save_for_backward(dst, src, seg, rows)
        return out.view(B, Q, H)

    @staticmethod
    def backward(ctx, dy):
        B, Q, H, Bu, K = ctx.meta
        dy2 = dy.reshape(B * Q, H).contiguous()
        d_enc = d_u = None
        if K == 0:
            if ctx.needs_input_grad[0]:
                d_enc = dy
            if ctx.needs_input_grad[1]:
                d_u = torch.zeros((Bu, Q, H), device=dy.device, dtype=dy.dtype)
            return d_enc, d_u, None
        dst, src, seg, rows = ctx.saved_tensors
        if ctx.needs_input_grad[0]:
            d_enc = ops.zero_rows_(dy2.clone(), dst).view(B, Q, H)
        if ctx.needs_input_grad[1]:
            if Bu == 1:
                d_u = ops.segment_sum_rows(dy2, seg, rows, Q).view(1, Q, H).to(dy.dtype)
            else:
                d_u = torch.zeros((B * Q, H), device=dy.device, dtype=dy.dtype)
                ops.copy_rows_(d_u, src, dy2, dst)
                d_u = d_u.view(B, Q, H)
        return d_enc, d_u, None


def numpy_to_pil(images):
    """[B, H, W, 3] floats in [0, 1] -> list of PIL images (diffusers `VaeImageProcessor.numpy_to_pil`: x255, round, uint8)."""
    from PIL import Image
    arr = (images * 255).round().astype("uint8")
    return [Image.fromarray(a) for a in arr]


class StableDiffusionHead(MultimodalHead):
    """Mirror of reference `StableDiffusionHead` (modeling_plugins.py:335-850): same constructor arguments, `projector` /
    `unet` attribute names (state-dict keys `projector.projector.weight`, `unet.*`), `pipeline(...)` signature.

    Built: the training `forward` (:493-577: VAE encode -> add_noise -> UNet fwd + dgrad-only backward -> MSE) and the sampler
    (`pipeline`, :672-850) on the native UNet with a CUDA-graph loop, `output_type="latent"`.
    `output_type` "latent" | "pt" | "np" | "pil" (VAE decode on the native decoder).
    `diffusion_name_or_path` may be a dict of UNet config overrides for random init (no checkpoints exist in the sandbox);
    a checkpoint directory is loaded through safetensors into the native module (identical key names).
    """

    def __init__(self, diffusion_name_or_path=None, projector_type="linear", projector_depth: int = 1,
                 projector_name_or_path: str = None, pretrained_model_name_or_path: str = None, embed_hidden_size: int = 4096,
                 drop_prob: float | None = None, noise_offset: float = 0.0, input_perturbation: float = 0.0,
                 snr_gamma: float | None = None, resolution: int = 512, center_crop: bool = True, random_flip: bool = True,
                 freeze_vae: bool = True, freeze_unet: bool = True, freeze_projector: bool = False, local_files_only: bool = False):
        super().__init__()
        from .unet import UNet2DConditionModel
        from .vae import AutoencoderKLDecoder, AutoencoderKLEncoder
        self.save_model_name = "stable_diffusion_head"
        self.diffusion_name_or_path = diffusion_name_or_path
        self.projector_type, self.projector_depth = projector_type, projector_depth
        self.projector_name_or_path = projector_name_or_path
        self.pretrained_model_name_or_path = pretrained_model_name_or_path
        self.embed_hidden_size = embed_hidden_size
        self.drop_prob, self.noise_offset, self.input_perturbation, self.snr_gamma = drop_prob, noise_offset, input_perturbation, snr_gamma
        self.resolution, self.center_crop, self.random_flip = resolution, center_crop, random_flip
        self.freeze_vae, self.freeze_unet, self.freeze_projector = freeze_vae, freeze_unet, freeze_projector
        if not freeze_unet:
            raise ValueError("the native UNet is a frozen tower (freeze_unet=True in every shipped config)")
        if isinstance(diffusion_name_or_path, str):
            import glob
            self.unet = UNet2DConditionModel()
            files = glob.glob(os.path.join(diffusion_name_or_path, "unet", "*.safetensors"))
            if not files:
                raise FileNotFoundError(f"no unet/*.safetensors under {diffusion_name_or_path}")
            from safetensors.torch import load_file
            self.unet.load_state_dict(load_file(files[0]))
        else:
            cfgd = dict(diffusion_name_or_path or {})
            vae_cfg = cfgd.pop("vae", None)
            self.unet = UNet2DConditionModel(cfgd)
        self.vae = AutoencoderKLEncoder(vae_cfg if not isinstance(diffusion_name_or_path, str) else None)
        if isinstance(diffusion_name_or_path, str):
            import glob
            from safetensors.torch import load_file
            vf = glob.glob(os.path.join(diffusion_name_or_path, "vae", "*.safetensors"))
            if vf:
                self.vae.load_state_dict(load_file(vf[0]), strict=False)      # decoder.* / post_quant_conv.* are not part of this path
        # decode half of the same AutoencoderKL (separate module so its keys stay `decoder.*` / `post_quant_conv.*`)
        self.vae_decoder = AutoencoderKLDecoder(vae_cfg if not isinstance(diffusion_name_or_path, str) else None)
        if isinstance(diffusion_name_or_path, str) and vf:
            self.vae_decoder.load_state_dict(load_file(vf[0]), strict=False)
        self.vae_decoder.requires_grad_(False)
        self.vae.requires_grad_(False)
        projector_cfg = dict(projector=projector_type, freeze_projector=freeze_projector, depth=projector_depth,
                             save_model_name=self.save_model_name, model_name_or_path=None)
        self.projector = build_projector(projector_cfg, in_hidden_size=embed_hidden_size,
                                         out_hidden_size=self.unet.cfg["cross_attention_dim"], bias=False)
        self._init_weights(self.projector)
        self.vae_scale_factor = 8
        if pretrained_model_name_or_path is not None:
            self.load_model(pretrained_model_name_or_path)
        self.projector.load_model(projector_name_or_path)
        self.unet.requires_grad_(False)
        self.projector.requires_grad_(not freeze_projector)

    @property
    def processor(self):
        return None

    @property
    def config(self):
        return dict(diffusion_name_or_path=self.diffusion_name_or_path, pretrained_model_name_or_path=self.pretrained_model_name_or_path,
                    embed_hidden_size=self.embed_hidden_size, drop_prob=self.drop_prob, noise_offset=self.noise_offset,
                    input_perturbation=self.input_perturbation, snr_gamma=self.snr_gamma, resolution=self.resolution,
                    freeze_vae=self.freeze_vae, freeze_unet=self.freeze_unet, freeze_projector=self.freeze_projector)

    def fsdp_ignored_modules(self) -> list:
        return [self.unet] + ([self.projector] if self.freeze_projector else [])

    def save_model(self, output_dir: str):
        torch.save(self.state_dict(), os.path.join(output_dir, f"{self.save_model_name}.bin"))

    def load_model(self, output_dir: str):
        f = os.path.join(output_dir, f"{self.save_model_name}.bin")
        if os.path.isfile(f):
            self.load_state_dict(torch.load(f, map_location="cpu", weights_only=True), strict=False)

    def _alphas_cumprod(self, device):
        if getattr(self, "_ac", None) is None or self._ac.device != device:
            betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2     # scaled_linear (SURVEY A.2)
            self._ac = torch.cumprod(1.0 - betas, dim=0).to(device)
        return self._ac

    def forward(self, images=None, encoder_hidden_states=None, u_encoder_hidden_states=None, dream_embeddings=None, *,
                latents=None, noise=None, timesteps=None, vae_noise=None, offset_noise=None, perturbation_noise=None, drop_mask=None):
        """Diffusion loss, reference :493-577: VAE encode (:511-512) -> noise draw, + `noise_offset` (:521-523), `input_perturbation`
        (:524-525, :533-534) -> timestep draw (:528) -> add_noise (:534-536) -> CFG-dropout mix when `drop_prob` is set and the null-prompt
        states are given (:539-543) -> projector (:546) -> UNet eps-prediction (:556) -> MSE in fp32 (:559) or min-SNR weighted
        (`snr_gamma`, :561-572).  Gradients flow through the frozen UNet into the conditioning.
        `latents` / `noise` / `timesteps` / `vae_noise` / `offset_noise` / `perturbation_noise` / `drop_mask` let tests inject the random
        draws (the reference uses the global generators, in this order).  `images=None` (the reference's DDP dummy branch, :500-508) is
        not needed by our reducer and returns None."""
        if images is None and latents is None:
            return None
        dev = encoder_hidden_states.device
        if latents is None:
            latents = self.vae.encode_sample(images, z=vae_noise)
        latents = latents.float().contiguous()
        assert encoder_hidden_states.shape[0] == latents.shape[0], \
            f"encoder_hidden_states.shape[0]: {encoder_hidden_states.shape[0]} != latents.shape[0]: {latents.shape[0]}"
        bsz = latents.shape[0]
        if noise is None:
            noise = torch.randn_like(latents)
        noise = noise.float()
        if self.noise_offset:                                                       # RNG post-processing on [B,4,h,w] fp32 (:521-523)
            if offset_noise is None:
                offset_noise = torch.randn((bsz, latents.shape[1], 1, 1), device=dev)
            noise = noise + self.noise_offset * offset_noise.float().view(bsz, latents.shape[1], 1, 1)
        noise = noise.contiguous()
        fwd_noise = noise
        if self.input_perturbation:                                                 # (:524-525): perturbed noise drives x_t, target stays `noise`
            if perturbation_noise is None:
                perturbation_noise = torch.randn_like(noise)
            fwd_noise = (noise + self.input_perturbation * perturbation_noise.float()).contiguous()
        if timesteps is None:
            timesteps = torch.randint(0, 1000, (bsz,), device=dev)
        t32 = timesteps.to(torch.int32).contiguous()
        ac = self._alphas_cumprod(dev)
        noisy = ops.add_noise(latents, fwd_noise, t32, ac)
        if u_encoder_hidden_states is not None and self.drop_prob is not None:      # train with classifier-free guidance (:539-543)
            if drop_mask is None:
                drop_mask = torch.bernoulli(torch.zeros(bsz) + self.drop_prob)       # drawn on the host, as the reference does (:541)
            encoder_hidden_states = _CfgDropFn.apply(encoder_hidden_states, u_encoder_hidden_states.to(encoder_hidden_states.dtype),
                                                     drop_mask.detach().to("cpu"))
        cond = self.projector(encoder_hidden_states)[-1]
        snr = None if self.snr_gamma is None else (ac, float(self.snr_gamma))
        return _DiffusionLossFn.apply(cond, self.unet, noisy, t32, noise, snr)      # epsilon prediction (:548-549)

    @torch.no_grad()
    def pipeline(self, height: int | None = None, width: int | None = None, num_inference_steps: int = 50, guidance_scale: float = 7.5,
                 num_images_per_prompt: int | None = 1, eta: float = 0.0, generator=None, latents=None, prompt_embeds=None,
                 negative_prompt_embeds=None, output_type: str | None = "latent", callback=None, callback_steps: int = 1,
                 cross_attention_kwargs=None, guidance_rescale: float = 0.0, scheduler: str = "ddpm", use_cuda_graph: bool = True):
        """reference :672-850.  `scheduler="ddpm"` is what the reference runs (its training DDPMScheduler, :379/:833);
        `"ddim"` (eta 0) is BASELINE.json's C4 sampler."""
        from .unet import DenoiseLoop, check_planes
        height = height or self.resolution
        width = width or self.resolution
        if height % 8 or width % 8:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        # stricter than the reference: every UNet / VAE plane must tile the implicit-GEMM conv (DESIGN.md, divergences)
        check_planes(height // 8, width // 8, len(self.unet.cfg["block_out_channels"]), f"UNet latents of a {height}x{width} image")
        if output_type != "latent":
            check_planes(height, width, len(self.vae_decoder.cfg["block_out_channels"]), f"VAE decoder planes of a {height}x{width} image")
        assert prompt_embeds is not None, "`prompt_embeds` must be provided by LLM."
        n_img = int(num_images_per_prompt or 1)
        if n_img > 1:                                           # (:760-772) each prompt's embeddings repeated per requested image
            prompt_embeds = prompt_embeds.repeat_interleave(n_img, dim=0)
            if negative_prompt_embeds is not None:
                negative_prompt_embeds = negative_prompt_embeds.repeat_interleave(n_img, dim=0)
            if latents is not None and latents.shape[0] != prompt_embeds.shape[0]:
                raise ValueError(f"latents batch {latents.shape[0]} != prompts x num_images_per_prompt = {prompt_embeds.shape[0]}")
        if output_type not in ("latent", "pt", "np", "pil"):
            raise ValueError(f"output_type must be one of 'latent', 'pt', 'np', 'pil', got {output_type!r}")
        cond = self.projector(prompt_embeds)[-1]
        if guidance_scale > 1.0:
            assert negative_prompt_embeds is not None, "When using classifier free guidance, `negative_prompt_embeds` must be provided by LLM."
            cond = torch.cat([self.projector(negative_prompt_embeds)[-1], cond])
        loop = DenoiseLoop(self.unet, cond, num_inference_steps, guidance_scale, scheduler, latents=latents, height=height, width=width,
                           use_cuda_graph=use_cuda_graph, generator=generator, guidance_rescale=guidance_rescale)
        lat = loop.run(callback=callback, callback_steps=callback_steps)
        if output_type == "latent":
            return lat
        image = self.vae_decoder.decode(lat)                                  # vae.decode(latents / scaling_factor), :842
        image = (image / 2 + 0.5).clamp(0, 1)                                 # VaeImageProcessor.postprocess denormalize
        if output_type == "pt":
            return image
        arr = image.permute(0, 2, 3, 1).cpu().numpy()
        return arr if output_type == "np" else numpy_to_pil(arr)
