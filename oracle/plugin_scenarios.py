"""TEST INFRASTRUCTURE — deterministic scenarios for the plugin-level oracles (splice / conditioning gather / loss combination /
diffusion loss / CFG rescale / config defaults), shared by
  * oracle/gen_golden_plugins.py   (mints tests/golden/plugins.npz and tests/golden/reference_config.json from the LIVE reference),
  * tests/test_golden_plugins.py, tests/test_oracle_pin_model.py, tests/test_oracle_pin_sdhead.py, tests/test_scheduler_cpu.py,
    tests/test_hf_surface_cpu.py   (oracle / product == golden, run anywhere).
`live_*` functions exec the reference's own methods verbatim from a reference checkout (modeling_dreamllm.py:1045-1158, :1353-1509;
modeling_plugins.py:468-577, :658-669; configuration_dreamllm.py:64-278) with stand-in sub-modules; `oracle_*` functions compute the
same quantities with the restatements.  Never imported by the product."""
from __future__ import annotations

import copy
import math
import os
import textwrap
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn.functional as F
from torch.nn import CrossEntropyLoss

from . import decoder_oracle as O
from . import splice_oracle as SO
from . import unet_oracle as UO

REF_MODEL = "/root/reference/omni/models/dreamllm/modeling_dreamllm.py"
REF_PLUGINS = "/root/reference/omni/models/dreamllm/modeling_plugins.py"
REF_CONFIG = os.path.join(os.path.dirname(REF_MODEL), "configuration_dreamllm.py")
TOK = {"<im_start>": 90, "<im_patch>": 91, "<im_end>": 92, "<dream_start>": 93, "<dream_end>": 94}
ST = {"additional_special_tokens": TOK, "<s>": 1, "</s>": 2}
P, Q, H, V = 5, 3, 16, 96
T = 1000
SMALL_UNET = dict(block_out_channels=(32, 64), attention_head_dim=(2, 4), cross_attention_dim=48, down_attn=(True, False),
                  up_attn=(False, True), norm_num_groups=8)
SPLICE_CASES = [(2, True), (3, True), (1, False), (0, True)]                       # (n_images, with_dream)
CAUSAL_CASES = [(None, 3), (0.1, 2)]                                               # (drop_prob, n_dm)
SDHEAD_CASES = [(0.0, 0.0, None, None), (0.1, 0.0, None, None), (0.0, 0.1, None, None), (0.0, 0.0, 5.0, None), (0.0, 0.0, None, 0.5),
                (0.05, 0.1, 5.0, 0.5)]                                             # (noise_offset, input_perturbation, snr_gamma, drop_prob)


def reference_available() -> bool:
    return all(os.path.isfile(f) for f in (REF_MODEL, REF_PLUGINS, REF_CONFIG))


# ------------------------------------------------------------------------------------------------ shared inputs
def make_ids():
    rows = [[1, 90] + [91] * P + [92, 7, 8, 93] + [91] * Q + [94, 2],
            [1, 5, 90] + [91] * P + [92, 90] + [91] * P + [92, 6, 2],          # two <im_start>; with 2 images only one is left for this row
            [1, 93] + [91] * Q + [94, 9, 93] + [91] * Q + [94, 2]]             # two dreams
    S = max(len(r) for r in rows)
    return torch.tensor([r + [0] * (S - len(r)) for r in rows])


def splice_inputs(n_images):
    g = torch.Generator().manual_seed(0)
    ids = make_ids()
    torch.manual_seed(0)
    emb = torch.nn.Embedding(V, H)
    dq = torch.randn(1, Q, H, generator=g)
    feats = torch.randn(max(n_images, 1), P, H, generator=g)
    return ids, emb, dq, feats


def causal_inputs():
    g = torch.Generator().manual_seed(1)
    ids = make_ids()
    B, S = ids.shape
    hidden = torch.randn(B, S, H, generator=g)
    u_hidden = torch.randn(1, Q + 4, H, generator=g)
    labels = ids.clone()
    labels[ids >= 90] = -100
    labels[ids == 0] = -100
    head_w = torch.randn(V, H, generator=g) * 0.1
    return ids, hidden, u_hidden, labels, head_w


def sdhead_parts():
    torch.manual_seed(0)
    unet = UO.UNet2DConditionModel(SMALL_UNET).eval()
    proj = torch.nn.Linear(40, 48)
    lat = torch.randn(3, 4, 8, 8)
    g = torch.Generator().manual_seed(1)
    enc = torch.randn(3, 5, 40, generator=g)
    u_row = torch.randn(1, 5, 40, generator=g)
    return unet, proj, lat, enc, u_row


def rescale_inputs():
    """(cfg, text) for `rescale_noise_cfg` at guidance 7.5"""
    g = torch.Generator().manual_seed(0)
    text, uncond = torch.randn(3, 4, 8, 8, generator=g) * 1.3, torch.randn(3, 4, 8, 8, generator=g)
    return uncond + 7.5 * (text - uncond), text


class Tok:
    """tokenizer stand-in: length + the special-token ids of TOK / ST"""

    def __init__(self, n):
        self.n = n
        self.pad_token_id = 0

    def __len__(self):
        return self.n

    def convert_tokens_to_ids(self, t):
        table = {**TOK, "<s>": 1, "</s>": 2}
        return [table[x] for x in t] if isinstance(t, list) else table[t]


CONFIG_TOKENS = {"additional_special_tokens": ["<im_start>", "<dream_start>"], "bos_token": "<s>"}


def sdhead_replay(seed, lat, noise_offset, input_perturbation, drop_prob):
    """the reference's RNG draws in its order (modeling_plugins.py:520-541)"""
    torch.manual_seed(seed)
    noise = torch.randn_like(lat)
    offset = torch.randn((3, 4, 1, 1)) if noise_offset else None
    pert = torch.randn_like(noise) if input_perturbation else None
    t = torch.randint(0, T, (3,)).long()
    mask = torch.bernoulli(torch.zeros(3) + drop_prob)[:, None, None] if drop_prob is not None else None
    return noise, offset, pert, t, mask


def sdhead_seed(lat, noise_offset, input_perturbation, drop_prob):
    if drop_prob is None:
        return 1234
    return next(s for s in range(1234, 1334) if 0 < float(sdhead_replay(s, lat, noise_offset, input_perturbation, drop_prob)[4].sum()) < 3)


# ------------------------------------------------------------------------------------------------ oracle side
def oracle_splice(n_images, with_dream):
    ids, emb, dq, feats = splice_inputs(n_images)
    with torch.no_grad():
        return SO.splice(ids, emb(ids), feats[:n_images] if n_images else None, dq if with_dream else None, 90, 93)


def oracle_causal(drop_prob, n_dm):
    ids, hidden, u_hidden, labels, head_w = causal_inputs()
    enc = SO.gather_conditioning(ids, hidden, 93, Q, n_dm)
    u_enc = None if drop_prob is None else u_hidden[:, 2:2 + Q].repeat(n_dm, 1, 1)
    lm = O.lm_loss(F.linear(hidden, head_w).float(), labels)
    vm = enc.float().pow(2).mean()                                      # the stand-in head's "loss"
    return dict(enc=enc, u_enc=u_enc, lm_loss=lm, loss=vm * 10.0 + lm * 1.0, null_ids=[[1, 93] + [91] * Q + [94, 2]])


def oracle_sdhead(noise_offset, input_perturbation, snr_gamma, drop_prob):
    unet, proj, lat, enc, u_row = sdhead_parts()
    seed = sdhead_seed(lat, noise_offset, input_perturbation, drop_prob)
    noise, offset, pert, t, mask = sdhead_replay(seed, lat, noise_offset, input_perturbation, drop_prob)
    cond = enc
    if mask is not None:
        cond = (1.0 - mask) * enc + mask * u_row.repeat(3, 1, 1)         # (:539-542) — the row select `_CfgDropFn` performs
    with torch.no_grad():
        return UO.diffusion_loss(unet, lat, proj(cond), noise, t, UO.alphas_cumprod(T), noise_offset=noise_offset,
                                 offset_noise=None if offset is None else offset.view(3, 4), input_perturbation=input_perturbation,
                                 perturbation_noise=pert, snr_gamma=snr_gamma)


# ------------------------------------------------------------------------------------------------ live reference side
class _Out(tuple):
    """BaseModelOutputWithPast stand-in: indexable + the attributes the reference reads."""
    def __new__(cls, hidden):
        o = super().__new__(cls, (hidden,))
        o.past_key_values = o.hidden_states = o.attentions = None
        o.additional_log_info = {}
        return o


def _exec_method(path, start_marker, end_marker, nth=0, names=("forward",)):
    src = open(path).read()
    a = -1
    for _ in range(nth + 1):
        a = src.index(start_marker, a + 1)
    b = src.index(end_marker, a)
    ns = dict(torch=torch, F=F, math=math, np=np, CrossEntropyLoss=CrossEntropyLoss, BaseModelOutputWithPast=None,
              CausalLMOutputWithPast=lambda **kw: SimpleNamespace(**kw), DEFAULT_IMAGE_START_TOKEN="<im_start>",
              DEFAULT_DREAM_START_TOKEN="<dream_start>", DEFAULT_DREAM_END_TOKEN="<dream_end>", DEFAULT_IMAGE_PATCH_TOKEN="<im_patch>",
              DEFAULT_BOS_TOKEN="<s>", DEFAULT_EOS_TOKEN="</s>",
              logger=SimpleNamespace(warning=lambda *a, **k: None, warning_once=lambda *a, **k: None, error=lambda *a, **k: None))
    exec("from __future__ import annotations\n" + textwrap.dedent(src[a:b]), ns)
    return [ns[n] for n in names]


_FWD_SIG = "    def forward(\n        self,\n        input_ids: torch.LongTensor = None,\n        images:"


def live_splice(n_images, with_dream):
    (fwd,) = _exec_method(REF_MODEL, _FWD_SIG, "    # `DreamEmbedding`")
    ids, emb, dq, feats = splice_inputs(n_images)
    seen = {}

    class M:
        training = False
        config = SimpleNamespace(special_tokens2ids_dict=ST)
        embed_tokens = emb
        dream_embedding = staticmethod(lambda bs=1: dq.repeat(bs, 1, 1))
        clip_vision_embedding = staticmethod(lambda images: feats[:n_images] if images is not None else torch.zeros(()))

        def _forward(self, **kw):
            seen.update(kw)
            return kw["inputs_embeds"]
    M.dream_embedding.embed_len = Q
    M.forward = fwd
    images = torch.zeros(n_images, 3, 2, 2) if n_images else None
    images_dm = torch.zeros(2, 3, 2, 2) if with_dream else None
    with torch.no_grad():
        out = M().forward(input_ids=ids, images=images, images_dm=images_dm)
    return out, seen


def live_causal(drop_prob, n_dm):
    (fwd,) = _exec_method(REF_MODEL, _FWD_SIG, "    def prepare_inputs_for_generation", nth=1)
    ids, hidden, u_hidden, labels, head_w = causal_inputs()
    calls, sd_calls = [], []

    def model(**kw):
        calls.append(kw)
        return _Out(hidden if len(calls) == 1 else u_hidden)
    model.config = SimpleNamespace(special_tokens2ids_dict=ST)
    model.dream_embedding = SimpleNamespace(embed_len=Q)

    def sd_head(images_dm, enc, u_enc, *rest):
        sd_calls.append((enc, u_enc))
        return enc.float().pow(2).mean()
    sd_head.drop_prob = drop_prob
    self = SimpleNamespace(training=True, model=model, stable_diffusion_head=sd_head, lm_head=lambda h: F.linear(h, head_w),
                           loss_weight_lm=1.0, loss_weight_vm=10.0, vocab_size=V,
                           config=SimpleNamespace(max_position_embeddings=2048, output_attentions=False, output_hidden_states=False,
                                                  use_return_dict=True, special_tokens2ids_dict=ST, pretraining_tp=1, vocab_size=V,
                                                  loss_scale_schedule="none"))
    out = fwd(self, input_ids=ids, images_dm=torch.zeros(n_dm, 3, 2, 2), labels=labels)
    enc, u_enc = sd_calls[0]
    return dict(enc=enc, u_enc=u_enc, lm_loss=torch.as_tensor(out.additional_log_info["lm_loss"]), loss=out.loss,
                null_ids=None if len(calls) == 1 else calls[1]["input_ids"].tolist(), n_model_calls=len(calls))


class _Sched:
    """DDPMScheduler stand-in: the attributes / methods the reference forward touches (:529, :534-536, :551-554, :473)."""

    def __init__(self):
        self.config = SimpleNamespace(num_train_timesteps=T, prediction_type="epsilon")
        self.alphas_cumprod = UO.alphas_cumprod(T)

    def add_noise(self, x0, noise, t):
        return UO.add_noise(x0, noise, t, self.alphas_cumprod)


def live_sdhead_object(noise_offset, input_perturbation, snr_gamma, drop_prob):
    snr, fwd = _exec_method(REF_PLUGINS, "    def _compute_snr(self, timesteps):", "    def check_inputs(", names=("_compute_snr", "forward"))
    unet, proj, lat, enc, u_row = sdhead_parts()
    head = type("RefStableDiffusionHead", (), {"_compute_snr": snr, "forward": fwd})()
    head.vae = SimpleNamespace(encode=lambda images: SimpleNamespace(latent_dist=SimpleNamespace(sample=lambda: lat / 0.18215)),
                               config=SimpleNamespace(scaling_factor=0.18215))
    head.noise_scheduler = _Sched()
    head.projector = lambda x: [proj(x)]
    head.unet = lambda x, t, c: SimpleNamespace(sample=unet(x, t, c))
    head.noise_offset, head.input_perturbation, head.snr_gamma, head.drop_prob = noise_offset, input_perturbation, snr_gamma, drop_prob
    head.embed_hidden_size, head.device, head.dtype = 40, torch.device("cpu"), torch.float32
    return head, lat, enc, u_row


def live_sdhead(noise_offset, input_perturbation, snr_gamma, drop_prob):
    head, lat, enc, u_row = live_sdhead_object(noise_offset, input_perturbation, snr_gamma, drop_prob)
    seed = sdhead_seed(lat, noise_offset, input_perturbation, drop_prob)
    u_enc = u_row.repeat(3, 1, 1) if drop_prob is not None else None
    torch.manual_seed(seed)
    with torch.no_grad():
        return head.forward(torch.zeros(3, 3, 64, 64), enc, u_enc)


def live_sdhead_dummy():
    """the reference's images=None branch (:500-509), which only feeds DDP's unused-parameter check"""
    head, _, _, _ = live_sdhead_object(0.0, 0.0, None, None)
    with torch.no_grad():
        return head.forward(None, None, None, dream_embeddings=torch.randn(1, 5, 40))


def live_rescale_noise_cfg():
    """`_rescale_noise_cfg` (modeling_plugins.py:658-669) on `rescale_inputs()` at guidance_rescale 0.7"""
    src = open(REF_PLUGINS).read()
    a = src.index("    def _rescale_noise_cfg(")
    b = src.index("    @torch.no_grad()", a)
    ns = {"torch": torch}
    exec(textwrap.dedent(src[a:b]), ns)
    cfg, text = rescale_inputs()
    return ns["_rescale_noise_cfg"](None, cfg, text, 0.7)


def live_config():
    """The reference's `DreamLLMConfig` (configuration_dreamllm.py:64-278) on the installed transformers: a default instance, and one
    after `update_special_tokens2ids_dict(CONFIG_TOKENS, Tok(96))`."""
    from transformers import PretrainedConfig

    class _Log:
        def warning(self, *a, **k):
            pass
        info = warning

    src = open(REF_CONFIG).read().split("\n")
    ns = dict(PretrainedConfig=PretrainedConfig, logger=_Log(), CLASS_KEY="_class_", NAME_KEY="_name_", PLUGIN_TYPE_KEY="_plugin_type_")
    exec("from __future__ import annotations\n" + "\n".join(src[63:278]), ns)
    ref = ns["DreamLLMConfig"]()
    defaults = copy.deepcopy({k: getattr(ref, k) for k in ref.to_dict()})
    ref.update_special_tokens2ids_dict(CONFIG_TOKENS, Tok(96))
    return defaults, ref.special_tokens2ids_dict
