"""Mint golden vectors for the decoder hot path from the REFERENCE'S OWN CODE.

Run in the build container only (needs /root/reference):   python -m oracle.gen_golden
Writes tests/golden/decoder_layer_*.npz.  Each file holds the seeds/shape needed to
regenerate inputs + weights (oracle.decoder_oracle.init_layer_params — deterministic CPU
RNG), a checksum of those, and the reference's outputs: y, dx, and slices of every dW.
tests/golden/kvcache_layer.npz holds the kv-cache decode scenario in fp32, and
tests/golden/decoder_bf16.npz the reference's bf16 outputs of a plain and a kv-cache run.

The reference classes are exec'd verbatim by oracle/ref_exec.py (modeling_dreamllm.py:69-655).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import decoder_oracle as O  # noqa: E402
from oracle import ref_exec  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = [
    # name, hidden, inter, heads, bsz, seq, seed, pad (number of right-pad tokens in sample 1)
    ("tiny", 256, 512, 2, 2, 48, 11, 0),
    ("ragged", 256, 384, 2, 2, 200, 12, 37),
    ("mid", 512, 1408, 4, 1, 384, 13, 0),
    # BASELINE.json configs[0] itself: Vicuna-7B layer, hidden 4096, 32 heads, seq 512, bs 1 (y / dx stored strided to keep the file small)
    ("c1", 4096, 11008, 32, 1, 512, 14, 0),
]
STRIDED = {"mid": (2, 2), "c1": (4, 8)}        # name -> (row step, column step) of the stored y / dx
BF16_CASE = (256, 512, 2, 2, 40, 5)            # hidden, inter, heads, bsz, seq, seed of the bf16 rounding-point pin
THREADS = 8     # intra-op threads the fixtures are minted with: the CPU fp32 GEMMs split their sums by thread count


def make_inputs(hidden, bsz, seq, seed):
    g = torch.Generator().manual_seed(seed + 1000)
    x = torch.randn(bsz, seq, hidden, generator=g)
    gy = torch.randn(bsz, seq, hidden, generator=g) / (bsz * seq * hidden) ** 0.5
    return x, gy


def checksum(t: torch.Tensor) -> float:
    return float(t.double().abs().sum())


def run_reference(ns, name, hidden, inter, heads, bsz, seq, seed, pad):
    cfg = ref_exec.make_config(hidden, inter, heads)
    layer = ns["DreamLLMDecoderLayer"](cfg).float()
    p = O.init_layer_params(hidden, inter, seed)
    sd = {k: v.clone() for k, v in p.items()}
    sd["self_attn.rotary_emb.inv_freq"] = layer.self_attn.rotary_emb.inv_freq.clone()
    layer.load_state_dict(sd)
    x, gy = make_inputs(hidden, bsz, seq, seed)
    x.requires_grad_(True)
    am = None
    if pad:
        am = torch.ones(bsz, seq, dtype=torch.long)
        am[1, seq - pad :] = 0
    mask = ref_exec.causal_mask_4d(bsz, seq, torch.float32, am)
    pos = torch.arange(seq)[None].expand(bsz, -1)
    y = layer(x, attention_mask=mask, position_ids=pos)[0]
    if am is not None:
        gy = gy * am[..., None]  # padded positions carry no loss (labels are -100 there)
    y.backward(gy)
    out = {
        "shape": np.array([hidden, inter, heads, bsz, seq, seed, pad], dtype=np.int64),
        "x_checksum": np.float64(checksum(x.detach())),
        "w_checksum": np.float64(sum(checksum(v) for v in p.values())),
        "y": y.detach().numpy().astype(np.float32),
        "dx": x.grad.numpy().astype(np.float32),
    }
    if name in STRIDED:
        rs, cs = STRIDED[name]
        out["stride"] = np.array([rs, cs], dtype=np.int64)
        out["y_abs_sum"], out["dx_abs_sum"] = np.float64(checksum(y.detach())), np.float64(checksum(x.grad))
        out["y"], out["dx"] = out["y"][:, ::rs, ::cs].copy(), out["dx"][:, ::rs, ::cs].copy()
    for k, prm in layer.named_parameters():
        g = prm.grad
        out["d_" + k] = (g[:8, :64] if g.dim() == 2 else g).numpy().astype(np.float32)
        out["dsum_" + k] = np.float64(g.double().sum())
    return out


def run_reference_cached(ns):
    """The reference layer (eager attention, :309-400) driven with `past_key_value` / `use_cache=True` over `cached_decode_scenario`:
    a LEFT-padded batch, prefill + single-token decode steps, 4-D masks from the reference's own `_prepare_4d_causal_attention_mask`."""
    from transformers.modeling_attn_mask_utils import _prepare_4d_causal_attention_mask
    hidden, inter, heads = 256, 512, 2
    p, calls = O.cached_decode_scenario(hidden, inter, heads)
    layer = ns["DreamLLMDecoderLayer"](ref_exec.make_config(hidden, inter, heads)).float()
    sd = {k: v.clone() for k, v in p.items()}
    sd["self_attn.rotary_emb.inv_freq"] = layer.self_attn.rotary_emb.inv_freq.clone()
    layer.load_state_dict(sd)
    past, out = None, {"shape": np.array([hidden, inter, heads], dtype=np.int64)}
    with torch.no_grad():
        for i, (x, am, pos) in enumerate(calls):
            past_len = 0 if past is None else past[0].shape[2]
            mask = _prepare_4d_causal_attention_mask(am, (x.shape[0], x.shape[1]), x, past_len)
            y, past = layer(x, attention_mask=mask, position_ids=pos, past_key_value=past, use_cache=True)
            out[f"y{i}"] = y.numpy().astype(np.float32)
            out[f"mask{i}"] = am.numpy()
    out["k_final"] = past[0][:, :, -4:].numpy().astype(np.float32)          # last rotated keys of the final cache
    return out


def _bf16_layer(ns, p, hidden, inter, heads):
    layer = ns["DreamLLMDecoderLayer"](ref_exec.make_config(hidden, inter, heads)).float()
    sd = {k: v.clone() for k, v in p.items()}
    sd["self_attn.rotary_emb.inv_freq"] = layer.self_attn.rotary_emb.inv_freq.clone()
    layer.load_state_dict(sd)
    return layer.to(torch.bfloat16)


def run_reference_bf16(ns):
    """The reference layer in bf16 on BF16_CASE: an oracle that shares its rounding points (norm cast before the weight multiply, bf16
    rope tables, fp32 softmax) reproduces this output bit for bit."""
    hidden, inter, heads, bsz, seq, seed = BF16_CASE
    layer = _bf16_layer(ns, O.init_layer_params(hidden, inter, seed), hidden, inter, heads)
    x, _ = make_inputs(hidden, bsz, seq, seed)
    pos = torch.arange(seq)[None].expand(bsz, -1)
    with torch.no_grad():
        y = layer(x.to(torch.bfloat16), attention_mask=ref_exec.causal_mask_4d(bsz, seq, torch.bfloat16), position_ids=pos)[0]
    return {"y": y.float().numpy()}


def run_reference_cached_bf16(ns):
    """`run_reference_cached` in bf16; only the rows of real tokens are stored (pad query rows differ by design between the
    reference's eager and flash paths)."""
    from transformers.modeling_attn_mask_utils import _prepare_4d_causal_attention_mask
    BF = torch.bfloat16
    hidden, inter, heads = 256, 512, 2
    p, calls = O.cached_decode_scenario(hidden, inter, heads)
    layer = _bf16_layer(ns, p, hidden, inter, heads)
    past, out = None, {}
    with torch.no_grad():
        for i, (x, am, pos) in enumerate(calls):
            past_len = 0 if past is None else past[0].shape[2]
            mask = _prepare_4d_causal_attention_mask(am, (x.shape[0], x.shape[1]), x.to(BF), past_len)
            y, past = layer(x.to(BF), attention_mask=mask, position_ids=pos, past_key_value=past, use_cache=True)
            out[f"kv_y{i}"] = y[am[:, -x.shape[1]:].bool()].float().numpy()
    return out


def main():
    assert ref_exec.available(), "needs /root/reference (build container only)"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(THREADS)
    ns = ref_exec.load_reference_namespace()
    only = set(sys.argv[1:])
    for case in CASES:
        if only and case[0] not in only:
            continue
        out = run_reference(ns, *case)
        path = os.path.join(OUT, f"decoder_layer_{case[0]}.npz")
        np.savez_compressed(path, **out)
        print(path, os.path.getsize(path) // 1024, "KiB")
    if not only or "kvcache" in only:
        path = os.path.join(OUT, "kvcache_layer.npz")
        np.savez_compressed(path, **run_reference_cached(ns))
        print(path, os.path.getsize(path) // 1024, "KiB")
    if not only or "bf16" in only:
        path = os.path.join(OUT, "decoder_bf16.npz")
        np.savez_compressed(path, **run_reference_bf16(ns), **run_reference_cached_bf16(ns))
        print(path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
