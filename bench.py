#!/usr/bin/env python
"""bench.py — the judged benchmark (contract in the task statement).

Headline workload = BASELINE.json configs[4] at its per-GPU shape (the only config that carries both halves of the metric
"interleaved tokens+pixels/sec @ Vicuna-7B+SD2.1 512px"): DreamLLM stage-1 *creation* training step — Vicuna-7B LLM (frozen) + dream
queries (trainable) + SD-2.1 head (VAE encode + UNet, frozen; projector trainable), 4 samples / GPU of
[bos, 32 text, <dream_start>, 64 x <im_patch>, <dream_end>, eos] with 512x512 targets: forward, backward (dgrad through all 32 LLM
layers and the whole UNet), gradient all-reduce (N > 1), global-norm clip + AdamW on the trainable parameters.
    value = (sum(attention_mask) + Nd * 512 * 512) / s        (SURVEY.md §8d), inputs resident in HBM
    e2e   = same through DreamLLMForCausalMLM.forward/backward with pinned HOST ids + images (12.6 MB H2D / step) and loss D2H

Nested records in the same JSON line, each with its own roofline:
    c2  configs[1]  Vicuna-7B text-only fwd+bwd, seq 2048, bs 8 / GPU  (tcgen05 GEMM roofline + whole-step tensor fraction; DDP at N > 1)
    c4  configs[3]  SD-2.1 UNet 64x64, 50-step DDIM, 77 dream-query embeddings, bs 16, CFG, whole loop in ONE CUDA graph
                    (step tensor fraction + per-kernel HBM fractions of GroupNorm / LayerNorm / GEGLU / sampler)
    c3  configs[2]  CLIP ViT-L/14-336 + linear projector + Vicuna-7B, 576 visual + 1024 text tokens, bs 4, fwd+bwd through the collator
    c1  configs[0]  one DreamLLMDecoderLayer fwd+bwd, hidden 4096 seq 512 bs 1, with the CPU reference timed in full beside it

  python bench.py --gpus N --steps K --warmup W            # our CUDA path (N>1 under torchrun, weak scaling)
  python bench.py --impl reference ...                     # the reference algorithm on the host CPU cores (oracle port), same workload
  python bench.py ... --dump-outputs DIR                   # also write what the last timed headline step computed, as DIR/*.npy

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "interleaved tokens+pixels/sec @ Vicuna-7B+SD2.1 512px, 1/2/4/8 B200"
UNIT = "tokens+pixels/s"
BF = torch.bfloat16

# Vicuna-7B DreamLLM (vocab 32000 + 8 special tokens, projects/dreamllm/train.py:74-89)
H, I, NH, L, V = 4096, 11008, 32, 32, 32008
# token ids: tokenization_dreamllm.py:78-94  ([PAD] 32000, <image>, <im_patch>, <im_start>, <im_end>, <dream>, <dream_start>, <dream_end>)
IM_PATCH, IM_START, IM_END, DREAM_START, DREAM_END = 32002, 32003, 32004, 32006, 32007
C5 = dict(bs=4, Q=64, txt=32, res=512)                      # per GPU; Q = reference default num_dream_queries (configs/common.py:18)
UNET_GF_PER_SAMPLE = 804.3e9                                # SURVEY §8 row U1 (analytic, 64x64 latents, Q = 77)
VAE_ENC_GF = 1116.7e9                                       # SURVEY §8(f) row 1


def llm_fwd_flops(tokens, seq, layers=L, with_head=True):
    """Algorithmic forward FLOPs (SURVEY.md §8d): dense GEMMs + causal attention counted at half (2*S*H per token)."""
    per_tok_layer = 2 * (4 * H * H + 3 * H * I) + 2 * seq * H
    return tokens * (layers * per_tok_layer + (2 * H * V if with_head else 0))


def c5_flops_per_gpu(bs, seq):
    """stage-1 step: LLM fwd + dgrad-only bwd (frozen weights: ~1x fwd), lm_head fwd (logits are computed, labels all -100), VAE encode
    fwd, UNet fwd + dgrad-only bwd (~1x fwd).  SURVEY §8d "Stage-1 step FLOPs"."""
    llm = llm_fwd_flops(bs * seq, seq, with_head=True)
    return 2 * llm + bs * (VAE_ENC_GF + 2 * UNET_GF_PER_SAMPLE)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def summary(self, lo=0, hi=None):
        sm, mx, reasons = [], None, set()
        for r in self.rows[lo:hi]:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        return self.summary()


_T0 = time.time()


def log(msg):
    """progress on stderr (stdout carries exactly one JSON line)"""
    if int(os.environ.get("RANK", 0)) == 0:
        print(f"[bench {time.time() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tf_sustained": d.get("bf16_tflops_sustained", 1442.3), "tf_burst": d.get("bf16_tflops", 1701.0),
                "hbm": d.get("hbm_gbs", 6569.6), "how": "measured (MEASURED_PEAKS.json)"}
    return {"tf_sustained": 1400.0, "tf_burst": 1590.0, "hbm": 6650.0, "how": "fallback (B200_PROFILING.md)"}


def gemm_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/*_gemm_traffic.json)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_gemm_traffic.json")))
    if not files:
        return None, "no ncu --set full capture committed"
    d = json.load(open(files[-1]))
    return d["dram_bytes_per_launch"], d["note"]


# =============================================================================================== CPU reference legs (oracle port)
_CPU_THREADS = None


def _cpu_threads():
    """Thread count for the CPU reference legs = whichever of {8, 16, 32, 64, all hardware threads} runs a reference decoder layer fastest
    on this box.  (Handing torch all 128+ hardware threads of the GPU host made the S = 100 layer 16x SLOWER than 8 threads do — 7.5 s
    vs 0.46 s — and the CPU baseline swung 4x between boxes in round 1; the reference deserves its best setting, and the number of
    threads actually used is what `cores` reports.)"""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        torch.set_num_threads(_CPU_THREADS)
        return _CPU_THREADS
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    from oracle import decoder_oracle as O
    p = {k: v.requires_grad_(False) for k, v in O.init_layer_params(H, I, 100, dtype=torch.bfloat16).items()}
    x = torch.randn(1, 100, H).to(torch.bfloat16).requires_grad_(True)
    cos, sin = O.rope_tables(H // NH, 2048, dtype=torch.bfloat16)
    pos, mask = torch.arange(100)[None], O.causal_additive_mask(1, 100, torch.bfloat16)
    best, best_t = None, None
    for t in sorted({c for c in (8, 16, 32, 64, n) if c <= n}):
        torch.set_num_threads(t)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            x.grad = None
            O.decoder_layer(x, p, NH, cos, sin, pos, mask).float().pow(2).mean().backward()
            ts.append(time.perf_counter() - t0)
        log(f"  cpu threads {t}: reference decoder layer (S=100) {min(ts[1:]):.3f}s")
        if best_t is None or min(ts[1:]) < best_t:
            best, best_t = t, min(ts[1:])
    _CPU_THREADS = best
    torch.set_num_threads(best)
    log(f"  cpu threads: using {best} of {n} hardware threads")
    return best


def _median_time(fn, warm, iters):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), ts


def cpu_llm_layer(seq, bs=1, frozen=False, dtype=torch.bfloat16, warm=1, iters=3):
    """One reference decoder layer (oracle port of modeling_dreamllm.py:599-654, eager attention) fwd+bwd on the host cores."""
    from oracle import decoder_oracle as O
    p = {k: v.requires_grad_(not frozen) for k, v in O.init_layer_params(H, I, 100, dtype=dtype).items()}
    g = torch.Generator().manual_seed(0)
    x = torch.randn(bs, seq, H, generator=g).to(dtype).requires_grad_(True)
    cos, sin = O.rope_tables(H // NH, 2048, dtype=dtype)
    pos = torch.arange(seq)[None]
    mask = O.causal_additive_mask(bs, seq, dtype)

    def step():
        x.grad = None
        O.decoder_layer(x, p, NH, cos, sin, pos, mask).float().pow(2).mean().backward()
    return _median_time(step, warm, iters)


def cpu_lm_head(seq, frozen=False, dtype=torch.bfloat16, warm=1, iters=3):
    from oracle import decoder_oracle as O
    g = torch.Generator().manual_seed(0)
    lm_w = (torch.randn(V, H, generator=g) * 0.02).to(dtype).requires_grad_(not frozen)
    norm_w = torch.ones(H, dtype=dtype, requires_grad=not frozen)
    x = torch.randn(1, seq, H, generator=g).to(dtype).requires_grad_(True)
    labels = torch.randint(0, 32000, (1, seq), generator=g)

    def step():
        logits = torch.nn.functional.linear(O.rmsnorm(x, norm_w), lm_w).float()
        O.lm_loss(logits, labels).backward()
    return _median_time(step, warm, iters)


def _fast_init(mod):
    """Random weights without nn.init's 17 s of kaiming draws (values are irrelevant to timing)."""
    mod = mod.to_empty(device="cpu")
    with torch.no_grad():
        for p in mod.parameters():
            p.uniform_(-0.02, 0.02)
        for b in mod.buffers():
            b.zero_()
    return mod


def cpu_reference_c5(warm=1, iters=3):
    """Reference algorithm for ONE sample of the headline workload on the host cores: 1 decoder layer at S = 100 (frozen weights, dgrad
    only — extrapolated x32), final norm + lm_head logits, VAE encode of one 512x512 image, UNet fwd + backward to the conditioning."""
    from oracle import unet_oracle as UO
    from oracle import vae_oracle as VO
    cores = _cpu_threads()
    S = 1 + C5["txt"] + 1 + C5["Q"] + 1 + 1
    t_layer, _ = cpu_llm_layer(S, frozen=True, warm=warm, iters=iters)
    log(f"  cpu: decoder layer {t_layer:.3f}s ({cores} threads)")
    t_head, _ = cpu_lm_head(S, frozen=True, warm=warm, iters=iters)
    log(f"  cpu: lm_head {t_head:.3f}s")
    with torch.device("meta"):
        unet, vae = UO.UNet2DConditionModel(), VO.AutoencoderKLEncoder()
    unet, vae = _fast_init(unet), _fast_init(vae)
    for p in list(unet.parameters()) + list(vae.parameters()):
        p.requires_grad_(False)
    g = torch.Generator().manual_seed(1)
    img = torch.rand(1, 3, 512, 512, generator=g) * 2 - 1
    cond = torch.randn(1, C5["Q"], 1024, generator=g).requires_grad_(True)
    tt = torch.tensor([500])

    def vae_step():
        with torch.no_grad():
            vae.encode_sample(img, torch.randn(1, 4, 64, 64, generator=g))

    def unet_step():
        cond.grad = None
        lat = torch.randn(1, 4, 64, 64, generator=g)
        unet(lat, tt, cond).float().pow(2).mean().backward()
    log("  cpu: UNet / VAE oracles built")
    t_vae, _ = _median_time(vae_step, warm, iters)
    log(f"  cpu: VAE encode {t_vae:.2f}s")
    t_unet, _ = _median_time(unet_step, warm, iters)
    log(f"  cpu: UNet fwd+bwd {t_unet:.2f}s")
    t_sample = L * t_layer + t_head + t_vae + t_unet
    units = S + C5["res"] * C5["res"]
    return {"value": units / t_sample, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": (f"oracle port on the host CPU, ONE sample of the headline workload (seq {S} + one 512x512 target), {warm} warm-up + "
                       f"{iters} timed, medians: decoder layer bf16 fwd+dgrad {t_layer:.3f}s x{L} (extrapolated) + norm/lm_head {t_head:.3f}s"
                       f" + VAE encode fp32 {t_vae:.2f}s + UNet fwd+bwd-to-cond fp32 {t_unet:.2f}s = {t_sample:.2f}s / sample"),
            "seconds_per_sample": t_sample}


def cpu_reference_c2(seq, warm=1, iters=3):
    cores = _cpu_threads()
    t_layer, _ = cpu_llm_layer(seq, warm=warm, iters=iters)
    t_head, _ = cpu_lm_head(seq, warm=warm, iters=iters)
    t_full = t_layer * L + t_head
    return {"value": seq / t_full, "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"oracle port (CPU torch bf16, eager attention): 1 decoder layer + lm_head/CE at bs=1 seq={seq}, fwd+bwd, {warm} warm-up + "
                      f"{iters} timed (median); layer {t_layer:.2f}s x{L} + head {t_head:.2f}s extrapolated to the 32-layer model"}


def cpu_reference_c1(warm=3, iters=5):
    """configs[0] in full: one decoder layer fwd+bwd, hidden 4096, seq 512, bs 1 — fp32 and bf16 on the host cores (BASELINE.md §5)."""
    cores = _cpu_threads()
    out = {"cores": cores, "torch": torch.__version__, "warmup": warm, "iters": iters}
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        med, ts = cpu_llm_layer(512, dtype=dt, warm=warm, iters=iters)
        out[f"{name}_ms"] = med * 1e3
        out[f"{name}_ms_all"] = [round(t * 1e3, 1) for t in ts]
    return out


def c5_config(args, world):
    S = 1 + C5["txt"] + 1 + C5["Q"] + 1 + 1
    return {"workload": f"BASELINE.json configs[4] per-GPU shape: DreamLLM stage-1 creation step (Vicuna-7B frozen + {C5['Q']} dream queries + "
                        f"SD-2.1 VAE-enc/UNet frozen + projector), {C5['bs']} samples/GPU, seq {S}, {C5['res']}x{C5['res']} targets, fwd + bwd + "
                        f"grad all-reduce + clip + AdamW, bf16",
            "global_batch": C5["bs"] * world, "seq_len": S, "dream_queries": C5["Q"], "layers": args.layers, "hidden": H, "vocab": V,
            "parallelism": f"dp{world}", "l2": "working set (13.5 GB LLM + 1.7 GB UNet weights streamed every step) >> 126 MB L2; no explicit flush",
            "nested": "c2 = configs[1], c4 = configs[3], c3 = configs[2], c1 = configs[0] (see keys of the same name)"}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    iters = max(1, min(args.steps, 3))
    cb = cpu_reference_c5(warm=1 if args.warmup else 0, iters=iters)
    units = C5["bs"] * args.gpus * (c5_config(args, args.gpus)["seq_len"] + C5["res"] ** 2)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * units / cb["value"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 (LLM) / fp32 (VAE, UNet on CPU)", "data": "synthetic", "config": c5_config(args, args.gpus),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if not args.fast:
        line["c1"] = {"cpu": cpu_reference_c1()}
    print(json.dumps(line), flush=True)


# =============================================================================================== our arm
class Env:
    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.args = args
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            from dreamllm_b200.ddp import configure_nccl_env
            configure_nccl_env()
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks = measured_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, k):
        """k calls of fn bracketed by barrier + synchronize on both sides, CUDA events, MAX over ranks -> total ms."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms)


def build_llm(env, layers):
    from dreamllm_b200.modeling_dreamllm import DreamLLMConfig, DreamLLMForCausalMLM
    cfg = DreamLLMConfig.vicuna_7b(num_hidden_layers=layers)
    torch.manual_seed(1234)
    old = torch.get_default_dtype()
    torch.set_default_dtype(BF)
    with torch.device(env.dev):
        model = DreamLLMForCausalMLM(cfg)
    torch.set_default_dtype(old)
    return model


def run_c5(env, model, steps, warmup, dump_dir=None):
    """Headline: stage-1 creation training step.  Whole fwd+bwd replayed as ONE CUDA graph (static layout: the collator's index maps are
    built once), then — outside the graph — gradient all-reduce (N > 1), global-norm clip and fused AdamW on the flat trainable bucket.
    `dump_dir`: write what the last timed step hands its caller — the loss, the trainable parameters after its AdamW update and the
    gradients it applied (flat, in `trainable` order, 2 x 17.8 MB) — as fp32 .npy files, so two builds can be compared output for output."""
    from dreamllm_b200 import ops
    from dreamllm_b200.modeling_plugins import DreamEmbedding, StableDiffusionHead, build_splice_plan
    dev, world, rank, dist = env.dev, env.world, env.rank, env.dist
    B, Q, TXT, R = C5["bs"], C5["Q"], C5["txt"], C5["res"]
    old = torch.get_default_dtype()
    torch.set_default_dtype(BF)
    with torch.device(dev):
        dream = DreamEmbedding(num_dream_queries=Q, embed_hidden_size=H)
        head = StableDiffusionHead(None, embed_hidden_size=H)
    torch.set_default_dtype(old)
    model.stable_diffusion_head = head
    model.model.attach_plugins(None, dream, image_start_id=IM_START, dream_start_id=DREAM_START)
    for p in model.parameters():                                  # stage-1 freezing (configs/stage1/base.py:29-36, :48-50)
        p.requires_grad_(False)
    dream.dream_queries.requires_grad_(True)
    head.projector.requires_grad_(True)
    model.train()
    trainable = [p for p in model.parameters() if p.requires_grad]
    # flat bf16 parameter / gradient buckets for the trainable set (4.46 M parameters = 8.9 MB)
    n_tr = sum(p.numel() for p in trainable)
    pad = (n_tr + 127) // 128 * 128
    flat_p, flat_g = torch.zeros(pad, device=dev, dtype=BF), torch.zeros(pad, device=dev, dtype=BF)
    off = 0
    gviews = []
    with torch.no_grad():
        for p in trainable:
            v = flat_p[off:off + p.numel()].view(p.shape)
            v.copy_(p.data)
            p.data = v
            gviews.append(flat_g[off:off + p.numel()].view(p.shape))
            off += p.numel()
    master, m_, v_ = flat_p.float(), torch.zeros(pad, device=dev), torch.zeros(pad, device=dev)
    ss = torch.zeros(1, device=dev)
    opt_step = [0]

    g = torch.Generator().manual_seed(1 + rank)
    S = 1 + TXT + 1 + Q + 1 + 1
    ids = torch.empty(B, S, dtype=torch.long)
    for b in range(B):
        ids[b] = torch.tensor([1] + torch.randint(3, 32000, (TXT,), generator=g).tolist() + [DREAM_START] + [IM_PATCH] * Q + [DREAM_END, 2])
    labels = torch.full((B, S), -100)                             # creation layout: all labels -100 (builder_dreamllm.py:210-218)
    imgs = (torch.rand(B, 3, R, R, generator=g) * 2 - 1).pin_memory()
    ids_pin = ids.pin_memory()
    plan = build_splice_plan(ids, -1, DREAM_START, 0, Q, 0, B, dev)
    x_static = ids.to(dev)
    im_static = imgs.to(dev)
    lab_dev = labels.to(dev)
    loss_static = torch.zeros(1, device=dev)

    def compute():
        for p in trainable:
            p.grad = None
        out = model(input_ids=x_static, images_dm=im_static.to(BF), labels=lab_dev, attention_mask_has_padding=False, splice_plan=plan)
        out.loss.backward()
        for p, gv in zip(trainable, gviews):
            gv.copy_(p.grad)
        loss_static.copy_(out.loss.detach().float().reshape(1))
        return out

    def optimizer():
        if world > 1:
            dist.all_reduce(flat_g, op=dist.ReduceOp.AVG)
        opt_step[0] += 1
        ss.zero_()
        ops.sumsq_bf16_(flat_g, ss, accumulate=True)
        ops.adamw_step_(flat_g, flat_p, m_, v_, master, lr=2e-3, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, step=opt_step[0],
                        grad_sumsq=ss, max_grad_norm=1.0)           # stage-1 LR 2e-3, max_grad_norm 1.0 (configs/stage1/base.py:74)

    graph, mode = None, "eager launches"
    ops.LAUNCHES.reset()
    log("  c5: first eager step")
    compute()
    optimizer()
    launches_per_step = ops.LAUNCHES.count
    for _ in range(max(warmup - 1, 1)):
        compute()
        optimizer()
    torch.cuda.synchronize()
    if os.environ.get("DLLM_STAGE1_GRAPH", "1") == "1":
        try:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                compute()
            torch.cuda.current_stream().wait_stream(s)
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_):
                compute()
            graph, mode = g_, "fwd+bwd captured in ONE CUDA graph, replayed; all-reduce + clip + AdamW launched after it"
        except Exception as ex:  # noqa: BLE001
            graph, mode = None, f"graph capture failed ({type(ex).__name__}: {str(ex)[:120]}); eager launches"
            torch.cuda.synchronize()

    def step_dev():
        if graph is not None:
            graph.replay()
        else:
            compute()
        optimizer()

    def step_e2e():
        x_static.copy_(ids_pin, non_blocking=True)                # H2D every step: ids + fp32 images from pinned host memory
        im_static.copy_(imgs, non_blocking=True)
        step_dev()
        return float(loss_static.item())                          # D2H every step

    log(f"  c5: {mode}")
    for _ in range(2):
        step_e2e()
    total = env.timed(step_dev, steps)
    total_e2e = env.timed(step_e2e, steps)
    if dump_dir:
        os.makedirs(dump_dir, exist_ok=True)
        for name, t in (("c5_loss", loss_static), ("c5_trainable_params", flat_p[:n_tr]), ("c5_trainable_grads", flat_g[:n_tr])):
            np.save(os.path.join(dump_dir, f"{name}.npy"), t.float().cpu().numpy())
    toks, pix = B * S * world, B * R * R * world
    ms, ms_e = total / steps, total_e2e / steps
    fl = c5_flops_per_gpu(B, S)
    return {"ms_per_step": ms, "value": (toks + pix) / ms * 1e3, "tokens_per_s": toks / ms * 1e3, "pixels_per_s": pix / ms * 1e3,
            "e2e": {"value": (toks + pix) / ms_e * 1e3, "unit": UNIT, "ms_per_step": ms_e,
                    "h2d_bytes_per_step": int(ids_pin.numel() * 8 + imgs.numel() * 4), "d2h_bytes_per_step": 4},
            "launches_per_step": launches_per_step, "launch_mode": mode, "vm_loss": float(loss_static.item()) / model.loss_weight_vm,
            "trainable_params": n_tr,
            "roofline": {"bound": "tensor", "scope": "whole step (LLM fwd+dgrad, VAE encode, UNet fwd+dgrad)",
                         "algorithmic_tflop_per_step_per_gpu": fl / 1e12, "achieved": fl / 1e12 / (ms / 1e3), "peak": env.peaks["tf_sustained"],
                         "unit": "TFLOP/s", "frac": fl / 1e12 / (ms / 1e3) / env.peaks["tf_sustained"],
                         "note": "small-M step (400 LLM tokens, 4 UNet samples): weight streaming (13.5 GB + 2 x 1.7 GB per step = "
                                 f"{(13.5 * 2 + 3.5) / (ms / 1e3) / 1e3:.2f} TB/s of the {env.peaks['hbm'] / 1e3:.2f} TB/s copy peak) bounds it"}}


def run_c2(env, model, steps, warmup, bs, seq, layers):
    from dreamllm_b200 import ops
    from dreamllm_b200.ddp import BucketedGradReducer
    dev, world, rank = env.dev, env.world, env.rank
    for p in model.parameters():
        p.requires_grad_(True)
        p.grad = None
    for p in list(model.stable_diffusion_head.parameters()) if hasattr(model, "stable_diffusion_head") else []:
        p.requires_grad_(False)
    params = [p for n, p in model.named_parameters() if not n.startswith("stable_diffusion_head") and "dream_embedding" not in n]
    reducer = BucketedGradReducer(params, bucket_cap_mb=512.0) if world > 1 else None
    gen = torch.Generator().manual_seed(1234 + rank)
    host_ids = torch.randint(0, 32000, (bs, seq), generator=gen).pin_memory()
    dev_ids = host_ids.to(dev)

    def step(ids):
        if reducer is not None:
            reducer.zero_grad()
        else:
            for p in params:
                p.grad = None
        out = model(input_ids=ids, labels=ids, attention_mask_has_padding=False)
        out.loss.backward()
        if reducer is not None:
            reducer.finalize()
        return out.loss

    for _ in range(warmup):
        step(dev_ids)
    env.barrier()
    ops.PROFILE.reset(enabled=True)
    ops.LAUNCHES.reset()
    total = env.timed(lambda: step(dev_ids), steps)
    launches = ops.LAUNCHES.count
    gs = ops.PROFILE.summary()
    ops.PROFILE.reset(enabled=False)

    def e2e_step():
        return float(step(host_ids.to(dev, non_blocking=True)).item())
    total_e = env.timed(e2e_step, steps)
    copies = reducer.copies if reducer is not None else None
    if reducer is not None:
        reducer.remove()
    for p in params:
        p.grad = None
    ms, ms_e = total / steps, total_e / steps
    toks = bs * seq * world
    fl = 3 * llm_fwd_flops(bs * seq, seq, layers)
    pk = env.peaks
    return {"workload": f"BASELINE.json configs[1]: Vicuna-7B text-only causal-LM fwd+bwd, seq={seq} bs={bs}/GPU bf16, no optimizer step (config is fwd+bwd)",
            "ms_per_step": ms, "tokens_per_s": toks / ms * 1e3, "e2e_tokens_per_s": toks / ms_e * 1e3,
            "h2d_bytes_per_step": int(host_ids.numel() * 8), "d2h_bytes_per_step": 4, "gpu_launches": launches,
            "ddp": None if world == 1 else {"bucket_mb": 512, "grad_bytes": 2 * sum(p.numel() for p in params), "grad_copies_into_buckets": copies},
            "roofline": {"bound": "tensor", "kernel": "dllm::gemm_kernel<2,*,*,bf16> (tcgen05 GEMM, all fwd/dgrad/wgrad launches)",
                         "achieved": gs["tflops"], "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                         "frac": gs["tflops"] / pk["tf_sustained"] if gs["tflops"] else None, "traffic": gemm_traffic()[0],
                         "traffic_note": gemm_traffic()[1], "peak_source": f"bf16_tflops_sustained, {pk['how']}",
                         "launches_timed": gs["n"], "gemm_share_of_step": gs["ms"] / total if total else None},
            "step_roofline": {"algorithmic_tflop_per_step_per_gpu": fl / 1e12, "achieved_tflops_per_gpu": fl / 1e12 / (ms / 1e3),
                              "frac_of_measured_sustained_peak": fl / 1e12 / (ms / 1e3) / pk["tf_sustained"],
                              "frac_of_measured_burst_peak": fl / 1e12 / (ms / 1e3) / pk["tf_burst"]}}


def hbm_kernel_fracs(env):
    """Live CUDA-event microbench of the UNet's HBM-bound kernels at the C4 shapes (32 UNet samples): algorithmic bytes / time vs the
    measured copy bandwidth.  Planes <= 84 MB partly live in the 126 MB L2 between passes, exactly as inside the step."""
    from dreamllm_b200 import ops
    dev = env.dev
    peak = env.peaks["hbm"]
    g = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *s: (torch.randn(*s, device=dev, generator=g) * 0.5).to(BF)   # noqa: E731
    out = {}

    def rec(name, fn, nbytes, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / iters * 1e-3
        out[name] = {"us": round(t * 1e6, 1), "gbps": round(nbytes / t / 1e9, 1), "frac": round(nbytes / t / 1e9 / peak, 3)}
    N = 32
    for C, HW in ((320, 4096), (640, 1024), (1280, 256)):
        Tn = N * HW
        xl, wl, bl = rnd(Tn, C), rnd(C), rnd(C)
        xg = xl.view(N, HW, C)
        rec(f"groupnorm_silu[{N}x{HW}x{C}]", lambda: ops.groupnorm(xg, wl, bl, 32, 1e-5, True), 3 * Tn * C * 2)
        rec(f"layernorm_fwd[{Tn}x{C}]", lambda: ops.layernorm_fwd(xl, wl, bl, 1e-5), 2 * Tn * C * 2)
        ff = rnd(Tn, 8 * C)
        rec(f"geglu[{Tn}x{4 * C}]", lambda: ops.geglu(ff), 3 * Tn * 4 * C * 2)
        del xl, ff
    x2 = rnd(N, 32, 32, 640)
    rec("upsample2x[32x32x32x640]", lambda: ops.upsample2x(x2), 5 * x2.numel() * 2)
    a = rnd(N, 64, 64, 320)
    rec("concat_channels[32x64x64x(320+320)]", lambda: ops.concat_channels(a, a), 4 * a.numel() * 2)
    return out


def run_c4(env, steps_inf=50, bs=16, Q=77, guidance=7.5, runs=3):
    from dreamllm_b200 import ops
    from dreamllm_b200.modeling_plugins import StableDiffusionHead
    from dreamllm_b200.unet import DenoiseLoop
    dev = env.dev
    torch.manual_seed(0)
    old = torch.get_default_dtype()
    torch.set_default_dtype(BF)
    with torch.device(dev):
        head = StableDiffusionHead(None)
    torch.set_default_dtype(old)
    g = torch.Generator(device=dev).manual_seed(1 + env.rank)
    pos = torch.randn(bs, Q, H, device=dev, generator=g).to(BF)
    neg = torch.randn(bs, Q, H, device=dev, generator=g).to(BF)
    cond = torch.cat([head.projector(neg)[-1], head.projector(pos)[-1]])
    loop = DenoiseLoop(head.unet, cond, steps_inf, guidance, "ddim", height=512, width=512, whole_loop_graph=True)
    ops.LAUNCHES.reset()
    log("  c4: capturing the whole 50-step loop into one CUDA graph")
    loop.run()
    torch.cuda.synchronize()
    log("  c4: captured + first replay done")
    launches = ops.LAUNCHES.count
    times = []
    for _ in range(runs):
        loop.reset()
        times.append(env.timed(loop.run, 1))
    ms = statistics.median(times)
    samples = 2 * bs
    flop = UNET_GF_PER_SAMPLE * samples * steps_inf
    pk = env.peaks
    hbm = hbm_kernel_fracs(env)
    worst = min(hbm.items(), key=lambda kv: kv[1]["frac"])
    finite = bool(torch.isfinite(loop.latents).all())
    del loop, head
    return {"workload": f"BASELINE.json configs[3]: SD-2.1 UNet 64x64 latents, {steps_inf}-step DDIM, {Q} dream-query embeddings, bs={bs}/GPU, "
                        f"guidance {guidance} ({samples} UNet samples/step), whole loop = ONE CUDA graph",
            "ms_total": ms, "ms_per_denoise_step": ms / steps_inf, "images_per_s": bs * env.world / (ms / 1e3),
            "pixels_per_s": bs * env.world * 512 * 512 / (ms / 1e3), "gpu_launches_captured": launches, "finite": finite,
            "roofline": {"bound": "tensor", "scope": "whole 50-step loop", "algorithmic_pflop": flop / 1e15,
                         "achieved": flop / 1e12 / (ms / 1e3), "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                         "frac": flop / 1e12 / (ms / 1e3) / pk["tf_sustained"]},
            "hbm_roofline": {"bound": "hbm", "peak": pk["hbm"], "unit": "GB/s", "kernels": hbm, "worst": worst[0], "frac": worst[1]["frac"]}}


def run_c3(env, model, steps, warmup):
    from types import SimpleNamespace

    from dreamllm_b200.clip_vision import CLIPVisionConfigLite
    from dreamllm_b200.collator import DataCollatorForDreamLLMDataset, to_device
    from dreamllm_b200.modeling_plugins import CLIPVisionEmbedding
    dev = env.dev
    B, TXT, R = 4, 1024, 336
    old = torch.get_default_dtype()
    torch.set_default_dtype(BF)
    with torch.device(dev):
        clip = CLIPVisionEmbedding(CLIPVisionConfigLite(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                                                        image_size=R, patch_size=14), projector_type="linear", embed_hidden_size=H)
    torch.set_default_dtype(old)
    model.model.attach_plugins(clip, None, image_start_id=IM_START, dream_start_id=DREAM_START)
    for n, p in model.named_parameters():
        p.requires_grad_(not n.startswith("stable_diffusion_head") and "dream_embedding" not in n and "clip_vision_model" not in n)
    model.train()
    P = clip.embed_len
    collate = DataCollatorForDreamLLMDataset(SimpleNamespace(pad_token_id=32000), image_start_id=IM_START, clip_embed_len=P, pin_memory=True)
    g = torch.Generator().manual_seed(1234 + env.rank)
    examples = []
    for _ in range(B):
        text = torch.randint(3, 32000, (TXT,), generator=g).tolist()
        ids = torch.tensor([1, IM_START] + [IM_PATCH] * P + [IM_END] + text + [2])
        labels = ids.clone()
        labels[: P + 3] = -100                                    # image positions carry no LM loss (builder_dreamllm.py:197-200)
        examples.append(dict(input_ids=ids, attention_mask=torch.ones_like(ids), labels=labels,
                             images=torch.randn(1, 3, R, R, generator=g).to(BF), images_dm=None))
    host = collate(examples)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in host.items()}
    tokens = host["num_tokens"] * env.world
    keep = ("input_ids", "images", "attention_mask", "labels", "input_ids_cpu", "splice_plan", "attention_mask_has_padding", "seqlens",
            "shifted_labels")
    params = [p for p in model.parameters() if p.requires_grad]

    def step():
        for p in params:
            p.grad = None
        out = model(**to_device({k: host[k] for k in keep}, dev))      # H2D every step (ids, images, index maps)
        out.loss.backward()
        return float(out.loss.item())                                  # D2H every step
    for _ in range(warmup):
        step()
    total = env.timed(step, steps)
    for p in params:
        p.grad = None
    ms = total / steps
    Sx = int(host["input_ids"].shape[1])
    fl = 3 * llm_fwd_flops(B * Sx, Sx) + B * (365.3e9 + 0.7e9 + 4.8e9)
    return {"workload": f"BASELINE.json configs[2]: CLIP ViT-L/14-336 (frozen) + linear projector + Vicuna-7B, {P} visual + {TXT} text tokens, bs={B}/GPU, "
                        f"seq {Sx}, fwd+bwd through the index-map collator incl. H2D of ids/images and loss D2H (no cross-rank gradient sum in this record)",
            "ms_per_step": ms, "tokens_per_s": tokens / ms * 1e3,
            "roofline": {"bound": "tensor", "scope": "whole step", "algorithmic_tflop_per_step_per_gpu": fl / 1e12,
                         "achieved": fl / 1e12 / (ms / 1e3), "peak": env.peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": fl / 1e12 / (ms / 1e3) / env.peaks["tf_sustained"]}}


def run_c1(env, model):
    """configs[0] on the GPU: one decoder layer of the 7B model, fwd+bwd, hidden 4096 seq 512 bs 1 (628.14 GFLOP, SURVEY §8d)."""
    layer = model.model.layers[0]
    for p in layer.parameters():
        p.requires_grad_(True)
    g = torch.Generator(device=env.dev).manual_seed(0)
    x = torch.randn(1, 512, H, device=env.dev, generator=g).to(BF).requires_grad_(True)

    def step():
        x.grad = None
        for p in layer.parameters():
            p.grad = None
        layer(x)[0].float().pow(2).mean().backward()
    for _ in range(10):
        step()
    # ~40 launches of 10-60 us each: the eager figure is partly host-launch-bound and noisy right after model construction, so it is the
    # median of 5 batches of 20; the same step captured as ONE CUDA graph (how the training loops run it) is reported beside it
    eager = sorted(env.timed(step, 20) / 20 for _ in range(5))
    ms_eager = eager[2]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
        graph = torch.cuda.CUDAGraph()
        x.grad = None
        for p in layer.parameters():
            p.grad = None
        with torch.cuda.graph(graph, stream=side):
            layer(x)[0].float().pow(2).mean().backward()
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(5):
        graph.replay()
    ms = sorted(env.timed(graph.replay, 20) / 20 for _ in range(5))[2]
    del graph
    for p in layer.parameters():
        p.grad = None
    fl = 628.14e9
    return {"workload": "BASELINE.json configs[0]: single DreamLLMDecoderLayer fwd+bwd, hidden=4096 seq=512 bs=1", "gpu_ms": ms,
            "gpu_ms_eager": ms_eager, "launch_mode": "fwd+bwd captured in one CUDA graph (median of 5 x 20 replays); eager median beside it",
            "roofline": {"bound": "tensor", "achieved": fl / 1e12 / (ms / 1e3), "peak": env.peaks["tf_burst"], "unit": "TFLOP/s",
                         "frac": fl / 1e12 / (ms / 1e3) / env.peaks["tf_burst"],
                         "note": "M = 512: the 512 x 4096 outputs are 64 tiles on 148 SMs (< 1/2 wave) — latency-, not tensor-bound (SURVEY §7)"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=L, help="dev only: fewer layers (reported in config; not a valid bench)")
    ap.add_argument("--bs", type=int, default=8, help="c2 batch per GPU")
    ap.add_argument("--seq", type=int, default=2048, help="c2 sequence length")
    ap.add_argument("--only", default="", help="dev only: comma list of records to run (c5,c2,c4,c3,c1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fast", action="store_true", help="skip the slow CPU legs (c1 in full, c2 sample)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, updated trainable parameters and gradients of the last timed "
                                                          "headline step to DIR/*.npy (fp32); inputs are seeded, identical run to run")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: dreamllm_b200 has no CPU fallback")
    env = Env(args)
    only = set(filter(None, args.only.split(","))) or {"c5", "c2", "c4", "c3", "c1"}
    log("building the 7B LLM")
    model = build_llm(env, args.layers)
    log("LLM built")
    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
    rec = {}
    marks = {}
    # order: c1 / c2 / c3 need every LLM weight trainable; c5 re-freezes the LLM, so it runs after them; c4 is independent
    for name, fn in (("c1", lambda: run_c1(env, model)),
                     ("c2", lambda: run_c2(env, model, args.steps, args.warmup, args.bs, args.seq, args.layers)),
                     ("c3", lambda: run_c3(env, model, args.steps, 2)),
                     ("c5", lambda: run_c5(env, model, args.steps, args.warmup, args.dump_outputs if rank == 0 else None)),
                     ("c4", lambda: run_c4(env))):
        if name not in only:
            continue
        lo = sampler.mark()
        log(f"{name}: start")
        try:
            rec[name] = fn()
            log(f"{name}: done")
        except Exception as ex:  # noqa: BLE001  (a failing secondary record must not lose the headline line)
            if name == "c5":
                raise
            rec[name] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        marks[name] = (lo, sampler.mark())
    clocks_all = sampler.stop() if rank == 0 else None
    if rank != 0:
        if env.world > 1:
            env.dist.destroy_process_group()
        return

    c5 = rec.get("c5")
    head_rec = c5 if c5 is not None else next(iter(rec.values()))
    line = {"metric": METRIC, "value": head_rec.get("value"), "unit": UNIT, "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head_rec.get("ms_per_step"), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (uniform token ids, U(-1,1) images, random-init N(0,0.02) weights)", "config": c5_config(args, env.world),
            "e2e": head_rec.get("e2e"), "clocks": sampler.summary(*marks.get("c5", (0, None))) if marks else clocks_all,
            "clocks_whole_run": clocks_all}
    if c5 is not None:
        line["tokens_per_s"], line["pixels_per_s"] = c5["tokens_per_s"], c5["pixels_per_s"]
        line["gpu_launches"] = int(c5["launches_per_step"] * args.steps * 2)       # timed device-resident + e2e regions
        line["launch_mode"] = c5["launch_mode"]
        line["step_roofline"] = c5["roofline"]
    # the dominant kernel of the path is the tcgen05 GEMM; its live-event roofline comes from the c2 record (large-M launches)
    if "c2" in rec and "roofline" in rec["c2"]:
        line["roofline"] = rec["c2"]["roofline"]
    elif c5 is not None:
        line["roofline"] = c5["roofline"]
    for k in ("c2", "c4", "c3", "c1"):
        if k in rec:
            line[k] = rec[k]
            if k in marks:
                line[k]["clocks"] = sampler.summary(*marks[k])
    if env.world == 1 and not args.no_cpu_baseline:
        log("cpu_baseline (oracle port, one sample of the headline workload): start")
        cb = cpu_reference_c5(warm=1, iters=3)
        log("cpu_baseline: done")
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if not args.fast:
            if "c1" in line and "error" not in line["c1"]:
                line["c1"]["cpu"] = cpu_reference_c1()
                line["c1"]["speedup_vs_cpu_bf16"] = line["c1"]["cpu"]["bf16_ms"] / line["c1"]["gpu_ms"]
            if "c2" in line and "error" not in line["c2"]:
                line["c2"]["cpu_baseline"] = cpu_reference_c2(args.seq, warm=1, iters=3)
    print(json.dumps(line), flush=True)
    if env.world > 1:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
