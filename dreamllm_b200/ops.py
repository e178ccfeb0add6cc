"""Thin torch-tensor wrappers over the C ABI (include/dreamllm_sm100.h).

torch is used here only for device memory and the current stream; every function hands raw device pointers to
libdreamllm_sm100.so and raises RuntimeError on a non-zero return code.  No function here has a torch / CPU
fallback: a CPU tensor is an error.
"""
from __future__ import annotations

import weakref

import torch

from ._lib import check, lib

BF16 = torch.bfloat16


class _LaunchCounter:
    """Counts OUR kernel launches (bench.py's `gpu_launches`)."""

    def __init__(self):
        self.count = 0

    def reset(self):
        self.count = 0

    def add(self, n=1):
        self.count += n


class _GemmProfile:
    """Optional live CUDA-event timing of every GEMM launch on the launching stream (bench.py roofline)."""

    def __init__(self):
        self.enabled = False
        self.records = []

    def reset(self, enabled=False):
        self.enabled = enabled
        self.records = []

    def summary(self):
        torch.cuda.synchronize()
        ms = sum(s.elapsed_time(e) for s, e, _ in self.records)
        fl = sum(f for _, _, f in self.records)
        return {"ms": ms, "tflops": (fl / 1e9 / ms) if ms > 0 else None, "n": len(self.records)}


LAUNCHES = _LaunchCounter()
PROFILE = _GemmProfile()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t) -> int:
    return 0 if t is None else t.data_ptr()


def _chk_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("dreamllm_b200 ops need CUDA tensors (there is no CPU fallback)")


# ----------------------------------------------------------------------------------------------- GEMM
ACT_NONE, ACT_QUICK_GELU, ACT_GELU, ACT_SILU = 0, 1, 2, 3


def gemm(a: torch.Tensor, b: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False, out: torch.Tensor | None = None,
         out_dtype=BF16, cta_pair: int = -1, bias: torch.Tensor | None = None, residual: torch.Tensor | None = None,
         act: int = 0) -> torch.Tensor:
    """C[M,N] = op(A) @ op(B) on tcgen05.

    a_mn=False: a is [M,K];  a_mn=True: a is [K,M] (uses a^T)
    b_mn=False: b is [N,K] (nn.Linear weight layout, C = A @ B^T);  b_mn=True: b is [K,N] (C = A @ B)
    Inputs are 2-D bf16 with unit inner stride (row stride may exceed the width: column-slice views are fine).
    """
    _chk_cuda(a, b, out)
    assert a.dtype == BF16 and b.dtype == BF16 and a.dim() == 2 and b.dim() == 2
    assert a.stride(1) == 1 and b.stride(1) == 1
    if a_mn:
        K, M = a.shape
    else:
        M, K = a.shape
    if b_mn:
        Kb, N = b.shape
    else:
        N, Kb = b.shape
    assert K == Kb, f"contraction mismatch {K} vs {Kb}"
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=out_dtype)
    assert out.shape == (M, N) and out.stride(1) == 1 and out.dtype in (BF16, torch.float32)
    if PROFILE.enabled:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    wsb = 0
    if not a_mn and out.dtype == BF16 and cta_pair < 0 and M <= 4096:          # small-M shapes: split-K when the library says it pays
        wsb = lib().dllm_gemm_splitk_workspace_bytes(M, N, K)
    if wsb:
        _chk_cuda(bias, residual)
        ldr = 0
        if bias is not None:
            assert bias.dtype == BF16 and bias.is_contiguous() and bias.numel() == N
        if residual is not None:
            assert residual.dtype == BF16 and residual.shape == (M, N) and residual.stride(1) == 1
            ldr = residual.stride(0)
        ws = torch.empty(wsb, device=a.device, dtype=torch.uint8)
        rc = lib().dllm_gemm_bf16_ws(_p(a), _p(b), _p(out), M, N, K, a.stride(0), b.stride(0), out.stride(0), int(b_mn), _p(bias),
                                     _p(residual), ldr, int(act), _p(ws), wsb, _stream())
        LAUNCHES.add(1)
    elif bias is None and residual is None and act == 0:
        rc = lib().dllm_gemm_bf16(_p(a), _p(b), _p(out), M, N, K, a.stride(0), b.stride(0), out.stride(0), int(a_mn),
                                  int(b_mn), int(out.dtype == torch.float32), cta_pair, _stream())
    else:
        _chk_cuda(bias, residual)
        if bias is not None:
            assert bias.dtype == BF16 and bias.is_contiguous() and bias.numel() == N
        ldr = 0
        if residual is not None:
            assert residual.dtype == BF16 and residual.shape == (M, N) and residual.stride(1) == 1
            ldr = residual.stride(0)
        rc = lib().dllm_gemm_bf16_ex(_p(a), _p(b), _p(out), M, N, K, a.stride(0), b.stride(0), out.stride(0), int(a_mn),
                                     int(b_mn), int(out.dtype == torch.float32), cta_pair, _p(bias), _p(residual), ldr,
                                     int(act), _stream())
    check(rc, "dllm_gemm_bf16")
    if PROFILE.enabled:
        e1.record()
        PROFILE.records.append((e0, e1, 2.0 * M * N * K))
    LAUNCHES.add(1)
    return out


def linear(x2d: torch.Tensor, weight: torch.Tensor, out=None, out_dtype=BF16, bias=None, residual=None, act=0) -> torch.Tensor:
    """y = act(x @ W^T + bias) + residual (nn.Linear forward with the fused epilogue)."""
    return gemm(x2d, weight, out=out, out_dtype=out_dtype, bias=bias, residual=residual, act=act)


def geglu_permute(weight: torch.Tensor, bias: torch.Tensor | None):
    """`GEGLU.proj` weight [2I, K] / bias [2I] -> row order [64 value rows | their 64 gate rows] per 128-row group (what `linear_geglu`
    expects).  I % 64 == 0."""
    I2, K = weight.shape
    inner = I2 // 2
    assert inner % 64 == 0
    wp = torch.stack([weight[:inner].view(inner // 64, 64, K), weight[inner:].view(inner // 64, 64, K)], dim=1).reshape(I2, K).contiguous()
    bp = None
    if bias is not None:
        bp = torch.stack([bias[:inner].view(inner // 64, 64), bias[inner:].view(inner // 64, 64)], dim=1).reshape(I2).contiguous()
    return wp, bp


def linear_geglu(x2d: torch.Tensor, w_perm: torch.Tensor, b_perm: torch.Tensor | None) -> torch.Tensor:
    """out[M, I] = h * gelu(gate), [h | gate] = x @ W^T + b, fused into the GEMM epilogue (weights from `geglu_permute`)."""
    _chk_cuda(x2d, w_perm, b_perm)
    M, K = x2d.shape
    N = w_perm.shape[0]
    assert x2d.dtype == BF16 and w_perm.dtype == BF16 and x2d.stride(1) == 1 and w_perm.is_contiguous() and w_perm.shape[1] == K
    out = torch.empty((M, N // 2), device=x2d.device, dtype=BF16)
    if PROFILE.enabled:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    check(lib().dllm_gemm_bf16_geglu(_p(x2d), _p(w_perm), _p(b_perm), _p(out), M, N, K, x2d.stride(0), w_perm.stride(0), out.stride(0),
                                     _stream()), "dllm_gemm_bf16_geglu")
    if PROFILE.enabled:
        e1.record()
        PROFILE.records.append((e0, e1, 2.0 * M * N * K))
    LAUNCHES.add(1)
    return out


def linear_dgrad(dy2d: torch.Tensor, weight: torch.Tensor, out=None) -> torch.Tensor:
    """dx = dy @ W."""
    return gemm(dy2d, weight, b_mn=True, out=out)


def linear_wgrad(dy2d: torch.Tensor, x2d: torch.Tensor, out=None, out_dtype=BF16) -> torch.Tensor:
    """dW = dy^T @ x."""
    return gemm(dy2d, x2d, a_mn=True, b_mn=True, out=out, out_dtype=out_dtype)


# ----------------------------------------------------------------------------------------------- norms
def rmsnorm_fwd(x2d, weight, eps, add=None, want_sum=True):
    """returns (y, rstd, x_sum) — x_sum = bf16(x + add) when `add` is given else x itself."""
    _chk_cuda(x2d, weight, add)
    T, H = x2d.shape
    assert x2d.is_contiguous() and x2d.dtype == BF16 and weight.dtype == BF16
    y = torch.empty_like(x2d)
    rstd = torch.empty(T, device=x2d.device, dtype=torch.float32)
    x_out = torch.empty_like(x2d) if add is not None else None
    if add is not None:
        assert add.is_contiguous() and add.shape == x2d.shape
    check(lib().dllm_rmsnorm_fwd(_p(x2d), _p(add), _p(weight), _p(x_out), _p(y), _p(rstd), T, H, float(eps), _stream()),
          "dllm_rmsnorm_fwd")
    LAUNCHES.add(1)
    return y, rstd, (x_out if add is not None else x2d)


def rmsnorm_bwd(dy2d, x2d, weight, rstd, dres=None, need_dw=True):
    """returns (dx, dweight|None); dx includes `dres` (the residual-branch gradient) when given."""
    _chk_cuda(dy2d, x2d, weight, rstd, dres)
    T, H = x2d.shape
    assert dy2d.is_contiguous() and x2d.is_contiguous()
    dx = torch.empty_like(x2d)
    dw = torch.empty_like(weight) if need_dw else None
    wsb = lib().dllm_rmsnorm_bwd_workspace_bytes(T, H) if need_dw else 0
    ws = torch.empty(max(wsb, 4), device=x2d.device, dtype=torch.uint8)
    check(lib().dllm_rmsnorm_bwd(_p(dy2d), _p(x2d), _p(weight), _p(rstd), _p(dres), _p(dx), _p(dw), 0, _p(ws), wsb, T, H,
                                 _stream()), "dllm_rmsnorm_bwd")
    LAUNCHES.add(3 if need_dw else 1)
    return dx, dw


# ----------------------------------------------------------------------------------------------- rope / swiglu / add
def rope_(buf2d, cos_t, sin_t, pos_i32, heads_total, head_dim, backward=False):
    """In place on the first heads_total*head_dim columns of buf2d ([T, ld])."""
    _chk_cuda(buf2d, cos_t, sin_t, pos_i32)
    T = buf2d.shape[0]
    assert buf2d.stride(1) == 1 and pos_i32.dtype == torch.int32 and pos_i32.numel() == T
    assert cos_t.dtype == BF16 and cos_t.is_contiguous() and cos_t.shape[1] == head_dim
    check(lib().dllm_rope_inplace(_p(buf2d), _p(cos_t), _p(sin_t), _p(pos_i32), buf2d.stride(0), T, heads_total, head_dim,
                                  -1 if backward else 1, _stream()), "dllm_rope_inplace")
    LAUNCHES.add(1)
    return buf2d


def swiglu_fwd(gu2d, inter):
    _chk_cuda(gu2d)
    T = gu2d.shape[0]
    assert gu2d.shape[1] == 2 * inter and gu2d.stride(1) == 1
    act = torch.empty((T, inter), device=gu2d.device, dtype=BF16)
    check(lib().dllm_swiglu_fwd(_p(gu2d), _p(act), gu2d.stride(0), T, inter, _stream()), "dllm_swiglu_fwd")
    LAUNCHES.add(1)
    return act


def swiglu_bwd(dact2d, gu2d, inter, out=None):
    _chk_cuda(dact2d, gu2d)
    T = gu2d.shape[0]
    assert dact2d.is_contiguous() and gu2d.is_contiguous()
    dgu = torch.empty_like(gu2d) if out is None else out
    check(lib().dllm_swiglu_bwd(_p(dact2d), _p(gu2d), _p(dgu), gu2d.stride(0), T, inter, _stream()), "dllm_swiglu_bwd")
    LAUNCHES.add(1)
    return dgu


def add(a, b, out=None):
    _chk_cuda(a, b)
    assert a.is_contiguous() and b.is_contiguous() and a.shape == b.shape
    out = torch.empty_like(a) if out is None else out
    check(lib().dllm_add_bf16(_p(a), _p(b), _p(out), a.numel(), _stream()), "dllm_add_bf16")
    LAUNCHES.add(1)
    return out


# ----------------------------------------------------------------------------------------------- loss / embedding
def cross_entropy_(logits2d, shifted_labels, dloss=1.0, write_grad=True):
    """loss (fp32 scalar tensor); when write_grad, logits2d is overwritten with dloss * dloss/dlogits."""
    _chk_cuda(logits2d, shifted_labels)
    T, V = logits2d.shape
    assert logits2d.dtype == BF16 and logits2d.stride(1) == 1 and shifted_labels.dtype == torch.int64
    assert shifted_labels.is_contiguous() and shifted_labels.numel() == T
    loss = torch.empty(1, device=logits2d.device, dtype=torch.float32)
    ws = torch.empty(T + 2, device=logits2d.device, dtype=torch.float32)
    check(lib().dllm_cross_entropy(_p(logits2d), _p(shifted_labels), _p(loss), float(dloss), _p(ws), logits2d.stride(0), T,
                                   V, int(write_grad), _stream()), "dllm_cross_entropy")
    LAUNCHES.add(3)
    return loss[0]


def embedding_fwd(ids, weight):
    _chk_cuda(ids, weight)
    ids = ids.contiguous()
    T = ids.numel()
    H = weight.shape[1]
    out = torch.empty((*ids.shape, H), device=weight.device, dtype=weight.dtype)
    check(lib().dllm_embedding_fwd(_p(ids), _p(weight), _p(out), T, H, _stream()), "dllm_embedding_fwd")
    LAUNCHES.add(1)
    return out


def embedding_bwd(ids, dy2d, vocab, out=None, padding_idx=None):
    """dW[v] = sum of dy rows whose id is v (deterministic: ids sorted, one segment per row).  `out` = preallocated [vocab, H] (e.g. the
    gradient-bucket slice); `padding_idx` row gets no gradient, as nn.Embedding (reference modeling_dreamllm.py:814)."""
    _chk_cuda(ids, dy2d, out)
    T, H = dy2d.shape
    sorted_ids, order = torch.sort(ids.reshape(-1), stable=True)
    if out is None:
        dW = torch.zeros((vocab, H), device=dy2d.device, dtype=dy2d.dtype)
    else:
        assert out.shape == (vocab, H) and out.is_contiguous() and out.dtype == dy2d.dtype
        dW = out.zero_()
    check(lib().dllm_embedding_bwd(_p(sorted_ids), _p(order), _p(dy2d), _p(dW), T, H, 0, _stream()), "dllm_embedding_bwd")
    LAUNCHES.add(1)
    if padding_idx is not None and 0 <= int(padding_idx) < vocab:
        dW[int(padding_idx)].zero_()
    return dW


# ----------------------------------------------------------------------------------------------- attention
def attn_fwd(q, k, v, causal=True, seqlens=None, scale=None):
    """q,k,v: [B, S, nh, d] views (last two dims dense, token stride shared) — e.g. slices of the fused qkv buffer.
    returns (out [B,S,nh*d], lse [B,nh,S])."""
    _chk_cuda(q, k, v, seqlens)
    B, S, nh, d = q.shape
    for t in (q, k, v):
        assert t.dtype == BF16 and t.stride(3) == 1 and t.stride(2) == d and t.stride(0) == S * t.stride(1)
    assert q.stride(1) == k.stride(1) == v.stride(1)
    out = torch.empty((B, S, nh * d), device=q.device, dtype=BF16)
    lse = torch.empty((B, nh, S), device=q.device, dtype=torch.float32)
    scale = float(d) ** -0.5 if scale is None else float(scale)
    check(lib().dllm_attn_fwd(_p(q), _p(k), _p(v), _p(out), _p(lse), _p(seqlens), B, S, nh, d, q.stride(1), nh * d,
                              int(causal), scale, _stream()), "dllm_attn_fwd")
    LAUNCHES.add(1)
    return out, lse


def attn_bwd(dout, q, k, v, out, lse, dq, dk, dv, causal=True, seqlens=None, scale=None):
    """dq/dk/dv: [B,S,nh,d] views to write into (e.g. slices of a fused dqkv buffer)."""
    _chk_cuda(dout, q, k, v, out, lse, dq, dk, dv, seqlens)
    B, S, nh, d = q.shape
    assert dout.is_contiguous() and out.is_contiguous()
    assert dq.stride(1) == dk.stride(1) == dv.stride(1)
    scale = float(d) ** -0.5 if scale is None else float(scale)
    wsb = lib().dllm_attn_bwd_workspace_bytes(B, S, nh, d)
    ws = torch.empty(max(wsb, 4), device=q.device, dtype=torch.uint8)
    check(lib().dllm_attn_bwd(_p(dout), _p(q), _p(k), _p(v), _p(out), _p(lse), _p(dq), _p(dk), _p(dv), _p(seqlens), _p(ws),
                              wsb, B, S, nh, d, q.stride(1), nh * d, dq.stride(1), int(causal), scale, _stream()),
          "dllm_attn_bwd")
    LAUNCHES.add(3)
    return dq, dk, dv


# ----------------------------------------------------------------------------------------------- CLIP / splice helpers
def layernorm_fwd(x2d, weight, bias, eps):
    _chk_cuda(x2d, weight, bias)
    T, H = x2d.shape
    assert x2d.is_contiguous() and x2d.dtype == BF16
    y = torch.empty_like(x2d)
    check(lib().dllm_layernorm_fwd(_p(x2d), _p(weight), _p(bias), _p(y), T, H, float(eps), _stream()), "dllm_layernorm_fwd")
    LAUNCHES.add(1)
    return y


def clip_patchify(images, patch, kpad):
    """images [N,3,R,R] bf16 NCHW -> [N*(R/patch)^2, kpad] unfolded patches (conv-weight flatten order, zero padded)."""
    _chk_cuda(images)
    N, C, R, R2 = images.shape
    assert C == 3 and R == R2 and images.is_contiguous() and images.dtype == BF16
    G = R // patch
    out = torch.empty((N * G * G, kpad), device=images.device, dtype=BF16)
    check(lib().dllm_clip_patchify(_p(images), _p(out), N, R, patch, kpad, _stream()), "dllm_clip_patchify")
    LAUNCHES.add(1)
    return out


def clip_assemble(patches2d, cls, pos, N, P):
    _chk_cuda(patches2d, cls, pos)
    C = patches2d.shape[1]
    out = torch.empty((N, P + 1, C), device=patches2d.device, dtype=BF16)
    check(lib().dllm_clip_assemble(_p(patches2d), _p(cls), _p(pos), _p(out), N, P, C, _stream()), "dllm_clip_assemble")
    LAUNCHES.add(1)
    return out


def copy_rows_(dst2d, dst_idx, src2d, src_idx, accumulate=False):
    _chk_cuda(dst2d, dst_idx, src2d, src_idx)
    assert dst2d.is_contiguous() and src2d.is_contiguous() and dst_idx.dtype == torch.int32 and src_idx.dtype == torch.int32
    R, H = dst_idx.numel(), dst2d.shape[1]
    assert src_idx.numel() == R and src2d.shape[1] == H
    check(lib().dllm_copy_rows(_p(dst2d), _p(dst_idx), _p(src2d), _p(src_idx), R, H, int(accumulate), _stream()), "dllm_copy_rows")
    LAUNCHES.add(1)
    return dst2d


def segment_sum_rows(src2d, seg, rows, Q):
    _chk_cuda(src2d, seg, rows)
    H = src2d.shape[1]
    out = torch.empty((Q, H), device=src2d.device, dtype=BF16)
    check(lib().dllm_segment_sum_rows(_p(out), _p(src2d), _p(seg), _p(rows), Q, H, _stream()), "dllm_segment_sum_rows")
    LAUNCHES.add(1)
    return out


def zero_rows_(dst2d, idx):
    _chk_cuda(dst2d, idx)
    check(lib().dllm_zero_rows(_p(dst2d), _p(idx), idx.numel(), dst2d.shape[1], _stream()), "dllm_zero_rows")
    LAUNCHES.add(1)
    return dst2d


# ----------------------------------------------------------------------------------------------- UNet ops (NHWC bf16)
def attn_fwd_cross(q, k, v, scale=None):
    """q [B,Sq,nh,d], k/v [B,Skv,nh,d] (views; k and v share a token stride). Non-causal. returns out [B,Sq,nh*d]."""
    _chk_cuda(q, k, v)
    B, Sq, nh, d = q.shape
    Skv = k.shape[1]
    assert k.stride(1) == v.stride(1) and q.stride(3) == 1 and k.stride(3) == 1 and q.stride(2) == d and k.stride(2) == d
    out = torch.empty((B, Sq, nh * d), device=q.device, dtype=BF16)
    lse = torch.empty((B, nh, Sq), device=q.device, dtype=torch.float32)
    scale = float(d) ** -0.5 if scale is None else float(scale)
    check(lib().dllm_attn_fwd_ex(_p(q), _p(k), _p(v), _p(out), _p(lse), 0, B, Sq, Skv, nh, d, q.stride(1), k.stride(1), nh * d, 0,
                                 scale, _stream()), "dllm_attn_fwd_ex")
    LAUNCHES.add(1)
    return out


def conv3x3_plane_supported(H: int, W: int) -> bool:
    """The planes `dllm_conv3x3_nhwc` accepts: a 128-pixel tile is Wb x Hb x Nb pixels, so W must divide 128 or be a multiple of it,
    and H must be a multiple of Hb = 128 / W (or divide it, when one tile spans several whole images)."""
    if H <= 0 or W <= 0 or (W % 128 if W > 128 else 128 % W):
        return False
    hb = 1 if W >= 128 else 128 // W
    return (hb % H == 0) if hb > H else (H % hb == 0)


def conv3x3(x_nhwc, w_k, bias=None, rowbias=None, residual=None):
    """x [N,H,W,Cin] bf16 contiguous; w_k [Cout, 9*Cin] ((r,s,c)-major); returns [N,H,W,Cout]."""
    _chk_cuda(x_nhwc, w_k, bias, rowbias, residual)
    N, H, W, Cin = x_nhwc.shape
    Cout = w_k.shape[0]
    assert x_nhwc.is_contiguous() and w_k.is_contiguous() and w_k.shape[1] == 9 * Cin
    y = torch.empty((N, H, W, Cout), device=x_nhwc.device, dtype=BF16)
    if residual is not None:
        assert residual.is_contiguous() and residual.numel() == y.numel()
    if rowbias is not None:
        assert rowbias.is_contiguous() and rowbias.shape == (N, Cout)
    wsb = lib().dllm_conv3x3_splitk_workspace_bytes(N, H, W, Cin, Cout) if N * H * W <= 4096 else 0
    if wsb:                                                    # small planes (8x8 / 16x16 of a few samples): split-K + reduce
        ws = torch.empty(wsb, device=x_nhwc.device, dtype=torch.uint8)
        check(lib().dllm_conv3x3_nhwc_ws(_p(x_nhwc), _p(w_k), _p(y), N, H, W, Cin, Cout, _p(bias), _p(rowbias), _p(residual), _p(ws), wsb,
                                         _stream()), "dllm_conv3x3_nhwc_ws")
        LAUNCHES.add(2)
        return y
    check(lib().dllm_conv3x3_nhwc(_p(x_nhwc), _p(w_k), _p(y), N, H, W, Cin, Cout, _p(bias), _p(rowbias), _p(residual), _stream()),
          "dllm_conv3x3_nhwc")
    LAUNCHES.add(1)
    return y


def groupnorm(x_nhwc, weight, bias, groups, eps, silu, return_stats=False):
    _chk_cuda(x_nhwc, weight, bias)
    N, C = x_nhwc.shape[0], x_nhwc.shape[-1]
    HW = x_nhwc.numel() // (N * C)
    assert x_nhwc.is_contiguous()
    wsb = lib().dllm_groupnorm_workspace_bytes(N, HW, groups)
    ws = torch.empty(wsb, device=x_nhwc.device, dtype=torch.uint8)
    y = torch.empty_like(x_nhwc)
    if not return_stats:
        check(lib().dllm_groupnorm_nhwc(_p(x_nhwc), _p(weight), _p(bias), _p(y), _p(ws), wsb, N, HW, C, groups, float(eps), int(silu),
                                        _stream()), "dllm_groupnorm_nhwc")
        LAUNCHES.add(3)
        return y
    stats = torch.empty((N, groups, 2), device=x_nhwc.device, dtype=torch.float32)
    check(lib().dllm_groupnorm_stats(_p(x_nhwc), _p(stats), _p(ws), wsb, N, HW, C, groups, float(eps), _stream()), "dllm_groupnorm_stats")
    check(lib().dllm_groupnorm_apply(_p(x_nhwc), _p(weight), _p(bias), _p(stats), _p(y), N, HW, C, groups, int(silu), _stream()),
          "dllm_groupnorm_apply")
    LAUNCHES.add(3)
    return y, stats


def groupnorm_bwd(dy, x_nhwc, weight, bias, stats, groups, silu, dres=None):
    _chk_cuda(dy, x_nhwc, stats, dres)
    N, C = x_nhwc.shape[0], x_nhwc.shape[-1]
    HW = x_nhwc.numel() // (N * C)
    assert dy.is_contiguous() and x_nhwc.is_contiguous() and (dres is None or dres.is_contiguous())
    wsb = lib().dllm_groupnorm_workspace_bytes(N, HW, groups)
    ws = torch.empty(wsb, device=dy.device, dtype=torch.uint8)
    dx = torch.empty_like(x_nhwc)
    check(lib().dllm_groupnorm_bwd_nhwc(_p(dy), _p(x_nhwc), _p(weight), _p(bias), _p(stats), _p(dres), _p(dx), _p(ws), wsb, N, HW, C,
                                        groups, int(silu), _stream()), "dllm_groupnorm_bwd_nhwc")
    LAUNCHES.add(3)
    return dx


def layernorm_bwd(dy2d, x2d, weight, eps, dres=None):
    _chk_cuda(dy2d, x2d, weight, dres)
    T, H = x2d.shape
    assert dy2d.is_contiguous() and x2d.is_contiguous() and (dres is None or dres.is_contiguous())
    dx = torch.empty_like(x2d)
    check(lib().dllm_layernorm_bwd(_p(dy2d), _p(x2d), _p(weight), _p(dres), _p(dx), T, H, float(eps), _stream()), "dllm_layernorm_bwd")
    LAUNCHES.add(1)
    return dx


def geglu_bwd(dout2d, in2d):
    T, I2 = in2d.shape
    assert dout2d.is_contiguous() and in2d.is_contiguous()
    din = torch.empty_like(in2d)
    check(lib().dllm_geglu_bwd(_p(dout2d), _p(in2d), _p(din), T, I2 // 2, _stream()), "dllm_geglu_bwd")
    LAUNCHES.add(1)
    return din


def attn_bwd_cross(dout, q, k, v, out, lse, dq, dk, dv, scale=None):
    """q/dq [B,Sq,nh,d]; k,v,dk,dv [B,Skv,nh,d] views (k,v share a token stride; dk,dv share one)."""
    _chk_cuda(dout, q, k, v, out, lse, dq, dk, dv)
    B, Sq, nh, d = q.shape
    Skv = k.shape[1]
    scale = float(d) ** -0.5 if scale is None else float(scale)
    wsb = lib().dllm_attn_bwd_workspace_bytes(B, Sq, nh, d)
    ws = torch.empty(max(wsb, 4), device=q.device, dtype=torch.uint8)
    assert dout.is_contiguous() and out.is_contiguous()
    check(lib().dllm_attn_bwd_ex(_p(dout), _p(q), _p(k), _p(v), _p(out), _p(lse), _p(dq), _p(dk), _p(dv), 0, _p(ws), wsb, B, Sq, Skv,
                                 nh, d, q.stride(1), k.stride(1), nh * d, dq.stride(1), dk.stride(1), 0, scale, _stream()),
          "dllm_attn_bwd_ex")
    LAUNCHES.add(3)


def attn_fwd_cross_lse(q, k, v, scale=None):
    _chk_cuda(q, k, v)
    B, Sq, nh, d = q.shape
    Skv = k.shape[1]
    out = torch.empty((B, Sq, nh * d), device=q.device, dtype=BF16)
    lse = torch.empty((B, nh, Sq), device=q.device, dtype=torch.float32)
    scale = float(d) ** -0.5 if scale is None else float(scale)
    check(lib().dllm_attn_fwd_ex(_p(q), _p(k), _p(v), _p(out), _p(lse), 0, B, Sq, Skv, nh, d, q.stride(1), k.stride(1), nh * d, 0,
                                 scale, _stream()), "dllm_attn_fwd_ex")
    LAUNCHES.add(1)
    return out, lse


def upsample2x_bwd(dy_nhwc):
    N, H2, W2, C = dy_nhwc.shape
    dx = torch.empty((N, H2 // 2, W2 // 2, C), device=dy_nhwc.device, dtype=BF16)
    check(lib().dllm_upsample2x_bwd_nhwc(_p(dy_nhwc), _p(dx), N, H2 // 2, W2 // 2, C, _stream()), "dllm_upsample2x_bwd_nhwc")
    LAUNCHES.add(1)
    return dx


def col2im_s2(dcols2d, N, H, W, C):
    dx = torch.empty((N, H, W, C), device=dcols2d.device, dtype=BF16)
    check(lib().dllm_col2im_s2_nhwc(_p(dcols2d), _p(dx), N, H, W, C, _stream()), "dllm_col2im_s2_nhwc")
    LAUNCHES.add(1)
    return dx


def split_channels(x_nhwc, c_first):
    """inverse of concat_channels: returns (x[..., :c_first], x[..., c_first:]) as contiguous tensors."""
    N, H, W, C = x_nhwc.shape
    rows = N * H * W
    a = torch.empty((N, H, W, c_first), device=x_nhwc.device, dtype=BF16)
    b = torch.empty((N, H, W, C - c_first), device=x_nhwc.device, dtype=BF16)
    check(lib().dllm_copy_cols2(_p(x_nhwc), _p(a), rows, C, c_first, 0, 0, c_first, _stream()), "dllm_copy_cols2")
    check(lib().dllm_copy_cols2(_p(x_nhwc), _p(b), rows, C, C - c_first, c_first, 0, C - c_first, _stream()), "dllm_copy_cols2")
    LAUNCHES.add(2)
    return a, b


def conv_out_bwd(deps_nchw_f32, weight, C):
    B, Cout, H, W = deps_nchw_f32.shape
    dx = torch.empty((B, H, W, C), device=weight.device, dtype=BF16)
    check(lib().dllm_conv_out_bwd(_p(deps_nchw_f32), _p(weight), _p(dx), B, C, H, W, Cout, _stream()), "dllm_conv_out_bwd")
    LAUNCHES.add(1)
    return dx


def timestep_embedding_batch(t_i32, dim):
    B = t_i32.numel()
    out = torch.empty((B, dim), device=t_i32.device, dtype=BF16)
    check(lib().dllm_timestep_embedding_batch(_p(t_i32), _p(out), B, dim, _stream()), "dllm_timestep_embedding_batch")
    LAUNCHES.add(1)
    return out


def add_noise(x0_f32, noise_f32, t_i32, alphas_cumprod_f32):
    out = torch.empty_like(x0_f32)
    B = x0_f32.shape[0]
    check(lib().dllm_add_noise(_p(x0_f32), _p(noise_f32), _p(t_i32), _p(alphas_cumprod_f32), _p(out), B, x0_f32.numel() // B, _stream()),
          "dllm_add_noise")
    LAUNCHES.add(1)
    return out


def mse_fwd_bwd(pred_f32, target_f32):
    loss = torch.empty(1, device=pred_f32.device, dtype=torch.float32)
    dpred = torch.empty_like(pred_f32)
    check(lib().dllm_mse_fwd_bwd(_p(pred_f32), _p(target_f32), _p(loss), _p(dpred), pred_f32.numel(), _stream()), "dllm_mse_fwd_bwd")
    LAUNCHES.add(1)
    return loss[0], dpred


def mse_minsnr_fwd_bwd(pred_f32, target_f32, t_i32, alphas_cumprod_f32, snr_gamma: float):
    """min-SNR weighted MSE (reference modeling_plugins.py:561-572): per-sample weight min(snr, gamma) / snr."""
    loss = torch.empty(1, device=pred_f32.device, dtype=torch.float32)
    dpred = torch.empty_like(pred_f32)
    B = pred_f32.shape[0]
    check(lib().dllm_mse_minsnr_fwd_bwd(_p(pred_f32), _p(target_f32), _p(t_i32), _p(alphas_cumprod_f32), float(snr_gamma), _p(loss),
                                        _p(dpred), B, pred_f32.numel() // B, _stream()), "dllm_mse_minsnr_fwd_bwd")
    LAUNCHES.add(1)
    return loss[0], dpred


def geglu(x2d):
    _chk_cuda(x2d)
    T, I2 = x2d.shape
    assert x2d.is_contiguous()
    out = torch.empty((T, I2 // 2), device=x2d.device, dtype=BF16)
    check(lib().dllm_geglu(_p(x2d), _p(out), T, I2 // 2, _stream()), "dllm_geglu")
    LAUNCHES.add(1)
    return out


def upsample2x(x_nhwc):
    N, H, W, C = x_nhwc.shape
    y = torch.empty((N, 2 * H, 2 * W, C), device=x_nhwc.device, dtype=BF16)
    check(lib().dllm_upsample2x_nhwc(_p(x_nhwc), _p(y), N, H, W, C, _stream()), "dllm_upsample2x_nhwc")
    LAUNCHES.add(1)
    return y


def im2col_s2(x_nhwc, pad=1):
    N, H, W, C = x_nhwc.shape
    out = torch.empty((N * (H // 2) * (W // 2), 9 * C), device=x_nhwc.device, dtype=BF16)
    check(lib().dllm_im2col_s2_nhwc(_p(x_nhwc), _p(out), N, H, W, C, int(pad), _stream()), "dllm_im2col_s2_nhwc")
    LAUNCHES.add(1)
    return out


def concat_channels(a_nhwc, b_nhwc):
    N, H, W, Ca = a_nhwc.shape
    Cb = b_nhwc.shape[-1]
    out = torch.empty((N, H, W, Ca + Cb), device=a_nhwc.device, dtype=BF16)
    rows = N * H * W
    check(lib().dllm_copy_cols(_p(a_nhwc), _p(out), rows, Ca, Ca + Cb, 0, _stream()), "dllm_copy_cols")
    check(lib().dllm_copy_cols(_p(b_nhwc), _p(out), rows, Cb, Ca + Cb, Ca, _stream()), "dllm_copy_cols")
    LAUNCHES.add(2)
    return out


_WCACHE = {}


def _cached_weight(key, w, build):
    """Derived weight layouts of frozen towers (built once; rebuilt if the parameter is written to, moved or replaced).

    The entry remembers WHICH tensor object it was built from (weak reference): `id(weight)` in the key, the data pointer and the version
    counter can all coincide for a new model's parameter once the old model has been freed (CPython reuses object slots, the caching
    allocator reuses blocks, and two freshly loaded parameters have the same version) — the cache then served the previous model's
    conv_in / conv_out matrices (seen as a rare, order-dependent failure of the UNet gradient test with an always identical error)."""
    ent = _WCACHE.get(key)
    tag = (w.data_ptr(), w._version, w.device, w.dtype)
    if ent is None or ent[0] != tag or ent[2]() is not w:
        with torch.no_grad():
            ent = (tag, build(w.detach()), weakref.ref(w, lambda _r, _k=key: _WCACHE.pop(_k, None)))
        _WCACHE[key] = ent
    return ent[1]


def conv_in(latents_nchw_f32, weight, bias, batch_out):
    """Conv2d(Cin <= 7, Cout, 3, pad 1) on fp32 NCHW latents / images -> NHWC bf16, as im2col ([M, 64] bf16) + tcgen05 GEMM with the bias
    epilogue (the direct kernel `dllm_conv_in` cost 1.4 ms per UNet step and 0.95 ms per VAE encode)."""
    Bs, Cin, H, W = latents_nchw_f32.shape
    Cout = weight.shape[0]
    if Cin * 9 > 64 or Cout % 8:
        y = torch.empty((batch_out, H, W, Cout), device=weight.device, dtype=BF16)
        check(lib().dllm_conv_in(_p(latents_nchw_f32), _p(weight), _p(bias), _p(y), batch_out, Bs, Cin, H, W, Cout, _stream()), "dllm_conv_in")
        LAUNCHES.add(1)
        return y

    def build(w):
        wk = torch.zeros((Cout, 64), device=w.device, dtype=BF16)
        wk[:, : Cin * 9] = w.reshape(Cout, Cin * 9).to(BF16)
        return wk
    wk = _cached_weight(("conv_in", id(weight)), weight, build)
    assert latents_nchw_f32.dtype == torch.float32 and latents_nchw_f32.is_contiguous()
    cols = torch.empty((batch_out * H * W, 64), device=weight.device, dtype=BF16)
    check(lib().dllm_im2col_in(_p(latents_nchw_f32), _p(cols), batch_out, Bs, Cin, H, W, _stream()), "dllm_im2col_in")
    LAUNCHES.add(1)
    return linear(cols, wk, bias=bias.to(BF16) if bias.dtype != BF16 else bias).view(batch_out, H, W, Cout)


def conv_out(x_nhwc, weight, bias, out=None):
    """Conv2d(C, Cout <= 8, 3, pad 1) NHWC bf16 -> fp32 NCHW, as the implicit-GEMM conv with Cout zero-padded to 8 + a channel-slicing
    layout pass (the direct kernel `dllm_conv_out` cost 0.68 ms per UNet step)."""
    N, H, W, C = x_nhwc.shape
    Cout = weight.shape[0]
    y = torch.empty((N, Cout, H, W), device=x_nhwc.device, dtype=torch.float32) if out is None else out
    if C % 64 or Cout > 8 or (W > 128 and W % 128) or (W <= 128 and 128 % W):
        check(lib().dllm_conv_out(_p(x_nhwc), _p(weight), _p(bias), _p(y), N, C, H, W, Cout, _stream()), "dllm_conv_out")
        LAUNCHES.add(1)
        return y

    def build(w):
        w8 = torch.zeros((8, 9 * C), device=w.device, dtype=BF16)
        w8[:Cout] = w.permute(0, 2, 3, 1).reshape(Cout, 9 * C).to(BF16)          # k = (r, s, c): the implicit-GEMM K order
        return w8

    def build_b(b):
        b8 = torch.zeros(8, device=b.device, dtype=BF16)
        b8[:Cout] = b.to(BF16)
        return b8
    w8 = _cached_weight(("conv_out_w", id(weight)), weight, build)
    b8 = _cached_weight(("conv_out_b", id(bias)), bias, build_b)
    y8 = conv3x3(x_nhwc, w8, bias=b8)
    check(lib().dllm_nhwc_to_nchw_f32(_p(y8), _p(y), N, H * W, 8, Cout, _stream()), "dllm_nhwc_to_nchw_f32")
    LAUNCHES.add(1)
    return y


def timestep_embedding(timesteps_i32, step_i32, B, dim):
    out = torch.empty((B, dim), device=timesteps_i32.device, dtype=BF16)
    check(lib().dllm_timestep_embedding(_p(timesteps_i32), _p(step_i32), _p(out), B, dim, _stream()), "dllm_timestep_embedding")
    LAUNCHES.add(1)
    return out


def sampler_step_(eps_f32, latents_f32, coef_f32, step_i32, guidance, use_cfg, mode=0, noise=None):
    n = latents_f32.numel()
    check(lib().dllm_sampler_step(_p(eps_f32), _p(latents_f32), _p(noise), _p(coef_f32), _p(step_i32), float(guidance), int(use_cfg),
                                  int(mode), n, _stream()), "dllm_sampler_step")
    LAUNCHES.add(2)
    return latents_f32


def softmax_rows_(x2d, scale):
    _chk_cuda(x2d)
    assert x2d.is_contiguous() and x2d.dtype == BF16
    check(lib().dllm_softmax_rows(_p(x2d), x2d.shape[0], x2d.shape[1], float(scale), _stream()), "dllm_softmax_rows")
    LAUNCHES.add(1)
    return x2d


def vae_sample(h_nchw_f32, wq, bq, z_f32, scaling):
    B, C2, H, W = h_nchw_f32.shape
    L = C2 // 2
    out = torch.empty((B, L, H, W), device=h_nchw_f32.device, dtype=torch.float32)
    check(lib().dllm_vae_sample(_p(h_nchw_f32), _p(wq), _p(bq), _p(z_f32), _p(out), B, L, H * W, float(scaling), _stream()), "dllm_vae_sample")
    LAUNCHES.add(1)
    return out


def attn_fwd_cache(q, k_cache, v_cache, kv_len, causal=True, scale=None, kv_mask=None):
    """q [B,Sq,nh,d] view; k_cache/v_cache [B, max_len, nh, d] (contiguous rows of nh*d), first kv_len rows valid.
    kv_mask: optional uint8 [B, mask_ld] (0 = padded key position), mask_ld a multiple of 64 covering kv_len."""
    _chk_cuda(q, k_cache, v_cache, kv_mask)
    B, Sq, nh, d = q.shape
    kv_rows = k_cache.shape[1]
    assert k_cache.stride(1) == v_cache.stride(1) and k_cache.stride(0) == kv_rows * k_cache.stride(1)
    out = torch.empty((B, Sq, nh * d), device=q.device, dtype=BF16)
    lse = torch.empty((B, nh, Sq), device=q.device, dtype=torch.float32)
    scale = float(d) ** -0.5 if scale is None else float(scale)
    if kv_mask is not None:
        assert kv_mask.dtype == torch.uint8 and kv_mask.dim() == 2 and kv_mask.shape[0] == B and kv_mask.stride(1) == 1
        check(lib().dllm_attn_fwd_cache_mask(_p(q), _p(k_cache), _p(v_cache), _p(out), _p(lse), _p(kv_mask), kv_mask.stride(0), B, Sq,
                                             int(kv_len), kv_rows, nh, d, q.stride(1), k_cache.stride(1), nh * d, int(causal), scale,
                                             _stream()), "dllm_attn_fwd_cache_mask")
    else:
        check(lib().dllm_attn_fwd_cache(_p(q), _p(k_cache), _p(v_cache), _p(out), _p(lse), B, Sq, int(kv_len), kv_rows, nh, d, q.stride(1),
                                        k_cache.stride(1), nh * d, int(causal), scale, _stream()), "dllm_attn_fwd_cache")
    LAUNCHES.add(1)
    return out


# ------------------------------------------------------------------------------------------------ optimizer shard (SURVEY §8f row 4)
_SUMSQ_WS = {}


def sumsq_bf16_(x_bf16, out_f32, accumulate: bool = True):
    """out[0] (+)= sum(x^2) in fp32 over a flat bf16 vector (numel % 8 == 0); deterministic two-stage reduction."""
    _chk_cuda(x_bf16, out_f32)
    assert x_bf16.dtype == BF16 and x_bf16.is_contiguous() and out_f32.dtype == torch.float32
    dev = x_bf16.device
    ws = _SUMSQ_WS.get(dev)
    if ws is None:
        ws = _SUMSQ_WS[dev] = torch.empty(lib().dllm_sumsq_workspace_bytes(), dtype=torch.uint8, device=dev)
    check(lib().dllm_sumsq_bf16(_p(x_bf16), x_bf16.numel(), _p(out_f32), int(accumulate), _p(ws), ws.numel(), _stream()),
          "dllm_sumsq_bf16")
    LAUNCHES.add(2)
    return out_f32


def adamw_step_(grad_bf16, param_bf16, exp_avg, exp_avg_sq, master_f32, *, lr, beta1, beta2, eps, weight_decay, step,
                grad_sumsq=None, max_grad_norm=0.0):
    """One fused AdamW step over a flat shard (reference: torch.optim.AdamW via HF Trainer `optim="adamw_torch"`).
    master_f32 is None  -> bf16-state mode: param / exp_avg / exp_avg_sq are bf16, per-op bf16 rounding as the reference's optimizer.
    master_f32 is given -> fp32 master / exp_avg / exp_avg_sq; param (bf16) is rewritten from the updated master."""
    _chk_cuda(grad_bf16, param_bf16, exp_avg, exp_avg_sq)
    n = grad_bf16.numel()
    bf16_state = master_f32 is None
    st = BF16 if bf16_state else torch.float32
    assert grad_bf16.dtype == BF16 and param_bf16.dtype == BF16 and exp_avg.dtype == st and exp_avg_sq.dtype == st
    assert param_bf16.numel() == n and exp_avg.numel() == n and exp_avg_sq.numel() == n
    assert all(t.is_contiguous() for t in (grad_bf16, param_bf16, exp_avg, exp_avg_sq))
    if not bf16_state:
        _chk_cuda(master_f32)
        assert master_f32.dtype == torch.float32 and master_f32.numel() == n and master_f32.is_contiguous()
    check(lib().dllm_adamw_step(_p(grad_bf16), _p(master_f32), _p(exp_avg), _p(exp_avg_sq), _p(param_bf16), n, int(bf16_state),
                                float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step), _p(grad_sumsq),
                                float(max_grad_norm), _stream()), "dllm_adamw_step")
    LAUNCHES.add(1)
