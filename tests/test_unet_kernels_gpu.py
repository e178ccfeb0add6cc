"""Every kernel of the diffusion side (UNet / VAE) against the same operation in float64 on the same bf16 inputs, element by element.

The whole-network tests (test_unet_gpu.py, test_sd_head_gpu.py) compare mean errors over a full UNet or VAE output and cannot see a
wrong halo column at a tile seam, a bad partial tile or a wrong group at a straddling vector.  Here each kernel is checked at the worst
element, at the shapes and tile geometries the real-width UNet and VAE launch (the coverage test at the end keeps the tables honest).

Bounds.  Where a kernel documents its bf16 rounding points the reference rounds at the same points, and the bound is a few bf16 ulps
of the value at each rounding point plus c * 2^-24 * sum|terms| for the fp32 accumulations.  Where the rounding points cannot be
matched (backward passes, softmax) our worst error against float64 must stay within 2x the worst error of torch's own bf16 run of the
same op.  Pure data movement must be bit-exact.  References run in float64 on the GPU with torch's own ops (never dreamllm_b200's).
"""
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as UO

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
F64 = torch.float64
DEV = "cuda"
U24 = 2.0 ** -24          # fp32 unit roundoff


# ------------------------------------------------------------------------------------------------ helpers
def _ops():
    from dreamllm_b200 import ops
    return ops


def _lib():
    from dreamllm_b200 import _lib
    return _lib.lib()


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn(shape, g, scale=1.0, shift=0.0):
    return (torch.randn(shape, generator=g, device=DEV) * scale + shift).to(BF)


def _rnd(x):
    """x rounded to bf16, kept in x's dtype"""
    return x.to(BF).to(x.dtype)


def _ulp(x):
    """bf16 spacing at |x| (8 significant bits)"""
    return torch.exp2(torch.floor(torch.log2(x.abs().to(F64).clamp_min(2.0 ** -120))) - 7)


def _check(got, ref, bound, what):
    """every element: |got - ref| <= bound (bound broadcastable); reports the worst offender"""
    got, ref = got.to(F64), ref.to(F64)
    err = (got - ref).abs()
    bound = torch.as_tensor(bound, dtype=F64, device=err.device).expand_as(err)
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = int(torch.argmax(torch.where(bad, err - bound, torch.zeros_like(err))).item())
        idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), err.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.numel()} elements out of bound; worst at {idx}: got {float(got[idx]):.6g} "
                             f"want {float(ref[idx]):.6g} err {float(err[idx]):.3g} bound {float(bound[idx]):.3g}")


def _like_for_like(got, ref, ours_bf16_ref, what, factor=2.0):
    """worst-element like-for-like: max|ours - fp64| <= factor * max|torch bf16 - fp64| (+ 2^-20 * max|fp64|, for ops that torch's
    bf16 run happens to get exactly right)"""
    e_o = float((got.to(F64) - ref.to(F64)).abs().max())
    e_t = float((ours_bf16_ref.to(F64) - ref.to(F64)).abs().max())
    assert e_o <= factor * e_t + 2.0 ** -20 * float(ref.abs().max()), f"{what}: worst error ours {e_o:.4g} vs torch bf16 {e_t:.4g} (x{factor} allowed)"


def _weight_holder():
    """the UNet's weight-layout methods read only `_wcache`"""
    return types.SimpleNamespace(_wcache={})


# ================================================================================================ 1. conv3x3 (implicit GEMM)
# (N, H, W, Cin, Cout, epilogue, path).  path "ops" = ops.conv3x3 (split-K when the library plans it for a plane of <= 4096 pixels),
# "direct" = dllm_conv3x3_nhwc without a workspace (never split: the kcta = 1 unsplit kernel is reachable only this way).  Epilogue:
# b = bias, rb = per-image row bias (the time embedding), res = residual.  The comment names the tile geometry conv3x3_nhwc_ws derives
# (Wb x Hb x Nb = one 128-pixel tile; kcta = 2 when M = N*H*W > 128) and the split-K decision.
CONV_CASES = [
    (1, 16, 512, 64, 320, "b,rb,res", "ops"),    # W = 512: 4 tiles per row, unsplit, partial N tile (320 of 512)
    (1, 32, 256, 128, 128, "b", "ops"),          # W = 256, Cout 128 (pick_bn 128), unsplit (VAE 256^2 class)
    (1, 64, 128, 64, 1280, "b,res", "ops"),      # W = 128, Hb = 1, unsplit
    (4, 64, 64, 320, 320, "b,rb", "ops"),        # C5 / C4 headline: W = 64, Hb = 2, unsplit, bias + time-embedding row bias
    (2, 64, 64, 320, 320, "b,res", "ops"),       # resnet conv2
    (2, 64, 64, 320, 8, "b", "ops"),             # conv_out (Cout zero-padded to 8) / upsampler conv
    (2, 64, 64, 640, 320, "", "ops"),            # dgrad-shaped: no epilogue
    (4, 32, 32, 320, 320, "b,rb", "ops"),        # W = 32, Hb = 4, M = 4096: split-K ...
    (5, 32, 32, 320, 320, "b,rb", "ops"),        # ... and the same geometry at M = 5120: unsplit
    (2, 32, 32, 1920, 640, "b,res", "ops"),      # split
    (2, 32, 32, 1280, 1280, "b", "ops"),         # M = 2048 but 40 tiles: unsplit
    (2, 32, 32, 640, 960, "", "ops"),            # split
    (2, 32, 32, 640, 1280, "", "ops"),           # unsplit
    (2, 16, 16, 640, 1280, "b,rb", "ops"),       # W = 16, Hb = 8, split
    (2, 16, 16, 2560, 1280, "b,res", "ops"),     # Cin 2560, split
    (2, 16, 16, 1280, 1280, "b", "ops"),         # split
    (2, 16, 16, 1280, 2560, "", "ops"),          # split
    (16, 16, 16, 640, 1280, "b,rb", "ops"),      # W = 16 at M = 4096 with 80 tiles: unsplit
    (3, 8, 8, 2560, 1280, "b,rb,res", "ops"),    # W = 8: Nb = 2, 3 images (last tile half empty), kcta 2, split
    (2, 8, 8, 1280, 1280, "b,rb", "ops"),        # M = 128: kcta 1, split
    (2, 8, 8, 2560, 1280, "b,res", "ops"),       # kcta 1, split
    (2, 8, 8, 1280, 2560, "", "ops"),            # kcta 1, split
    (1, 8, 8, 1920, 640, "b", "ops"),            # kcta 1, one image in a 2-image tile, split
    (5, 4, 4, 1280, 1280, "b,rb", "ops"),        # W = 4: Nb = 8, 5 images, kcta 1, split
    (2, 8, 8, 960, 320, "b,rb,res", "direct"),   # kcta 1 unsplit
    (5, 4, 4, 1280, 640, "b,rb", "direct"),      # kcta 1 unsplit, Nb = 8 with 5 images
    (3, 8, 8, 640, 128, "b", "direct"),          # kcta 2 unsplit, Nb = 2 with 3 images
    (1, 64, 64, 512, 512, "b", "ops"),           # VAE 64^2: M = 4096, split
    (1, 64, 64, 512, 512, "b,res", "ops"),       # VAE 64^2 resnet conv2, split
]


def _conv_epi(epi, N, Cout, g, M):
    bias = _randn((Cout,), g, 0.5) if "b" in epi.split(",") else None
    rowbias = _randn((N, Cout), g, 0.5) if "rb" in epi.split(",") else None
    residual = _randn((M, Cout), g) if "res" in epi.split(",") else None
    return bias, rowbias, residual


def _conv_ref(x, w, bias, rowbias, residual, stride=1, pad=1):
    """float64 conv2d of the bf16 operands with the kernel's rounding points: mid = bf16(acc + bias + rowbias[n]); out = bf16(mid + res).
    Returns (out NHWC fp64, bound).  Bound: each rounding point may differ by 2 bf16 ulps (each side rounds by <= 1/2 ulp, and a
    binade crossing doubles one side's ulp), plus 16 * 2^-24 * sum|x*w| for the fp32 (tensor-core / split-K) accumulation."""
    xc = x.permute(0, 3, 1, 2).to(F64)
    wc = w.to(F64)
    acc = F.conv2d(xc, wc, stride=stride, padding=pad).permute(0, 2, 3, 1)
    mag = F.conv2d(xc.abs(), wc.abs(), stride=stride, padding=pad).permute(0, 2, 3, 1)
    mid = acc
    if bias is not None:
        mid = mid + bias.to(F64)
    if rowbias is not None:
        mid = mid + rowbias.to(F64)[:, None, None, :]
    mid_r = _rnd(mid)
    bound = 16 * U24 * mag + 2 * _ulp(mid_r)
    if residual is None:
        return mid_r, bound
    out = _rnd(mid_r + residual.to(F64).view(mid_r.shape))
    return out, bound + 2 * _ulp(out)


def _conv_call(x, wk, bias, rowbias, residual, path):
    ops = _ops()
    if path == "ops":
        return ops.conv3x3(x, wk, bias=bias, rowbias=rowbias, residual=residual)
    N, H, W, Cin = x.shape
    Cout = wk.shape[0]
    y = torch.empty((N, H, W, Cout), device=DEV, dtype=BF)
    p = lambda t: 0 if t is None else t.data_ptr()   # noqa: E731
    from dreamllm_b200._lib import check
    check(_lib().dllm_conv3x3_nhwc(x.data_ptr(), wk.data_ptr(), y.data_ptr(), N, H, W, Cin, Cout, p(bias), p(rowbias), p(residual),
                                   torch.cuda.current_stream().cuda_stream), "dllm_conv3x3_nhwc")
    return y


def _conv_class(N, H, W, Cin, Cout, epi, path="ops"):
    """(Wb, Hb, Nb, split, kcta, epilogue set) — the tile geometry conv3x3_nhwc_ws derives; the split decision is the library's own
    (`ops.conv3x3` passes a workspace for planes of <= 4096 pixels and the library splits when its plan says so)."""
    Wb, Hb, Nb = min(W, 128), (1 if W >= 128 else 128 // W), 1
    if Hb > H:
        Nb, Hb = Hb // H, H
    M = N * H * W
    split = path == "ops" and M <= 4096 and _lib().dllm_conv3x3_splitk_workspace_bytes(N, H, W, Cin, Cout) > 0
    return (Wb, Hb, Nb, bool(split), 2 if M > 128 else 1, frozenset(e for e in epi.split(",") if e))


@pytest.mark.parametrize("N,H,W,Cin,Cout,epi,path", CONV_CASES)
def test_conv3x3_fwd_vs_fp64(N, H, W, Cin, Cout, epi, path):
    from dreamllm_b200.unet import UNet2DConditionModel
    g = _gen(N * 7919 + H * 131 + W + Cin * 3 + Cout)
    x = _randn((N, H, W, Cin), g)
    w = _randn((Cout, Cin, 3, 3), g, (9 * Cin) ** -0.5)
    bias, rowbias, residual = _conv_epi(epi, N, Cout, g, N * H * W)
    wk = UNet2DConditionModel._conv_w(_weight_holder(), types.SimpleNamespace(weight=w))
    got = _conv_call(x, wk, bias, rowbias, residual, path)
    ref, bound = _conv_ref(x, w, bias, rowbias, residual)
    _check(got, ref, bound, f"conv3x3 {N}x{H}x{W} {Cin}->{Cout} [{epi}] {path} class {_conv_class(N, H, W, Cin, Cout, epi, path)}")


DGRAD_CASES = [
    (2, 64, 64, 320, 640),       # unsplit
    (2, 32, 32, 960, 640),       # dx has 960 channels: split
    (2, 32, 32, 1920, 640),      # 1920 channels: unsplit
    (2, 16, 16, 2560, 1280),     # split
    (3, 8, 8, 1280, 1280),       # Nb = 2 with a half-empty last tile
    (1, 8, 8, 1920, 640),        # kcta 1
]


@pytest.mark.parametrize("N,H,W,Cin,Cout", DGRAD_CASES)
def test_conv3x3_dgrad_vs_fp64_autograd(N, H, W, Cin, Cout):
    """dx = conv3x3(dy, _conv_w_dgrad(w)) against the float64 autograd input gradient of F.conv2d(x, w, padding=1).  One rounding point
    (the output): 2 ulps + 16 * 2^-24 * sum|dy * w|."""
    from dreamllm_b200.unet import UNet2DConditionModel
    g = _gen(N + H + Cin + Cout)
    dy = _randn((N, H, W, Cout), g)
    w = _randn((Cout, Cin, 3, 3), g, (9 * Cout) ** -0.5)
    w2 = UNet2DConditionModel._conv_w_dgrad(_weight_holder(), types.SimpleNamespace(weight=w))
    got = _ops().conv3x3(dy, w2)
    dyc = dy.permute(0, 3, 1, 2).to(F64)

    def input_grad(d, wt):
        xx = torch.zeros((N, Cin, H, W), device=DEV, dtype=F64, requires_grad=True)
        F.conv2d(xx, wt, padding=1).backward(d)
        return xx.grad.permute(0, 2, 3, 1)
    ref = input_grad(dyc, w.to(F64))
    mag = input_grad(dyc.abs(), w.to(F64).abs())
    ref_r = _rnd(ref)
    _check(got, ref_r, 16 * U24 * mag + 2 * _ulp(ref_r), f"dgrad {N}x{H}x{W} {Cout}->{Cin}")


@pytest.mark.parametrize("N,H,W,C,Cout,pad", [(2, 64, 64, 320, 320, 1), (2, 16, 16, 1280, 1280, 1), (3, 8, 8, 640, 640, 1),
                                               (1, 64, 64, 128, 128, 0), (1, 32, 32, 512, 512, 0)])
def test_downsample_im2col_s2_and_gemm_vs_strided_conv(N, H, W, C, Cout, pad):
    """Downsample2D: im2col_s2 is bit-exact against F.unfold (k = (r, s, c) order); im2col + ops.linear against a float64 stride-2 conv —
    padding 1 for the UNet; F.pad(0, 1, 0, 1) then padding 0 for the VAE (pad = 0)."""
    from dreamllm_b200.unet import UNet2DConditionModel
    ops = _ops()
    g = _gen(H * C + pad)
    x = _randn((N, H, W, C), g)
    w = _randn((Cout, C, 3, 3), g, (9 * C) ** -0.5)
    b = _randn((Cout,), g, 0.5)
    cols = ops.im2col_s2(x, pad=pad)
    xc = x.permute(0, 3, 1, 2)
    xp = F.pad(xc, (1, 1, 1, 1)) if pad else F.pad(xc, (0, 1, 0, 1))
    un = F.unfold(xp.float(), 3, stride=2)                                   # [N, C*9 (c, r, s), L]
    want = un.view(N, C, 9, -1).permute(0, 3, 2, 1).reshape(-1, 9 * C).to(BF)
    assert torch.equal(cols, want)
    wk = UNet2DConditionModel._conv_w(_weight_holder(), types.SimpleNamespace(weight=w))
    got = ops.linear(cols, wk, bias=b).view(N, H // 2, W // 2, Cout)
    ref, bound = _conv_ref(xp.permute(0, 2, 3, 1), w, b, None, None, stride=2, pad=0)
    _check(got, ref, bound, f"downsample {H}x{W} {C} pad {pad}")


@pytest.mark.parametrize("N,H,W,C", [(2, 64, 64, 320), (2, 16, 16, 1280), (3, 8, 8, 640)])
def test_col2im_s2_vs_fold(N, H, W, C):
    """col2im_s2 (Downsample2D backward) against F.fold of the float64 columns: one rounding of a <= 4-term fp32 sum."""
    g = _gen(N * H + C)
    Ho, Wo = H // 2, W // 2
    dcols = _randn((N * Ho * Wo, 9 * C), g)
    got = _ops().col2im_s2(dcols, N, H, W, C)
    c = dcols.to(F64).view(N, Ho * Wo, 9, C).permute(0, 3, 2, 1).reshape(N, C * 9, Ho * Wo)
    ref = F.fold(c, (H, W), 3, padding=1, stride=2).permute(0, 2, 3, 1)
    mag = F.fold(c.abs(), (H, W), 3, padding=1, stride=2).permute(0, 2, 3, 1)
    ref_r = _rnd(ref)
    _check(got, ref_r, 4 * U24 * mag + 2 * _ulp(ref_r), f"col2im_s2 {H}x{W}x{C}")


# ================================================================================================ 2. GroupNorm (+SiLU), forward and backward
# (N, H, W, C): G = 32.  cpg = C / 32: 10, 30 and 60 put an 8-channel vector across two groups; C = 128 (cpg 4) takes the per-channel
# group path, C = 256 (cpg 8) is its boundary; C = 2560 runs one row lane per CTA (RL = 1), C = 1920 two.  (1, 1, 4295, C) is a plane of
# 4096 + 64*3 + 7 pixels (not a multiple of any rows-per-CTA); 512^2 makes gn_rows grow the rows per CTA.
GN_CASES = [
    (2, 64, 64, 320), (2, 32, 32, 640), (2, 32, 32, 960), (2, 16, 16, 1280), (2, 16, 16, 1920), (1, 8, 8, 2560), (3, 8, 8, 2560),
    (1, 512, 512, 128), (1, 256, 256, 256), (1, 128, 128, 512), (1, 64, 64, 512), (3, 1, 4295, 640), (1, 1, 4103, 320), (1, 64, 64, 128),
]
GN_OFFSET = [(2, 32, 32, 320), (1, 64, 64, 128)]   # per-group mean about 30x the spread: the one-pass E[x^2] - mean^2 variance
GN_C = sorted({c[3] for c in GN_CASES + GN_OFFSET})


def _gn_input(N, H, W, C, g, offset):
    """per-(image, group) mean and spread both vary, so that using a neighbouring group's statistics is visible"""
    G = 32
    s = torch.rand((N, 1, 1, G, 1), generator=g, device=DEV) * 1.5 + 0.5
    m = (torch.rand((N, 1, 1, G, 1), generator=g, device=DEV) * 4 - 2) if not offset else 30 * s * torch.sign(torch.randn((N, 1, 1, G, 1), generator=g, device=DEV))
    z = torch.randn((N, H, W, G, C // G), generator=g, device=DEV)
    return (m + s * z).reshape(N, H, W, C).to(BF)


def _gn_ref(x, w, b, eps, silu):
    """float64 GroupNorm of the bf16 input; returns (t = x_hat * w + b before rounding, mean, rstd, x_hat, stats pieces) per element"""
    N, H, W, C = x.shape
    G = 32
    xg = x.to(F64).view(N, H * W, G, C // G)
    mean = xg.mean(dim=(1, 3), keepdim=True)
    var = xg.var(dim=(1, 3), unbiased=False, keepdim=True)
    ex2 = (xg * xg).mean(dim=(1, 3), keepdim=True)
    mabs = xg.abs().mean(dim=(1, 3), keepdim=True)
    rstd = (var + eps).rsqrt()
    xh = (xg - mean) * rstd
    t = (xh.reshape(N, H, W, C) * w.to(F64) + b.to(F64))
    return t, mean, rstd, xh.reshape(N, H, W, C), ex2, var, mabs


def _gn_t_bound(x, w, b, eps, ref):
    """error of the kernel's pre-rounding t = (x - mean) * rstd * w + b.  Statistics are fp32 sums over up to 2^18 elements in
    order-fixed trees: |d mean| <= 128 * 2^-24 * mean|x|, and the one-pass variance E[x^2] - mean^2 has |d var| <= 128 * 2^-24 * E[x^2],
    so |d rstd| / rstd <= 64 * 2^-24 * E[x^2] / (var + eps); plus 4 * 2^-24 of the fp32 arithmetic on |x_hat * w| + |b|."""
    t, mean, rstd, xh, ex2, var, mabs = ref
    N, H, W, C = x.shape
    shp = (N, 1, 1, 32, 1)
    eta_m = (128 * U24 * mabs).view(shp)
    eta_r = (64 * U24 * ex2 / (var + eps)).view(shp)
    rs = rstd.view(shp)
    xh5 = xh.view(N, H, W, 32, C // 32)
    wa = w.to(F64).abs().view(1, 1, 1, 32, C // 32)
    e = wa * (xh5.abs() * eta_r + rs * eta_m) + 4 * U24 * ((xh5 * w.to(F64).view(1, 1, 1, 32, C // 32)).abs() + b.to(F64).abs().view(1, 1, 1, 32, C // 32))
    return e.reshape(N, H, W, C)


def _gn_fwd_check(N, H, W, C, silu, offset):
    ops = _ops()
    g = _gen(N * H * W + C + int(silu) + 10 * int(offset))
    x = _gn_input(N, H, W, C, g, offset)
    w = _randn((C,), g, 0.3, 1.0)
    b = _randn((C,), g, 0.3)
    eps = 1e-5 if C != 128 else 1e-6
    ref = _gn_ref(x, w, b, eps, silu)
    t, mean, rstd = ref[0], ref[1], ref[2]
    t_r = _rnd(t)
    # one rounding point at t (documented: the GroupNorm output is rounded before SiLU): 2 ulps of t_r on top of t's own error
    bt = _gn_t_bound(x, w, b, eps, ref) + 2 * _ulp(t_r)
    if silu:
        want = _rnd(F.silu(t_r))
        # silu is 1.1-Lipschitz; expf (fast-math) adds 2^-20 relative; the output rounds once more
        bound = 1.1 * bt + 2.0 ** -20 * want.abs() + 2 * _ulp(want)
    else:
        want, bound = t_r, bt
    y = ops.groupnorm(x, w, b, 32, eps, silu)
    _check(y, want, bound, f"groupnorm fused {N}x{H}x{W}x{C} silu={silu} offset={offset}")
    y2, stats = ops.groupnorm(x, w, b, 32, eps, silu, return_stats=True)
    assert torch.equal(y2, y), "stats + apply path differs from the fused path"
    m_ref, r_ref = mean.view(N, 32), rstd.view(N, 32)
    _check(stats[..., 0], m_ref, 128 * U24 * ref[6].view(N, 32) + 1e-30, "groupnorm mean")
    _check(stats[..., 1], r_ref, r_ref * (64 * U24 * (ref[4] / (ref[5] + eps)).view(N, 32) + 4 * U24), "groupnorm rstd")
    return x, w, b, eps, stats


@pytest.mark.parametrize("N,H,W,C", GN_CASES)
@pytest.mark.parametrize("silu", [True, False])
def test_groupnorm_fwd_vs_fp64(N, H, W, C, silu):
    _gn_fwd_check(N, H, W, C, silu, False)


@pytest.mark.parametrize("N,H,W,C", GN_OFFSET)
def test_groupnorm_fwd_large_mean_vs_fp64(N, H, W, C):
    _gn_fwd_check(N, H, W, C, True, True)


@pytest.mark.parametrize("N,H,W,C", [c for c in GN_CASES if c[1] * c[2] <= 128 * 128] + GN_OFFSET[:1])
@pytest.mark.parametrize("silu,with_dres", [(True, False), (True, True), (False, True)])
def test_groupnorm_bwd_vs_fp64_autograd(N, H, W, C, silu, with_dres):
    """groupnorm_bwd against float64 autograd of silu?(group_norm(x)) (+ dres); like-for-like against torch's bf16 group_norm backward"""
    ops = _ops()
    g = _gen(N * H * W + C + 3 * int(silu) + int(with_dres))
    offset = (N, H, W, C) in GN_OFFSET
    x = _gn_input(N, H, W, C, g, offset)
    w = _randn((C,), g, 0.3, 1.0)
    b = _randn((C,), g, 0.3)
    dy = _randn((N, H, W, C), g)
    dres = _randn((N, H, W, C), g) if with_dres else None
    eps = 1e-5
    _, stats = ops.groupnorm(x, w, b, 32, eps, silu, return_stats=True)
    got = ops.groupnorm_bwd(dy, x, w, b, stats, 32, silu, dres=dres)

    def run(dt):
        xx = x.permute(0, 3, 1, 2).to(dt, copy=True).requires_grad_(True)
        y = F.group_norm(xx, 32, w.to(dt), b.to(dt), eps)
        if silu:
            y = F.silu(y)
        y.backward(dy.permute(0, 3, 1, 2).to(dt))
        d = xx.grad.permute(0, 2, 3, 1)
        return d + dres.to(dt) if with_dres else d
    _like_for_like(got, run(F64), run(BF), f"groupnorm_bwd {N}x{H}x{W}x{C} silu={silu} dres={with_dres}")


# ================================================================================================ 3. LayerNorm forward / backward
LN_H = [320, 512, 640, 1024, 1280, 1536]      # 8-element vectors per row: 40..192, i.e. the VPL = 2 / 4 / 6 warp kernels and their limits


@pytest.mark.parametrize("H", LN_H)
@pytest.mark.parametrize("T", [1, 7, 16387])
def test_layernorm_fwd_bwd_vs_fp64(H, T):
    ops = _ops()
    g = _gen(H * 3 + T)
    x = (torch.randn((T, H), generator=g, device=DEV) * (torch.rand((T, 1), generator=g, device=DEV) * 2 + 0.2)
         + torch.randn((T, 1), generator=g, device=DEV) * 3).to(BF)
    w = _randn((H,), g, 0.3, 1.0)
    b = _randn((H,), g, 0.3)
    dy = _randn((T, H), g)
    dres = _randn((T, H), g)
    eps = 1e-5

    def run(dt, with_dres):
        xx = x.to(dt, copy=True).requires_grad_(True)
        y = F.layer_norm(xx, (H,), w.to(dt), b.to(dt), eps)
        y.backward(dy.to(dt))
        return y.detach(), (xx.grad + dres.to(dt) if with_dres else xx.grad)
    y = ops.layernorm_fwd(x, w, b, eps)
    y64, _ = run(F64, False)
    yb, _ = run(BF, False)
    _like_for_like(y, y64, yb, f"layernorm_fwd T={T} H={H}")
    for with_dres in (False, True):
        got = ops.layernorm_bwd(dy, x, w, eps, dres=dres if with_dres else None)
        _like_for_like(got, run(F64, with_dres)[1], run(BF, with_dres)[1], f"layernorm_bwd T={T} H={H} dres={with_dres}")


# ================================================================================================ 4. GEGLU
def _gelu_bracket(gate):
    """bf16(gelu(gate)) as the kernel may round it: exact-erf GELU in float64, widened by the fp32 evaluation error
    (erff <= 2 ulp, a few fp32 operations: 2^-18 * (|g| + |gelu|)), then rounded at both ends.  tanh-GELU is outside this bracket
    wherever it moves the rounded value."""
    g64 = gate.to(F64)
    ge = F.gelu(g64)
    e = 2.0 ** -18 * (g64.abs() + ge.abs())
    return _rnd((ge - e).float()), _rnd((ge + e).float())


@pytest.mark.parametrize("T,I", [(1, 8), (7, 320), (4096, 1280), (262147, 16)])
def test_geglu_fwd_exact_erf_rounding(T, I):
    """out = bf16(h * bf16(gelu(gate))): the product of two bf16 numbers is exact in fp32, so the output must equal the rounding of
    h * (the bracketed bf16 gelu) — bit-exact up to where fp32 erf can sit on the other side of a rounding boundary.
    T = 262147 rows take the launch-splitting branch (more than 65535 row blocks)."""
    g = _gen(T + I)
    x = _randn((T, 2 * I), g, 2.0)
    got = _ops().geglu(x)
    h, gate = x[:, :I].float(), x[:, I:]
    lo, hi = _gelu_bracket(gate)
    a, c = _rnd(h * lo), _rnd(h * hi)
    lo_o, hi_o = torch.minimum(a, c), torch.maximum(a, c)
    gf = got.float()
    bad = (gf < lo_o) | (gf > hi_o)
    assert not bool(bad.any()), (f"geglu T={T} I={I}: {int(bad.sum())} elements outside the exact-erf rounding bracket, e.g. got "
                                 f"{float(gf[bad][0])} bracket [{float(lo_o[bad][0])}, {float(hi_o[bad][0])}]")


@pytest.mark.parametrize("T,I", [(7, 320), (4096, 1280), (1000, 2560)])
def test_geglu_bwd_vs_fp64_autograd(T, I):
    g = _gen(T * 3 + I)
    x = _randn((T, 2 * I), g, 2.0)
    dout = _randn((T, I), g)
    got = _ops().geglu_bwd(dout, x)

    def run(dt):
        xx = x.to(dt, copy=True).requires_grad_(True)
        (xx[:, :I] * F.gelu(xx[:, I:])).backward(dout.to(dt))
        return xx.grad
    _like_for_like(got, run(F64), run(BF), f"geglu_bwd T={T} I={I}")


@pytest.mark.parametrize("M,K,I", [(1077, 320, 1280), (130, 640, 2560)])
def test_linear_geglu_m_tail_vs_fp64(M, K, I):
    """FF-in GEMM with GEGLU in its epilogue at an M that leaves a partial last tile.  Rounding points: h = bf16(acc_h + b_h),
    gate = bf16(acc_g + b_g), bf16(gelu(gate)), bf16(h * gelu).  Bound: 2 ulps at h and gate on top of 16 * 2^-24 * sum|x*w|,
    propagated through |gelu'| <= 1.13 and the product, plus 2 ulps of gelu and of the output."""
    ops = _ops()
    g = _gen(M + K + I)
    x = _randn((M, K), g)
    w = _randn((2 * I, K), g, K ** -0.5)
    b = _randn((2 * I,), g, 0.3)
    wp, bp = ops.geglu_permute(w, b)
    got = ops.linear_geglu(x, wp, bp)
    x64, w64 = x.to(F64), w.to(F64)
    f = _rnd(x64 @ w64.t() + b.to(F64))
    mag = x64.abs() @ w64.abs().t()
    ef = 16 * U24 * mag + 2 * _ulp(f)
    h, gt, eh, eg = f[:, :I], f[:, I:], ef[:, :I], ef[:, I:]
    ge = _rnd(F.gelu(gt))
    ege = 1.13 * eg + 2 * _ulp(ge)
    out = _rnd(h * ge)
    bound = eh * ge.abs() + (h.abs() + eh) * ege + 2 * _ulp(out)
    _check(got, out, bound, f"linear_geglu M={M}")


# ================================================================================================ 5. data movement (bit-exact) and the rest
@pytest.mark.parametrize("N,H,W,C", [(2, 32, 32, 1280), (3, 8, 8, 640), (1, 64, 64, 8)])
def test_upsample2x_fwd_exact_bwd_one_rounding(N, H, W, C):
    ops = _ops()
    g = _gen(N + H + C)
    x = _randn((N, H, W, C), g)
    y = ops.upsample2x(x)
    want = F.interpolate(x.permute(0, 3, 1, 2).float(), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1).to(BF)
    assert torch.equal(y, want)
    dy = _randn((N, 2 * H, 2 * W, C), g)
    got = ops.upsample2x_bwd(dy)
    xx = torch.zeros((N, C, H, W), device=DEV, dtype=F64, requires_grad=True)
    F.interpolate(xx, scale_factor=2.0, mode="nearest").backward(dy.permute(0, 3, 1, 2).to(F64))
    ref = xx.grad.permute(0, 2, 3, 1)
    # a 4-term fp32 sum rounded once: 2 ulps, plus 4 * 2^-24 of the summed magnitudes for the fp32 adds
    ref_r = _rnd(ref)
    mag = 4 * F.avg_pool2d(dy.permute(0, 3, 1, 2).to(F64).abs(), 2).permute(0, 2, 3, 1)
    _check(got, ref_r, 2 * _ulp(ref_r) + 4 * U24 * mag, f"upsample2x_bwd {H}x{W}x{C}")


@pytest.mark.parametrize("Ca,Cb", [(1280, 640), (8, 320), (640, 1280), (320, 8)])
def test_concat_split_channels_exact(Ca, Cb):
    ops = _ops()
    g = _gen(Ca + 7 * Cb)
    a = _randn((3, 8, 16, Ca), g)
    b = _randn((3, 8, 16, Cb), g)
    c = ops.concat_channels(a, b)
    assert torch.equal(c, torch.cat([a, b], dim=-1))
    a2, b2 = ops.split_channels(c, Ca)
    assert torch.equal(a2, a) and torch.equal(b2, b)


@pytest.mark.parametrize("Bsrc,batch_out,Cin,Cout,H,W", [(2, 4, 4, 320, 64, 64), (1, 1, 3, 128, 128, 96), (3, 3, 4, 512, 32, 48),
                                                         (2, 4, 8, 320, 16, 16)])
def test_conv_in_vs_fp64(Bsrc, batch_out, Cin, Cout, H, W):
    """conv_in: fp32 NCHW input rounded to bf16, conv + bias rounded once.  Cin <= 7 takes im2col + GEMM (image n reads latents
    n % Bsrc: the CFG duplication); Cin = 8 takes the direct kernel."""
    g = _gen(Bsrc + batch_out + Cin + Cout)
    x = torch.randn((Bsrc, Cin, H, W), generator=g, device=DEV)
    w = _randn((Cout, Cin, 3, 3), g, (9 * Cin) ** -0.5)
    b = _randn((Cout,), g, 0.5)
    got = _ops().conv_in(x, w, b, batch_out)
    xr = _rnd(x.to(F64))[torch.arange(batch_out, device=DEV) % Bsrc]
    ref, bound = _conv_ref(xr.permute(0, 2, 3, 1).to(BF), w, b, None, None)
    _check(got, ref, bound, f"conv_in Cin={Cin} {H}x{W} batch {batch_out}/{Bsrc}")


@pytest.mark.parametrize("N,H,W,C,Cout", [(2, 64, 64, 320, 4), (1, 64, 64, 512, 8), (2, 32, 32, 128, 3), (2, 48, 48, 320, 4),
                                          (1, 40, 24, 128, 3), (1, 48, 16, 64, 8)])
def test_conv_out_vs_fp64(N, H, W, C, Cout):
    """conv_out -> fp32 NCHW holding bf16(acc + bias): implicit-GEMM path when W tiles 128 and C % 64 == 0, else the direct kernel
    (W = 48 and 40: not a divisor of 128)."""
    g = _gen(N + H + W + C + Cout)
    x = _randn((N, H, W, C), g)
    w = _randn((Cout, C, 3, 3), g, (9 * C) ** -0.5)
    b = _randn((Cout,), g, 0.5)
    got = _ops().conv_out(x, w, b)
    ref, bound = _conv_ref(x, w, b, None, None)
    _check(got, ref.permute(0, 3, 1, 2), bound.permute(0, 3, 1, 2), f"conv_out {H}x{W} {C}->{Cout}")


@pytest.mark.parametrize("N,H,W,C", [(2, 64, 64, 320), (1, 16, 24, 64)])
def test_conv_out_bwd_vs_fp64_autograd(N, H, W, C):
    g = _gen(N + H + W + C)
    deps = torch.randn((N, 4, H, W), generator=g, device=DEV)
    w = _randn((4, C, 3, 3), g, 0.05)
    got = _ops().conv_out_bwd(deps, w, C)

    def input_grad(d, wt):
        xx = torch.zeros((N, C, H, W), device=DEV, dtype=F64, requires_grad=True)
        F.conv2d(xx, wt, padding=1).backward(d)
        return xx.grad.permute(0, 2, 3, 1)
    ref = _rnd(input_grad(deps.to(F64), w.to(F64)))
    mag = input_grad(deps.to(F64).abs(), w.to(F64).abs())
    _check(got, ref, 2 * _ulp(ref) + 16 * U24 * mag, f"conv_out_bwd {H}x{W}x{C}")


@pytest.mark.parametrize("cols", [8, 72, 4096, 4104])
def test_softmax_rows_vs_fp64(cols):
    g = _gen(cols)
    rows = 37
    x = torch.randn((rows, cols), generator=g, device=DEV) * 3
    x[::5] *= 40                                             # rows of large logits
    x = x.to(BF)
    scale = cols ** -0.5 if cols > 8 else 1.0
    got = _ops().softmax_rows_(x.clone(), scale)
    ref = torch.softmax(x.to(F64) * scale, dim=-1)
    tb = torch.softmax(x.float() * scale, dim=-1).to(BF)
    _like_for_like(got, ref, tb, f"softmax_rows cols={cols}")


def test_vae_sample_vs_fp64_past_both_clamps():
    """moments = bf16(Wq h + bq) (fp32 sums), logvar clamped to [-30, 20], out = (mean + exp(logvar / 2) z) * scaling.  Bound: mean and
    logvar each 2 ulps + 8 * 2^-24 * sum|w h|; exp's argument error carries to the product; fast-math expf adds 2^-20 relative."""
    g = _gen(5)
    B, L, H, W = 3, 4, 16, 24
    h = torch.randn((B, 2 * L, H, W), generator=g, device=DEV)
    wq = _randn((2 * L, 2 * L), g, 0.3)
    bq = torch.tensor([0.1, -0.2, 0.3, 0.0, -36.0, 26.0, 0.5, -1.0], device=DEV).to(BF)   # logvar of channel 0 / 1 pushed past both clamps
    z = torch.randn((B, L, H, W), generator=g, device=DEV)
    got = _ops().vae_sample(h, wq, bq, z, 0.18215)
    mom = torch.einsum("oc,bchw->bohw", wq.to(F64), h.to(F64)) + bq.to(F64).view(1, -1, 1, 1)
    mag = torch.einsum("oc,bchw->bohw", wq.to(F64).abs(), h.to(F64).abs()) + bq.to(F64).abs().view(1, -1, 1, 1)
    mean, lv = _rnd(mom[:, :L]), _rnd(mom[:, L:]).clamp(-30, 20)
    assert bool((lv == -30).any()) and bool((lv == 20).any())
    em = 2 * _ulp(mean) + 8 * U24 * mag[:, :L]
    el = 2 * _ulp(lv) + 8 * U24 * mag[:, L:]
    sd = torch.exp(0.5 * lv)
    ref = (mean + sd * z.to(F64)) * 0.18215
    bound = (em + sd * z.to(F64).abs() * (0.5 * el * 1.01 + 2.0 ** -20 * (1 + 0.5 * lv.abs())) + 4 * U24 * ref.abs() / 0.18215) * 0.18215
    _check(got, ref, bound, "vae_sample")


def test_timestep_embedding_vs_formula():
    """Timesteps(320, flip_sin_to_cos, shift 0) in float64: [cos(t f_i) | sin(t f_i)], f_i = exp(-ln(1e4) i / 160).  The library is
    built with --use_fast_math, so cosf / sinf are the approximate intrinsics; at arguments up to 999 rad their range reduction (and
    the fp32 product t * f_i, 2^-24 * 999 rad) costs up to ~1e-4 absolute, so the bound is one bf16 ulp at magnitude 1 (2^-7)."""
    ops = _ops()
    t = torch.tensor([0, 1, 999, 500, 37], dtype=torch.int32, device=DEV)
    half = 160
    f = torch.exp(-torch.log(torch.tensor(1e4, dtype=F64)) * torch.arange(half, dtype=F64) / half).to(DEV)
    arg = t.to(F64)[:, None] * f[None]
    want = torch.cat([torch.cos(arg), torch.sin(arg)], dim=-1)
    _check(ops.timestep_embedding_batch(t, 320), want, 2.0 ** -7, "timestep_embedding_batch")
    for step in (0, 2, 4):
        got = ops.timestep_embedding(t, torch.tensor([step], dtype=torch.int32, device=DEV), 3, 320)
        _check(got, want[step].expand(3, -1), 2.0 ** -7, f"timestep_embedding step {step}")


def _ac64():
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=F64) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


@pytest.mark.parametrize("kind", ["ddim", "ddpm"])
@pytest.mark.parametrize("guidance", [1.0, 7.5])
def test_sampler_step_vs_oracle_first_and_last(kind, guidance):
    """fused CFG + scheduler update against oracle/unet_oracle.py's ddim_step / ddpm_step in float64, at the first and the last step of a
    50-step schedule.  Bound: fp32 coefficients and five fp32 operations, 2^-19 of the magnitudes of the update's terms."""
    from dreamllm_b200.unet import scheduler_tables
    ops = _ops()
    n_steps = 50
    ts, coef = scheduler_tables(n_steps, kind)
    ratio = 1000 // n_steps
    ac = _ac64()
    g = _gen(int(guidance * 10) + (kind == "ddpm"))
    B = 2
    shape = (B, 4, 8, 16)
    use_cfg = guidance > 1
    eps = torch.randn(((2 * B) if use_cfg else B,) + shape[1:], generator=g, device=DEV)
    noise = torch.randn((n_steps,) + shape, generator=g, device=DEV) if kind == "ddpm" else None
    for i in (0, n_steps - 1):
        lat = torch.randn(shape, generator=g, device=DEV)
        got = lat.clone()
        step = torch.tensor([i], dtype=torch.int32, device=DEV)
        ops.sampler_step_(eps, got, coef.to(DEV), step, guidance, use_cfg, 0 if kind == "ddim" else 1, noise)
        assert int(step) == i + 1
        e = UO.cfg_combine(eps[:B], eps[B:], guidance).to(F64) if use_cfg else eps.to(F64)
        t = int(ts[i])
        acd = ac.to(DEV)
        if kind == "ddim":
            want = UO.ddim_step(lat.to(F64), e, t, ratio, acd)
        else:
            want = UO.ddpm_step(lat.to(F64), e, t, ratio, acd, noise[i].to(F64))
        c = coef[i].to(F64).to(DEV)
        ea = (eps[:B].abs() + guidance * (eps[B:] - eps[:B]).abs()).to(F64) if use_cfg else eps.abs().to(F64)
        x0a = (lat.abs().to(F64) + c[1] * ea) / c[0]
        mag = c[2] * x0a + c[3] * (ea if kind == "ddim" else lat.abs().to(F64)) + (c[4] * noise[i].abs().to(F64) if noise is not None else 0)
        _check(got, want, 2.0 ** -19 * mag, f"sampler_step {kind} g={guidance} step {i}")


@pytest.mark.parametrize("n", [3 * 4 * 17 * 19, 1, 1023, 65537])
def test_mse_fwd_bwd_vs_fp64(n):
    g = _gen(n)
    p = torch.randn(n, generator=g, device=DEV)
    t = torch.randn(n, generator=g, device=DEV)
    loss, dp = _ops().mse_fwd_bwd(p, t)
    d = p.to(F64) - t.to(F64)
    want = (d * d).mean()
    assert abs(float(loss) - float(want)) <= 64 * U24 * float(want) + 1e-30, (float(loss), float(want))
    _check(dp, 2 * d / n, 4 * U24 * (2 * d / n).abs(), f"mse dpred n={n}")


# ================================================================================================ 6. supported image sizes
def test_unsupported_image_sizes_fail_before_any_launch_and_supported_ones_match_the_oracle():
    """Image sides that are multiples of 64 from 256 to 1024: every unsupported size raises ValueError from `pipeline` before a single
    kernel launch; a supported non-square size runs the sampler and matches the oracle."""
    from dreamllm_b200.modeling_plugins import StableDiffusionHead
    from dreamllm_b200.unet import DenoiseLoop, check_planes
    ops = _ops()
    SMALL_UNET = dict(block_out_channels=(64, 128, 256, 256), attention_head_dim=(1, 2, 4, 4), cross_attention_dim=128)
    cfg = dict(SMALL_UNET)
    cfg["vae"] = dict(block_out_channels=(64, 128, 128, 128))
    torch.manual_seed(0)
    head = StableDiffusionHead(cfg, embed_hidden_size=256)
    ref_unet = UO.UNet2DConditionModel(SMALL_UNET).eval()
    ref_unet.load_state_dict(head.unet.state_dict())
    wproj = head.projector.projector.weight.detach().float().clone()
    head = head.to(device=DEV, dtype=BF)
    emb = torch.randn(1, 8, 256, generator=torch.Generator().manual_seed(1))
    sizes = list(range(256, 1025, 64))
    supported = []
    for hh in sizes:
        for ww in sizes:
            try:
                check_planes(hh // 8, ww // 8, 4, "")
                check_planes(hh, ww, 4, "")
                supported.append((hh, ww))
                continue
            except ValueError:
                pass
            torch.cuda.synchronize()
            n0 = ops.LAUNCHES.count
            with pytest.raises(ValueError, match="not supported"):
                head.pipeline(height=hh, width=ww, num_inference_steps=2, guidance_scale=1.0, prompt_embeds=emb.cuda().to(BF))
            assert ops.LAUNCHES.count == n0
    assert supported == [(a, b) for a in (256, 512, 1024) for b in (256, 512, 1024)]
    # a supported, non-square size end to end: 2 DDIM steps at 256 x 512 against the oracle
    N = 2
    lat0 = torch.randn(1, 4, 32, 64, generator=torch.Generator().manual_seed(2))
    cond = torch.nn.functional.linear(emb, wproj)
    ac, ts = UO.alphas_cumprod(), UO.set_timesteps(N)
    lat = lat0.clone()
    with torch.no_grad():
        for t in ts.tolist():
            lat = UO.ddim_step(lat, ref_unet(lat, torch.tensor(t), cond), t, 1000 // N, ac)
    got = head.pipeline(height=256, width=512, num_inference_steps=N, guidance_scale=1.0, prompt_embeds=emb.cuda().to(BF),
                        latents=lat0.cuda(), scheduler="ddim").cpu()
    rel = float((got - lat).abs().mean() / lat.abs().mean())
    assert rel < 5e-2, rel
    with pytest.raises(ValueError, match="not supported"):
        DenoiseLoop(head.unet, cond.cuda().to(BF), 2, 1.0, "ddim", height=384, width=512)


# ================================================================================================ 7. coverage of the real models
def _gn_class(C):
    cpg = C // 32
    return (C, "per-channel" if cpg < 8 else ("aligned" if cpg % 8 == 0 else "straddle"))


def test_tables_cover_every_conv_and_groupnorm_the_real_models_launch(monkeypatch):
    """Record every conv3x3 / GroupNorm call of a real-width UNet forward_train + backward_cond (N = 2, 64^2 latents, Q = 64) and a
    real-width VAE encode of one 512^2 image; every conv tile-geometry class and every GroupNorm (C, channels-per-group class) they
    launch must be in this file's tables."""
    from dreamllm_b200.unet import UNet2DConditionModel
    from dreamllm_b200.vae import AutoencoderKLEncoder
    ops = _ops()
    convs, gns = set(), set()
    conv3x3, groupnorm, groupnorm_bwd = ops.conv3x3, ops.groupnorm, ops.groupnorm_bwd

    def rec_conv(x, w_k, bias=None, rowbias=None, residual=None):
        N, H, W, Cin = x.shape
        epi = ",".join(n for n, t in (("b", bias), ("rb", rowbias), ("res", residual)) if t is not None)
        convs.add(_conv_class(N, H, W, Cin, w_k.shape[0], epi))
        return conv3x3(x, w_k, bias=bias, rowbias=rowbias, residual=residual)

    def rec_gn(x, *a, **k):
        gns.add(_gn_class(x.shape[-1]))
        return groupnorm(x, *a, **k)

    def rec_gn_bwd(dy, x, *a, **k):
        gns.add(_gn_class(x.shape[-1]))
        return groupnorm_bwd(dy, x, *a, **k)
    monkeypatch.setattr(ops, "conv3x3", rec_conv)
    monkeypatch.setattr(ops, "groupnorm", rec_gn)
    monkeypatch.setattr(ops, "groupnorm_bwd", rec_gn_bwd)
    with torch.device(DEV):
        torch.manual_seed(0)
        unet = UNet2DConditionModel().to(BF)
    g = _gen(0)
    B, Q = 2, 64
    lat = torch.randn((B, 4, 64, 64), generator=g, device=DEV)
    t = torch.tensor([10, 900], dtype=torch.int32, device=DEV)
    cond = _randn((B, Q, 1024), g)
    eps, tape = unet.forward_train(lat, t, cond)
    unet.backward_cond(torch.randn_like(eps) * 1e-3, tape)
    del unet, tape, eps
    with torch.device(DEV):
        vae = AutoencoderKLEncoder().to(BF)
    vae.encode_sample(torch.rand((1, 3, 512, 512), generator=g, device=DEV) * 2 - 1)
    torch.cuda.synchronize()
    table = {_conv_class(*c[:6], c[6]) for c in CONV_CASES} | {_conv_class(N, H, W, Cout, Cin, "") for N, H, W, Cin, Cout in DGRAD_CASES}
    missing = convs - table
    assert not missing, f"conv3x3 classes launched by the real models but not in CONV_CASES / DGRAD_CASES: {sorted(missing, key=str)}"
    gmiss = gns - {_gn_class(C) for C in GN_C}
    assert not gmiss and {c for c, _ in gns} <= set(GN_C), f"GroupNorm classes not in GN_CASES: {gmiss}"
