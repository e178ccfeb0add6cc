"""Pin the CPU oracle (oracle/decoder_oracle.py) to the reference: against tests/golden/*.npz minted from the reference's own code
(oracle/gen_golden.py) — fp32 outputs and gradients, and bf16 outputs that the oracle must reproduce bit for bit.
"""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import decoder_oracle as O
from oracle import gen_golden

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "decoder_layer_*.npz")))
BF16 = os.path.join(os.path.dirname(__file__), "golden", "decoder_bf16.npz")


def _run_oracle(hidden, inter, heads, bsz, seq, seed, pad):
    p = {k: v.requires_grad_(True) for k, v in O.init_layer_params(hidden, inter, seed).items()}
    x, gy = gen_golden.make_inputs(hidden, bsz, seq, seed)
    x.requires_grad_(True)
    am = None
    if pad:
        am = torch.ones(bsz, seq, dtype=torch.long)
        am[1, seq - pad:] = 0
        gy = gy * am[..., None]
    cos, sin = O.rope_tables(hidden // heads, 2048)
    pos = torch.arange(seq)[None].expand(bsz, -1)
    mask = O.causal_additive_mask(bsz, seq, torch.float32, am)
    y = O.decoder_layer(x, p, heads, cos, sin, pos, mask)
    y.backward(gy)
    return x, p, y


@pytest.fixture
def minting_threads():
    """Run at the thread count the fixtures were minted with: at hidden 4096 a different count moves fp32 outputs by ~1e-5 (summation
    order), which the stored tolerances rightly do not absorb."""
    n = torch.get_num_threads()
    torch.set_num_threads(gen_golden.THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_matches_golden(path, minting_threads):
    g = np.load(path)
    hidden, inter, heads, bsz, seq, seed, pad = [int(v) for v in g["shape"]]
    x, p, y = _run_oracle(hidden, inter, heads, bsz, seq, seed, pad)
    # inputs regenerate bit-identically (CPU RNG) — otherwise the fixture is meaningless
    assert gen_golden.checksum(x.detach()) == pytest.approx(float(g["x_checksum"]), rel=1e-12)
    assert sum(gen_golden.checksum(v.detach()) for v in p.values()) == pytest.approx(float(g["w_checksum"]), rel=1e-12)
    yn, dxn = y.detach().numpy(), x.grad.numpy()
    if "stride" in g.files:                                   # BASELINE-shape case: strided storage + whole-tensor |.| sums
        rs, cs = [int(v) for v in g["stride"]]
        assert float(np.abs(yn.astype(np.float64)).sum()) == pytest.approx(float(g["y_abs_sum"]), rel=1e-6)
        assert float(np.abs(dxn.astype(np.float64)).sum()) == pytest.approx(float(g["dx_abs_sum"]), rel=1e-5)
        yn, dxn = yn[:, ::rs, ::cs], dxn[:, ::rs, ::cs]
    np.testing.assert_allclose(yn, g["y"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(dxn, g["dx"], rtol=1e-4, atol=1e-7)
    for k, v in p.items():
        gr = v.grad
        sl = (gr[:8, :64] if gr.dim() == 2 else gr).numpy()
        np.testing.assert_allclose(sl, g["d_" + k], rtol=1e-4, atol=1e-7, err_msg=k)
        assert float(gr.double().sum()) == pytest.approx(float(g["dsum_" + k]), rel=1e-3, abs=1e-6)


def test_golden_present():
    assert len(GOLDEN) >= 3


def test_oracle_matches_live_reference_bf16_rounding_points():
    """bf16 run: the oracle must share the reference's rounding points (norm cast before the weight multiply, bf16 rope tables, fp32
    softmax) — bit for bit against the reference layer's own bf16 output (oracle/gen_golden.py::run_reference_bf16)."""
    hidden, inter, heads, bsz, seq, seed = gen_golden.BF16_CASE
    p = O.init_layer_params(hidden, inter, seed)
    x, _ = gen_golden.make_inputs(hidden, bsz, seq, seed)
    xb = x.to(torch.bfloat16)
    pos = torch.arange(seq)[None].expand(bsz, -1)
    y_ref = torch.from_numpy(np.load(BF16)["y"]).to(torch.bfloat16)
    pb = {k: v.to(torch.bfloat16) for k, v in p.items()}
    # reference casts the fp32-built tables to the activation dtype at use (:126-127)
    cos, sin = O.rope_tables(hidden // heads, 2048, dtype=torch.bfloat16)
    y = O.decoder_layer(xb, pb, heads, cos, sin, pos, O.causal_additive_mask(bsz, seq, torch.bfloat16))
    assert torch.equal(y, y_ref)


def test_lm_loss_masked_mean():
    torch.manual_seed(0)
    logits = torch.randn(2, 7, 11)
    labels = torch.randint(0, 11, (2, 7))
    labels[0, 3:] = -100
    want = torch.nn.functional.cross_entropy(logits[:, :-1].reshape(-1, 11), labels[:, 1:].reshape(-1), ignore_index=-100)
    assert torch.allclose(O.lm_loss(logits, labels), want, atol=1e-6)
    # no valid label: plain mean of (zero) CE terms — reference :1468-1469
    assert float(O.lm_loss(logits, torch.full((2, 7), -100))) == 0.0


def test_kvcache_oracle_matches_reference_golden():
    """kv-cache decode (SURVEY §8f row 2): the oracle's `past_kv` path (restating :344-355 + the past-aware 4-D mask of :965-967) against
    tests/golden/kvcache_layer.npz — the reference's own DreamLLMDecoderLayer driven with `past_key_value` / `use_cache=True` over a
    LEFT-padded batch (prefill + 3 single-token steps), minted by oracle/gen_golden.py::run_reference_cached."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "kvcache_layer.npz"))
    hidden, inter, heads = [int(v) for v in g["shape"]]
    p, calls = O.cached_decode_scenario(hidden, inter, heads)
    outs = O.run_cached_scenario(p, calls, heads)
    assert len(outs) == 4
    for i, ((x, am, pos), y) in enumerate(zip(calls, outs)):
        assert np.array_equal(am.numpy(), g[f"mask{i}"])
        valid = am[:, -x.shape[1]:].bool()                 # rows of this call that are real tokens
        np.testing.assert_allclose(y.detach()[valid].numpy(), g[f"y{i}"][valid.numpy()], rtol=1e-5, atol=1e-6, err_msg=f"call {i}")
    # pad QUERY rows differ by design between the reference's two paths (SURVEY §8 row a3'): eager = uniform attention, flash = zeros


def test_kvcache_oracle_matches_live_reference_bf16():
    """Same scenario, bf16, against the reference layer's bf16 outputs (oracle/gen_golden.py::run_reference_cached_bf16): shared
    rounding points => identical outputs on the valid rows."""
    BF = torch.bfloat16
    hidden, inter, heads = 256, 512, 2
    p, calls = O.cached_decode_scenario(hidden, inter, heads)
    outs = O.run_cached_scenario(p, calls, heads, dtype=BF)
    g = np.load(BF16)
    assert len(outs) == 4
    for i, ((x, am, pos), y) in enumerate(zip(calls, outs)):
        valid = am[:, -x.shape[1]:].bool()
        assert torch.equal(torch.from_numpy(g[f"kv_y{i}"]).to(BF), y[valid]), f"call {i}"
