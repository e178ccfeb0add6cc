"""Pins the diffusion-loss restatement (oracle/unet_oracle.py `diffusion_loss`, `add_noise`, and the CFG-dropout row mix) to the
reference code: `StableDiffusionHead._compute_snr` and `.forward` were exec'd verbatim from the reference's modeling_plugins.py
(:468-577) and run on CPU with stand-in `vae` / `noise_scheduler` / `projector` / `unet` objects built from the oracle's modules
(oracle/plugin_scenarios.py); tests/golden/plugins.npz holds the losses they returned (`python -m oracle.gen_golden_plugins`).  Same
seed => the reference's own RNG draws (randn_like, randn, randint, bernoulli — in its order) are reproduced and fed to the
restatement, so every branch (`noise_offset`, `input_perturbation`, `snr_gamma`, `drop_prob`) is compared to the reference's
arithmetic.  What stays from-spec is only the inside of diffusers' UNet / VAE / scheduler classes (not installable here — DESIGN.md §2)."""
import os

import numpy as np
import pytest
import torch

from oracle import plugin_scenarios as PS

GOLD = os.path.join(os.path.dirname(__file__), "golden", "plugins.npz")


@pytest.mark.parametrize("noise_offset,input_perturbation,snr_gamma,drop_prob", PS.SDHEAD_CASES)
def test_diffusion_loss_restatement_equals_live_reference_forward(noise_offset, input_perturbation, snr_gamma, drop_prob):
    i = PS.SDHEAD_CASES.index((noise_offset, input_perturbation, snr_gamma, drop_prob))
    want = torch.tensor(float(np.load(GOLD)[f"sdhead_{i}"]), dtype=torch.float32)
    got = PS.oracle_sdhead(noise_offset, input_perturbation, snr_gamma, drop_prob)
    torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-7)


def test_dummy_forward_of_the_reference_is_a_zero():
    """(:500-509) the reference's images=None branch only feeds DDP's unused-parameter check; our reducer needs no such pass."""
    assert float(np.load(GOLD)["sdhead_dummy"]) == 0.0
