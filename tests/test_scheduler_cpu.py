"""Host side of the sampler (dreamllm_b200/unet.py `scheduler_tables`): the per-step coefficient table the fused CFG + scheduler kernel
reads (`sampler_step_kernel`, csrc/unet_ops.cu) reproduces the oracle's DDIM / DDPM steps (oracle/unet_oracle.py, SURVEY Appendix A.2)
when the kernel's three-line update is applied in fp32 on the CPU.  The kernel itself is checked on the GPU (tests/test_unet_gpu.py)."""
import pytest
import torch

from dreamllm_b200.unet import scheduler_tables
from oracle import unet_oracle as UO


def _kernel_update(xt, eps_u, eps_c, c, guidance, mode, noise=None):
    """sampler_step_kernel, restated: CFG combine, x0 from eps, DDIM (mode 0) or DDPM (mode 1) update."""
    e = eps_u + guidance * (eps_c - eps_u) if eps_c is not None else eps_u
    x0 = (xt - c[1] * e) / c[0]
    if mode == 0:
        return c[2] * x0 + c[3] * e
    return c[2] * x0 + c[3] * xt + (c[4] * noise if noise is not None else 0.0)


@pytest.mark.parametrize("n_steps", [1, 3, 20, 50, 999])
@pytest.mark.parametrize("kind", ["ddim", "ddpm"])
def test_tables_reproduce_oracle_scheduler_steps(n_steps, kind):
    ts, coef = scheduler_tables(n_steps, kind)
    assert ts.dtype == torch.int32 and coef.shape == (n_steps, 5) and coef.dtype == torch.float32
    assert torch.equal(ts.long(), UO.set_timesteps(n_steps))                         # leading spacing + steps_offset 1
    ac = UO.alphas_cumprod()
    ratio = 1000 // n_steps
    g = torch.Generator().manual_seed(n_steps)
    x = torch.randn(2, 4, 8, 8, generator=g)
    x_ref = x.clone()
    guidance = 7.5
    for i in list(range(n_steps))[:: max(1, n_steps // 25)] + [n_steps - 1]:        # a spread of steps incl. the last (t_prev < 0)
        t = int(ts[i])
        eu, ec = torch.randn(2, 4, 8, 8, generator=g), torch.randn(2, 4, 8, 8, generator=g)
        noise = torch.randn(2, 4, 8, 8, generator=g)
        e = UO.cfg_combine(eu, ec, guidance)
        if kind == "ddim":
            want = UO.ddim_step(x_ref, e, t, ratio, ac)
            got = _kernel_update(x, eu, ec, coef[i], guidance, 0)
        else:
            want = UO.ddpm_step(x_ref, e, t, ratio, ac, noise)
            got = _kernel_update(x, eu, ec, coef[i], guidance, 1, noise)
        torch.testing.assert_close(got, want, rtol=2e-4, atol=2e-4)


def test_last_ddpm_step_adds_no_noise_only_at_t0():
    ts, coef = scheduler_tables(999, "ddpm")
    assert int(ts[-1]) == 1 and float(coef[-1, 4]) > 0        # steps_offset = 1: the last timestep is t = 1, still stochastic
    with pytest.raises(ValueError, match="num_train_timesteps"):
        scheduler_tables(1000, "ddim")                        # leading spacing + offset 1 would index alphas_cumprod[1000]
    ts, coef = scheduler_tables(50, "ddim")
    assert float(coef[:, 4].abs().max()) == 0.0               # eta = 0


def test_rescale_noise_cfg_equals_live_reference():
    """`rescale_noise_cfg` vs the reference's `_rescale_noise_cfg` (modeling_plugins.py:658-669) on the same inputs, as
    tests/golden/plugins.npz recorded it (`python -m oracle.gen_golden_plugins`); formula check elsewhere."""
    import os

    import numpy as np

    from dreamllm_b200.unet import rescale_noise_cfg
    from oracle.plugin_scenarios import rescale_inputs
    cfg, text = rescale_inputs()
    got = rescale_noise_cfg(cfg, text, 0.7)
    std = lambda x: x.flatten(1).std(dim=1).view(-1, 1, 1, 1)
    torch.testing.assert_close(got, 0.7 * cfg * std(text) / std(cfg) + 0.3 * cfg, rtol=1e-5, atol=1e-6)
    assert torch.equal(rescale_noise_cfg(cfg, text, 0.0), cfg)
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "plugins.npz"))
    assert torch.equal(got, torch.from_numpy(gold["rescale_noise_cfg"]))
