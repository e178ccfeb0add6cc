"""Pins the splice / conditioning-gather / loss-combination restatements to the reference model wrappers: `DreamLLMModel.forward`
(modeling_dreamllm.py:1045-1158) and `DreamLLMForCausalMLM.forward` (:1353-1509), exec'd verbatim from the reference and run on CPU with
stand-in sub-modules (oracle/plugin_scenarios.py), recorded what they returned and passed on in tests/golden/plugins.npz
(`python -m oracle.gen_golden_plugins`).

Chain of custody this closes:  reference == oracle/splice_oracle.py == SplicePlan index maps (tests/test_collator_cpu.py, CPU)
== CUDA copy_rows / segment_sum_rows / gather_rows kernels (tests/test_clip_splice_gpu.py, GPU)."""
import os

import numpy as np
import pytest
import torch

from oracle import plugin_scenarios as PS

GOLD = os.path.join(os.path.dirname(__file__), "golden", "plugins.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.mark.parametrize("n_images,with_dream", PS.SPLICE_CASES)
def test_splice_oracle_equals_live_reference_model_forward(gold, n_images, with_dream):
    i = PS.SPLICE_CASES.index((n_images, with_dream))
    assert torch.equal(torch.from_numpy(gold[f"splice_{i}"]), PS.oracle_splice(n_images, with_dream))
    assert not gold[f"splice_{i}_ids_forwarded"]                       # the reference hands `_forward` embeddings only


@pytest.mark.parametrize("drop_prob,n_dm", PS.CAUSAL_CASES)
def test_conditioning_gather_null_prompt_and_loss_equal_live_reference_causal_lm_forward(gold, drop_prob, n_dm):
    i = PS.CAUSAL_CASES.index((drop_prob, n_dm))
    ours = PS.oracle_causal(drop_prob, n_dm)
    # (1) conditioning gather == oracle (== SplicePlan.cond_rows, tests/test_collator_cpu.py)
    assert torch.equal(torch.from_numpy(gold[f"causal_{i}_enc"]), ours["enc"])
    # (2) null prompt: the id layout our `_null_prompt_states` builds, hidden rows [2, 2+Q), broadcast over the batch (:1420-1439)
    if drop_prob is None:
        assert f"causal_{i}_u_enc" not in gold.files and int(gold[f"causal_{i}_n_model_calls"]) == 1
    else:
        assert gold[f"causal_{i}_null_ids"].tolist() == ours["null_ids"]
        assert torch.equal(torch.from_numpy(gold[f"causal_{i}_u_enc"]), ours["u_enc"])
    # (3) losses: masked-mean CE over shifted labels (:1456-1470) and vm * w_vm + lm * w_lm (:1486-1488)
    for k in ("lm_loss", "loss"):
        want = torch.tensor(float(gold[f"causal_{i}_{k}"]), dtype=torch.float32)
        torch.testing.assert_close(want, ours[k], rtol=1e-6, atol=1e-7)
