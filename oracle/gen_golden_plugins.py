"""Mint tests/golden/plugins.npz and tests/golden/reference_config.json from the REFERENCE'S OWN CODE (needs a reference checkout).

    python -m oracle.gen_golden_plugins

Scenarios and the verbatim exec of the reference methods live in oracle/plugin_scenarios.py.  Stored: the reference's spliced embeddings
(`DreamLLMModel.forward`, and whether it handed `_forward` token ids), conditioning rows / losses / number of model calls
(`DreamLLMForCausalMLM.forward`), diffusion losses (`StableDiffusionHead.forward`, all six option branches, and its images=None branch),
`_rescale_noise_cfg`, and the `DreamLLMConfig` defaults and special-token map.  The tests check the oracles and the product against
these files wherever they run."""
from __future__ import annotations

import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import plugin_scenarios as PS  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
OUT = os.path.join(GOLDEN, "plugins.npz")
OUT_CONFIG = os.path.join(GOLDEN, "reference_config.json")


def main():
    assert PS.reference_available(), "needs /root/reference"
    d = {}
    for i, (n_images, with_dream) in enumerate(PS.SPLICE_CASES):
        out, seen = PS.live_splice(n_images, with_dream)
        d[f"splice_{i}"] = out.numpy()
        d[f"splice_{i}_ids_forwarded"] = np.bool_(seen["input_ids"] is not None)
    for i, (drop_prob, n_dm) in enumerate(PS.CAUSAL_CASES):
        r = PS.live_causal(drop_prob, n_dm)
        d[f"causal_{i}_enc"] = r["enc"].numpy()
        d[f"causal_{i}_lm_loss"] = np.float64(float(r["lm_loss"]))
        d[f"causal_{i}_loss"] = np.float64(float(r["loss"]))
        d[f"causal_{i}_n_model_calls"] = np.int64(r["n_model_calls"])
        if r["u_enc"] is not None:
            d[f"causal_{i}_u_enc"] = r["u_enc"].numpy()
            d[f"causal_{i}_null_ids"] = np.asarray(r["null_ids"])
    for i, case in enumerate(PS.SDHEAD_CASES):
        d[f"sdhead_{i}"] = np.float64(float(PS.live_sdhead(*case)))
    d["sdhead_dummy"] = np.float64(float(PS.live_sdhead_dummy()))
    d["rescale_noise_cfg"] = PS.live_rescale_noise_cfg().numpy()
    np.savez_compressed(OUT, **d)
    print(f"wrote {OUT}: {len(d)} arrays, {os.path.getsize(OUT)} bytes")
    defaults, special = PS.live_config()
    with open(OUT_CONFIG, "w") as f:
        json.dump({"defaults": defaults, "special_tokens2ids_dict": special}, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {OUT_CONFIG}")


if __name__ == "__main__":
    main()
