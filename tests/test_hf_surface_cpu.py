"""CPU tests of the drop-in boundary that is not arithmetic (SURVEY.md §8b): DreamLLMConfig + plugin registration / instantiation,
the HF on-disk layout (`save_pretrained` / `from_pretrained`), `resize_token_embeddings`, generation helpers.  Modules are built on CPU
(construction, state dicts and (de)serialisation need no kernels; forward does and is covered by the -m gpu tests)."""
import json
import os

import pytest
import torch

from dreamllm_b200.configuration_dreamllm import ConfigAndInitKwargs, DreamLLMConfig, deep_instantiate
from dreamllm_b200.modeling_dreamllm import DreamLLMForCausalMLM, KVCache
from dreamllm_b200.modeling_plugins import DreamEmbedding
from oracle.plugin_scenarios import CONFIG_TOKENS, Tok

REF_CFG = os.path.join(os.path.dirname(__file__), "golden", "reference_config.json")
TINY = dict(vocab_size=96, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2)


def test_config_defaults_equal_the_live_reference_config():
    """Every default against the reference's own class (configuration_dreamllm.py:64-278) on the installed transformers, as
    tests/golden/reference_config.json recorded it (`python -m oracle.gen_golden_plugins`)."""
    with open(REF_CFG) as f:
        gold = json.load(f)
    ref, ours = gold["defaults"], DreamLLMConfig()
    for k, v in ours.to_dict().items():
        if k in ("model_type", "rope_scaling"):            # transformers 5 rewrites rope_scaling=None into rope_parameters
            continue
        assert ref[k] == v, k
    assert ref["model_type"] == ours.model_type == "dreamllm"
    ours.update_special_tokens2ids_dict(CONFIG_TOKENS, Tok(96))
    assert gold["special_tokens2ids_dict"] == ours.special_tokens2ids_dict == {"additional_special_tokens": {"<im_start>": 90,
                                                                                                             "<dream_start>": 93},
                                                                              "<s>": 1}


def test_plugin_registration_and_instantiation():
    cfg = DreamLLMConfig(**TINY)
    name = cfg.update_plugins(ConfigAndInitKwargs(_class_=DreamEmbedding, _name_="dream_embedding", _plugin_type_="embedding",
                                                  pretrained_model_name_or_path=None, num_dream_queries=4, embed_hidden_size=128))
    assert name == "dream_embedding" and cfg.plugins_type == {"dream_embedding": "embedding"}
    assert cfg.plugins_init_kwargs["dream_embedding"]["_target_"] == "dreamllm_b200.modeling_plugins.DreamEmbedding"   # swap = change this
    cfg.update_plugins(dict(_class_=DreamEmbedding, _name_="dream_embedding", _plugin_type_="embedding", num_dream_queries=6))
    assert cfg.plugins_init_kwargs["dream_embedding"]["num_dream_queries"] == 6 and \
        cfg.plugins_init_kwargs["dream_embedding"]["embed_hidden_size"] == 128                # second call updates, keeps the rest (:249-252)
    with pytest.raises(AssertionError):
        cfg.update_plugins(dict(_class_=DreamEmbedding, _name_="x"))
    obj = deep_instantiate(cfg.plugins_init_kwargs["dream_embedding"])
    assert isinstance(obj, DreamEmbedding) and obj.embed_len == 6 and obj.dream_queries.shape == (1, 6, 128)
    nested = deep_instantiate({"a": [{"_target_": "collections.OrderedDict", "x": 1}], "b": 2})
    assert nested["a"][0] == {"x": 1} and nested["b"] == 2
    cfg.reset_plugins_init_kwargs("/some/dir")
    assert cfg.plugins_init_kwargs["dream_embedding"]["pretrained_model_name_or_path"] == "/some/dir"
    with pytest.raises(ValueError):
        DreamLLMConfig(rope_scaling={"type": "ntk", "factor": 2.0})


def test_config_json_round_trip_and_foreign_keys(tmp_path):
    cfg = DreamLLMConfig(**TINY, loss_weight_vm=3.0, some_future_key=[1, 2])
    cfg.update_plugins(dict(_class_=DreamEmbedding, _name_="dream_embedding", _plugin_type_="embedding", num_dream_queries=4,
                            embed_hidden_size=128, pretrained_model_name_or_path=None))
    cfg.save_pretrained(tmp_path)
    raw = json.load(open(tmp_path / "config.json"))
    assert raw["model_type"] == "dreamllm" and raw["plugins_init_kwargs"]["dream_embedding"]["_target_"].endswith("DreamEmbedding")
    back = DreamLLMConfig.from_pretrained(str(tmp_path))
    assert back.to_dict() == cfg.to_dict() and back.some_future_key == [1, 2] and back.loss_weight_vm == 3.0
    # a config.json written by transformers >= 5 (rope_parameters instead of rope_theta / rope_scaling)
    raw.pop("rope_theta"), raw.pop("rope_scaling")
    raw["rope_parameters"] = {"rope_theta": 500000.0, "rope_type": "default"}
    raw["transformers_version"] = "5.5.0"
    assert DreamLLMConfig.from_dict(raw).rope_theta == 500000.0
    with pytest.raises(OSError):
        DreamLLMConfig.from_pretrained(str(tmp_path / "nope"))


def _tiny_model(with_plugin=True):
    cfg = DreamLLMConfig(**TINY)
    cfg.update_special_tokens2ids_dict({"additional_special_tokens": ["<im_start>", "<im_patch>", "<im_end>", "<dream_start>", "<dream_end>"],
                                        "bos_token": "<s>", "eos_token": "</s>"}, Tok(96))
    if with_plugin:
        cfg.update_plugins(dict(_class_=DreamEmbedding, _name_="dream_embedding", _plugin_type_="embedding", num_dream_queries=4,
                                embed_hidden_size=128, pretrained_model_name_or_path=None))
    torch.manual_seed(0)
    m = DreamLLMForCausalMLM(cfg)
    m.init_plugin_modules()
    return m


@pytest.mark.parametrize("safe,shard", [(True, None), (False, None), (True, 200_000)])
def test_save_and_from_pretrained_round_trip(tmp_path, safe, shard):
    m = _tiny_model()
    with torch.no_grad():
        m.model.dream_embedding.dream_queries.normal_()
    assert m.model.dream_start_id == 93 and m.model.image_start_id == 90 and m.model.dream_end_id == 94
    assert "model.dream_embedding.dream_queries" in m._keys_to_ignore_on_save or \
        "model.dream_embedding.dream_queries" in m.model._keys_to_ignore_on_save
    kw = {} if shard is None else dict(max_shard_size=shard)
    m.save_pretrained(str(tmp_path), safe_serialization=safe, **kw)
    files = sorted(os.listdir(tmp_path))
    assert "config.json" in files and "dream_embedding.bin" in files                    # plugin saved by its own save_model
    if shard:
        assert "model.safetensors.index.json" in files and sum(f.startswith("model-000") for f in files) > 1
        wm = json.load(open(tmp_path / "model.safetensors.index.json"))["weight_map"]
        assert not any(k.startswith("model.dream_embedding") for k in wm)               # plugin keys stay out of the LLM checkpoint
    m2 = DreamLLMForCausalMLM.from_pretrained(str(tmp_path), Tok(96))
    a, b = m.state_dict(), m2.state_dict()
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert isinstance(m2.model.dream_embedding, DreamEmbedding)
    assert m2.config.plugins_init_kwargs["dream_embedding"]["pretrained_model_name_or_path"] == str(tmp_path)   # :1325-1328
    with pytest.raises(AssertionError, match="tokenizer should not be None"):
        DreamLLMForCausalMLM.from_pretrained(str(tmp_path))


def test_state_dict_keys_are_the_reference_keys():
    """SURVEY §8b: checkpoint compatibility with Vicuna / LLaMA and released DreamLLM weights."""
    m = _tiny_model()
    keys = set(m.state_dict().keys())
    want = {"model.embed_tokens.weight", "model.norm.weight", "lm_head.weight", "model.dream_embedding.dream_queries"}
    for i in range(2):
        want |= {f"model.layers.{i}.self_attn.{p}_proj.weight" for p in "qkvo"}
        want |= {f"model.layers.{i}.mlp.{p}_proj.weight" for p in ("gate", "up", "down")}
        want |= {f"model.layers.{i}.input_layernorm.weight", f"model.layers.{i}.post_attention_layernorm.weight",
                 f"model.layers.{i}.self_attn.rotary_emb.inv_freq"}
    assert keys == want


def test_from_pretrained_grows_vocab_and_tolerates_missing_inv_freq(tmp_path):
    m = _tiny_model(with_plugin=False)
    m.save_pretrained(str(tmp_path))
    from safetensors.torch import load_file, save_file
    sd = {k: v for k, v in load_file(str(tmp_path / "model.safetensors")).items() if not k.endswith("inv_freq")}
    save_file(sd, str(tmp_path / "model.safetensors"))
    m2 = DreamLLMForCausalMLM.from_pretrained(str(tmp_path), Tok(100))
    assert m2.get_input_embeddings().weight.shape == (100, 128) and m2.get_output_embeddings().weight.shape == (100, 128)
    assert m2.config.vocab_size == m2.vocab_size == m2.model.vocab_size == 100
    assert torch.equal(m2.get_input_embeddings().weight[:96], m.get_input_embeddings().weight)
    assert torch.equal(m2.lm_head.weight[:96], m.lm_head.weight)
    sd["bogus.weight"] = torch.zeros(1)
    save_file(sd, str(tmp_path / "model.safetensors"))
    with pytest.raises(RuntimeError, match="unexpected"):
        DreamLLMForCausalMLM.from_pretrained(str(tmp_path), Tok(96))


def test_generation_helpers():
    m = _tiny_model(with_plugin=False)
    ids = torch.arange(10).view(2, 5)
    mask = torch.tensor([[1, 1, 1, 1, 1], [1, 1, 1, 0, 0]])
    out = m.prepare_inputs_for_generation(ids, attention_mask=mask, images="IMG", use_cache=True)
    assert torch.equal(out["input_ids"], ids) and out["images"] == "IMG" and out["use_cache"] is True
    assert out["position_ids"].tolist() == [[0, 1, 2, 3, 4], [0, 1, 2, 1, 1]]                  # (:1527-1531)
    cache = KVCache(2, 2, 16, 2, 64, "cpu", dtype=torch.float32)
    cache.len = 4
    out = m.prepare_inputs_for_generation(ids, past_key_values=cache, attention_mask=mask)
    assert out["input_ids"].shape == (2, 1) and torch.equal(out["input_ids"], ids[:, 4:]) and out["position_ids"].shape == (2, 1)
    legacy = tuple((torch.zeros(2, 2, 4, 64), torch.zeros(2, 2, 4, 64)) for _ in range(2))
    assert m.prepare_inputs_for_generation(ids, past_key_values=legacy)["input_ids"].shape == (2, 1)
    cache.k[0][0, :cache.len] += 1.0                       # only the valid prefix [:len] is ever written / moved
    beam = torch.tensor([1, 0])
    cache = m._reorder_cache(cache, beam)
    assert float(cache.k[0][1].sum()) > 0 and float(cache.k[0][0].sum()) == 0
    re = m._reorder_cache(tuple((torch.arange(2.).view(2, 1, 1, 1), torch.arange(2.).view(2, 1, 1, 1)) for _ in range(2)), beam)
    assert re[0][0].flatten().tolist() == [1.0, 0.0]
    assert m.fsdp_ignored_modules() == []


def test_average_init_of_added_token_rows():
    from dreamllm_b200.modeling_dreamllm import average_init_token_embeddings
    m = _tiny_model(with_plugin=False)
    e0, h0 = m.get_input_embeddings().weight.detach().clone(), m.lm_head.weight.detach().clone()
    average_init_token_embeddings(m, 8)
    e, h = m.get_input_embeddings().weight, m.lm_head.weight
    assert torch.equal(e[:-8], e0[:-8]) and torch.equal(h[:-8], h0[:-8])
    torch.testing.assert_close(e[-8:], e0[:-8].mean(0, keepdim=True).expand(8, -1))
    torch.testing.assert_close(h[-3], h0[:-8].mean(0))
    with pytest.raises(AssertionError):
        average_init_token_embeddings(m, 0)
