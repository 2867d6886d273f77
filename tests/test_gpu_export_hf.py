"""Unified-HF export (SURVEY.md 8(f1)) byte for byte against the reference's ``export_hf_checkpoint`` of the SAME
calibrated state (tests/golden/ref_export.*.npz, made by oracle/gen_golden.py export with the real reference on CPU):
FP8, NVFP4 (dynamic and static weights) and INT4-AWQ (re-smoothing of q/k/v and gate/up to one averaged
pre_quant_scale, folded into the preceding norm)."""

import json
import os

import _golden
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TD = {"torch.bfloat16": torch.bfloat16, "torch.float32": torch.float32, "torch.float16": torch.float16,
      "torch.uint8": torch.uint8, "torch.float8_e4m3fn": torch.float8_e4m3fn, "torch.int8": torch.int8}


@pytest.fixture(scope="module")
def fx():
    return _golden.load("ref_export")


def build_calibrated(fx, key, preset):
    """The mirror model in the state the reference's export started from."""
    from transformers import LlamaConfig, LlamaForCausalLM

    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import replace_quant_module, set_quantizer_by_cfg
    from model_optimizer_b200.nn import TensorQuantizer

    cfg = LlamaConfig(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, vocab_size=128, max_position_embeddings=128, tie_word_embeddings=False,
                      architectures=["LlamaForCausalLM"])
    model = LlamaForCausalLM(cfg).to(torch.bfloat16).eval()
    with torch.no_grad():
        for name, p in model.named_parameters():
            raw = torch.from_numpy(fx[f"{key}/in/param/{name}"].copy())
            p.copy_(raw.view(torch.bfloat16).reshape(p.shape))
    model = model.cuda()
    replace_quant_module(model)
    set_quantizer_by_cfg(model, cfgs.get_preset(preset)["quant_cfg"])
    mods = dict(model.named_modules())
    n = 0
    for k in fx.files:
        pre = f"{key}/in/q/"
        if not k.startswith(pre):
            continue
        qname, buf = k[len(pre):].rsplit(".", 1)
        q = mods.get(qname)
        if not isinstance(q, TensorQuantizer):
            continue
        dt = TD[str(fx[f"{key}/in/qdtype/{qname}.{buf}"])]
        t = torch.from_numpy(fx[k]).to(dt).cuda()
        if buf == "_amax":
            q.amax = t
        elif buf == "_global_amax":
            q.register_buffer("_global_amax", t)
        else:
            q._enable_pre_quant_scale = True
            q.pre_quant_scale = t
        n += 1
    assert n > 0
    with torch.no_grad():                                   # first forward of static-block quantizers fixes their layout
        for m in model.modules():
            wq = getattr(m, "weight_quantizer", None)
            if isinstance(wq, TensorQuantizer) and wq.is_enabled and wq.is_static_block_quant:
                wq(m.weight)
    return model


@pytest.mark.parametrize("key,preset", [("FP8_DEFAULT_CFG", "FP8_DEFAULT_CFG"), ("NVFP4_DEFAULT_CFG", "NVFP4_DEFAULT_CFG"),
                                        ("INT4_AWQ_CFG", "INT4_AWQ_CFG"),
                                        ("NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG@max", "NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG")])
def test_export_state_dict_bytes_equal_reference(fx, key, preset, tmp_path):
    from safetensors.torch import load_file

    from model_optimizer_b200.export_hf import export_hf_checkpoint

    model = build_calibrated(fx, key, preset)
    sd, cfg = export_hf_checkpoint(model, str(tmp_path))
    want_cfg = json.loads(str(fx[f"{key}/cfg"]))
    assert cfg["quantization"] == want_cfg["quantization"]
    got = load_file(os.path.join(tmp_path, "model.safetensors"))          # through the file: what a consumer reads
    want_keys = sorted(k[len(f"{key}/out/"):] for k in fx.files if k.startswith(f"{key}/out/"))
    assert sorted(got) == want_keys, (sorted(set(got) ^ set(want_keys))[:10])
    bad = []
    for k in want_keys:
        dt, shape = json.loads(str(fx[f"{key}/meta/{k}"]))
        t = got[k]
        assert str(t.dtype) == dt and list(t.shape) == shape, (k, t.dtype, tuple(t.shape), dt, shape)
        raw = t.contiguous().reshape(-1).view(torch.uint8).numpy() if t.numel() else np.zeros(0, np.uint8)
        if not np.array_equal(raw, fx[f"{key}/out/{k}"]):
            bad.append((k, int((raw != fx[f"{key}/out/{k}"]).sum()), raw.size))
    assert not bad, bad[:8]
    assert os.path.exists(os.path.join(tmp_path, "hf_quant_config.json"))


def test_export_awq_resmooth_structure(fx):
    """After export the fused groups carry no pre_quant_scale (folded into the norms), o_proj / down_proj keep theirs."""
    from model_optimizer_b200.export_hf import export_hf_state_dict

    model = build_calibrated(fx, "INT4_AWQ_CFG", "INT4_AWQ_CFG")
    sd, _ = export_hf_state_dict(model)
    pqs = sorted(k for k in sd if k.endswith("pre_quant_scale"))
    assert pqs == sorted(f"model.layers.{i}.{n}.pre_quant_scale" for i in range(2)
                         for n in ("self_attn.o_proj", "mlp.down_proj"))
    assert sd["model.layers.0.self_attn.q_proj.weight"].dtype == torch.uint8
    assert tuple(sd["model.layers.0.self_attn.q_proj.weight"].shape) == (64, 128)      # [out / 2, in]
