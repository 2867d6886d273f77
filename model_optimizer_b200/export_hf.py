"""Unified-HF checkpoint export -- the step right after the hot path (SURVEY.md 8(f1)).

Mirror of ``modelopt/torch/export/unified_export_hf.py`` for dense decoder-only HF models (``LlamaForCausalLM``
layout) and the formats this engine packs (FP8, NVFP4 dynamic / static, INT4-AWQ):

  * ``requantize_resmooth_fused_llm_layers`` (:421-540) -- linears that read the same tensor (q/k/v, gate/up) are found
    with forward hooks on a dummy forward, then ``preprocess_linear_fusion`` (quant_utils.py:1475-1545) re-smooths
    them to ONE averaged ``pre_quant_scale`` (weights rescaled and re-calibrated), unifies the input amax and the
    per-tensor weight amax / NVFP4 global amax, and ``fuse_prequant_layernorm`` (:1442-1472) folds the shared
    pre_quant_scale into the preceding norm;
  * ``_export_quantized_weight`` (:569-800) per linear: ``weight`` (packed), ``weight_scale``, ``weight_scale_2``,
    ``input_scale`` -- every pack is one kernel of this engine (``export.py``);
  * ``postprocess_state_dict`` (quant_utils.py:1054-1110): quantizer state dropped, ``input_quantizer._pre_quant_scale``
    renamed to ``pre_quant_scale``;
  * ``hf_quant_config.json`` (quant_utils.py:1583-1700, convert_hf_quant_config_format) and ``model.safetensors``.

Pinned byte for byte against the reference's own export of the same calibrated state (tests/golden/ref_export.*.npz).
"""

from __future__ import annotations

import json
import os
from collections import defaultdict

import torch
from torch import nn

from . import export as ex
from . import model_calib
from .nn import TensorQuantizer, is_quantized_linear

_ALGO = {ex.QUANTIZATION_FP8: "FP8", ex.QUANTIZATION_NVFP4: "NVFP4", ex.QUANTIZATION_W4A16_NVFP4: "W4A16_NVFP4",
         ex.QUANTIZATION_INT4_AWQ: "W4A16_AWQ", ex.QUANTIZATION_INT8_SQ: "W8A8_SQ_PER_CHANNEL"}


def _is_layernorm(m: nn.Module) -> bool:
    name = type(m).__name__.lower()
    return ("layernorm" in name or "rmsnorm" in name) and getattr(m, "weight", None) is not None


def _enabled(q) -> bool:
    return isinstance(q, TensorQuantizer) and q.is_enabled


# ---- shared-input discovery (unified_export_hf.py:279-349) ------------------------------------------------------
@torch.no_grad()
def collect_shared_input_modules(model: nn.Module, dummy_forward):
    """-> ({input tensor id: [linears]}, {norm output tensor id: norm}); quantizers disabled during the probe."""
    input_to_linear: dict = defaultdict(list)
    output_to_norm: dict = {}
    keep = []                                   # keep the probed tensors alive so that ids stay unique
    handles = []

    def in_hook(mod, args, out):
        if args and isinstance(args[0], torch.Tensor):
            keep.append(args[0])
            input_to_linear[id(args[0])].append(mod)

    def out_hook(mod, args, out):
        if isinstance(out, torch.Tensor):
            keep.append(out)
            output_to_norm[id(out)] = mod

    for _, m in model.named_modules():
        if _is_layernorm(m):
            handles.append(m.register_forward_hook(out_hook))
        elif is_quantized_linear(m) and (_enabled(m.input_quantizer) or _enabled(m.weight_quantizer)):
            handles.append(m.register_forward_hook(in_hook))
    qs = [q for q in model.modules() if isinstance(q, TensorQuantizer)]
    saved = [q._disabled for q in qs]
    try:
        for q in qs:
            q._disabled = True
        dummy_forward()
    finally:
        for q, d in zip(qs, saved):
            q._disabled = d
        for h in handles:
            h.remove()
    return input_to_linear, output_to_norm


# ---- fusion preprocessing (quant_utils.py:1285-1302, 1442-1545) ---------------------------------------------------
@torch.no_grad()
def _update_pre_quant_scale(module, new_pqs):
    old = module.input_quantizer._pre_quant_scale
    dtype = module.weight.dtype
    w = (module.weight.to(torch.float32) * old.to(dtype=torch.float32, device=module.weight.device)
         / new_pqs.to(dtype=torch.float32, device=module.weight.device)).to(dtype)
    module.weight.copy_(w)
    module.input_quantizer.pre_quant_scale = new_pqs
    wq = module.weight_quantizer                       # redo the weight collection
    wq.reset_amax()
    model_calib.max_calibrate(wq, lambda q: q(module.weight), distributed_sync=False)
    model_calib._finalize_static_nvfp4(module)         # promoted (fp32) state like the reference's quantizer class


@torch.no_grad()
def preprocess_linear_fusion(modules, resmooth_only=False):
    fmts = [ex.get_quantization_format(m) for m in modules]
    assert all(f == fmts[0] for f in fmts), "Modules have different quantization formats"
    iq0 = modules[0].input_quantizer
    if iq0.pre_quant_scale is not None:
        avg = torch.mean(torch.stack([m.input_quantizer.pre_quant_scale for m in modules]), dim=0)
        for m in modules:
            if not torch.equal(m.input_quantizer.pre_quant_scale, avg):
                _update_pre_quant_scale(m, avg)
    if resmooth_only:
        return
    if iq0.is_enabled and iq0.amax is not None:
        assert iq0.amax.numel() == 1, "Only support scalar input quant amax"
        amax = torch.max(torch.stack([m.input_quantizer.amax.reshape(()) for m in modules]))
        for m in modules:
            m.input_quantizer.amax = amax.reshape(m.input_quantizer.amax.shape)
    wq0 = modules[0].weight_quantizer
    if getattr(wq0, "_global_amax", None) is not None:          # static NVFP4: one global amax for the fused group
        g = torch.max(torch.stack([m.weight_quantizer._global_amax.reshape(()) for m in modules]))
        for m in modules:
            m.weight_quantizer._global_amax.copy_(g)
            m.weight_quantizer._state_gen += 1
    elif wq0.is_enabled and wq0.amax is not None and wq0.amax.numel() == 1:
        amax = torch.max(torch.stack([m.weight_quantizer.amax.reshape(()) for m in modules]))
        for m in modules:
            m.weight_quantizer.amax = amax.reshape(m.weight_quantizer.amax.shape)


@torch.no_grad()
def fuse_prequant_layernorm(norm: nn.Module, modules):
    iq = modules[0].input_quantizer
    if not hasattr(iq, "_pre_quant_scale"):
        return
    pqs = iq._pre_quant_scale.to(norm.weight.device)
    norm.weight.copy_((norm.weight * pqs).to(norm.weight.dtype))
    if getattr(norm, "bias", None) is not None:
        norm.bias.copy_(norm.bias * pqs)
    for m in modules:
        delattr(m.input_quantizer, "_pre_quant_scale")
        m.fused_with_prequant = True


@torch.no_grad()
def requantize_resmooth_fused_llm_layers(model: nn.Module):
    device = next(model.parameters()).device

    def dummy():
        model(torch.ones([1, 2], dtype=torch.long, device=device))

    input_to_linear, output_to_norm = collect_shared_input_modules(model, dummy)
    fused = []
    for tid, modules in input_to_linear.items():
        fmt = ex.get_quantization_format(modules[0])
        if len(modules) > 1 and fmt not in (ex.QUANTIZATION_FP8, ex.QUANTIZATION_NONE):
            preprocess_linear_fusion(modules)
            fused.append(modules)
            if fmt is not None and "awq" in fmt and tid in output_to_norm:
                fuse_prequant_layernorm(output_to_norm[tid], modules)
    return fused


# ---- per-linear export (unified_export_hf.py:569-800) ---------------------------------------------------------------
@torch.no_grad()
def export_linear_tensors(module) -> dict:
    """{suffix: tensor} for one quantized linear, the reference's names, dtypes and shapes."""
    fmt = ex.get_quantization_format(module)
    wq, iq = module.weight_quantizer, module.input_quantizer
    w = module.weight.detach()
    out = {}
    if fmt == ex.QUANTIZATION_FP8:
        amax = wq._amax.to(torch.float32)
        wsf = ex._tdiv(amax, wq.maxbound).reshape(())                    # 0-dim: `weight / scale` stays in the weight dtype
        out["weight_scale"] = wsf
        out["weight"] = ex.to_quantized_weight(w, wsf, fmt)
        if getattr(iq, "_amax", None) is not None and iq.is_enabled:
            out["input_scale"] = ex._tdiv(iq._amax.to(torch.float32), iq.maxbound).squeeze()
        return out
    if fmt in (ex.QUANTIZATION_NVFP4, ex.QUANTIZATION_W4A16_NVFP4):
        packed, scales, wsf2 = ex.export_nvfp4_weight(module)
        out.update(weight=packed, weight_scale=scales, weight_scale_2=wsf2.reshape(()))
    elif fmt == ex.QUANTIZATION_INT4_AWQ:
        amax = wq.export_amax()                                            # [out, in / block]
        wsf = ex._tdiv(amax.float(), wq.maxbound).reshape(w.shape[0], -1)
        out.update(weight=ex.pack_int4_in_uint8(w, wsf), weight_scale=wsf)
    else:
        raise NotImplementedError(f"unified-HF export of format {fmt!r}")
    if iq.is_enabled and iq.amax is not None:
        out["input_scale"] = ex.get_activation_scaling_factor(module).squeeze()
    return out


def get_quant_config(model: nn.Module) -> dict:
    """hf_quant_config.json (quant_utils.py:1583-1700 + process_layer_quant_config :660-770) for a uniformly
    quantized model; ``exclude_modules``: modules that carry quantizers but stay unquantized, and embeddings (the
    reference attaches -- disabled -- quantizers to ``nn.Embedding``)."""
    fmts, excluded, group = set(), [], None
    for name, m in model.named_modules():
        if is_quantized_linear(m):
            f = ex.get_quantization_format(m)
            if f is None:
                excluded.append(name)
            else:
                fmts.add(f)
                bs = m.weight_quantizer.block_sizes
                if bs and (bs.get(-1) or bs.get(m.weight.dim() - 1)):
                    group = bs.get(-1) or bs.get(m.weight.dim() - 1)
        elif isinstance(m, nn.Embedding):
            excluded.append(name)
    if len(fmts) != 1:
        raise NotImplementedError(f"mixed-precision export ({sorted(map(str, fmts))})")
    fmt = fmts.pop()
    q = {"quant_algo": _ALGO[fmt], "kv_cache_quant_algo": None}
    if fmt in (ex.QUANTIZATION_NVFP4, ex.QUANTIZATION_W4A16_NVFP4):
        q["group_size"] = group
    elif fmt == ex.QUANTIZATION_INT4_AWQ:
        q.update(group_size=group, has_zero_point=False, pre_quant_scale=True)
    q["exclude_modules"] = sorted(excluded)
    return {"producer": {"name": "modelopt", "version": "b200quant"}, "quantization": q}


@torch.no_grad()
def export_hf_state_dict(model: nn.Module):
    """-> (state_dict with the unified-HF names, hf_quant_config dict).  Modifies the model's quantizer state the
    way the reference's export does (re-smoothing, unified amax)."""
    requantize_resmooth_fused_llm_layers(model)
    cfg = get_quant_config(model)
    sd = {}
    handled = set()
    for name, m in model.named_modules():
        if is_quantized_linear(m) and ex.get_quantization_format(m) is not None:
            for suffix, t in export_linear_tensors(m).items():
                sd[f"{name}.{suffix}"] = t
            pqs = getattr(m.input_quantizer, "_pre_quant_scale", None)
            if pqs is not None:
                sd[f"{name}.pre_quant_scale"] = pqs.detach()
            if m.bias is not None:
                sd[f"{name}.bias"] = m.bias.detach()
            handled.add(name)
    for key, t in model.state_dict().items():
        mod = key.rsplit(".", 1)[0]
        if mod in handled or "_quantizer" in key:
            continue
        sd[key] = t.detach()
    return sd, cfg


def export_hf_checkpoint(model: nn.Module, export_dir: str):
    """``export_hf_checkpoint`` (unified_export_hf.py:1540-1649): ``model.safetensors`` + ``hf_quant_config.json``
    (+ the HF ``config.json`` when the model has one)."""
    from safetensors.torch import save_file

    sd, cfg = export_hf_state_dict(model)
    os.makedirs(export_dir, exist_ok=True)
    save_file({k: v.contiguous().cpu() for k, v in sd.items()}, os.path.join(export_dir, "model.safetensors"),
              metadata={"format": "pt"})
    with open(os.path.join(export_dir, "hf_quant_config.json"), "w") as f:
        json.dump(cfg, f, indent=4)
    if hasattr(model, "config") and hasattr(model.config, "to_json_file"):
        model.config.to_json_file(os.path.join(export_dir, "config.json"))
    return sd, cfg


__all__ = ["export_hf_checkpoint", "export_hf_state_dict", "export_linear_tensors", "get_quant_config",
           "requantize_resmooth_fused_llm_layers", "preprocess_linear_fusion", "fuse_prequant_layernorm",
           "collect_shared_input_modules"]
