"""GPU parity for the scale-search kernels and the host-side mirror (TensorQuantizer / calibrators /
quantize()) against the oracle and the whole-algorithm reference fixtures."""

import copy
import os

import _golden
import numpy as np
import pytest
import torch
from torch import nn

from oracle import oracle_np as o

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TD = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}


@pytest.fixture(scope="module")
def algos():
    return np.load(os.path.join(ROOT, "tests", "golden", "ref_algos.npz"))


@pytest.fixture(scope="module")
def ops():
    from model_optimizer_b200 import ops as _ops

    return _ops


def dev(x, d):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to("cuda").to(TD[d])


def host(t):
    return t.detach().float().cpu().numpy()


def rnd(shape, d, seed):
    return o.round_to(np.random.default_rng(seed).standard_normal(shape).astype(np.float32), d)


def bit_equal(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    return bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


# ---- kernels -----------------------------------------------------------------------------------
@pytest.mark.parametrize("d", ["bf16", "f16", "f32"])
def test_scale_cols_and_awq_step(ops, d):
    w = rnd((96, 512), d, 1)
    s = o.round_to(np.abs(rnd((512,), d, 2)) + np.float32(0.5), d)
    assert bit_equal(host(ops.scale_cols(dev(w, d), dev(s, d))), o.scale_cols(w, s, d))
    for bs, bits, narrow in ((128, 4, False), (64, 4, True), (16, 8, False), (512, 3, False)):
        got = host(ops.awq_scale_fake_quant(dev(w, d), dev(s, d), bs, bits, narrow))
        assert bit_equal(got, o.awq_scale_fake_quant(w, s, bs, bits, narrow, d)), (bs, bits, narrow)
    x = rnd((7, 40), d, 3)  # odd shape -> scalar kernel
    sx = o.round_to(np.abs(rnd((40,), d, 4)) + np.float32(0.1), d)
    assert bit_equal(host(ops.scale_cols(dev(x, d), dev(sx, d))), o.scale_cols(x, sx, d))


def test_awq_weight_scale(ops):
    for d in ("bf16", "f32"):
        w = rnd((300, 1024), d, 5)
        sums = torch.zeros(1024, dtype=torch.float32, device="cuda")
        ops.awq_weight_scale_sums_(sums, dev(w, d), 128)
        got = o.round_to(host(sums) / np.float32(300), d)
        ref = o.awq_weight_scale(w, 128, d)
        # fp32 accumulation order differs from torch's mean: <= 1 ulp of the weight dtype
        tol = 2.0**-7 if d == "bf16" else 1e-6
        assert np.allclose(got, ref, rtol=tol), np.max(np.abs(got - ref) / ref)


def test_mse_sweep(ops, algos):
    x, a0, mult = algos["mse/x"], algos["mse/amax0"], algos["mse/mult"]
    loss = torch.zeros(len(mult), dtype=torch.float64, device="cuda")
    ops.mse_sweep_(loss, dev(x, "bf16"), dev(a0, "f32").reshape(1), dev(mult, "f32"), 8, False, False)
    got = loss.cpu().numpy()
    assert np.allclose(got, algos["mse/losses"], rtol=2e-5)
    assert np.allclose(got, o.mse_sweep_losses(x, a0, mult, 8, False, False), rtol=1e-6)
    assert int(np.argmin(got)) == int(np.argmin(algos["mse/losses"]))
    loss8 = torch.zeros(len(mult), dtype=torch.float64, device="cuda")
    ops.mse_sweep_(loss8, dev(x, "bf16"), dev(a0, "f32").reshape(1), dev(mult, "f32"), 0)
    assert np.allclose(loss8.cpu().numpy(), o.mse_sweep_losses(x, a0, mult, 0), rtol=1e-6)


def test_nvfp4_fp8_scale_sweep(ops, algos):
    w, g = algos["sweep/w"], algos["sweep/global_amax"]
    got = host(ops.nvfp4_fp8_scale_sweep(dev(w, "bf16"), dev(g, "f32").reshape(1), candidates="ieee"))
    assert bit_equal(got, o.nvfp4_fp8_scale_sweep(w, g))
    # default candidates: as torch builds them on the GPU (multiply by fl(1 / 448))
    assert bit_equal(host(ops.fp8_scale_candidates("cuda")), o.fp8_scale_candidates(cuda_rule=True))
    got_dev = host(ops.nvfp4_fp8_scale_sweep(dev(w, "bf16"), dev(g, "f32").reshape(1)))
    assert bit_equal(got_dev, o.nvfp4_fp8_scale_sweep(w, g, cuda_rule=True))
    assert np.mean(got != algos["sweep/best_amax"]) <= 0.01  # reference Python sweep (CPU: IEEE candidates)
    w2 = rnd((64, 1024), "bf16", 8)
    w2[0] = 0
    g2 = o.reduce_amax(w2)
    assert bit_equal(host(ops.nvfp4_fp8_scale_sweep(dev(w2, "bf16"), dev(g2, "f32").reshape(1), candidates="ieee")),
                     o.nvfp4_fp8_scale_sweep(w2, g2))


# ---- host mirror ---------------------------------------------------------------------------------
def build_mlp(algos, key, d):
    m = nn.Sequential(nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, 32))
    with torch.no_grad():
        m[0].weight.copy_(torch.from_numpy(algos[f"{key}/w0"]))
        m[0].bias.copy_(torch.from_numpy(algos[f"{key}/b0"]))
        m[2].weight.copy_(torch.from_numpy(algos[f"{key}/w2"]))
        m[2].bias.copy_(torch.from_numpy(algos[f"{key}/b2"]))
    return m.to(TD[d]).cuda()


@pytest.mark.parametrize("cname", ["INT8_DEFAULT_CFG", "FP8_DEFAULT_CFG"])
@pytest.mark.parametrize("d", ["f32", "bf16"])
def test_quantize_max_presets_match_reference(algos, cname, d):
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    key = f"{cname}/{d}"
    model = build_mlp(algos, key, d)
    data = [dev(x, d) for x in algos[f"{key}/data"]]

    def loop(m):
        for x in data:
            m(x)

    with torch.no_grad():
        quantize(model, cfgs.get_preset(cname), loop)
        for li in (0, 2):
            for qn in ("input_quantizer", "weight_quantizer"):
                ref = algos[f"{key}/l{li}.{qn}.amax"]
                got = getattr(model[li], qn).amax
                assert got.dtype == TD[d]
                assert bit_equal(host(got).reshape(ref.shape), ref), (li, qn)
        y = host(model(data[0]))
    tol = 2e-4 if d == "f32" else 6e-2
    assert np.allclose(y, algos[f"{key}/y"], atol=tol, rtol=tol)


def test_smoothquant_matches_reference(algos):
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    for d in ("f32", "bf16"):
        key = f"INT8_SMOOTHQUANT_CFG/{d}"
        model = build_mlp(algos, key, d)
        data = [dev(x, d) for x in algos[f"{key}/data"]]
        with torch.no_grad():
            quantize(model, cfgs.get_preset("INT8_SMOOTHQUANT_CFG"), lambda m: [m(x) for x in data])
            for li in (0, 2):
                lin = model[li]
                tol = 1e-6 if d == "f32" else 2.0**-7
                assert np.allclose(host(lin.input_quantizer.pre_quant_scale), algos[f"{key}/l{li}.input_quantizer.pqs"], rtol=tol)
                assert np.allclose(host(lin.weight), algos[f"{key}/l{li}.weight_after"], rtol=tol, atol=1e-7)
                assert np.allclose(host(lin.input_quantizer.amax), algos[f"{key}/l{li}.input_quantizer.amax"], rtol=tol)
                assert np.allclose(host(lin.weight_quantizer.amax).ravel(), algos[f"{key}/l{li}.weight_quantizer.amax"].ravel(), rtol=tol)
            y = host(model(data[0]))
        tol = 1e-3 if d == "f32" else 8e-2
        assert np.allclose(y, algos[f"{key}/y"], atol=tol, rtol=tol)


def test_awq_lite_matches_reference(algos):
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    d = "f32"
    key = f"INT4_AWQ_CFG/{d}"
    model = build_mlp(algos, key, d)
    data = [dev(x, d) for x in algos[f"{key}/data"]]
    with torch.no_grad():
        quantize(model, cfgs.get_preset("INT4_AWQ_CFG"), lambda m: [m(x) for x in data])
        for li in (0, 2):
            lin = model[li]
            ref = algos[f"{key}/l{li}.input_quantizer.pqs"]
            got = host(lin.input_quantizer.pre_quant_scale)
            assert np.allclose(got, ref, rtol=1e-4), (li, np.max(np.abs(got - ref) / ref))
            assert np.allclose(host(lin.weight), algos[f"{key}/l{li}.weight_after"], rtol=1e-4, atol=1e-7)
        y = host(model(data[0]))
    assert np.allclose(y, algos[f"{key}/y"], atol=2e-3, rtol=2e-3)


def test_nvfp4_preset_and_real_quantize():
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize
    from model_optimizer_b200.qtensor import NVFP4QTensor

    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(256, 512), nn.GELU(), nn.Linear(512, 128)).to(torch.bfloat16).cuda()
    data = [torch.randn(32, 256, device="cuda", dtype=torch.bfloat16) for _ in range(3)]
    with torch.no_grad():
        quantize(model, cfgs.get_preset("NVFP4_DEFAULT_CFG"), lambda m: [m(x) for x in data])
        iq = model[0].input_quantizer
        want = max(float(x.abs().max()) for x in data)
        assert iq.amax.numel() == 1 and abs(float(iq.amax) - want) == 0
        x = data[0]
        xq = iq(x)
        ref = o.fake_quant_nvfp4(host(x), np.float32(want), "bf16")
        assert bit_equal(host(xq), ref)
        w = model[0].weight
        q, sf, sf2 = NVFP4QTensor.quantize(w, 16)
        p, s, s2 = o.pack_nvfp4(host(w))
        assert np.array_equal(q._quantized_data.cpu().numpy(), p)
        assert np.array_equal(sf.view(torch.uint8).cpu().numpy(), s)
        deq = q.dequantize(scale=sf, double_scale=sf2, block_sizes={-1: 16})
        assert bit_equal(host(deq), o.unpack_nvfp4(p, s, s2, "bf16"))


def test_histogram_calibrator_matches_oracle():
    from model_optimizer_b200.calib import HistogramCalibrator

    xs = [o.round_bf16(rnd((64, 512), "bf16", s) * np.float32(1 + 0.7 * s)) for s in range(3)]
    cal = HistogramCalibrator(8, None, False)
    ref = o.HistogramCalibrator(2048)
    for x in xs:
        cal.collect(dev(x, "bf16"))
        ref.collect(x)
    assert np.array_equal(cal._calib_hist.cpu().numpy(), ref.hist)
    assert cal._num_bins == ref.num_bins and np.array_equal(cal.calib_bin_edges, ref.edges)
    # the three searches == the oracle restatement (pinned to the reference by tests/test_oracle_calibrators.py)
    for pct in (99.9, 99.99, 50.0):
        assert float(cal.compute_amax("percentile", percentile=pct)) == float(o.hist_amax_percentile(ref.hist, ref.edges, pct))
    assert float(cal.compute_amax("mse")) == float(o.hist_amax_mse(ref.hist, ref.edges, 8, False, 1, 128))
    assert float(cal.compute_amax("mse", stride=5, start_bin=64)) == float(o.hist_amax_mse(ref.hist, ref.edges, 8, False, 5, 64))
    assert float(cal.compute_amax("entropy", start_bin=128, stride=16)) == \
        float(o.hist_amax_entropy(ref.hist, ref.edges, 8, False, 16, 128))


def test_cpu_tensor_is_rejected(ops):
    from model_optimizer_b200._lib import B200QuantError

    with pytest.raises(B200QuantError):
        ops.fake_quant_fp8(torch.randn(8), torch.tensor(1.0))


def test_sharded_engine_graph_step_matches_oracle():
    from model_optimizer_b200.engine import TINY, ShardedPTQEngine

    eng = ShardedPTQEngine(TINY, tokens=64, qformat="nvfp4", dtype=torch.bfloat16, device="cuda")
    acts = eng.alloc_activations(seed=3)
    outs = eng.alloc_outputs(4)
    eng.capture(acts, outs)
    assert float(eng.arena.freeze().abs().sum()) == 0.0
    eng.step_graph()
    eng.step_graph()  # running max over two identical batches == one batch
    torch.cuda.synchronize()
    want = np.array([float(o.reduce_amax(host(x))) for x in acts], dtype=np.float32)
    got = host(eng.arena.freeze())
    assert np.array_equal(got, want)
    assert np.array_equal(host(eng.amax_arena), o.round_bf16(want))
    res = eng.fake_quant(acts, outs)  # eager launches, ring of 4 output buffers: check the last four
    torch.cuda.synchronize()
    for (qn, q, _), x, y in list(zip(eng.quantizers, acts, res))[-4:]:
        ref = o.fake_quant_nvfp4(host(x), np.float32(host(q._amax)), "bf16")
        assert bit_equal(host(y), ref), qn
    assert eng.launches_per_step() == 3          # grouped (pointer-array) launches: collect, export, fake quant


def test_export_quantized_linear_formats(algos):
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200 import export as ex
    from model_optimizer_b200.model_quant import quantize

    torch.manual_seed(1)
    x = [torch.randn(64, 256, device="cuda", dtype=torch.bfloat16) for _ in range(2)]
    for preset, fmt in (("FP8_DEFAULT_CFG", "fp8"), ("NVFP4_DEFAULT_CFG", "nvfp4"), ("INT4_AWQ_CFG", "int4_awq")):
        model = nn.Sequential(nn.Linear(256, 512), nn.GELU(), nn.Linear(512, 256)).to(torch.bfloat16).cuda()
        with torch.no_grad():
            quantize(model, cfgs.get_preset(preset), lambda m: [m(t) for t in x])
        lin = model[0]
        out = ex.export_quantized_linear(lin)
        assert out["quantization"] == fmt
        w = host(lin.weight)
        if fmt == "fp8":
            amax = o.reduce_amax(w)
            sf = np.float32(amax) / np.float32(448.0)
            assert np.float32(host(out["weight_scale"])) == sf
            ref = o.pack_fp8(w, sf, 1, "bf16", "f32", scale_is_0dim=False)  # (1,) fp32 scale: fp32 quotient
            assert np.array_equal(out["weight"].view(torch.uint8).cpu().numpy(), ref)
            assert "input_scale" in out
            deq = ex.from_quantized_weight(out["weight"], out["weight_scale"], "fp8", torch.bfloat16)
            assert np.allclose(host(deq), w, rtol=0.07, atol=float(sf))
        elif fmt == "nvfp4":
            p, s, s2 = o.pack_nvfp4(w)
            assert np.array_equal(out["weight"].cpu().numpy(), p)
            assert np.array_equal(out["weight_scale"].view(torch.uint8).cpu().numpy(), s)
            assert np.float32(host(out["weight_scale_2"])) == np.float32(s2)
            assert float(out["input_scale"]) > 0
        else:
            wsf = host(out["weight_scale"])
            bam = o.reduce_block_amax(w, 128)
            assert np.array_equal(wsf, (bam / np.float32(7.0)).astype(np.float32))
            ref = o.pack_int4_export(w, wsf, "bf16", "f32")
            assert np.array_equal(out["weight"].cpu().numpy(), ref)
            assert "pre_quant_scale" in out and out["pre_quant_scale"].numel() == 256


def test_nvfp4_act_headroom_calibrator():
    from model_optimizer_b200.calib import NVFP4ActHeadroomCalibrator

    xs = [o.round_bf16(rnd((128, 1024), "bf16", s) * np.float32(0.5 + s)) for s in range(3)]
    xs[1][0, :16] = 0
    cal = NVFP4ActHeadroomCalibrator()
    hist = np.zeros(512, dtype=np.int64)
    rmax = np.float32(0)
    for x in xs:
        cal.collect(dev(x, "bf16"))
        h, m = o.nvfp4_block_log2_hist(x)
        hist += h
        rmax = max(rmax, m)
    got = cal._hist.cpu().numpy()
    assert got.sum() == hist.sum()
    assert np.abs(got - hist).sum() <= 4      # values on a bin edge may move with the last ulp of log2f
    assert np.float32(cal._running_max.item()) == rmax
    amax = float(cal.compute_amax())
    assert amax >= float(rmax) * 0.5 and np.isfinite(amax)


def test_fp8_per_channel_per_token_dynamic_preset():
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(128, 256)).to(torch.bfloat16).cuda()
    x = torch.randn(4, 8, 128, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        quantize(model, cfgs.get_preset("FP8_PER_CHANNEL_PER_TOKEN_CFG"), lambda m: m(x))
        lin = model[0]
        assert lin.input_quantizer._dynamic and lin.input_quantizer.amax is None
        xq = lin.input_quantizer(x)
        xh = host(x).reshape(-1, 128)
        # 3-D activation: the per-token amax [B, T, 1] has two non-singleton dims, for which the reference runs
        # _fp8_eager (tensor_quant.py:78-79); a 2-D activation [tokens, H] goes to fake_e4m3fy_with_axis
        ref = o.fake_quant_fp8(xh, o.reduce_amax(xh, axis=1), 128, "bf16", eager=True).reshape(4, 8, 128)
        assert bit_equal(host(xq), ref)
        from model_optimizer_b200.nn import TensorQuantizer

        fresh = TensorQuantizer({"num_bits": (4, 3), "type": "dynamic", "block_sizes": {-1: None}, "axis": None})
        x2 = x.reshape(-1, 128)      # the kept axes are fixed at the first call: a fresh quantizer for the 2-D case
        assert bit_equal(host(fresh(x2)), o.fake_quant_fp8(xh, o.reduce_amax(xh, axis=1), 128, "bf16"))
        wa = lin.weight_quantizer.amax
        assert tuple(wa.shape) == (256, 1)
        assert bit_equal(host(wa), o.reduce_amax(host(lin.weight), axis=1))


def test_awq_clip_picks_per_block_amax_within_range():
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(256, 128)).to(torch.bfloat16).cuda()
    with torch.no_grad():
        model[0].weight[:, ::37] *= 6  # outliers make clipping pay off in some blocks
    data = [torch.randn(64, 256, device="cuda", dtype=torch.bfloat16) for _ in range(2)]
    cfg = cfgs.get_preset("INT4_BLOCKWISE_WEIGHT_ONLY_CFG")
    cfg["algorithm"] = {"method": "awq_clip"}
    with torch.no_grad():
        quantize(model, cfg, lambda m: [m(t) for t in data])
    wq = model[0].weight_quantizer
    full = o.reduce_block_amax(host(model[0].weight), 128).reshape(-1, 1)
    got = host(wq.amax)
    assert got.shape == full.shape
    ratio = got / full
    assert np.all(ratio >= 0.5 - 1e-2) and np.all(ratio <= 1.0 + 1e-6)
    assert np.any(ratio < 0.999)


def test_hf_llama_shaped_model_ptq_presets():
    """Llama family through the API surface: every nn.Linear of a (tiny, random) HF LlamaForCausalLM gets
    calibrated quantizers, lm_head stays untouched, amaxes equal a recomputation from hooks."""
    pytest.importorskip("transformers")
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.llama_ptq import build_llama, run_llama_ptq
    from model_optimizer_b200.nn import QuantLinear

    for preset in ("NVFP4_DEFAULT_CFG", "FP8_DEFAULT_CFG", "INT8_DEFAULT_CFG"):
        model = build_llama(hidden=256, intermediate=512, layers=2, heads=4, kv_heads=2, vocab=512, max_pos=128)
        seen = {}

        def hook(name):
            def f(mod, inp):
                seen[name] = max(seen.get(name, 0.0), float(inp[0].abs().max()))
            return f

        hs = [m.register_forward_pre_hook(hook(n)) for n, m in model.named_modules() if isinstance(m, nn.Linear)]
        res = run_llama_ptq(preset, n_samples=8, seq_len=64, batch=4, model=model, vocab=512)
        for h in hs:
            h.remove()
        assert res["n_quantizers"] == 2 * 7 * 2 and res["amax_finite"]
        assert isinstance(model.lm_head, QuantLinear) and not model.lm_head.weight_quantizer.is_enabled
        lin = model.model.layers[1].mlp.down_proj
        assert float(lin.input_quantizer.amax) == seen["model.layers.1.mlp.down_proj"]
        wa = lin.weight_quantizer.amax
        if preset == "INT8_DEFAULT_CFG":
            assert tuple(wa.shape) == (256, 1)
            assert torch.equal(wa.squeeze(1), lin.weight.abs().amax(dim=1))
        else:
            assert float(wa) == float(lin.weight.abs().max())
        out = model(torch.randint(0, 512, (2, 64), device="cuda")).logits
        assert torch.isfinite(out).all()


def test_quantized_weight_cache_tracks_state():
    from model_optimizer_b200.nn import QuantLinear

    torch.manual_seed(0)
    lin = QuantLinear.convert(nn.Linear(64, 32).to(torch.bfloat16).cuda())
    lin.weight_quantizer.amax = lin.weight.detach().abs().amax(dim=1, keepdim=True)
    lin.input_quantizer.disable()
    x = torch.randn(4, 64, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        y1 = lin(x)
        cached = lin._weight_cache[1]
        y2 = lin(x)
        assert lin._weight_cache[1] is cached and torch.equal(y1, y2)
        lin.weight.mul_(0.5)                      # in-place change bumps the version -> recompute
        y3 = lin(x)
        assert lin._weight_cache[1] is not cached and not torch.equal(y1, y3)
        c2 = lin._weight_cache[1]
        lin.weight_quantizer.amax = lin.weight_quantizer.amax * 2  # state change -> recompute
        lin(x)
        assert lin._weight_cache[1] is not c2
    y4 = lin(x)                                   # grad mode: never cached
    assert lin._weight_cache is None and y4.requires_grad


def test_real_quantize_paths_return_reference_packs():
    """fake_quant=False: TensorQuantizer._real_quantize (tensor_quantizer.py:796-888) -> QTensor packs."""
    from model_optimizer_b200.nn import TensorQuantizer

    w = o.round_bf16(rnd((64, 256), "bf16", 21))
    wt = dev(w, "bf16")
    q = TensorQuantizer({"num_bits": (2, 1), "block_sizes": {-1: 16, "type": "dynamic", "scale_bits": (4, 3)},
                         "fake_quant": False})
    qt = q(wt)
    p, s, s2 = o.pack_nvfp4(w)
    assert np.array_equal(qt._quantized_data.cpu().numpy(), p)
    assert np.array_equal(q._scale.view(torch.uint8).cpu().numpy(), s) and np.float32(host(q._double_scale)) == np.float32(s2)
    deq = qt.dequantize(scale=q._scale, double_scale=q._double_scale, block_sizes={-1: 16})
    assert bit_equal(host(deq), o.unpack_nvfp4(p, s, s2, "bf16"))

    q = TensorQuantizer({"num_bits": 4, "block_sizes": {-1: 128}, "fake_quant": False})
    qt = q(wt)
    rp, rs = o.pack_int4_blockwise_cuda(w, 128, "bf16")
    assert np.array_equal(qt._quantized_data.cpu().numpy().reshape(-1), rp)
    assert bit_equal(host(q._scale), rs)
    deq = qt.dequantize(scale=q._scale, block_sizes={-1: 128})
    assert bit_equal(host(deq).reshape(-1), o.unpack_int4_blockwise(rp, rs, 128, "bf16"))

    q = TensorQuantizer({"num_bits": (4, 3), "axis": None, "fake_quant": False})
    qt = q(wt)
    sc = o.round_bf16(o.reduce_amax(w) / np.float32(448))
    assert bit_equal(host(q._scale), sc)
    assert np.array_equal(qt._quantized_data.view(torch.uint8).cpu().numpy(), o.pack_fp8(w, sc, 1, "bf16", "bf16"))


def test_nvfp4_static_mse_fp8_sweep_preset_end_to_end():
    """NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG: static block-16 weights, max-calibrate -> promote (fp32 per-block
    amax + global amax) -> per-block FP8-scale sweep -> static fake quant (config.py:1726, model_calib.py:733-827)."""
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    torch.manual_seed(3)
    model = nn.Sequential(nn.Linear(256, 128)).to(torch.bfloat16).cuda()
    x = torch.randn(16, 256, device="cuda", dtype=torch.bfloat16)
    with torch.no_grad():
        quantize(model, cfgs.get_preset("NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG"), lambda m: m(x))
        lin = model[0]
        wq = lin.weight_quantizer
        w = host(lin.weight)
        g = o.reduce_amax(w)
        assert wq._amax.dtype == torch.float32 and wq._global_amax.dtype == torch.float32
        assert np.float32(host(wq._global_amax)) == np.float32(g)
        best = o.nvfp4_fp8_scale_sweep(w, g, cuda_rule=True)      # candidates as torch builds them on the GPU
        assert bit_equal(host(wq._amax).ravel(), best)
        wfq = wq(lin.weight)
        ref = o.fake_quant_nvfp4_static(w, best, g, True, 448.0, "bf16")
        assert bit_equal(host(wfq), ref)
        iq = lin.input_quantizer
        assert iq.amax.numel() == 1 and float(iq.amax) == float(x.abs().max())
        assert torch.isfinite(model(x)).all()


def test_more_presets_on_llama_shaped_model():
    """The pattern-only / algorithm variants of the NVFP4 presets and the MX presets on a tiny HF Llama:
    the right quantizers end up enabled, AWQ leaves a pre_quant_scale, logits stay finite and close."""
    pytest.importorskip("transformers")
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.llama_ptq import build_llama
    from model_optimizer_b200.model_quant import quantize

    torch.manual_seed(0)
    ids = [torch.randint(0, 512, (4, 64), device="cuda") for _ in range(2)]

    def loop(m):
        for t in ids:
            m(t)

    base = build_llama(hidden=256, intermediate=512, layers=2, heads=4, kv_heads=2, vocab=512, max_pos=128)
    sd = {k: v.clone() for k, v in base.state_dict().items()}
    with torch.no_grad():
        ref_logits = base(ids[0]).logits.float()
    for preset in ("NVFP4_AWQ_LITE_CFG", "NVFP4_AWQ_CLIP_CFG", "W4A16_NVFP4_CFG", "NVFP4_MLP_ONLY_CFG",
                   "W4A8_NVFP4_FP8_CFG", "MXFP8_DEFAULT_CFG", "MXFP4_MLP_WEIGHT_ONLY_CFG", "W4A8_MXFP4_FP8_CFG"):
        model = build_llama(hidden=256, intermediate=512, layers=2, heads=4, kv_heads=2, vocab=512, max_pos=128)
        model.load_state_dict(sd)
        with torch.no_grad():
            quantize(model, cfgs.get_preset(preset), loop)
            logits = model(ids[0]).logits.float()
        assert torch.isfinite(logits).all(), preset
        err = (logits - ref_logits).norm() / ref_logits.norm()
        assert err < 0.5, (preset, float(err))
        layer = model.model.layers[0]
        q, down = layer.self_attn.q_proj, layer.mlp.down_proj
        if preset == "NVFP4_AWQ_LITE_CFG":
            assert down.input_quantizer.pre_quant_scale is not None and q.input_quantizer.amax is not None
        if preset == "W4A16_NVFP4_CFG":
            assert q.weight_quantizer.is_enabled and not q.input_quantizer.is_enabled
        if preset in ("NVFP4_MLP_ONLY_CFG", "MXFP4_MLP_WEIGHT_ONLY_CFG"):
            assert down.weight_quantizer.is_enabled and not q.weight_quantizer.is_enabled
        if preset == "MXFP4_MLP_WEIGHT_ONLY_CFG":
            assert down.weight_quantizer.is_mx_format and not down.input_quantizer.is_enabled
        if preset == "W4A8_MXFP4_FP8_CFG":
            assert q.weight_quantizer.is_mx_format and q.input_quantizer.num_bits == (4, 3)
            assert q.input_quantizer.amax is None  # algorithm None: the FP8 input quantizer stays dynamic
        if preset == "MXFP8_DEFAULT_CFG":
            assert q.weight_quantizer.amax is None and q.input_quantizer.is_mx_format


def test_bias_calibrator_and_affine_quantizer():
    """a22: BiasCalibrator statistics through the fused max/min/sum kernel vs the reference run on CPU (fixture),
    vs torch on the GPU, and an affine (bias-shifted) INT8 quantizer end to end."""
    import os

    from model_optimizer_b200.calib import BiasCalibrator
    from model_optimizer_b200.nn import TensorQuantizer

    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_bias.npz"))
    keys = sorted({k.rsplit("/x0", 1)[0] for k in G.files if k.endswith("/x0")})
    assert len(keys) == 8
    for key in keys:
        _, dname, _, ax = key.split("/")
        axis = None if ax == "none" else tuple(int(a) for a in ax.split("_"))
        dt = torch.bfloat16 if dname == "bf16" else torch.float32
        x0, x1 = torch.from_numpy(G[key + "/x0"]).cuda().to(dt), torch.from_numpy(G[key + "/x1"]).cuda().to(dt)
        cal = BiasCalibrator("max_min", axis)
        cal.collect(x0)
        assert np.array_equal(host(cal.compute_bias()), G[key + "/max_min/b0"]), key
        cal.collect(x1)
        assert np.array_equal(host(cal.compute_bias()), G[key + "/max_min/b1"]), key
        cal = BiasCalibrator("mean", axis)
        cal.collect(x0)
        ref = G[key + "/mean/b0"]
        tol = (2.0 ** -7 if dname == "bf16" else 2.0 ** -21) * np.maximum(np.abs(ref), np.abs(G[key + "/x0"]).mean())
        assert np.all(np.abs(host(cal.compute_bias()) - ref) <= tol), key
    # larger, aligned (vector kernel) + unaligned (generic kernel) shapes against torch on the GPU
    from model_optimizer_b200.calib.bias import compute_maxmin

    g = torch.Generator(device="cuda").manual_seed(0)
    for shape, axis in (((4, 8, 300, 128), (-2, -4)), ((4, 8, 300, 128), None), ((7, 33, 50), (0, 1)), ((64, 1000), (0,))):
        x = (torch.randn(shape, device="cuda", generator=g) * 3 + 0.5).to(torch.bfloat16)
        mx, mn = compute_maxmin(x, axis)
        red = tuple(range(x.dim())) if axis is None else tuple(i for i in range(x.dim()) if i in axis or (i - x.dim()) in axis)
        want_mx = torch.amax(x, dim=red, keepdim=axis is not None)
        want_mn = torch.amin(x, dim=red, keepdim=axis is not None)
        assert torch.equal(mx, want_mx) and torch.equal(mn, want_mn), (shape, axis)
    # affine INT8 quantizer: static bias is collected, subtracted before and added after the fake quant
    x = (torch.randn(2, 4, 64, 32, device="cuda", generator=g) + 2.0).to(torch.bfloat16)
    tq = TensorQuantizer({"num_bits": 8, "axis": None, "bias": {-2: None, -4: None, "type": "static", "method": "max_min"}})
    tq.enable_calib()
    tq.disable_quant()
    tq(x)
    tq.load_calib_amax()
    tq.load_calib_bias()
    tq.enable_quant()
    tq.disable_calib()
    b = tq.bias_value
    assert tuple(b.shape) == (1, 4, 1, 32)
    xb = x - b
    assert float(tq.amax) == float(xb.abs().max())
    want = o.fake_quant_int(host(xb), np.float32(float(tq.amax)), 8, False, False, 1, "bf16")
    got = tq(x)
    assert torch.equal(got, torch.from_numpy(want).cuda().to(torch.bfloat16) + b)
    assert float((got.float() - x.float()).abs().max()) < float(tq.amax) / 127 * 0.75 + 0.02


def test_fp8_block_scales_eager_rule_and_2d_blocks(ops):
    """FP8 with static 1-D / 2-D block scales (FP8_2D_BLOCKWISE_WEIGHT_ONLY_CFG): the quantizer's tile amax, the
    eager-rule fake quant the reference runs for multi-dim amax (tensor_quant.py:78-79), FP8QTensor pack / dequant
    with block_sizes and the fp8_pb_wo export -- against the reference run on CPU (tests/golden/ref_fp8_blocks.*.npz)."""
    import os

    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200 import export as ex
    from model_optimizer_b200.model_quant import quantize
    from model_optimizer_b200.nn import TensorQuantizer
    from model_optimizer_b200.qtensor import FP8QTensor

    G = _golden.load("ref_fp8_blocks")
    keys = sorted({k.rsplit("/x", 1)[0] for k in G.files if k.endswith("/x")})
    assert len(keys) == 12
    for key in keys:
        _, dname, _, blk, _ = key.split("/")
        b1, b2 = (int(v) for v in blk.split("x"))
        dt = torch.bfloat16 if dname == "bf16" else torch.float32
        x = torch.from_numpy(G[key + "/x"]).cuda().to(dt)
        blocks = {-1: b2, -2: b1}
        tq = TensorQuantizer({"num_bits": (4, 3), "axis": None, "block_sizes": dict(blocks)})
        tq.enable_calib()
        tq.disable_quant()
        tq(x)
        tq.load_calib_amax()
        tq.enable_quant()
        tq.disable_calib()
        assert tuple(tq.amax.shape) == tuple(G[key + "/amax"].shape), key
        assert np.array_equal(host(tq.amax), G[key + "/amax"]), key
        assert bit_equal(host(tq(x)), G[key + "/fq"]), key
        q, sc = FP8QTensor.quantize(x, block_sizes=dict(blocks))
        assert np.array_equal(host(sc), G[key + "/scale"]), key
        assert np.array_equal(q._quantized_data.view(torch.uint8).cpu().numpy(), G[key + "/q"]), key
        assert bit_equal(host(q.dequantize(dtype=dt, scale=sc, block_sizes=dict(blocks))), G[key + "/deq"]), key
        wsf = (tq.amax.float() / torch.tensor(448.0, device="cuda")).squeeze()
        q2, _ = FP8QTensor.quantize(x, wsf, block_sizes=dict(blocks))
        assert np.array_equal(q2._quantized_data.view(torch.uint8).cpu().numpy(), G[key + "/q_export"]), key
    # eager rule vs the oracle on a per-tensor / per-row amax too
    x = rnd((96, 256), "bf16", 3)
    am = np.float32(np.abs(x).max())
    assert bit_equal(host(ops.fake_quant_fp8(dev(x, "bf16"), dev(am, "f32").reshape(1), eager=True)),
                     o.fake_quant_fp8(x, am, 1, "bf16", eager=True))
    rows = o.reduce_amax(x, axis=1).reshape(-1)
    assert bit_equal(host(ops.fake_quant_fp8(dev(x, "bf16"), dev(rows, "f32"), outer=256, eager=True)),
                     o.fake_quant_fp8(x, rows, 256, "bf16", eager=True))
    # the preset end to end + export
    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(384, 256, bias=False)).cuda().to(torch.bfloat16)
    w = model[0].weight.detach().clone()
    quantize(model, cfgs.get_preset("FP8_2D_BLOCKWISE_WEIGHT_ONLY_CFG"), lambda m: m(torch.randn(4, 384, device="cuda", dtype=torch.bfloat16)))
    wq = model[0].weight_quantizer
    assert tuple(wq.amax.shape) == (2, 1, 3, 1) and not model[0].input_quantizer.is_enabled
    wh = host(w)
    amax = np.abs(wh.reshape(2, 128, 3, 128)).max(axis=(1, 3))
    assert np.array_equal(host(wq.amax).reshape(2, 3), amax)
    d = ex.export_quantized_linear(model[0])
    assert d["quantization"] == "fp8_pb_wo" and tuple(d["weight_scale"].shape) == (2, 3)
    wsf = (amax.astype(np.float32) / np.float32(448.0)).astype(np.float32)
    assert np.array_equal(host(d["weight_scale"]), wsf)
    rows32 = np.broadcast_to(wsf[:, None, :], (2, 128, 3)).reshape(-1)
    want = o.pack_fp8(wh.reshape(2, 128, 3, 128).reshape(-1), rows32, 128, "bf16", "f32").reshape(256, 384)
    assert np.array_equal(d["weight"].view(torch.uint8).cpu().numpy(), want)


def test_int8_qtensor_matches_reference(ops):
    """INT8QTensor (a15): per-tensor / per-channel / 1-D and 2-D block scales, computed or given -- codes, scales and
    dequantized values against the reference run on CPU (tests/golden/ref_int8.npz); plus the kernel against the
    oracle on a large tensor with non-finite values."""
    import os

    from model_optimizer_b200.qtensor import INT8QTensor

    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_int8.npz"))
    bases = sorted({k.rsplit("/x", 1)[0] for k in G.files if k.endswith("/x")})
    assert len(bases) == 12
    dts = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}
    n = 0
    for base in bases:
        dname = base.split("/")[1]
        dt = dts[dname]
        x = torch.from_numpy(G[base + "/x"]).cuda().to(dt)
        for mode, kw in (("tensor", {}), ("axis0", {"axis": 0}), ("block128", {"block_sizes": {-1: 128}}),
                         ("block8x64", {"block_sizes": {-1: 64, -2: 8}})):
            key = f"{base}/{mode}"
            if key + "/q" not in G.files:
                continue
            q, sc = INT8QTensor.quantize(x.clone(), **kw)
            assert q._quantized_data.dtype == torch.int8
            assert np.array_equal(host(sc).reshape(G[key + "/scale"].shape), G[key + "/scale"]), key
            assert np.array_equal(q._quantized_data.cpu().numpy().reshape(G[key + "/q"].shape), G[key + "/q"]), key
            dkw = {"block_sizes": kw["block_sizes"]} if "block_sizes" in kw else {}
            assert bit_equal(host(q.dequantize(dtype=dt, scale=sc, **dkw)), G[key + "/deq"]), key
            n += 1
        sc32 = torch.from_numpy(G[base + "/given_f32/scale"]).cuda()
        q, _ = INT8QTensor.quantize(x.clone(), sc32)
        assert np.array_equal(q._quantized_data.cpu().numpy(), G[base + "/given_f32/q"]), base
    assert n >= 40
    # kernel vs oracle: 1 M elements, ragged tail, inf / NaN / huge values, per-row scales
    x = rnd((1024, 1031), "bf16", 9)
    x[3, 5], x[4, 6], x[5, 7], x[6, 8] = np.inf, -np.inf, np.nan, 3.0e38
    rows = o.round_bf16(o.reduce_amax(np.where(np.isfinite(x), x, 0), axis=1).reshape(-1) / np.float32(127.0))
    got = ops.pack_int8(dev(x, "bf16"), dev(rows, "bf16"), outer=1031).cpu().numpy()
    want = o.pack_int8(x.reshape(-1), rows, 1031, "bf16", "bf16").reshape(x.shape)
    assert np.array_equal(got, want)
    back = ops.unpack_int8(torch.from_numpy(want).cuda(), dev(rows, "bf16"), torch.bfloat16, outer=1031)
    assert bit_equal(host(back), o.unpack_int8(want.reshape(-1), rows, 1031, "bf16").reshape(x.shape))
