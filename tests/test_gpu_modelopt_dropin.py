"""The north-star boundary on the GPU: the REAL ``modelopt.torch.quantization.quantize()`` (the unmodified
reference installed into ``baseline/_ref`` by ``__graft_entry__.build()``), once stock -- the reference's own CUDA
extensions (compiled from its sources, ``oracle/build_ref_ext.py``) and its Triton kernels (JIT on the box) -- and
once with this engine plugged in through ``backend.install()`` + ``with_b200_backend`` (backend entry point,
``B200MaxCalibrator`` via the ``calibrator`` field, extension shims, FP8-sweep factory, QTensor packs).

Same tiny HF Llama, same seeded calibration batches.  Bars (written per test):
  * every ``_amax`` / ``_global_amax`` / ``_pre_quant_scale`` buffer bit-equal;
  * fake-quant outputs of every quantizer on a fresh input bit-equal for INT8 / FP8 / INT4, and equal up to exact
    E2M1 rounding ties for NVFP4 (the reference's Triton kernels divide with ``div.full.f32``; its own test skips
    tie vectors, tests/gpu/torch/quantization/test_tensor_quant_cuda.py:243-245);
  * ``mtq.compress`` packed weights and scales bit-exact;
  * ``backend.stats`` proves the b200 arm actually ran the kernels (no silent stock path).

Those tests need the reference installed and are skipped without it.  The two that compare this repo's own code
with the reference (``quantize()`` mirror, Hessian sweep) fall back to what the reference produced on the same inputs,
stored in tests/golden/ref_gpu_dropin/ (see tests/_refgold.py).  The stored mirror results come from a stock run
recorded with one torch / cuBLAS build (the tiny Llama's forward feeds the calibration), so a torch upgrade may call
for a re-record (B200Q_RECORD_GOLDEN) even where this engine is still correct."""

import copy
import json
import os

import numpy as np
import pytest
import torch
from _refgold import RefResults, Store

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPORT = {}


@pytest.fixture(scope="module")
def env():
    from baseline import ref_env

    if not ref_env.available():
        pytest.skip("baseline/_ref not populated (run __graft_entry__.build() where /root/reference exists)")
    mtq = ref_env.activate()
    loaded = ref_env.use_prebuilt_extensions()
    from model_optimizer_b200 import backend

    REPORT["reference_extensions_prebuilt"] = loaded
    return mtq, backend


def _reference_installed():
    from baseline import ref_env

    return ref_env.available()


@pytest.fixture(scope="module")
def store():
    s = Store("ref_gpu_dropin", _reference_installed())
    yield s
    s.save()


@pytest.fixture
def refs(store, request):
    return RefResults(store, request.node.name)


def _stock_quantize(base, preset):
    """The stock reference's ``mtq.quantize`` of ``base`` with ``preset`` (live runs only)."""
    from baseline import ref_env

    mtq = ref_env.activate()
    ref_env.use_prebuilt_extensions()
    from model_optimizer_b200 import backend

    backend.uninstall()
    return mtq.quantize(copy.deepcopy(base), copy.deepcopy(getattr(mtq, preset)), forward_loop)


def tiny_llama(seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM

    cfg = LlamaConfig(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, vocab_size=256, max_position_embeddings=128, tie_word_embeddings=False)
    torch.manual_seed(seed)
    return LlamaForCausalLM(cfg).to(device="cuda", dtype=torch.bfloat16).eval()


def calib_batches(n=4, b=2, t=48, seed=1):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 256, (b, t), generator=g).cuda() for _ in range(n)]


def forward_loop(model):
    for ids in calib_batches():
        model(ids)


def quantizer_buffers(model):
    out = {}
    for name, m in model.named_modules():
        if type(m).__name__ in ("TensorQuantizer", "StaticBlockScaleQuantizer"):
            for b in ("_amax", "_global_amax", "_pre_quant_scale"):
                t = getattr(m, b, None)
                if isinstance(t, torch.Tensor):
                    out[f"{name}.{b}"] = t.detach().clone()
    return out


def run_pair(env, preset_name, algorithm=None, mutate=None):
    """-> (stock model, b200 model, stats of the b200 arm)."""
    mtq, backend = env
    base = tiny_llama()
    cfg = copy.deepcopy(getattr(mtq, preset_name))
    if algorithm is not None:
        cfg["algorithm"] = algorithm
    if mutate is not None:
        mutate(cfg)
    backend.uninstall()
    stock = mtq.quantize(copy.deepcopy(base), copy.deepcopy(cfg), forward_loop)
    backend.install()
    backend.stats.clear()
    try:
        mine = mtq.quantize(copy.deepcopy(base), backend.with_b200_backend(cfg), forward_loop)
        st = dict(backend.stats)
    finally:
        backend.uninstall()
    return stock, mine, st


def assert_buffers_equal(stock, mine, what):
    a, b = quantizer_buffers(stock), quantizer_buffers(mine)
    assert a.keys() == b.keys(), (what, sorted(set(a) ^ set(b))[:8])
    assert len(a) > 0 or "MX" in what, what              # MX formats keep no amax state
    bad = [k for k in a if a[k].shape != b[k].shape or a[k].dtype != b[k].dtype or not torch.equal(a[k], b[k])]
    assert not bad, (what, len(bad), bad[:6],
                     [(a[k].flatten()[:3].tolist(), b[k].flatten()[:3].tolist()) for k in bad[:3]])
    return len(a)


def mismatch_stats(ref, got):
    ref, got = ref.float(), got.float()
    zero = (ref == 0) & (got == 0)
    diff = (ref != got) & ~zero
    r, g_ = ref[diff].abs(), got[diff].abs()
    hi, lo = torch.maximum(r, g_), torch.minimum(r, g_)
    bounded = bool(((lo == 0) | (hi / lo <= 2.05)).all())
    return int(diff.sum()), bounded


def _same_to_1ulp(a, b):
    """fp32 equality up to one unit in the last place."""
    ai, bi = a.contiguous().view(torch.int32).long(), b.contiguous().view(torch.int32).long()
    return (ai - bi).abs() <= 1


def compare_outputs(env, stock, mine, exact, what):
    """Logits of both quantized models on a fresh batch (each arm through its own kernels)."""
    mtq, backend = env
    ids = calib_batches(n=1, seed=7)[0]
    with torch.no_grad():
        y0 = stock(ids).logits
        backend.install()
        try:
            y1 = mine(ids).logits
        finally:
            backend.uninstall()
    if exact:
        assert torch.equal(y0, y1), (what, float((y0.float() - y1.float()).abs().max()))
        return 0.0
    # NVFP4 arms differ by exact-tie roundings of a few % of the elements (one E2M1 step each, see
    # per_quantizer_outputs); through two random-init layers that is a ~10 % relative logit difference -- the
    # parity statement is the per-quantizer one, this only guards against gross divergence
    rel = float((y0.float() - y1.float()).norm() / y0.float().norm())
    assert rel < 0.3, (what, rel)
    return rel


def per_quantizer_outputs(env, stock, mine, exact, what):
    """Feed every enabled quantizer of both arms the same fresh tensor (its own weight for weight quantizers)."""
    mtq, backend = env
    mods0, mods1 = dict(stock.named_modules()), dict(mine.named_modules())
    g = torch.Generator(device="cuda").manual_seed(3)
    n_total = n_bad = 0
    for name, q0 in mods0.items():
        if type(q0).__name__ not in ("TensorQuantizer", "StaticBlockScaleQuantizer") or not q0.is_enabled:
            continue
        q1 = mods1[name]
        qname = name
        while qname.rsplit(".", 1)[-1].isdigit():          # a member of a SequentialQuantizer: "...weight_quantizer.0"
            qname = qname.rsplit(".", 1)[0]
        parent = mods0[qname.rsplit(".", 1)[0]]
        if qname.endswith("weight_quantizer"):
            x = parent.weight.detach()
        else:
            x = torch.randn(2, 48, parent.in_features, device="cuda", generator=g).to(torch.bfloat16) * 0.7
        with torch.no_grad():
            y0 = q0(x)
            backend.install()
            try:
                y1 = q1(x)
            finally:
                backend.uninstall()
        assert y0.shape == y1.shape and y0.dtype == y1.dtype, (what, name)
        n, bounded = mismatch_stats(y0, y1)
        n_total += y0.numel()
        n_bad += n
        if exact:
            assert n == 0, (what, name, n)
        else:
            # NVFP4 vs the reference's Triton kernels: exact E2M1 / E4M3 rounding ties only (every mismatch within
            # one code step).  5 % like tests/test_gpu_vs_reference_triton.py: torch evaluates the global scale
            # `amax / (6 * 448)` on the GPU as a reciprocal multiply (one ulp off the IEEE value this engine uses),
            # which moves the tie set of 8-bit-mantissa data
            assert bounded and n <= 0.05 * y0.numel(), (what, name, n, y0.numel())
    assert n_total > 0
    return n_bad, n_total


# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("preset,exact", [("INT8_DEFAULT_CFG", True), ("FP8_DEFAULT_CFG", True),
                                          ("INT4_BLOCKWISE_WEIGHT_ONLY_CFG", True), ("NVFP4_DEFAULT_CFG", False),
                                          ("FP8_PER_CHANNEL_PER_TOKEN_CFG", True), ("MXFP8_DEFAULT_CFG", True)])
def test_max_calibration_presets(env, preset, exact):
    stock, mine, st = run_pair(env, preset)
    n = assert_buffers_equal(stock, mine, preset)
    if preset not in ("INT4_BLOCKWISE_WEIGHT_ONLY_CFG", "MXFP8_DEFAULT_CFG", "FP8_PER_CHANNEL_PER_TOKEN_CFG"):
        assert st.get("calib.max", 0) > 0, st            # activations calibrated through the b200 collect kernel
    env[1].stats.clear()
    bad, tot = per_quantizer_outputs(env, stock, mine, exact, preset)
    rel = compare_outputs(env, stock, mine, exact, preset)
    assert env[1].stats.get("entrypoint", 0) > 0, dict(env[1].stats)     # fake quant ran through the b200 backend
    st["forward"] = dict(env[1].stats)
    REPORT[preset] = {"buffers_equal": n, "fake_quant_mismatch": [bad, tot], "logit_rel_diff": rel, "stats": st}


def test_int4_awq_lite(env):
    """awq_lite (model_calib.py:1395-1722) with the INT4 block-128 weight fake quant on this engine: the loss per
    alpha, hence best_alpha and the folded pre_quant_scale, must come out the same."""
    stock, mine, st = run_pair(env, "INT4_AWQ_CFG")
    n = assert_buffers_equal(stock, mine, "INT4_AWQ_CFG")
    pqs = [k for k in quantizer_buffers(mine) if k.endswith("_pre_quant_scale")]
    assert pqs, "awq_lite produced no pre_quant_scale"
    # the smoothed weights themselves
    for (n0, p0), (n1, p1) in zip(stock.named_parameters(), mine.named_parameters()):
        assert n0 == n1 and torch.equal(p0, p1), n0
    bad, tot = per_quantizer_outputs(env, stock, mine, True, "INT4_AWQ_CFG")
    rel = compare_outputs(env, stock, mine, True, "INT4_AWQ_CFG")
    REPORT["INT4_AWQ_CFG"] = {"buffers_equal": n, "pre_quant_scales": len(pqs), "fake_quant_mismatch": [bad, tot],
                              "logit_rel_diff": rel, "stats": st}


def test_int8_smoothquant(env):
    stock, mine, st = run_pair(env, "INT8_SMOOTHQUANT_CFG")
    n = assert_buffers_equal(stock, mine, "INT8_SMOOTHQUANT_CFG")
    for (n0, p0), (n1, p1) in zip(stock.named_parameters(), mine.named_parameters()):
        assert n0 == n1 and torch.equal(p0, p1), n0
    rel = compare_outputs(env, stock, mine, True, "INT8_SMOOTHQUANT_CFG")
    REPORT["INT8_SMOOTHQUANT_CFG"] = {"buffers_equal": n, "logit_rel_diff": rel, "stats": st}


def test_nvfp4_static_weights_max(env):
    """Static NVFP4 weights (per-block amax + shared global amax of q/k/v and gate/up,
    utils/shared_input.py:314-346) after plain max calibration: per-block ``_amax`` and the tied ``_global_amax``
    are exact; fake quant goes through the rebound ``static_blockwise_fp4_fake_quant``."""
    stock, mine, st = run_pair(env, "NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG", algorithm="max")
    n = assert_buffers_equal(stock, mine, "nvfp4_static_max")
    mods = dict(mine.named_modules())
    attn = mods["model.layers.0.self_attn"]
    g = [getattr(attn, p).weight_quantizer._global_amax for p in ("q_proj", "k_proj", "v_proj")]
    assert torch.equal(g[0], g[1]) and torch.equal(g[1], g[2])
    env[1].stats.clear()
    bad, tot = per_quantizer_outputs(env, stock, mine, False, "nvfp4_static_max")
    rel = compare_outputs(env, stock, mine, False, "nvfp4_static_max")
    assert env[1].stats.get("fn.static_blockwise_fp4_fake_quant", 0) > 0, dict(env[1].stats)
    st["forward"] = dict(env[1].stats)
    REPORT["nvfp4_static_max"] = {"buffers_equal": n, "fake_quant_mismatch": [bad, tot], "logit_rel_diff": rel,
                                  "stats": st}


def test_nvfp4_static_mse_fp8_sweep(env):
    """mse_calibrate(fp8_scale_sweep=True): stock = the reference's Triton sweep, b200 = the registered factory
    (``_register_fp8_sweep_calibrator``) running ``b200q_nvfp4_fp8_scale_sweep``.  The winner is an argmin over 126
    fp32 losses summed in a different order: >= 99 % identical per-block winners, everything else bit-equal.
    ``best_amax = global_amax * c`` with c = e4m3 / 448: the reference builds c with torch on the GPU (a multiply by
    fl(1/448)), this engine with an IEEE division -- the same winner can differ in the last bit of the fp32 amax
    (inside the north star's "fp32 amax/scale within 1 ulp"); adjacent candidates are >= 6 % apart."""
    stock, mine, st = run_pair(env, "NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG")
    assert st.get("calib.fp8_sweep", 0) > 0, st
    a, b = quantizer_buffers(stock), quantizer_buffers(mine)
    assert a.keys() == b.keys()
    same = total = bitsame = 0
    for k in a:
        if k.endswith("weight_quantizer._amax"):
            assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype == torch.float32, k
            same += int(_same_to_1ulp(a[k], b[k]).sum())
            bitsame += int((a[k] == b[k]).sum())
            total += a[k].numel()
        else:
            assert torch.equal(a[k], b[k]), k
    assert total > 0 and same / total >= 0.99, (same, total)
    rel = compare_outputs(env, stock, mine, False, "nvfp4_static_mse")
    REPORT["nvfp4_static_mse_fp8_sweep"] = {"same_block_winner": [same, total], "bit_identical_amax": bitsame,
                                            "logit_rel_diff": rel, "stats": st}


@pytest.mark.parametrize("preset", ["INT8_DEFAULT_CFG", "FP8_DEFAULT_CFG", "INT4_BLOCKWISE_WEIGHT_ONLY_CFG"])
def test_mse_calibrate_multiplier_search(env, preset):
    """mse_calibrate (model_calib.py:733-827) without the FP8 sweep: the 39-step multiplier search of every weight
    amax (per-channel INT8 rows, per-tensor FP8, INT4 block-128 rows).  Stock = the reference's MseCalibrator
    (39 x fake quant through its CUDA extension + ATen reductions); b200 = one sweep kernel per weight.  The
    losses are fp32 sums in a different order, so a winner may differ where two multipliers tie to ~1e-6:
    >= 99.5 % identical amax entries, all within one multiplier step."""
    stock, mine, st = run_pair(env, preset, algorithm="mse")
    assert st.get("calib.mse", 0) > 0, st
    a, b = quantizer_buffers(stock), quantizer_buffers(mine)
    assert a.keys() == b.keys()
    same = total = 0
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, k
        if k.endswith("weight_quantizer._amax"):
            same += int((a[k] == b[k]).sum())
            total += a[k].numel()
            r = (a[k].float() / b[k].float())
            assert float(r.max()) < 1.6 and float(r.min()) > 0.6, (k, float(r.min()), float(r.max()))
        else:
            assert torch.equal(a[k], b[k]), k
    assert total > 0 and same / total >= 0.995, (same, total)
    REPORT[f"mse_{preset}"] = {"same_amax": [same, total], "stats": st}


@pytest.mark.parametrize("preset", ["FP8_DEFAULT_CFG", "NVFP4_DEFAULT_CFG", "INT4_BLOCKWISE_WEIGHT_ONLY_CFG",
                                    "FP8_2D_BLOCKWISE_WEIGHT_ONLY_CFG"])
def test_compress_packs_bit_exact(env, preset):
    """mtq.compress -> TensorQuantizer._real_quantize (:796-887) -> QTensor.quantize: packed bytes and scales."""
    mtq, backend = env
    stock, mine, _ = run_pair(env, preset)
    mtq.compress(stock)
    backend.install()
    backend.stats.clear()
    try:
        mtq.compress(mine)
        st = dict(backend.stats)
    finally:
        backend.uninstall()
    key = {"FP8_DEFAULT_CFG": "qtensor.fp8_quantize", "FP8_2D_BLOCKWISE_WEIGHT_ONLY_CFG": "qtensor.fp8_quantize",
           "NVFP4_DEFAULT_CFG": "qtensor.nvfp4_quantize", "INT4_BLOCKWISE_WEIGHT_ONLY_CFG": "ext.INT4_quantize"}[preset]
    assert st.get(key, 0) > 0, st
    n = 0
    m1 = dict(mine.named_modules())
    for name, m0 in stock.named_modules():
        w0 = m0._parameters.get("weight") if hasattr(m0, "_parameters") else None
        if type(w0).__name__ != "QTensorWrapper":        # RealQuantLinear keeps the pack as its weight parameter
            continue
        w1 = m1[name]._parameters["weight"]
        assert type(w1).__name__ == "QTensorWrapper", name
        assert w0.metadata["shape"] == w1.metadata["shape"] and w0.metadata["dtype"] == w1.metadata["dtype"]
        assert w0.metadata["qtensor_class"] is w1.metadata["qtensor_class"], name      # the REFERENCE's QTensor class
        q0, q1 = w0.data, w1.data
        assert q0.shape == q1.shape and q0.dtype == q1.dtype, (name, q0.shape, q1.shape, q0.dtype, q1.dtype)
        assert torch.equal(q0.view(torch.uint8), q1.view(torch.uint8)), (name, preset)
        for b in ("_scale", "_double_scale"):
            s0, s1 = getattr(m0.weight_quantizer, b, None), getattr(m1[name].weight_quantizer, b, None)
            assert (s0 is None) == (s1 is None), (name, b)
            if s0 is not None:
                assert s0.shape == s1.shape and s0.dtype == s1.dtype, (name, b, s0.shape, s1.shape, s0.dtype, s1.dtype)
                v0 = s0.view(torch.uint8) if s0.dtype == torch.float8_e4m3fn else s0
                v1 = s1.view(torch.uint8) if s1.dtype == torch.float8_e4m3fn else s1
                assert torch.equal(v0, v1), (name, b, preset)
        n += 1
    assert n > 0, "no compressed weights found"
    REPORT[f"compress_{preset}"] = {"packed_weights_equal": n, "stats": st}


@pytest.mark.parametrize("preset,exact", [("INT8_DEFAULT_CFG", True), ("FP8_DEFAULT_CFG", True),
                                          ("NVFP4_DEFAULT_CFG", True), ("INT8_SMOOTHQUANT_CFG", True),
                                          ("INT4_AWQ_CFG", True), ("NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG", False),
                                          ("NVFP4_W4A4_WEIGHT_LOCAL_HESSIAN_CFG", False)])
def test_mirror_quantize_matches_reference(refs, preset, exact):
    """The repo's own ``quantize()`` (the mirror of the reference interface) against the stock reference on the
    same tiny Llama: every linear's ``_amax`` / ``_global_amax`` / ``_pre_quant_scale`` and the smoothed weights.
    Against the stored reference, INT4-AWQ's smoothed weights are compared on a sample of their rows."""
    import model_optimizer_b200.config as cfgs
    from model_optimizer_b200.model_quant import quantize

    base = tiny_llama()
    stock = _stock_quantize(base, preset) if refs.store.live else None
    mine = quantize(copy.deepcopy(base), copy.deepcopy(getattr(cfgs, preset)), forward_loop)
    a = {k: v for k, v in quantizer_buffers(stock).items() if "_bmm_quantizer" not in k and "softmax" not in k} \
        if stock is not None else {}
    b = {}
    for name, m in mine.named_modules():
        if type(m).__name__ == "TensorQuantizer":
            for bn in ("_amax", "_global_amax", "_pre_quant_scale"):
                t = getattr(m, bn, None)
                if isinstance(t, torch.Tensor):
                    b[f"{name}.{bn}"] = t.detach()
    keys = [str(k) for k in refs.array(lambda: np.array(sorted(a)))]
    assert set(keys) == b.keys(), sorted(set(keys) ^ set(b))[:10]
    same = total = 0
    awq = preset == "INT4_AWQ_CFG"
    for k in keys:
        y = b[k].reshape(-1)
        if awq or (k.endswith("weight_quantizer._amax") and not exact):
            x = refs.rows(y, lambda: a[k].reshape(-1), whole=True)[0].reshape(-1)
        else:
            x = refs.bits(y, lambda: a[k].reshape(-1))
        assert x.numel() == y.numel(), (k, x.shape, y.shape)
        assert x.dtype == y.dtype, (k, x.dtype, y.dtype)
        if awq:
            # AWQ-lite: act_scale is a mean of |x| over tokens -- ATen's reduction order in the reference, one column
            # kernel here: fp32 sums within ~1e-6, so the folded bf16 scales / smoothed weights / their amax may
            # differ by one bf16 ulp (DESIGN.md section 4 tolerance class); best_alpha must agree (checked below)
            eq = (x.float() - y.float()).abs() <= x.float().abs() * 2.0 ** -6
            assert bool(eq.all()), (preset, k, int((~eq).sum()))
        elif k.endswith("weight_quantizer._amax") and not exact:
            eq = _same_to_1ulp(x, y)                                # FP8 sweep winners (see the sweep test)
        else:
            eq = x == y
            assert bool(eq.all()), (preset, k, int((~eq).sum()), x[:3].tolist(), y[:3].tolist())
        same += int(eq.sum())
        total += eq.numel()
    # sweeps: argmin over 126 fp32 losses (Hessian: a 16 x 16 quadratic form summed in another order than tl.dot)
    assert same / total >= (0.97 if "HESSIAN" in preset else 0.99), (same, total)
    names = [str(n) for n in refs.array(lambda: np.array([n for n, _ in stock.named_parameters()]))]
    params0 = dict(stock.named_parameters()) if stock is not None else {}
    assert names == [n for n, _ in mine.named_parameters()]
    for n0, p1 in mine.named_parameters():
        if awq:
            p0, p1 = refs.rows(p1.detach(), lambda: params0[n0].detach())
            assert torch.allclose(p0.float(), p1.float(), rtol=2.0 ** -6, atol=1e-6), n0
            # identical best_alpha <=> the scale vectors agree to rounding (a different alpha moves them by >> 1 ulp)
        else:
            assert torch.equal(refs.bits(p1.detach(), lambda: params0[n0].detach()), p1), n0   # smoothquant folded weights
    REPORT[f"mirror_{preset}"] = {"buffers": len(keys), "same_entries": [same, total]}


def test_hessian_sweep_vs_reference_triton_kernel(refs):
    """``nvfp4_fp8_scale_sweep_hessian`` (kernels/quantization/gemm/nvfp4_fp8_sweep.py:235-290), the reference's own
    Triton kernel JIT-compiled on this box, against ``b200q_nvfp4_fp8_scale_sweep_hessian`` on the same weight and
    per-cin-block Hessian.  Winners may differ only where two candidates' fp32 losses are equal to ~1e-6."""
    from model_optimizer_b200 import ops

    def reference(w, gam, hess):
        from baseline import ref_env

        ref_env.activate()
        from modelopt.torch.kernels.quantization.gemm import nvfp4_fp8_scale_sweep_hessian

        return nvfp4_fp8_scale_sweep_hessian(w.reshape(-1, 16), gam, hess, 16)

    g = torch.Generator(device="cuda").manual_seed(11)
    rep = {}
    for dtype in (torch.bfloat16, torch.float32):
        w = (torch.randn(384, 512, device="cuda", generator=g) * 0.05).to(dtype)
        x = torch.randn(2048, 512, device="cuda", generator=g) * (1 + 3 * torch.rand(512, device="cuda", generator=g))
        xt = x.float().T.reshape(512 // 16, 16, -1)
        hess = (xt @ xt.transpose(-1, -2)) / x.shape[0]
        gam = w.abs().max().float()
        got = ops.nvfp4_fp8_scale_sweep(w, gam.reshape(1), hessian=hess)
        ref = refs.rows(got.reshape(-1), lambda: reference(w, gam, hess).reshape(-1), whole=True)[0].reshape(got.shape)
        same = float(_same_to_1ulp(ref, got).float().mean())
        # the plain (unweighted) winner must differ from the Hessian one for a good share of the blocks
        plain = ops.nvfp4_fp8_scale_sweep(w, gam.reshape(1))
        moved = float((plain != got).float().mean())
        rep[str(dtype)] = {"same_winner": same, "differs_from_plain_mse": moved}
        assert same >= 0.985, (dtype, same)
        assert moved > 0.05, moved
    REPORT["hessian_sweep_vs_triton"] = rep


def test_zz_write_report():
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "modelopt_dropin.json"), "w") as f:
        json.dump(REPORT, f, indent=1, default=str)
