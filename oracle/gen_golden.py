"""Generate tests/golden/ref_*.npz by running the REAL reference on CPU in this container.

Run from the repo root (only where /root/reference exists):  python oracle/gen_golden.py
The fixtures are committed; the GPU box never needs /root/reference.

Test infrastructure, not product code.  The import shim below (fake dist version, stub
``omegaconf`` / ``pulp``) is the one documented in SURVEY.md Appendix D.
"""

from __future__ import annotations

import importlib.metadata as md
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _golden  # noqa: E402  (the fixtures' file format: split into parts under 1 MB)


def _install_shim():
    orig = md.version
    md.version = lambda n: "0.0.0+ref" if n == "nvidia-modelopt" else orig(n)

    class _Any(types.ModuleType):
        def __getattr__(self, k):
            if k.startswith("__"):
                raise AttributeError(k)
            return type(k, (), {})

    oc = _Any("omegaconf")
    oc.DictConfig = type("DictConfig", (dict,), {})
    oc.ListConfig = type("ListConfig", (list,), {})
    sys.modules["omegaconf"] = oc
    sys.modules["pulp"] = _Any("pulp")
    sys.path.insert(0, "/root/reference")


def bits16(t):
    import torch

    return t.contiguous().view(torch.int16).numpy().view(np.uint16).copy()


def make_inputs(seed, shape, kind, dtype):
    """Synthetic inputs (SURVEY.md 8d): gaussian, heavy tail, exact ties, zeros / one-hot blocks."""
    import torch

    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g)
    if kind == "heavy":
        x = x * (1 + 20 * (torch.rand(shape, generator=g) < 1e-2).float())
    elif kind == "ties":
        # multiples of E2M1 / integer rounding boundaries times power-of-two scales
        vals = torch.tensor([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0, 6.0, 0.5, 1.5, 2.0, 3.0, 4.0, 0.0, 7.0, 0.125])
        idx = torch.randint(0, 16, shape, generator=g)
        sgn = torch.randint(0, 2, shape, generator=g) * 2 - 1
        x = vals[idx] * sgn * (2.0 ** torch.randint(-3, 3, (shape[0], 1), generator=g))
    elif kind == "sparse":
        x = x * (torch.rand(shape, generator=g) < 0.05).float()
        x[0] = 0
        x[1, :16] = 0
        x[2, 5] = 3.0
        x[3] = x[3] * 1e-30
        x[4, 0] = -0.0
    return x.to(dtype)


def main():
    _install_shim()
    import torch

    torch.manual_seed(0)
    import modelopt.torch.quantization  # noqa: F401
    from modelopt.torch.export.quant_utils import pack_int4_in_uint8
    from modelopt.torch.kernels.quantization.gemm.fp4_kernel import compute_fp4_scales
    from modelopt.torch.quantization import tensor_quant as tq
    from modelopt.torch.quantization.calib import HistogramCalibrator, MaxCalibrator
    from modelopt.torch.quantization.qtensor import FP8QTensor, INT4QTensor, NVFP4QTensor
    from modelopt.torch.quantization.utils import reduce_amax, reduce_block_amax

    os.makedirs(OUT, exist_ok=True)
    shape = (48, 256)
    out = {}
    cases = []
    for dname, dtype in (("bf16", torch.bfloat16), ("f16", torch.float16), ("f32", torch.float32)):
        for kind in ("gauss", "heavy", "ties", "sparse"):
            if dname != "bf16" and kind in ("heavy",):
                continue
            seed = len(cases) + 1
            x = make_inputs(seed, shape, kind, dtype)
            key = f"{dname}_{kind}"
            cases.append(key)
            xf = x.float()
            out[f"{key}/x"] = xf.numpy().copy()

            # --- collect -------------------------------------------------------------------
            out[f"{key}/amax_tensor"] = reduce_amax(x).float().numpy()
            out[f"{key}/amax_rows"] = reduce_amax(x, axis=1).float().numpy()          # [48,1]
            out[f"{key}/amax_cols"] = reduce_amax(x, axis=0).float().numpy()          # [1,256]
            out[f"{key}/amax_block16"] = reduce_block_amax(x, {-1: 16}).float().numpy()
            out[f"{key}/amax_block128"] = reduce_block_amax(x, {-1: 128}).float().numpy()
            if kind != "sparse" or dname == "bf16":
                cal = MaxCalibrator(8, None, False)
                cal.collect(x)
                cal.collect(x * 0.5)
                out[f"{key}/maxcal"] = cal.compute_amax().float().numpy()
                cal0 = MaxCalibrator(8, 0, False)
                cal0.collect(x)
                out[f"{key}/maxcal_axis0"] = cal0.compute_amax().float().numpy()

            amax_t = reduce_amax(x)
            amax_r = reduce_amax(x, axis=1)
            # --- integer fake quant (CPU twin; differs from the CUDA kernel only for unsigned /
            #     tiny amax, SURVEY.md A.6) -------------------------------------------------------
            for bits, narrow in ((8, False), (8, True), (4, False), (3, True)):
                out[f"{key}/int{bits}_n{int(narrow)}_tensor"] = (
                    tq._tensor_quant(x, amax_t, bits, False, narrow).float().numpy()
                )
            out[f"{key}/int8_rows"] = tq._tensor_quant(x, amax_r, 8, False, False).float().numpy()
            xb = x.reshape(-1, 128)
            out[f"{key}/int4_block128"] = (
                tq._tensor_quant(xb, reduce_amax(xb, axis=1), 4, False, False).float().numpy().reshape(shape)
            )
            # --- fp8 fake quant -------------------------------------------------------------
            out[f"{key}/fp8_tensor"] = tq.fp8_eager(x, amax_t).float().numpy()
            out[f"{key}/fp8_rows"] = tq.fp8_eager(x, amax_r).float().numpy()
            out[f"{key}/fp8_noamax"] = tq.fp8_eager(x, None).float().numpy()
            # --- nvfp4 ----------------------------------------------------------------------
            if kind != "sparse":
                q, sf, sf2 = NVFP4QTensor.quantize(x.clone(), 16)
                out[f"{key}/nvfp4_packed"] = q._quantized_data.numpy().copy()
                out[f"{key}/nvfp4_scales"] = sf.view(torch.uint8).numpy().copy()
                out[f"{key}/nvfp4_wsf2"] = sf2.float().numpy()
                deq = q.dequantize(dtype=dtype, scale=sf, double_scale=sf2, block_sizes={-1: 16})
                out[f"{key}/nvfp4_deq"] = deq.float().numpy()
                # static scales (CPU path of compute_fp4_scales -> fp8_eager)
                bam = reduce_block_amax(x, {-1: 16}).float()
                out[f"{key}/fp4_scales_static"] = compute_fp4_scales(bam, amax_t.float(), True).numpy()
                out[f"{key}/fp4_scales_static_46"] = compute_fp4_scales(bam, amax_t.float(), True, 256.0).numpy()

                class _Q:  # minimal static-quantizer stand-in for the static pack branch
                    pass

                wq = _Q()
                wq.block_sizes = {-1: 16}
                wq._amax = bam.reshape(-1, 1)
                wq.global_amax = amax_t.float()
                wq._global_amax = amax_t.float()
                wsf, wsf2 = NVFP4QTensor.get_weights_scaling_factor_from_quantizer(wq, x)
                qs, _, _ = NVFP4QTensor.quantize(x.clone(), 16, wsf, wsf2)
                out[f"{key}/nvfp4s_packed"] = qs._quantized_data.numpy().copy()
                out[f"{key}/nvfp4s_scales"] = wsf.view(torch.uint8).numpy().copy()
                out[f"{key}/nvfp4s_wsf2"] = wsf2.float().numpy()
            # --- int4 packs -----------------------------------------------------------------
            if kind in ("gauss", "heavy", "ties"):
                qi, sc = INT4QTensor.quantize(x.clone(), 128)   # CPU branch (RNE before clamp)
                out[f"{key}/int4cpu_packed"] = qi._quantized_data.numpy().reshape(-1).copy()
                out[f"{key}/int4cpu_scales"] = sc.float().numpy()
                wscale = (reduce_block_amax(x, {-1: 128}).float() / 7.0)
                out[f"{key}/int4exp_scale"] = wscale.numpy()
                out[f"{key}/int4exp_packed"] = pack_int4_in_uint8(x, wscale).numpy().copy()
                wscale_same = (reduce_block_amax(x, {-1: 128}) / 7.0)
                out[f"{key}/int4exp_scale_same"] = wscale_same.float().numpy()
                out[f"{key}/int4exp_packed_same"] = pack_int4_in_uint8(x, wscale_same).numpy().copy()
            # --- fp8 packs ------------------------------------------------------------------
            if kind != "sparse":
                qf, sc = FP8QTensor.quantize(x.clone())
                out[f"{key}/fp8pack_tensor"] = qf._quantized_data.view(torch.uint8).numpy().copy()
                out[f"{key}/fp8pack_tensor_scale"] = sc.float().numpy()
                qf, sc = FP8QTensor.quantize(x.clone(), axis=0)
                out[f"{key}/fp8pack_rows"] = qf._quantized_data.view(torch.uint8).numpy().copy()
                out[f"{key}/fp8pack_rows_scale"] = sc.float().numpy()
                s0 = amax_t.float() / 448.0   # export path: 0-dim fp32 scale
                out[f"{key}/fp8pack_export"] = (x / s0).to(torch.float8_e4m3fn).view(torch.uint8).numpy().copy()
                out[f"{key}/fp8pack_export_scale"] = s0.numpy()
                # what unified_export_hf really passes: get_scaling_factor() keeps export_amax()'s shape (1,), so
                # `weight / scale` promotes to fp32 (export/quant_utils.py:225-242, 854-866)
                from modelopt.torch.export.quant_utils import to_quantized_weight
                out[f"{key}/fp8pack_export1"] = to_quantized_weight(x, s0.reshape(1), "fp8").view(torch.uint8).numpy().copy()
            # --- histogram --------------------------------------------------------------------
            if dname == "bf16" and kind in ("gauss", "heavy"):
                hc = HistogramCalibrator(8, None, False, num_bins=2048)
                hc.collect(x)
                out[f"{key}/hist1"] = hc._calib_hist.numpy().copy()
                out[f"{key}/hist1_edges_last"] = hc._calib_bin_edges[-1].numpy().copy()
                hc.collect(x * 1.5)
                out[f"{key}/hist2"] = hc._calib_hist.numpy().copy()
                out[f"{key}/hist2_edges_last"] = hc._calib_bin_edges[-1].numpy().copy()

    out["cases"] = np.array(cases)
    print("wrote", _golden.save("ref_small", out, OUT), len(out), "arrays")




def main_algos():
    """Second fixture file: whole-algorithm outputs of the reference on CPU (config 1 plumbing, MSE
    sweeps, the NVFP4 FP8-scale sweep, AWQ-lite / SmoothQuant end to end on a tiny MLP)."""
    _install_shim()
    import torch
    import torch.nn as nn

    import modelopt.torch.quantization as mtq
    from modelopt.torch.quantization import tensor_quant as tq
    from modelopt.torch.quantization.calib.mse import MseCalibrator, NVFP4MSECalibrator
    from modelopt.torch.quantization.utils import reduce_amax, reduce_block_amax

    out = {}
    torch.manual_seed(0)

    # ---- config 1: 2-layer MLP, INT8 per-tensor mtq.quantize() + MaxCalibrator on CPU ---------------
    def mlp(dtype):
        torch.manual_seed(1)
        m = nn.Sequential(nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, 32)).to(dtype)
        return m

    def calib_batches(dtype, n=4):
        g = torch.Generator().manual_seed(7)
        return [torch.randn(16, 64, generator=g).to(dtype) for _ in range(n)]

    for cname in ("INT8_DEFAULT_CFG", "FP8_DEFAULT_CFG", "INT8_SMOOTHQUANT_CFG", "INT4_AWQ_CFG"):
        for dname, dtype in (("f32", torch.float32), ("bf16", torch.bfloat16)):
            if cname == "FP8_DEFAULT_CFG" and dname == "bf16":
                pass
            model = mlp(dtype)
            data = calib_batches(dtype)
            key = f"{cname}/{dname}"
            out[f"{key}/w0"] = model[0].weight.detach().float().numpy().copy()
            out[f"{key}/b0"] = model[0].bias.detach().float().numpy().copy()
            out[f"{key}/w2"] = model[2].weight.detach().float().numpy().copy()
            out[f"{key}/b2"] = model[2].bias.detach().float().numpy().copy()
            out[f"{key}/data"] = torch.stack(data).float().numpy()

            def loop(m):
                for d in data:
                    m(d)

            import copy

            cfg = copy.deepcopy(getattr(mtq, cname))
            model = mtq.quantize(model, cfg, loop)
            for li in (0, 2):
                lin = model[li]
                for qn in ("input_quantizer", "weight_quantizer"):
                    q = getattr(lin, qn)
                    if getattr(q, "_amax", None) is not None:
                        out[f"{key}/l{li}.{qn}.amax"] = q._amax.detach().float().numpy().copy()
                    if getattr(q, "_pre_quant_scale", None) is not None:
                        out[f"{key}/l{li}.{qn}.pqs"] = q._pre_quant_scale.detach().float().numpy().copy()
                out[f"{key}/l{li}.weight_after"] = lin.weight.detach().float().numpy().copy()
            with torch.no_grad():
                out[f"{key}/y"] = model(data[0]).float().numpy().copy()

    # ---- MSE calibrator (per-tensor, INT8 via the CPU twin) -----------------------------------------
    x = make_inputs(3, (64, 256), "heavy", torch.bfloat16)
    amax = reduce_amax(x)
    cal = MseCalibrator(amax=amax, axis=None, quant_func=lambda t, a: tq._tensor_quant(t, a, 8, False, False))
    cal.collect(x)
    out["mse/x"] = x.float().numpy()
    out["mse/amax0"] = amax.float().numpy()
    out["mse/mult"] = cal._candidates.numpy().copy()
    out["mse/losses"] = torch.stack(cal._losses_sum).double().numpy()
    out["mse/best"] = cal.compute_amax().float().numpy()

    # ---- NVFP4 FP8-scale sweep: the reference 126-step Python sweep on CPU ------------------------------
    w = make_inputs(5, (32, 256), "gauss", torch.bfloat16)
    bam = reduce_block_amax(w, {-1: 16}).float().reshape(-1, 1)
    g = reduce_amax(w).float()

    def qf(t, a):  # static NVFP4 fake quant in pure torch (what the quantizer's quant_func computes)
        scale = (a.float() / 6.0)
        s = torch.where(scale == 0, torch.ones_like(scale), scale)
        absx = t.abs() / s
        b = torch.tensor([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0])
        vals = torch.tensor([0, 0.5, 1, 1.5, 2, 3, 4, 6.0])
        idx = torch.bucketize(absx, b, right=False)
        tie_up = (absx == 0.75) | (absx == 1.75) | (absx == 3.5)
        q = vals[idx + tie_up.long()]
        return torch.sign(t) * q * s

    ncal = NVFP4MSECalibrator(amax=bam, global_amax=g, axis=0, quant_func=qf)
    ncal.collect(w.reshape(-1, 16))
    out["sweep/w"] = w.float().numpy()
    out["sweep/global_amax"] = g.numpy()
    out["sweep/best_amax"] = ncal.compute_amax().float().numpy().ravel()

    np.savez_compressed(os.path.join(OUT, "ref_algos.npz"), **out)
    print("wrote", os.path.join(OUT, "ref_algos.npz"), len(out), "arrays")


def main_presets():
    """Dump the reference's preset PTQ configs (config.py:1681-1778) as JSON for config parity tests."""
    _install_shim()
    import json

    import modelopt.torch.quantization as mtq

    names = ["INT8_DEFAULT_CFG", "INT8_SMOOTHQUANT_CFG", "INT8_WEIGHT_ONLY_CFG", "FP8_DEFAULT_CFG",
             "FP8_PER_CHANNEL_PER_TOKEN_CFG", "NVFP4_DEFAULT_CFG", "NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG",
             "NVFP4_W4A4_WEIGHT_LOCAL_HESSIAN_CFG", "INT4_BLOCKWISE_WEIGHT_ONLY_CFG", "INT4_AWQ_CFG", "NVFP4_AWQ_LITE_CFG", "NVFP4_AWQ_CLIP_CFG",
             "W4A16_NVFP4_CFG", "W4A8_NVFP4_FP8_CFG", "NVFP4_EXPERTS_ONLY_CFG", "NVFP4_MLP_ONLY_CFG",
             "NVFP4_OMLP_ONLY_CFG", "NVFP4_MLP_WEIGHT_ONLY_CFG", "MXFP8_DEFAULT_CFG", "MXFP6_DEFAULT_CFG",
             "MXFP4_DEFAULT_CFG", "MXINT8_DEFAULT_CFG", "W4A8_MXFP4_FP8_CFG", "MXFP4_MLP_WEIGHT_ONLY_CFG",
             "FP8_2D_BLOCKWISE_WEIGHT_ONLY_CFG"]

    def norm(o):
        if isinstance(o, dict):
            return {str(k): norm(v) for k, v in o.items()}
        if isinstance(o, (list, tuple)):
            return [norm(v) for v in o]
        return o

    out = {n: norm(getattr(mtq, n)) for n in names}
    with open(os.path.join(OUT, "ref_presets.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote ref_presets.json")


def _load_ref_libs():
    """oracle/_ref/libmxref*.so: the reference's own C++ (built by `make -C oracle`, see the Makefile)."""
    import ctypes

    import torch

    libdir = os.path.join(os.path.dirname(torch.__file__), "lib")
    for n in ["libc10.so", "libtorch_cpu.so", "libc10_cuda.so", "libtorch_cuda.so", "libtorch.so", "libtorch_python.so"]:
        try:
            ctypes.CDLL(os.path.join(libdir, n), mode=ctypes.RTLD_GLOBAL)
        except OSError:
            pass
    ref = os.path.join(ROOT, "oracle", "_ref")
    h = ctypes.CDLL(os.path.join(ref, "libmxref.so"))
    h.ref_convert_to_exmy_n.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_int]
    cu = ctypes.CDLL(os.path.join(ref, "libmxref_cu.so"))
    cu.ref_mx_block.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    return h, cu


def main_mx():
    """MX formats: element rounding + fused_amax_convert block math from the reference's C++ (host build),
    MXFP8 / MXFP4 QTensor round trips from the reference's Python."""
    _install_shim()
    import torch
    from modelopt.torch.quantization.qtensor.mxfp4_tensor import MXFP4QTensor
    from modelopt.torch.quantization.qtensor.mxfp8_tensor import MXFP8QTensor

    h, cu = _load_ref_libs()
    out = {}
    rng = np.random.default_rng(7)
    # (1) convert_to_exmy on a dense set of values incl. every tie of the small formats
    for fmt in range(9):
        xs = [rng.standard_normal(2000).astype(np.float32) * 3, (rng.standard_normal(500) * 300).astype(np.float32),
              np.array([0.0, -0.0, np.inf, -np.inf, 1e-9, -1e-9, 1e30], np.float32),
              np.arange(0, 64, 0.03125, dtype=np.float32), -np.arange(0, 64, 0.03125, dtype=np.float32),
              np.arange(0, 1, 1 / 1024, dtype=np.float32), np.arange(0, 70000, 128, dtype=np.float32),
              np.arange(0, 1 / 64, 1 / 131072, dtype=np.float32)]
        x = np.concatenate(xs)
        x = np.concatenate([x, np.nextafter(x, np.float32(1e9)), np.nextafter(x, np.float32(-1e9))]).astype(np.float32)
        if fmt != 2:                      # INT8 of NaN / |x| >= 2^31 is undefined in the reference (int conversion:
            x = np.concatenate([x, np.array([np.nan], np.float32)])    # x86 gives INT_MIN, the GPU saturates)
        else:
            x = x[np.abs(x) < 2.0e9]
        y = np.empty_like(x)
        h.ref_convert_to_exmy_n(x.ctypes.data, y.ctypes.data, x.size, fmt)
        out[f"cvt/{fmt}/x"] = x.view(np.uint32)
        out[f"cvt/{fmt}/y"] = y.view(np.uint32)
    # (2) fused_amax_convert block math (E8M0 scale), all formats x block sizes x dtypes
    tdt = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}
    for fmt in range(9):
        for bs in (8, 16, 32):
            for dname, dt in tdt.items():
                for kind, shape in (("gauss", (6, 96)), ("heavy", (6, 96)), ("ties", (6, 64)), ("sparse", (6, 64)),
                                    ("ragged", (5, 72 + bs // 2))):
                    x = make_inputs(100 * fmt + bs, shape, "gauss" if kind == "ragged" else kind, torch.float32)
                    if kind == "gauss":
                        x = x * (2.0 ** torch.randint(-30, 30, (shape[0], 1), generator=torch.Generator().manual_seed(bs)))
                        x[0, :bs] = 0
                        x[1, 0] = 448.0 * 4      # exact power-of-two ratios amax / dmax
                        x[2, 0] = 6.0 / 64
                    x = x.to(dt)
                    if fmt == 2:      # INT8 of +-inf is undefined on the host (int conversion): keep it finite
                        x = torch.nan_to_num(x, posinf=torch.finfo(dt).max, neginf=-torch.finfo(dt).max)
                    xf = x.float().numpy()
                    y = np.zeros_like(xf)
                    for r in range(xf.shape[0]):
                        for c0 in range(0, xf.shape[1], bs):
                            blk = np.ascontiguousarray(xf[r, c0:c0 + bs])
                            yb = np.empty_like(blk)
                            cu.ref_mx_block(blk.ctypes.data, yb.ctypes.data, blk.size, fmt, 9)
                            y[r, c0:c0 + bs] = yb
                    yt = torch.from_numpy(y).to(dt)              # y[real_idx] = quantize(...): float -> T
                    key = f"fq/{fmt}/{bs}/{dname}/{kind}"
                    out[key + "/x"] = xf.view(np.uint32)
                    out[key + "/y"] = yt.float().numpy().view(np.uint32)
    # (3) QTensor round trips
    for dname, dt in tdt.items():
        for kind, shape in (("gauss", (8, 96)), ("heavy", (8, 96)), ("ties", (8, 64)), ("sparse", (8, 64))):
            x = make_inputs(11, shape, kind, torch.float32)
            if kind == "gauss":
                x = x * (2.0 ** torch.randint(-40, 40, (shape[0], 1), generator=torch.Generator().manual_seed(3)))
                x[1, 0] = 448.0 * 8
                x[2, 0] = 6.0 / 32
            x = x.to(dt)
            # an inf block amax is undefined in MXFP4QTensor (inf -> uint8 cast of the exponent): keep x finite
            x = torch.nan_to_num(x, posinf=torch.finfo(dt).max, neginf=-torch.finfo(dt).max)
            key = f"qt/{dname}/{kind}"
            out[key + "/x"] = x.float().numpy().view(np.uint32)
            q8, s8 = MXFP8QTensor.quantize(x)
            out[key + "/mxfp8/q"] = q8._quantized_data.view(torch.uint8).numpy().copy()
            out[key + "/mxfp8/scale"] = s8.numpy().copy()
            out[key + "/mxfp8/deq"] = q8.dequantize(dtype=dt, scale=s8).float().numpy().view(np.uint32)
            for bs in (32, 16):
                q4, s4 = MXFP4QTensor.quantize(x, bs)
                out[key + f"/mxfp4_{bs}/q"] = q4._quantized_data.numpy().copy()
                out[key + f"/mxfp4_{bs}/scale"] = s4.numpy().copy()
                out[key + f"/mxfp4_{bs}/deq"] = q4.dequantize(dtype=dt, scale=s4, block_sizes={-1: bs}).float().numpy().view(np.uint32)
        # ragged last dim: MXFP8 pads to 32 and crops; row 0 holds an inf, row 1 a NaN (defined for MXFP8)
        x = make_inputs(12, (4, 80), "gauss", dt)
        x[0, 3] = float("inf")
        x[1, 70] = float("nan")
        q8, s8 = MXFP8QTensor.quantize(x)
        out[f"qt/{dname}/ragged/x"] = x.float().numpy().view(np.uint32)
        out[f"qt/{dname}/ragged/mxfp8/q"] = q8._quantized_data.view(torch.uint8).numpy().copy()
        out[f"qt/{dname}/ragged/mxfp8/scale"] = s8.numpy().copy()
        out[f"qt/{dname}/ragged/mxfp8/deq"] = q8.dequantize(dtype=dt, scale=s8).float().numpy().view(np.uint32)
    print("wrote", _golden.save("ref_mx", out, OUT), len(out), "arrays")


def main_bias():
    """BiasCalibrator (calib/bias.py) on CPU: running max_min / mean statistics over two batches."""
    _install_shim()
    import torch
    from modelopt.torch.quantization.calib.bias import BiasCalibrator

    out = {}
    tdt = {"bf16": torch.bfloat16, "f32": torch.float32}
    for dname, dt in tdt.items():
        for shape, axis in (((3, 4, 10, 16), (-2, -4)), ((3, 4, 10, 16), None), ((6, 10, 32), (0, 1)), ((5, 7, 24), (-2,))):
            g = torch.Generator().manual_seed(len(shape) * 7 + (0 if axis is None else len(axis)))
            xs = [(torch.randn(shape, generator=g) * 3 + 0.7).to(dt), (torch.randn(shape, generator=g) * 2 - 1.1).to(dt)]
            key = f"bias/{dname}/{'x'.join(map(str, shape))}/{'none' if axis is None else '_'.join(map(str, axis))}"
            out[key + "/x0"] = xs[0].float().numpy()
            out[key + "/x1"] = xs[1].float().numpy()
            for method in ("max_min", "mean"):
                cal = BiasCalibrator(method=method, axis=axis)
                cal.collect(xs[0])
                out[key + f"/{method}/b0"] = cal.compute_bias().float().numpy()
                cal.collect(xs[1])
                out[key + f"/{method}/b1"] = cal.compute_bias().float().numpy()
    np.savez_compressed(os.path.join(OUT, "ref_bias.npz"), **out)
    print("wrote", os.path.join(OUT, "ref_bias.npz"), len(out), "arrays")


def main_nvfp4_blocks():
    """NVFP4QTensor with block sizes other than 16 (W4A8_NVFP4_FP8_CFG / NVFP4_MLP_WEIGHT_ONLY_CFG use 32)."""
    _install_shim()
    import torch
    from modelopt.torch.quantization.qtensor.nvfp4_tensor import NVFP4QTensor

    out = {}
    for dname, dt in {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}.items():
        for kind in ("gauss", "heavy", "ties", "sparse"):
            x = make_inputs(21, (8, 256), kind, dt)
            for bs in (32, 64):
                key = f"nvfp4b/{dname}/{kind}/{bs}"
                q, sf, sf2 = NVFP4QTensor.quantize(x, bs)
                out[key + "/x"] = x.float().numpy()
                out[key + "/packed"] = q._quantized_data.numpy().copy()
                out[key + "/scale"] = sf.view(torch.uint8).numpy().copy()
                out[key + "/sf2"] = sf2.float().numpy()
                out[key + "/deq"] = q.dequantize(dtype=dt, scale=sf, double_scale=sf2, block_sizes={-1: bs}).float().numpy()
    np.savez_compressed(os.path.join(OUT, "ref_nvfp4_blocks.npz"), **out)
    print("wrote", os.path.join(OUT, "ref_nvfp4_blocks.npz"), len(out), "arrays")


def main_fp8_blocks():
    """FP8 with 2-D / 1-D static block scales: TensorQuantizer fake quant (runs _fp8_eager, tensor_quant.py:78-79)
    and FP8QTensor.quantize / dequantize with block_sizes (qtensor/fp8_tensor.py:41-155), on CPU."""
    _install_shim()
    import torch
    from modelopt.torch.quantization.nn import TensorQuantizer
    from modelopt.torch.quantization.config import QuantizerAttributeConfig
    from modelopt.torch.quantization.qtensor.fp8_tensor import FP8QTensor

    out = {}
    for dname, dt in {"bf16": torch.bfloat16, "f32": torch.float32}.items():
        for shape, blocks in (((256, 384), {-1: 128, -2: 128}), ((40, 72), {-1: 16, -2: 8}), ((37, 50), {-1: 16, -2: 8})):
            for kind in ("gauss", "heavy"):
                x = make_inputs(31, shape, kind, dt)
                key = f"fp8b/{dname}/{shape[0]}x{shape[1]}/{blocks[-2]}x{blocks[-1]}/{kind}"
                tq = TensorQuantizer(QuantizerAttributeConfig(num_bits=(4, 3), axis=None, block_sizes=dict(blocks)))
                tq.enable_calib()
                tq.disable_quant()
                tq(x)
                tq.load_calib_amax()
                tq.enable_quant()
                tq.disable_calib()
                out[key + "/x"] = x.float().numpy()
                out[key + "/amax"] = tq.amax.float().numpy()
                out[key + "/fq"] = tq(x).float().numpy()
                q, sc = FP8QTensor.quantize(x, block_sizes=dict(blocks))
                out[key + "/q"] = q._quantized_data.view(torch.uint8).numpy().copy()
                out[key + "/scale"] = sc.float().numpy()
                out[key + "/deq"] = q.dequantize(dtype=dt, scale=sc, block_sizes=dict(blocks)).float().numpy()
                # export-style: fp32 scales from the calibrated amax (to_quantized_weight, quant_utils.py:874-877)
                wsf = (tq.amax.float() / 448.0).squeeze()
                q2, _ = FP8QTensor.quantize(x, wsf, block_sizes=dict(blocks))
                out[key + "/q_export"] = q2._quantized_data.view(torch.uint8).numpy().copy()
    print("wrote", _golden.save("ref_fp8_blocks", out, OUT), len(out), "arrays")


def main_int8():
    """INT8QTensor.quantize / dequantize (qtensor/int8_tensor.py:36-124) on CPU: per-tensor, per-channel (axis 0),
    1-D and 2-D block scales, computed or given scales."""
    _install_shim()
    import torch
    from modelopt.torch.quantization.qtensor.int8_tensor import INT8QTensor

    out = {}
    for dname, dt in {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}.items():
        for shape in ((24, 256), (37, 128)):
            for kind in ("gauss", "heavy"):
                x = make_inputs(41, shape, kind, dt)
                base = f"int8/{dname}/{shape[0]}x{shape[1]}/{kind}"
                out[base + "/x"] = x.float().numpy()
                for mode, kw in (("tensor", {}), ("axis0", {"axis": 0}), ("block128", {"block_sizes": {-1: 128}}),
                                 ("block8x64", {"block_sizes": {-1: 64, -2: 8}})):
                    if mode == "block8x64" and shape[0] % 8:
                        continue
                    q, sc = INT8QTensor.quantize(x.clone(), **kw)
                    key = f"{base}/{mode}"
                    out[key + "/q"] = q._quantized_data.view(torch.int8).numpy().copy()
                    out[key + "/scale"] = sc.float().numpy()
                    dkw = {"block_sizes": kw["block_sizes"]} if "block_sizes" in kw else {}
                    out[key + "/deq"] = q.dequantize(dtype=dt, scale=sc, **dkw).float().numpy()
                # given fp32 scales (an exported amax / 127): promotes the quotient to float32
                sc32 = (x.float().abs().amax(dim=1, keepdim=True) / 127.0)
                q, _ = INT8QTensor.quantize(x.clone(), sc32)
                out[base + "/given_f32/q"] = q._quantized_data.view(torch.int8).numpy().copy()
                out[base + "/given_f32/scale"] = sc32.numpy()
    np.savez_compressed(os.path.join(OUT, "ref_int8.npz"), **out)
    print("wrote", os.path.join(OUT, "ref_int8.npz"), len(out), "arrays")


def main_block_setup():
    """Static block-quant reshape bookkeeping of the reference TensorQuantizer (_setup_for_blockquant,
    nn/modules/tensor_quantizer.py:975-1045) for a grid of shapes / block configs -> JSON."""
    _install_shim()
    import json

    import torch
    from modelopt.torch.quantization.config import QuantizerAttributeConfig
    from modelopt.torch.quantization.nn import TensorQuantizer

    cases = []
    for shape in ((256, 384), (40, 72), (37, 50), (3, 20, 48), (2, 3, 16, 30)):
        for blocks in ({-1: 16}, {-1: 128}, {-1: 16, -2: 8}, {-1: 128, -2: 128}, {-2: 8}, {-1: 7, -2: 5}):
            if any(-k > len(shape) for k in blocks):
                continue
            tq = TensorQuantizer(QuantizerAttributeConfig(num_bits=8, axis=None, block_sizes=dict(blocks)))
            x = torch.zeros(shape)
            tq._setup_for_blockquant(x)
            y = tq._process_for_blockquant(x)
            cases.append({
                "shape": list(shape), "blocks": {str(k): v for k, v in blocks.items()},
                "axis": list(tq._axis), "reshape": list(tq._block_reshape_size), "processed": list(y.shape),
                "padding": list(getattr(tq, "_padding", ())), "original": list(tq._original_shape),
                "slices": [[sl.start, sl.stop] if isinstance(sl, slice) else None for sl in getattr(tq, "_slices", ())],
            })
    with open(os.path.join(OUT, "ref_block_setup.json"), "w") as f:
        json.dump(cases, f, indent=0)
    print("wrote ref_block_setup.json", len(cases))


def main_enabled_quantizers():
    """Which weight / input quantizers end up enabled on a tiny HF Llama per preset (conversion.py set_quantizer_by_cfg)."""
    _install_shim()
    import json

    import modelopt.torch.quantization as mtq
    from modelopt.torch.quantization.conversion import replace_quant_module, set_quantizer_by_cfg
    from modelopt.torch.quantization.nn import TensorQuantizer
    from transformers import LlamaConfig, LlamaForCausalLM

    cfg = LlamaConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, vocab_size=128, max_position_embeddings=64)
    out = {}
    for preset in ("NVFP4_DEFAULT_CFG", "NVFP4_MLP_ONLY_CFG", "NVFP4_OMLP_ONLY_CFG", "MXFP4_MLP_WEIGHT_ONLY_CFG",
                   "INT4_AWQ_CFG", "FP8_2D_BLOCKWISE_WEIGHT_ONLY_CFG", "W4A16_NVFP4_CFG", "INT8_DEFAULT_CFG"):
        m = LlamaForCausalLM(cfg)
        replace_quant_module(m)
        set_quantizer_by_cfg(m, getattr(mtq, preset)["quant_cfg"])
        out[preset] = sorted(n for n, q in m.named_modules() if isinstance(q, TensorQuantizer) and q.is_enabled
                             and (n.endswith("weight_quantizer") or n.endswith("input_quantizer")))
    with open(os.path.join(OUT, "ref_enabled_quantizers.json"), "w") as f:
        json.dump(out, f, indent=0)
    print("wrote ref_enabled_quantizers.json")


def main_calibrators():
    """Third calibrator fixture (VERDICT r01 item 2): the reference's host-side amax searches on CPU --
    ``HistogramCalibrator.compute_amax`` entropy / mse / percentile (calib/histogram.py:137-343),
    ``NVFP4ActHeadroomCalibrator`` histogram + ``compute_amax`` (calib/nvfp4_act_headroom.py:116-205) and the
    per-channel ``MseCalibrator`` (calib/mse.py:31-172) -> tests/golden/ref_calibrators.npz.

    ``_compute_amax_mse`` as shipped calls ``fake_tensor_quant(centers, amax, num_bits, unsigned)`` and
    ``scaled_e4m3(centers, amax, E, M)`` (histogram.py:307-310) against signatures whose third positional argument
    is ``bias`` (tensor_quant.py:343-355, 407-417): as executed it subtracts ``num_bits`` as a bias and quantizes with
    ``num_bits=int(unsigned)`` (a shift by -1 in the CUDA kernel), and raises TypeError for (4, 3).  The fixture
    runs the reference function with that call site repaired (``bias=None`` inserted) -- the documented intent,
    and what the reference's own tests assert (tests/unit/torch/quantization/test_calibrator.py:240-290)."""
    _install_shim()
    import torch

    import modelopt.torch.quantization  # noqa: F401
    from modelopt.torch.quantization import tensor_quant as tq
    from modelopt.torch.quantization.calib import HistogramCalibrator
    from modelopt.torch.quantization.calib import histogram as H
    from modelopt.torch.quantization.calib.mse import MseCalibrator
    from modelopt.torch.quantization.calib.nvfp4_act_headroom import NVFP4ActHeadroomCalibrator
    from modelopt.torch.quantization.utils import reduce_amax

    H.fake_tensor_quant = lambda c, a, nb, u: tq.fake_tensor_quant(c, a, None, nb, u)      # repaired call sites
    H.scaled_e4m3 = lambda c, a, e, m: tq.scaled_e4m3(c, a, None, e, m)
    out = {}
    # ---- histogram searches ---------------------------------------------------------------------------------
    cases = [("g2048_i8", 2048, 8, False, "heavy", 128), ("g512_i8", 512, 8, False, "gauss", 32),
             ("g512_u8", 512, 8, True, "gauss", 32), ("g512_i4", 512, 4, False, "heavy", 32),
             ("g2048_fp8", 2048, (4, 3), False, "heavy", 128)]
    for name, nbins, bits, unsigned, kind, start in cases:
        cal = HistogramCalibrator(bits, None, unsigned, num_bins=nbins)
        xs = [make_inputs(21 + i, (64, 512), kind, torch.bfloat16).float() * (1.0 + 0.6 * i) for i in range(2)]
        if unsigned:
            xs = [x.abs() for x in xs]
        for x in xs:
            cal.collect(x)                                   # second batch grows the range (:121-130)
        hist = cal._calib_hist.int().numpy().copy()
        edges = cal._calib_bin_edges.numpy().copy()
        out[f"hist/{name}/hist"] = hist
        out[f"hist/{name}/edges"] = edges
        out[f"hist/{name}/cfg"] = np.array([nbins, bits if isinstance(bits, int) else 0, int(unsigned), start])
        for pct in (99.99, 99.9, 90.0, 50.0):
            out[f"hist/{name}/percentile_{pct}"] = np.float32(float(cal.compute_amax("percentile", percentile=pct)))
        out[f"hist/{name}/mse"] = np.float32(float(cal.compute_amax("mse", start_bin=start)))
        out[f"hist/{name}/mse_stride4"] = np.float32(float(cal.compute_amax("mse", start_bin=start, stride=4)))
        if isinstance(bits, int):
            out[f"hist/{name}/entropy"] = np.float32(float(cal.compute_amax("entropy", start_bin=start)))
            out[f"hist/{name}/entropy_stride3"] = np.float32(
                float(cal.compute_amax("entropy", start_bin=start, stride=3)))
        print("hist", name, {k.split("/")[-1]: float(v) for k, v in out.items() if k.startswith(f"hist/{name}/") and v.ndim == 0})
    # ---- NVFP4 activation headroom ---------------------------------------------------------------------------
    xs = [make_inputs(31 + i, (96, 1024), "heavy" if i == 1 else "gauss", torch.bfloat16) * (0.3 + 0.9 * i)
          for i in range(3)]
    xs[1][0, :16] = 0
    xs[2][5:9] = xs[2][5:9] * 1e-4
    out["headroom/x"] = torch.stack(xs).float().numpy()
    for name, kw in (("default", {}), ("upper100", {"upper_percentile": 100.0}),
                     ("rho64_a5", {"rho": 64.0, "anchor_percentile": 5.0, "upper_percentile": 99.0})):
        cal = NVFP4ActHeadroomCalibrator(**kw)
        for x in xs:
            cal.collect(x)
        out[f"headroom/{name}/hist"] = cal._hist.numpy().copy()
        out[f"headroom/{name}/running_max"] = np.float32(float(cal._running_max))
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out[f"headroom/{name}/amax"] = np.float32(float(cal.compute_amax()))
        print("headroom", name, out[f"headroom/{name}/amax"], out[f"headroom/{name}/running_max"])
    # ---- per-channel MseCalibrator (the CPU twin of the quantizer's quant_func) --------------------------------
    for name, shape, bits, narrow, fp8 in (("int8_rows", (48, 256), 8, False, False), ("int4_blocks", (96, 128), 4, False, False),
                                           ("fp8_rows", (24, 512), 0, False, True)):
        x = make_inputs(41, shape, "heavy", torch.bfloat16)
        amax = reduce_amax(x, axis=1)                           # [R, 1] in bf16, like the quantizer's _amax buffer
        qf = (lambda t, a: tq.fp8_eager(t, a)) if fp8 else (lambda t, a, b=bits, n=narrow: tq._tensor_quant(t, a, b, False, n))
        cal = MseCalibrator(amax=amax, axis=0, quant_func=qf)
        cal.collect(x)
        out[f"mse_rows/{name}/x"] = x.float().numpy()
        out[f"mse_rows/{name}/amax0"] = amax.float().numpy()
        out[f"mse_rows/{name}/mult"] = cal._candidates.numpy().copy()
        out[f"mse_rows/{name}/losses"] = torch.stack(cal._losses_sum).float().numpy()
        best = cal.compute_amax()
        out[f"mse_rows/{name}/best"] = best.float().numpy()
        out[f"mse_rows/{name}/best_dtype"] = np.array(str(best.dtype))
        print("mse_rows", name, best.dtype, best.flatten()[:4].tolist())
    np.savez_compressed(os.path.join(OUT, "ref_calibrators.npz"), **out)
    print("wrote ref_calibrators.npz", len(out), "arrays")


def main_export():
    """Unified-HF export fixture (SURVEY.md 8(f1)): the reference's ``export_hf_checkpoint``
    (export/unified_export_hf.py:133, 569-700, 940-1100; quant_utils.py:1054-1570) on a tiny HF Llama after
    ``mtq.quantize`` on CPU, for FP8 / NVFP4 / NVFP4 static (MSE FP8 sweep) / INT4-AWQ.  Stored per preset:
      in/...   the calibrated state the export starts from (weights after AWQ smoothing, every quantizer's
               ``_amax`` / ``_global_amax`` / ``_pre_quant_scale``), so that a test can load it instead of
               re-calibrating on different hardware;
      out/...  every tensor of the exported ``model.safetensors`` as raw bytes + dtype + shape;
      cfg      ``hf_quant_config.json``.
    -> tests/golden/ref_export.*.npz"""
    _install_shim()
    import copy
    import json
    import tempfile

    import torch
    from safetensors.torch import load_file
    from transformers import LlamaConfig, LlamaForCausalLM

    import modelopt.torch.quantization as mtq
    from modelopt.torch.export import export_hf_checkpoint

    cfg = LlamaConfig(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, vocab_size=128, max_position_embeddings=128, tie_word_embeddings=False,
                      architectures=["LlamaForCausalLM"], dtype=torch.bfloat16)
    torch.manual_seed(0)
    base = LlamaForCausalLM(cfg).to(torch.bfloat16).eval()
    g = torch.Generator().manual_seed(1)
    data = [torch.randint(0, 128, (2, 48), generator=g) for _ in range(4)]

    def loop(m):
        for d in data:
            m(d)

    def raw(t):
        t = t.detach().contiguous().reshape(-1)
        return t.view(torch.uint8).numpy().copy() if t.numel() else np.zeros(0, np.uint8)

    out = {}
    presets = [("FP8_DEFAULT_CFG", None), ("NVFP4_DEFAULT_CFG", None), ("INT4_AWQ_CFG", None),
               ("NVFP4_W4A4_WEIGHT_MSE_FP8_SWEEP_CFG", "max")]
    for preset, algo in presets:
        m = copy.deepcopy(base)
        qcfg = copy.deepcopy(getattr(mtq, preset))
        if algo is not None:
            qcfg["algorithm"] = algo          # the sweep itself needs a GPU; the static export path does not
        mtq.quantize(m, qcfg, loop)
        key = preset if algo is None else f"{preset}@{algo}"
        for name, p in m.named_parameters():
            out[f"{key}/in/param/{name}"] = raw(p)
        for name, mod in m.named_modules():
            if type(mod).__name__ in ("TensorQuantizer", "StaticBlockScaleQuantizer"):
                for b in ("_amax", "_global_amax", "_pre_quant_scale"):
                    t = getattr(mod, b, None)
                    if isinstance(t, torch.Tensor):
                        out[f"{key}/in/q/{name}.{b}"] = t.detach().float().numpy().copy()
                        out[f"{key}/in/qdtype/{name}.{b}"] = np.array(str(t.dtype))
        with tempfile.TemporaryDirectory() as d:
            export_hf_checkpoint(m, export_dir=d)
            sd = load_file(os.path.join(d, "model.safetensors"))
            for k, v in sd.items():
                out[f"{key}/out/{k}"] = raw(v)
                out[f"{key}/meta/{k}"] = np.array(json.dumps([str(v.dtype), list(v.shape)]))
            out[f"{key}/cfg"] = np.array(json.dumps(json.load(open(os.path.join(d, "hf_quant_config.json")))))
        print("export", key, len(sd), "tensors", json.loads(str(out[f"{key}/cfg"]))["quantization"])
    print("wrote", _golden.save("ref_export", out, OUT), len(out), "arrays")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "algos":
        main_algos()
    elif len(sys.argv) > 1 and sys.argv[1] == "presets":
        main_presets()
    elif len(sys.argv) > 1 and sys.argv[1] == "mx":
        main_mx()
    elif len(sys.argv) > 1 and sys.argv[1] == "bias":
        main_bias()
    elif len(sys.argv) > 1 and sys.argv[1] == "nvfp4_blocks":
        main_nvfp4_blocks()
    elif len(sys.argv) > 1 and sys.argv[1] == "fp8_blocks":
        main_fp8_blocks()
    elif len(sys.argv) > 1 and sys.argv[1] == "block_setup":
        main_block_setup()
    elif len(sys.argv) > 1 and sys.argv[1] == "int8":
        main_int8()
    elif len(sys.argv) > 1 and sys.argv[1] == "enabled":
        main_enabled_quantizers()
        main_calibrators()
    elif len(sys.argv) > 1 and sys.argv[1] == "calibrators":
        main_calibrators()
    elif len(sys.argv) > 1 and sys.argv[1] == "export":
        main_export()
    else:
        main()
        main_algos()
        main_presets()
        main_mx()
        main_bias()
        main_nvfp4_blocks()
        main_fp8_blocks()
        main_block_setup()
        main_enabled_quantizers()
        main_calibrators()

