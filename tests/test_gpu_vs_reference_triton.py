"""Side by side on the GPU: the REFERENCE's Triton kernels -- AOT-compiled for sm_100 by
oracle/build_ref_triton.py from the @triton.jit functions under /root/reference into oracle/_ref/*.cubin
(which travel with the snapshot) -- launched through the CUDA driver API next to this engine's kernels.

  fp4_fake_quant_kernel                    NVFP4 dynamic fake quant, the default GPU path (fp4_kernel_hopper.py:33)
  static_blockwise_fp4_fake_quant_kernel   NVFP4 static fake quant (fp4_kernel.py:194)
  _fp8_scale_sweep_kernel                  126-candidate FP8 scale sweep (nvfp4_fp8_sweep.py:58)

Triton divides with `div.full.f32` (2-ulp approximate); this engine restates the formulas with IEEE division.
They can therefore differ exactly where a quotient sits within an ulp or two of a rounding boundary -- for
16-bit data that includes the many EXACT real-arithmetic ties (see test_gpu_vs_reference_ext.py), for fp32
data it is a handful of elements.  The tests bound and report those rates; everything else must be equal.
Where the cubins are absent the reference side is what they produced on the same inputs, stored in
tests/golden/ref_gpu_triton/ (see tests/_refgold.py), and the mismatches in the stored rows count against the bound
for the whole tensor; only the speed comparison needs the cubins and is skipped then."""

import ctypes
import json
import os

import numpy as np
import pytest
import torch
from _refgold import RefResults, Store

from oracle import oracle_np as o

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
DN = {torch.bfloat16: "bf16", torch.float16: "f16", torch.float32: "f32"}
REPORT = {}
LIVE = os.path.exists(os.path.join(REF, "triton_kernels.json")) and os.path.exists(
    os.path.join(REF, "modelopt_cuda_ext_fp8.so"))


class RefTritonKernel:
    def __init__(self, key):
        idx = os.path.join(REF, "triton_kernels.json")
        if not os.path.exists(idx):
            pytest.skip("oracle/_ref/triton_kernels.json not built (python oracle/build_ref_triton.py)")
        from cuda.bindings import driver as cu

        self.cu = cu
        self.meta = json.load(open(idx))["kernels"][key]
        torch.zeros(1, device="cuda")                       # make torch's primary context current
        with open(os.path.join(REF, self.meta["file"]), "rb") as f:
            self.image = f.read()
        err, self.mod = cu.cuModuleLoadData(self.image)
        assert err == cu.CUresult.CUDA_SUCCESS, err
        err, self.fn = cu.cuModuleGetFunction(self.mod, self.meta["name"].encode())
        assert err == cu.CUresult.CUDA_SUCCESS, err

    def __call__(self, grid, *args):
        vals, types = [], []
        for a, t in zip(args, self.meta["arg_types"]):
            vals.append(int(a))
            types.append(ctypes.c_void_p if t.startswith("*") else ctypes.c_int32)
        for _ in range(self.meta["n_params"] - len(args)):  # Triton's global / profile scratch pointers (unused)
            vals.append(0)
            types.append(ctypes.c_void_p)
        gx, gy, gz = (list(grid) + [1, 1])[:3]
        stream = self.cu.CUstream(torch.cuda.current_stream().cuda_stream)
        (err,) = self.cu.cuLaunchKernel(self.fn, gx, gy, gz, 32 * self.meta["num_warps"], 1, 1, self.meta["shared"],
                                        stream, (tuple(vals), tuple(types)), 0)
        assert err == self.cu.CUresult.CUDA_SUCCESS, err


@pytest.fixture(scope="module")
def store():
    s = Store("ref_gpu_triton", LIVE)
    yield s
    s.save()


@pytest.fixture
def refs(store, request):
    return RefResults(store, request.node.name)


@pytest.fixture(scope="module")
def ops():
    from model_optimizer_b200 import ops as _ops

    return _ops


def inputs(shape, dtype, seed, kind="gauss"):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, device="cuda", generator=g)
    if kind == "heavy":
        x = x * (1 + 20 * (torch.rand(shape, device="cuda", generator=g) < 1e-3).float())
    elif kind == "scaled":
        x = x * torch.exp2(torch.randint(-12, 8, (shape[0], 1), device="cuda", generator=g).float())
    return x.to(dtype)


def ref_global_scale(global_amax):
    return global_amax.float() / (6.0 * 448.0)        # :140, evaluated by torch on the GPU like the reference


def ref_fp4_fake_quant_block(x, global_amax):
    """fp4_fake_quant_block (fp4_kernel_hopper.py:102-170) with the compiled reference kernel."""
    k = RefTritonKernel(f"fp4_fake_quant_{DN[x.dtype]}")
    x2 = x.reshape(-1, x.shape[-1]).contiguous()
    y = torch.empty_like(x2)
    m, n = x2.shape
    gs = ref_global_scale(global_amax).to(x.device)
    k(((m + 15) // 16, (n + 63) // 64), x2.data_ptr(), y.data_ptr(), m, n, gs.data_ptr(), x2.stride(0), x2.stride(1),
      y.stride(0), y.stride(1))
    return y.view(x.shape)


def mismatch_stats(ref, got):
    ref, got = ref.to(torch.bfloat16).float(), got.to(torch.bfloat16).float()   # compare at bf16 resolution
    zero = (ref == 0) & (got == 0)
    diff = (ref != got) & ~zero
    r, g_ = ref[diff].abs(), got[diff].abs()
    hi, lo = torch.maximum(r, g_), torch.minimum(r, g_)
    bounded = bool(((lo == 0) | (hi / lo <= 2.05)).all())
    return int(diff.sum()), bounded


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_nvfp4_dynamic_vs_reference_triton(ops, refs, dtype):
    rep = {}
    for kind, shape in (("gauss", (1024, 4096)), ("heavy", (1024, 4096)), ("scaled", (512, 4096)), ("ragged", (300, 200))):
        x = inputs(shape, dtype, 11, "gauss" if kind == "ragged" else kind)
        g = x.abs().max().float().reshape(1)
        got = ops.fake_quant_nvfp4(x, g)
        ref, got = refs.rows(got, lambda: ref_fp4_fake_quant_block(x, g))
        gs = ref_global_scale(g)
        gs_ieee = g / torch.tensor(6.0 * 448.0, device="cuda")
        n, bounded = mismatch_stats(ref, got)
        rep[kind] = {"elements": x.numel(), "compared": ref.numel(), "mismatches": n, "rate": n / ref.numel(),
                     "global_scale_same_as_ieee": bool(torch.equal(gs, gs_ieee))}
        assert bounded, (dtype, kind)
        if torch.equal(gs, gs_ieee):
            assert n <= (1e-4 if dtype == torch.float32 else 0.02) * x.numel(), (dtype, kind, n)
        else:                       # torch's GPU `tensor / python_scalar` is a reciprocal multiply: one ulp in the scale
            assert n <= 0.05 * x.numel(), (dtype, kind, n)
    REPORT[f"nvfp4_dynamic_{DN[dtype]}"] = rep


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_nvfp4_static_vs_reference_triton(ops, refs, dtype):
    """static_blockwise_fp4_fake_quant (fp4_kernel.py:253-316): scales from compute_fp4_scales evaluated the way
    the reference does on the GPU (torch ops + its own FP8 extension), then its Triton kernel."""
    import importlib.machinery
    import importlib.util

    def reference(x, amax, g):
        p = os.path.join(REF, "modelopt_cuda_ext_fp8.so")
        if not os.path.exists(p):
            pytest.skip("reference fp8 extension not built")
        loader = importlib.machinery.ExtensionFileLoader("modelopt_cuda_ext_fp8", p)
        ext8 = importlib.util.module_from_spec(importlib.util.spec_from_loader("modelopt_cuda_ext_fp8", loader))
        loader.exec_module(ext8)
        k = RefTritonKernel(f"fp4_static_{DN[dtype]}")
        scale = amax / 6.0                                                     # :232
        scale = ext8.fake_e4m3fy(scale, (g * (448.0 / 448.0) / 6.0).reshape(1))   # :243-244 -> scaled_e4m3_impl
        xf = x.contiguous().view(-1)
        y = torch.empty_like(xf)
        k((amax.numel(),), xf.data_ptr(), y.data_ptr(), scale.contiguous().data_ptr(), amax.numel())
        return y.view(x.shape)

    rep = {}
    for kind in ("gauss", "heavy", "scaled"):
        x = inputs((1024, 2048), dtype, 12, kind)
        amax = x.view(-1, 16).abs().amax(dim=-1).float()
        g = amax.max()
        got = ops.fake_quant_nvfp4_static(x, amax, g.reshape(1), True, 448.0)
        ref, got = refs.rows(got, lambda: reference(x, amax, g))
        n, bounded = mismatch_stats(ref, got)
        rep[kind] = {"elements": x.numel(), "compared": ref.numel(), "mismatches": n, "rate": n / ref.numel()}
        assert bounded, (dtype, kind)
        assert n <= (1e-3 if dtype == torch.float32 else 0.02) * x.numel(), (dtype, kind, n)
    REPORT[f"nvfp4_static_{DN[dtype]}"] = rep


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fp8_scale_sweep_vs_reference_triton(ops, refs, dtype):
    """nvfp4_fp8_scale_sweep (nvfp4_fp8_sweep.py:127-160).  The winner is an argmin over 126 fp32 losses; the two
    implementations sum 16 squared errors in a different order and divide differently, so near-equal losses can
    swap: report the agreement rate."""
    w = inputs((1024, 1024), dtype, 13, "gauss")
    g = w.abs().max().float().reshape(1)
    n_blocks = w.numel() // 16

    def reference():
        k = RefTritonKernel(f"fp8_sweep_{DN[dtype]}")
        cand = torch.from_numpy(o.fp8_scale_candidates().astype(np.float32)).cuda()
        best = torch.empty(n_blocks, dtype=torch.float32, device="cuda")
        k(((n_blocks + 63) // 64,), w.contiguous().data_ptr(), cand.data_ptr(), g.data_ptr(), best.data_ptr(), n_blocks)
        return best

    got = ops.nvfp4_fp8_scale_sweep(w, g, candidates="ieee").reshape(-1)      # the cubin is fed the same IEEE candidates
    best, _ = refs.rows(got, reference)                                         # all blocks: small enough to store whole
    best = best.reshape(-1)
    same = float((best == got).float().mean())
    REPORT[f"fp8_sweep_{DN[dtype]}"] = {"blocks": n_blocks, "same_winner": same}
    assert same >= 0.97, same
    # the winners that differ must be near-equal in quality: compare the block MSE they produce
    bad = best != got
    if bad.any():
        wb = w.float().view(-1, 16)[bad]

        def mse(amax):
            s = (amax / 6.0).unsqueeze(1)
            a = wb.abs() / s
            q = torch.where(a <= 0.25, 0.0, torch.where(a < 0.75, 0.5, torch.where(a <= 1.25, 1.0, torch.where(
                a < 1.75, 1.5, torch.where(a <= 2.5, 2.0, torch.where(a < 3.5, 3.0, torch.where(a <= 5.0, 4.0, 6.0)))))))
            return ((wb.abs() - q * s) ** 2).sum(1)

        rel = (mse(best[bad]) - mse(got[bad])).abs() / mse(got[bad]).clamp_min(1e-30)
        assert float(rel.max()) < 1e-3, float(rel.max())


def test_speed_nvfp4_triton_side_by_side(ops):
    """4096 x 4096 bf16, 16 distinct inputs, both as CUDA-graph replays."""
    from _gpu_timing import _time_graph

    k = RefTritonKernel("fp4_fake_quant_bf16")
    gen = torch.Generator(device="cuda").manual_seed(0)
    xs = [torch.randn(4096, 4096, device="cuda", generator=gen).to(torch.bfloat16) for _ in range(16)]
    ys = [torch.empty_like(xs[0]) for _ in range(4)]
    g = xs[0].abs().max().float().reshape(1)
    gs = g / (6.0 * 448.0)

    def ref(i):
        y = ys[i % 4]
        k((256, 64), xs[i].data_ptr(), y.data_ptr(), 4096, 4096, gs.data_ptr(), 4096, 1, 4096, 1)

    t_ref = _time_graph(ref, 16)
    t_our = _time_graph(lambda i: ops.fake_quant_nvfp4(xs[i], g, out=ys[i % 4]), 16)
    REPORT["speed_nvfp4_4096x4096_bf16"] = {"reference_triton_us": round(t_ref, 2), "b200_us": round(t_our, 2),
                                            "speedup": round(t_ref / t_our, 2)}
    assert t_our < t_ref


def test_zz_write_report():
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "vs_reference_triton.json"), "w") as f:
        json.dump(REPORT, f, indent=1)
