"""Side by side on the GPU: the REFERENCE's own CUDA extensions (built for sm_100a by oracle/build_ref_ext.py
from the sources under /root/reference into oracle/_ref/*.so, which travel with the snapshot) against this
engine's kernels, on the same seeded inputs.  This is what pins the paths the CPU cannot execute:

  modelopt_cuda_ext      fake_tensor_quant / _with_axis / _ (in place), INT4_quantize, INT4_dequantize
  modelopt_cuda_ext_fp8  fake_e4m3fy / _with_axis
  modelopt_cuda_ext_mx   fused_amax_convert (built with --use_fast_math, like the reference builds it)

Where those builds are absent the reference side is what they produced on the same inputs, stored in
tests/golden/ref_gpu_ext/ (see tests/_refgold.py); only the speed comparison needs them and is skipped then.
Bar: bit-exact, except where noted in the test."""

import importlib.machinery
import importlib.util
import json
import os

import numpy as np
import pytest
import torch
from _refgold import RefResults, Store

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
DT = [torch.bfloat16, torch.float16, torch.float32]
REPORT = {}
EXTS = ("modelopt_cuda_ext", "modelopt_cuda_ext_fp8", "modelopt_cuda_ext_mx")
LIVE = all(os.path.exists(os.path.join(REF, n + ".so")) for n in EXTS)
_LOADED = {}


def load_ext(name):
    path = os.path.join(REF, name + ".so")
    if not os.path.exists(path):
        pytest.skip(f"{path} not built (python oracle/build_ref_ext.py where /root/reference exists)")
    loader = importlib.machinery.ExtensionFileLoader(name, path)
    mod = importlib.util.module_from_spec(importlib.util.spec_from_loader(name, loader))
    loader.exec_module(mod)
    return mod


def E(name):
    """The reference extension ``name`` (live runs only)."""
    if name not in _LOADED:
        _LOADED[name] = load_ext(name)
    return _LOADED[name]


@pytest.fixture(scope="module")
def ops():
    from model_optimizer_b200 import ops as _ops

    return _ops


@pytest.fixture(scope="module")
def store():
    s = Store("ref_gpu_ext", LIVE)
    yield s
    s.save()


@pytest.fixture
def refs(store, request):
    return RefResults(store, request.node.name)


@pytest.fixture(scope="module")
def ext():
    return load_ext("modelopt_cuda_ext")


@pytest.fixture(scope="module")
def ext_fp8():
    return load_ext("modelopt_cuda_ext_fp8")


@pytest.fixture(scope="module")
def ext_mx():
    return load_ext("modelopt_cuda_ext_mx")


def inputs(shape, dtype, seed, kind="gauss"):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, device="cuda", generator=g)
    if kind == "heavy":
        x = x * (1 + 20 * (torch.rand(shape, device="cuda", generator=g) < 1e-3).float())
    elif kind == "scaled":
        x = x * torch.exp2(torch.randint(-18, 12, (shape[0], 1), device="cuda", generator=g).float())
    elif kind == "ties":   # values that sit exactly on rounding boundaries after scaling by a power of two
        v = torch.tensor([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0, 6.0, 0.5, 1.5, 2.0, 3.0, 4.0, 7.0, 0.125, 448.0],
                         device="cuda")
        x = v[torch.randint(0, 16, shape, device="cuda", generator=g)] \
            * (torch.randint(0, 2, shape, device="cuda", generator=g) * 2 - 1) \
            * torch.exp2(torch.randint(-3, 3, (shape[0], 1), device="cuda", generator=g).float())
    return x.to(dtype)


def nbad(a, b):
    a, b = a.float(), b.float()
    ok = (a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))
    return int((~ok).sum())


def exact(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, what
    n = nbad(a, b)
    assert n == 0, f"{what}: {n}/{a.numel()} elements differ from the reference CUDA extension"


@pytest.mark.parametrize("dtype", DT)
def test_int_fake_quant_vs_reference_ext(ops, refs, dtype):
    for kind in ("gauss", "heavy", "ties"):
        x = inputs((257, 384), dtype, 1, kind)
        amax = x.abs().max().float().reshape(1)
        for bits in (3, 4, 5, 7, 8, 11):
            for unsigned in (False, True):
                for narrow in (True, False):
                    xin = x.abs() if unsigned else x
                    got = ops.fake_quant_int(xin, amax, bits, unsigned, narrow)
                    ref = refs.bits(got, lambda: E("modelopt_cuda_ext").fake_tensor_quant(xin, amax, bits, unsigned, narrow))
                    exact(got, ref, f"int{bits} u{unsigned} n{narrow} {kind}")
        # clipping amax, tiny amax (-> zeros), amax in the input dtype, in-place entry point
        for a in (amax * 0.37, amax * 0 + 2.0 ** -25, amax * 0 + 2.0 ** -24, amax.to(dtype)):
            got = ops.fake_quant_int(x, a, 8, False, False)
            exact(got, refs.bits(got, lambda: E("modelopt_cuda_ext").fake_tensor_quant(x, a, 8, False, False)), f"amax {a}")

        def in_place():
            y = x.clone()
            E("modelopt_cuda_ext").fake_tensor_quant_(y, amax, 8, False, True)
            return y

        got = ops.fake_quant_int(x, amax, 8, False, True)
        exact(got, refs.bits(got, in_place), "in place")
        # per-axis
        for axis in (0, 1):
            am = x.abs().amax(dim=1 - axis).float()
            got = ops.fake_quant_int(x, am, 8, False, False, outer=x.stride(axis))
            ref = refs.bits(got, lambda: E("modelopt_cuda_ext").fake_tensor_quant_with_axis(x, am, axis, 8, False, False))
            exact(got, ref, f"axis {axis} {kind}")
        # INT4 block-128 == axis 0 of the [n/128, 128] view (tensor_quantizer.py:1008-1016)
        xb = x.reshape(-1, 128)
        am = xb.abs().amax(dim=1).float()
        got = ops.fake_quant_int(xb, am, 4, False, False, outer=128)
        exact(got, refs.bits(got, lambda: E("modelopt_cuda_ext").fake_tensor_quant_with_axis(xb, am, 0, 4, False, False)),
              f"int4 block128 {kind}")


@pytest.mark.parametrize("dtype", DT)
def test_fp8_fake_quant_vs_reference_ext(ops, refs, dtype):
    for kind in ("gauss", "heavy", "ties", "scaled"):
        x = inputs((257, 384), dtype, 2, kind)
        amax = x.abs().max().float().reshape(1)
        for a in (amax, amax * 0.5, amax * 0 + 2.0 ** -25, amax.to(dtype)):
            got = ops.fake_quant_fp8(x, a)
            exact(got, refs.bits(got, lambda: E("modelopt_cuda_ext_fp8").fake_e4m3fy(x, a)), f"fp8 {kind} amax {float(a)}")
        for axis in (0, 1):
            am = x.abs().amax(dim=1 - axis).float()
            got = ops.fake_quant_fp8(x, am, outer=x.stride(axis))
            exact(got, refs.bits(got, lambda: E("modelopt_cuda_ext_fp8").fake_e4m3fy_with_axis(x, am, axis)), f"fp8 axis {axis}")


@pytest.mark.parametrize("dtype", DT)
def test_int4_compress_pack_vs_reference_ext(ops, refs, dtype):
    """INT4QTensor.quantize's CUDA branch (qtensor/int4_tensor.py:52-68): scales = 7 / block amax in the
    input dtype, bytes from INT4_quantize_kernel (arithmetic in the tensor dtype, roundf)."""
    for kind in ("gauss", "heavy", "ties"):
        for bs in (128, 32):
            x = inputs((96, 256), dtype, 3, kind).reshape(-1)
            scales = 7 / x.view(-1, bs).abs().amax(dim=-1, keepdim=True)       # what the reference computes in torch
            got, got_scales = ops.pack_int4_blockwise(x, bs)
            ref = refs.bits(got.reshape(-1), lambda: E("modelopt_cuda_ext").INT4_quantize(x, scales, bs).reshape(-1))
            exact(got_scales.reshape(scales.shape), scales, f"scales {kind} {bs}")
            assert torch.equal(got.reshape(-1), ref), f"packed bytes {kind} bs{bs} {dtype}"
            deq = ops.unpack_int4_blockwise(got, got_scales, bs).reshape(-1)
            exact(deq, refs.bits(deq, lambda: E("modelopt_cuda_ext").INT4_dequantize(ref, scales, bs).reshape(-1)),
                  f"dequant {kind} {bs}")


@pytest.mark.parametrize("dtype", DT)
def test_nf4_pack_vs_reference_ext(ops, refs, dtype):
    """NF4QTensor.quantize's CUDA branch: scales = block |x| max, bytes from NF4_quantize_kernel; and
    NF4_dequantize (always bfloat16).  Also arbitrary caller-given scales (|v| far outside the table)."""
    from oracle import oracle_np as o

    for kind in ("gauss", "heavy", "ties", "scaled"):
        for bs in (64, 32, 16):
            x = inputs((96, 256), dtype, 6, kind).reshape(-1)
            if kind == "ties":
                x[:512] = 0          # zero blocks: 0 / 0 -> NaN -> code 0
            scales = x.view(-1, bs).abs().amax(dim=-1, keepdim=True)
            got, got_scales = ops.pack_nf4(x, bs)
            ref = refs.bits(got, lambda: E("modelopt_cuda_ext").NF4_quantize(x, scales, bs).reshape(-1))
            exact(got_scales.reshape(scales.shape), scales, f"scales {kind} {bs}")
            assert torch.equal(got, ref), f"packed bytes {kind} bs{bs} {dtype}"
            want, _ = o.pack_nf4(x.float().cpu().numpy(), bs, {torch.bfloat16: "bf16", torch.float16: "f16", torch.float32: "f32"}[dtype])
            assert np.array_equal(got.cpu().numpy(), want), f"oracle {kind} bs{bs} {dtype}"
            deq = ops.unpack_nf4(got, got_scales, bs)
            deq_ref = refs.bits(deq, lambda: E("modelopt_cuda_ext").NF4_dequantize(ref, scales, bs).reshape(-1))
            assert deq.dtype == torch.bfloat16 and deq_ref.dtype == torch.bfloat16
            exact(deq, deq_ref, f"dequant {kind} {bs}")
            assert np.array_equal(deq.float().cpu().numpy(), o.unpack_nf4(want, scales.float().cpu().numpy(), bs)), "oracle deq"
        # given scales, some tiny / huge so that |x / scale| leaves the table range, plus inf / NaN inputs
        x = inputs((64, 256), dtype, 7, "gauss").reshape(-1)
        x[5], x[77], x[300] = float("inf"), float("-inf"), float("nan")
        g = torch.Generator(device="cuda").manual_seed(8)
        sc = (x.view(-1, 32).abs().amax(dim=-1, keepdim=True) * torch.exp2(torch.randint(-12, 3, (x.numel() // 32, 1), device="cuda", generator=g).float())).to(dtype)
        sc = torch.nan_to_num(sc, nan=1.0, posinf=1.0)
        got = ops.pack_nf4(x, 32, sc)[0]
        assert torch.equal(got, refs.bits(got, lambda: E("modelopt_cuda_ext").NF4_quantize(x, sc, 32).reshape(-1))), \
            f"given scales {dtype}"


FMT = ["E4M3", "E5M2", "INT8", "E0M3", "E1M2", "E3M0", "E2M1", "E3M2", "E2M3"]


@pytest.mark.parametrize("dtype", DT)
def test_mx_fake_quant_vs_reference_ext(ops, refs, dtype):
    """fused_amax_convert with an E8M0 scale.  The reference's `sign` is uninitialised for zero inputs
    (tensor_quant_mx.cu:39-43): zeros are compared by value.  The extension is built with --use_fast_math, so
    denormal scales / values may be flushed there: the 'scaled' case stays inside the normal range."""
    tot = bad = 0
    for name in FMT:
        for bs in (32, 16, 8):
            for kind in ("gauss", "heavy", "scaled", "ties"):
                x = inputs((129, 256), dtype, 4, kind)
                got = ops.fake_quant_mx(x, bs, name)
                ref = refs.bits(got, lambda: E("modelopt_cuda_ext_mx").fused_amax_convert(
                    x, bs, getattr(E("modelopt_cuda_ext_mx").Types, name), E("modelopt_cuda_ext_mx").Types.E8M0, None),
                    zero_sign=True)
                zero = (ref == 0) & (got == 0)        # sign of zero is unspecified in the reference
                n = nbad(torch.where(zero, torch.zeros_like(got), got), torch.where(zero, torch.zeros_like(ref), ref))
                tot += x.numel()
                bad += n
                assert n == 0, f"MX {name} bs{bs} {kind} {dtype}: {n}/{x.numel()} differ from fused_amax_convert"
    REPORT[f"mx_e8m0_{dtype}"] = {"elements": tot, "mismatches": bad}


def test_nvfp4_vs_reference_mx_twin(ops, refs):
    """The reference has TWO NVFP4 fake quants: the Triton kernel this engine restates (IEEE division; equal
    bit for bit to the NVFP4QTensor round trip, see tests/golden) and fused_amax_convert(E2M1, E4M3,
    global_amax) (two-level scale in double precision, reciprocal multiply, fast math; tensor_quant_mx.cu:153-183).
    * fp32 data (generic mantissas): the two agree except for a handful of elements within an ulp of a boundary.
    * 16-bit data: |x| / scale and block_amax * 448 / global_amax are very often EXACT rounding ties in real
      arithmetic (8 / 11-bit mantissas sharing factors with the global amax); which side a kernel lands on is
      decided by the last bit of its fp32 intermediates -- the reference's own test skips such vectors for Triton
      (tests/gpu/torch/quantization/test_tensor_quant_cuda.py:243-245).  There, every mismatch must stay within
      one E2M1 step / one E4M3 scale step and the rate must stay small; the rates are written to the report.
    Against the stored reference, the mismatches in the stored rows count against the bound for the whole tensor."""
    rep = {}
    for dtype in (torch.float32, torch.bfloat16, torch.float16):
        for kind in ("gauss", "heavy"):
            x = inputs((2048, 4096), dtype, 5, kind)
            g = x.abs().max().float().reshape(1)
            got = ops.fake_quant_nvfp4(x, g)
            ref, got = refs.rows(got, lambda: E("modelopt_cuda_ext_mx").fused_amax_convert(
                x, 16, E("modelopt_cuda_ext_mx").Types.E2M1, E("modelopt_cuda_ext_mx").Types.E4M3, g))
            # compare at bf16 resolution: the two fp32 block scales differ in the last bit by construction
            ref, got = ref.to(torch.bfloat16).float(), got.to(torch.bfloat16).float()
            diff = (ref != got)
            r, o_ = ref[diff].abs(), got[diff].abs()
            hi, lo = torch.maximum(r, o_), torch.minimum(r, o_)
            bounded = (lo == 0) | (hi / lo <= 2.05)
            n = int(diff.sum())
            rep[f"{dtype}_{kind}"] = {"elements": x.numel(), "compared": ref.numel(), "mismatches": n, "rate": n / ref.numel()}
            assert bool(bounded.all()), (dtype, kind)
            if dtype == torch.float32:
                assert n <= 1e-4 * x.numel(), (dtype, kind, n)
            else:
                assert n <= 0.02 * x.numel(), (dtype, kind, n)
    REPORT["nvfp4_vs_mx_twin"] = rep


from _gpu_timing import _time_eager, _time_graph  # noqa: E402


def test_speed_side_by_side(ops, ext, ext_fp8, ext_mx):
    """Same box, same harness (SURVEY 8d): the reference's CUDA kernels vs this engine's on the BASELINE tensor
    (4096 x 4096 bf16), 16 distinct inputs (512 MB >> L2), CUDA-graph replays so neither side pays launch
    latency.  INT4_quantize launches on the default stream (tensor_quant_gpu.cu:360) and cannot be captured:
    both sides of that pair are timed eagerly."""
    nbuf = 16
    gen = torch.Generator(device="cuda").manual_seed(0)
    xs = [torch.randn(4096, 4096, device="cuda", generator=gen).to(torch.bfloat16) for _ in range(nbuf)]
    ys = [torch.empty_like(xs[0]) for _ in range(4)]
    amax = xs[0].abs().max().float().reshape(1)
    rows = xs[0].abs().amax(dim=1).float()
    T = ext_mx.Types
    sc = [7 / x.view(-1, 128).abs().amax(dim=-1, keepdim=True) for x in xs[:2]]
    pairs = {
        "int8_per_tensor": (lambda i: ext.fake_tensor_quant(xs[i], amax, 8, False, False),
                            lambda i: ops.fake_quant_int(xs[i], amax, 8, False, False, out=ys[i % 4])),
        "int8_per_row": (lambda i: ext.fake_tensor_quant_with_axis(xs[i], rows, 0, 8, False, False),
                         lambda i: ops.fake_quant_int(xs[i], rows, 8, False, False, outer=4096, out=ys[i % 4])),
        "fp8_per_tensor": (lambda i: ext_fp8.fake_e4m3fy(xs[i], amax),
                           lambda i: ops.fake_quant_fp8(xs[i], amax, out=ys[i % 4])),
        "mxfp8_b32": (lambda i: ext_mx.fused_amax_convert(xs[i], 32, T.E4M3, T.E8M0, None),
                      lambda i: ops.fake_quant_mx(xs[i], 32, "E4M3", out=ys[i % 4])),
        "mxfp4_b32": (lambda i: ext_mx.fused_amax_convert(xs[i], 32, T.E2M1, T.E8M0, None),
                      lambda i: ops.fake_quant_mx(xs[i], 32, "E2M1", out=ys[i % 4])),
        "nvfp4_b16": (lambda i: ext_mx.fused_amax_convert(xs[i], 16, T.E2M1, T.E4M3, amax),
                      lambda i: ops.fake_quant_nvfp4(xs[i], amax, out=ys[i % 4])),
    }
    rep = {}
    for name, (ref_fn, our_fn) in pairs.items():
        t_ref, t_our = _time_graph(ref_fn, nbuf), _time_graph(our_fn, nbuf)
        rep[name] = {"reference_us": round(t_ref, 2), "b200_us": round(t_our, 2), "speedup": round(t_ref / t_our, 2)}
        assert t_our < t_ref, (name, t_our, t_ref)
    flat = [x.reshape(-1) for x in xs[:2]]
    t_ref = _time_eager(lambda i: ext.INT4_quantize(flat[i % 2], sc[i % 2], 128), nbuf)
    t_our = _time_eager(lambda i: ops.pack_int4_blockwise(flat[i % 2], 128), nbuf)
    rep["int4_pack_b128(eager, incl. launch)"] = {"reference_us": round(t_ref, 2), "b200_us": round(t_our, 2),
                                                  "speedup": round(t_ref / t_our, 2)}
    REPORT["speed_4096x4096_bf16"] = rep
    print(json.dumps(rep, indent=1))


def test_zz_write_report():
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "vs_reference_ext.json"), "w") as f:
        json.dump({k: (v if isinstance(v, dict) else str(v)) for k, v in REPORT.items()}, f, indent=1, default=str)
