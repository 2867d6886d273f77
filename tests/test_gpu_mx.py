"""GPU parity of the MX (E8M0 block scale) kernels, called through the C-ABI, against
(a) tests/golden/ref_mx.*.npz -- outputs of the reference's own C++ (host builds of tensor_quant_mx.h/.cu)
    and of its MXFP8 / MXFP4 QTensor Python, and
(b) the NumPy oracle on larger / irregular tensors.  Bar: bit-exact."""

import os

import _golden
import numpy as np
import pytest
import torch

from oracle import oracle_np as o

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = _golden.load("ref_mx")
TD = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}
FMT_NAMES = ["E4M3", "E5M2", "INT8", "E0M3", "E1M2", "E3M0", "E2M1", "E3M2", "E2M3"]


@pytest.fixture(scope="module")
def ops():
    from model_optimizer_b200 import ops as _ops

    return _ops


def f(a):
    return np.asarray(a).view(np.float32)


def dev(x, d):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to("cuda").to(TD[d])


def host(t):
    return t.detach().float().cpu().numpy()


def same(a, b, what=""):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.dtype.kind == "f":
        a, b = a.astype(np.float32), b.astype(np.float32)
        ok = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    else:
        ok = a == b
    n = int(np.sum(~ok))
    if n:
        i = tuple(np.argwhere(~ok)[0])
        raise AssertionError(f"{what}: {n}/{a.size} mismatches, first at {i}: got {a[i]!r} want {b[i]!r}")


@pytest.mark.parametrize("fmt", range(9))
@pytest.mark.parametrize("bs", [8, 16, 32])
def test_fake_quant_mx_golden(ops, fmt, bs):
    for dname in TD:
        for kind in ("gauss", "heavy", "ties", "sparse", "ragged"):
            key = f"fq/{fmt}/{bs}/{dname}/{kind}"
            x = f(G[key + "/x"])
            y = ops.fake_quant_mx(dev(x, dname), bs, FMT_NAMES[fmt])
            same(host(y), f(G[key + "/y"]), key)


@pytest.mark.parametrize("fmt", range(9))
@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
def test_fake_quant_mx_oracle_large(ops, fmt, dname):
    g = np.random.default_rng(100 + fmt)
    x = g.standard_normal((512, 2048)).astype(np.float32) * np.exp2(g.integers(-20, 12, (512, 1))).astype(np.float32)
    x = x * (1 + 30 * (g.random(x.shape) < 1e-3)).astype(np.float32)
    x[3, :64] = 0
    x[4, 5] = -0.0
    x = o.round_to(x, dname)
    for bs in (32, 16):
        y = ops.fake_quant_mx(dev(x, dname), bs, fmt)
        same(host(y), o.fake_quant_mx(x, bs, fmt, dtype=dname), f"fmt{fmt} bs{bs} {dname}")


@pytest.mark.parametrize("fmt", [0, 1, 3, 4, 5, 6, 7, 8])   # INT8 of NaN / inf is undefined in the reference
def test_fake_quant_mx_nonfinite(ops, fmt):
    g = np.random.default_rng(7)
    x = o.round_bf16(g.standard_normal((64, 256)).astype(np.float32))
    x[0, 3] = np.nan
    x[1, 40] = np.inf
    x[2, 70] = -np.inf
    x[3, :32] = np.nan
    x[5, 100], x[5, 101] = np.nan, np.inf
    for bs in (32, 16, 8):
        y = ops.fake_quant_mx(dev(x, "bf16"), bs, fmt)
        same(host(y), o.fake_quant_mx(x, bs, fmt, dtype="bf16"), f"fmt{fmt} bs{bs}")


def test_fake_quant_mx_inplace_unaligned_and_errors(ops):
    from model_optimizer_b200._lib import B200QuantError

    g = np.random.default_rng(3)
    x = o.round_bf16(g.standard_normal((33, 96)).astype(np.float32))
    want = o.fake_quant_mx(x, 32, o.MX_E4M3, dtype="bf16")
    t = dev(x, "bf16")
    ops.fake_quant_mx(t, 32, "E4M3", out=t)
    same(host(t), want, "in place")
    buf = torch.zeros(33 * 96 + 1, dtype=torch.bfloat16, device="cuda")
    v = buf[1:].view(33, 96)
    v.copy_(dev(x, "bf16"))
    same(host(ops.fake_quant_mx(v, 32, "E4M3")), want, "unaligned view")
    with pytest.raises(B200QuantError):
        ops.fake_quant_mx(t, 64, "E4M3")
    with pytest.raises(B200QuantError):
        ops.fake_quant_mx(t, 32, 9)
    e = torch.empty(0, 32, dtype=torch.bfloat16, device="cuda")
    assert ops.fake_quant_mx(e, 32, "E2M1").shape == (0, 32)


@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
def test_mxfp8_pack_golden_and_oracle(ops, dname):
    for kind in ("gauss", "heavy", "ties", "sparse", "ragged"):
        key = f"qt/{dname}/{kind}"
        x = f(G[key + "/x"])
        q, s = ops.pack_mxfp8(dev(x, dname))
        same(q.view(torch.uint8).cpu().numpy(), G[key + "/mxfp8/q"], key + " q")
        same(s.cpu().numpy(), G[key + "/mxfp8/scale"], key + " scale")
        same(host(ops.unpack_mxfp8(q, s, TD[dname])), f(G[key + "/mxfp8/deq"]), key + " deq")
        q2, _ = ops.pack_mxfp8(dev(x, dname), s)
        same(q2.view(torch.uint8).cpu().numpy(), G[key + "/mxfp8/q"], key + " with scale")
    g = np.random.default_rng(1)
    x = g.standard_normal((256, 4096)).astype(np.float32) * np.exp2(g.integers(-30, 20, (256, 1))).astype(np.float32)
    x = o.round_to(x, dname)
    q, s = ops.pack_mxfp8(dev(x, dname))
    wq, ws = o.pack_mxfp8(x)
    same(q.view(torch.uint8).cpu().numpy(), wq, "large q")
    same(s.cpu().numpy(), ws, "large scale")
    same(host(ops.unpack_mxfp8(q, s, TD[dname])), o.unpack_mxfp8(wq, ws, dtype=dname), "large deq")


@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("bs", [32, 16])
def test_mxfp4_pack_golden_and_oracle(ops, dname, bs):
    for kind in ("gauss", "heavy", "ties", "sparse"):
        key = f"qt/{dname}/{kind}"
        x = f(G[key + "/x"])
        q, s = ops.pack_mxfp4(dev(x, dname), bs)
        same(q.cpu().numpy(), G[key + f"/mxfp4_{bs}/q"], key + " q")
        same(s.cpu().numpy(), G[key + f"/mxfp4_{bs}/scale"], key + " scale")
        same(host(ops.unpack_mxfp4(q, s, bs, TD[dname])), f(G[key + f"/mxfp4_{bs}/deq"]), key + " deq")
    g = np.random.default_rng(2)
    lo, hi = (-30, 20) if dname != "f16" else (-12, 12)      # an inf block amax is undefined in MXFP4QTensor
    x = g.standard_normal((256, 4096)).astype(np.float32) * np.exp2(g.integers(lo, hi, (256, 1))).astype(np.float32)
    # exact E2M1 rounding ties (they round DOWN in MXFP4QTensor) in every block of the first rows
    ties = np.array([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0, 6.0], np.float32)
    x[:8, ::4] = ties[g.integers(0, 8, (8, 1024))] * np.where(g.random((8, 1024)) < 0.5, -1, 1)
    x[:8, 1] = 6.0
    x[9, :64] = 0
    x = o.round_to(x, dname)
    q, s = ops.pack_mxfp4(dev(x, dname), bs)
    wq, ws = o.pack_mxfp4(x, bs)
    same(s.cpu().numpy(), ws, "large scale")
    same(q.cpu().numpy(), wq, "large q")
    same(host(ops.unpack_mxfp4(q, s, bs, TD[dname])), o.unpack_mxfp4(wq, ws, bs, dtype=dname), "large deq")


def test_mx_full_size_properties(ops):
    """4096 x 4096 bf16 (BASELINE tensor): idempotence of the fake quant and pack/unpack == fake quant
    for MXFP8 (where the QTensor and the fused kernel agree: no ties-down rule, same scale)."""
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(4096, 4096, device="cuda", generator=gen, dtype=torch.float32).to(torch.bfloat16)
    for name in ("E4M3", "E2M1", "E3M2", "INT8"):
        y = ops.fake_quant_mx(x, 32, name)
        # value equality: a negative value that rounded to -0.0 comes back as +0.0 on the second pass
        assert torch.equal(ops.fake_quant_mx(y, 32, name), y), name
    q, s = ops.pack_mxfp8(x)
    deq = ops.unpack_mxfp8(q, s, torch.bfloat16)
    y = ops.fake_quant_mx(x, 32, "E4M3")
    nz = y != 0                     # negative values that round to zero: -0.0 (fused) vs the same from e4m3
    assert torch.equal(deq[nz].view(torch.int16), y[nz].view(torch.int16))
    assert (deq[~nz] == 0).all()


def test_convert_to_exmy_host(ops):
    for fmt in range(9):
        x, y = f(G[f"cvt/{fmt}/x"])[::5], f(G[f"cvt/{fmt}/y"])[::5]
        got = np.array([ops.convert_to_exmy(float(v), fmt) for v in x], dtype=np.float32)
        same(got, y, f"fmt {fmt}")


def test_tensor_quantizer_mx_dispatch_and_presets(ops):
    import torch.nn as nn

    from model_optimizer_b200.config import get_preset
    from model_optimizer_b200.model_quant import quantize
    from model_optimizer_b200.nn import TensorQuantizer
    from model_optimizer_b200.qtensor import MXFP4QTensor, MXFP8QTensor

    g = np.random.default_rng(9)
    x = o.round_bf16(g.standard_normal((4, 40, 128)).astype(np.float32) * 3)
    for nb, fmt in (((4, 3), o.MX_E4M3), ((3, 2), o.MX_E3M2), ((2, 1), o.MX_E2M1), (8, o.MX_INT8)):
        tq = TensorQuantizer({"num_bits": nb, "block_sizes": {-1: 32, "type": "dynamic", "scale_bits": (8, 0)}})
        assert tq.is_mx_format and tq.amax is None
        same(host(tq(dev(x, "bf16"))), o.fake_quant_mx(x, 32, fmt, dtype="bf16"), str(nb))
    t = dev(x, "bf16").requires_grad_(True)
    tq(t).sum().backward()            # MX is always pass-through in backward
    assert torch.equal(t.grad, torch.ones_like(t))
    # real quantization
    w = dev(x[0], "bf16")
    tq8 = TensorQuantizer({"num_bits": (4, 3), "fake_quant": False,
                           "block_sizes": {-1: 32, "type": "dynamic", "scale_bits": (8, 0)}})
    q8 = tq8(w)
    assert isinstance(q8, MXFP8QTensor) and tq8._scale.dtype == torch.uint8
    wq, ws = o.pack_mxfp8(x[0])
    same(q8._quantized_data.view(torch.uint8).cpu().numpy(), wq, "real mxfp8")
    tq4 = TensorQuantizer({"num_bits": (2, 1), "fake_quant": False,
                           "block_sizes": {-1: 32, "type": "dynamic", "scale_bits": (8, 0)}})
    q4 = tq4(w)
    assert isinstance(q4, MXFP4QTensor)
    same(q4._quantized_data.cpu().numpy(), o.pack_mxfp4(x[0], 32)[0], "real mxfp4")
    # presets through quantize(): calibration-free (algorithm None), weights and inputs fake-quantized
    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(128, 64, bias=False), nn.Linear(64, 128, bias=False)).cuda().to(torch.bfloat16)
    ref_w = [m.weight.detach().clone() for m in model]
    inp = dev(x, "bf16")
    for preset, fmt in (("MXFP8_DEFAULT_CFG", o.MX_E4M3), ("MXFP4_DEFAULT_CFG", o.MX_E2M1),
                        ("MXFP6_DEFAULT_CFG", o.MX_E3M2), ("MXINT8_DEFAULT_CFG", o.MX_INT8)):
        m2 = nn.Sequential(nn.Linear(128, 64, bias=False), nn.Linear(64, 128, bias=False)).cuda().to(torch.bfloat16)
        for a, b in zip(m2, ref_w):
            a.weight.data.copy_(b)
        m2 = quantize(m2, get_preset(preset), lambda m: m(inp))
        xq = torch.from_numpy(o.fake_quant_mx(x, 32, fmt, dtype="bf16")).cuda().to(torch.bfloat16)
        wq0 = torch.from_numpy(o.fake_quant_mx(host(ref_w[0]), 32, fmt, dtype="bf16")).cuda().to(torch.bfloat16)
        h = torch.nn.functional.linear(xq, wq0)
        same(host(m2[0](inp)), host(h), preset)
        if preset in ("MXFP8_DEFAULT_CFG", "MXFP4_DEFAULT_CFG"):
            from model_optimizer_b200 import export as ex

            d = ex.export_quantized_linear(m2[0])
            w0 = host(ref_w[0])
            if preset == "MXFP8_DEFAULT_CFG":
                assert d["quantization"] == "mxfp8"
                wq, ws = o.pack_mxfp8(w0)
                same(d["weight"].view(torch.uint8).cpu().numpy(), wq, "export mxfp8 weight")
                same(d["weight_scale"].cpu().numpy(), ws, "export mxfp8 scale")
                same(ex.get_weight_scaling_factor(m2[0]).cpu().numpy(), ws, "wsf mxfp8")
                same(ex.to_quantized_weight(ref_w[0], d["weight_scale"], "mxfp8").view(torch.uint8).cpu().numpy(), wq, "tqw")
            else:
                assert d["quantization"] == "mxfp4"
                wq, ws = o.pack_mxfp4(w0, 32)
                same(d["weight"].cpu().numpy(), wq, "export mxfp4 weight")
                same(d["weight_scale"].cpu().numpy(), ws.reshape(w0.shape[0], -1), "export mxfp4 scale")
                same(ex.to_quantized_weight(ref_w[0], None, "mxfp4", block_size=32).cpu().numpy(), wq, "tqw4")


def test_nf4_real_quantize_round_trip(ops):
    from model_optimizer_b200.nn import TensorQuantizer
    from model_optimizer_b200.qtensor import NF4QTensor

    g = np.random.default_rng(4)
    w = o.round_bf16(g.standard_normal((64, 256)).astype(np.float32) * 0.05)
    for dname in ("bf16", "f16", "f32"):
        wt = dev(w, dname)
        packed, scales = ops.pack_nf4(wt, 32)
        wp, ws = o.pack_nf4(w, 32, dname)
        same(packed.cpu().numpy(), wp, f"nf4 pack {dname}")
        same(host(scales).reshape(-1), ws.reshape(-1), f"nf4 scales {dname}")
        same(host(ops.unpack_nf4(packed, scales, 32)), o.unpack_nf4(wp, ws, 32), f"nf4 unpack {dname}")
    tq = TensorQuantizer({"num_bits": 4, "fake_quant": False,
                          "block_sizes": {-1: 32, "scale_bits": 8, "scale_block_sizes": {-1: 64}}})
    wt = dev(w, "bf16")
    q = tq(wt)
    assert isinstance(q, NF4QTensor) and tq._scale.dtype == torch.int8 and tq._double_scale.numel() == 64 * 256 // 32 // 64
    deq = tq.dequantize(q)
    assert deq.shape == wt.shape and deq.dtype == wt.dtype
    rel = (deq.float() - wt.float()).norm() / wt.float().norm()
    assert rel < 0.12, float(rel)            # 4-bit NormalFloat + int8 double-quantized scales
