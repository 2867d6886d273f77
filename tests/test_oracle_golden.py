"""The oracle (oracle/oracle_np.py) must reproduce, bit for bit, what the REAL reference produced
in this container (tests/golden/ref_small.*.npz, written by oracle/gen_golden.py) and the
reference's own known-answer vectors.  CPU only."""

import numpy as np
import pytest

from oracle import oracle_np as o


def _cases(golden):
    return [str(c) for c in golden["cases"]]


def _dt(key):
    return key.split("_")[0]


def eq(a, b):
    """bit-exact (NaN == NaN; -0.0 != +0.0)."""
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.dtype.kind == "f" or b.dtype.kind == "f":
        a = np.ascontiguousarray(a, dtype=np.float32)
        b = np.ascontiguousarray(b, dtype=np.float32)
        ok = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    else:
        ok = a == b
    nbad = int(np.sum(~ok))
    assert nbad == 0, f"{nbad} mismatches"


def eqz(a, b):
    """bit-exact up to the sign of zero."""
    eq(np.asarray(a, dtype=np.float32) + np.float32(0), np.asarray(b, dtype=np.float32) + np.float32(0))


def test_cases_present(golden):
    assert len(_cases(golden)) >= 9


def test_amax(golden):
    for k in _cases(golden):
        x = golden[f"{k}/x"]
        eq(o.reduce_amax(x), golden[f"{k}/amax_tensor"])
        eq(o.reduce_amax(x, axis=1), golden[f"{k}/amax_rows"])
        eq(o.reduce_amax(x, axis=0), golden[f"{k}/amax_cols"])
        eq(o.reduce_block_amax(x, 16), golden[f"{k}/amax_block16"])
        eq(o.reduce_block_amax(x, 128), golden[f"{k}/amax_block128"])


def test_max_calibrator(golden):
    for k in _cases(golden):
        if f"{k}/maxcal" not in golden:
            continue
        x = golden[f"{k}/x"]
        c = o.MaxCalibrator(None)
        c.collect(x)
        c.collect(o.round_to(x * np.float32(0.5), _dt(k)))
        eq(c.compute_amax(), golden[f"{k}/maxcal"])
        c0 = o.MaxCalibrator(0)
        c0.collect(x)
        eq(c0.compute_amax(), golden[f"{k}/maxcal_axis0"])


@pytest.mark.parametrize("bits,narrow", [(8, False), (8, True), (4, False), (3, True)])
def test_int_fake_quant_cpu_twin(golden, bits, narrow):
    for k in _cases(golden):
        x = golden[f"{k}/x"]
        amax = o.reduce_amax(x)
        ref = golden[f"{k}/int{bits}_n{int(narrow)}_tensor"]
        eq(o.tensor_quant_cpu(x, amax, bits, False, narrow, _dt(k)), ref)
        if amax > 2.0**-24:  # CUDA and CPU rules coincide away from the zero-amax corner
            eq(o.fake_quant_int(x, amax, bits, False, narrow, 1, _dt(k)), ref)


def test_int_fake_quant_axis(golden):
    for k in _cases(golden):
        x = golden[f"{k}/x"]
        amax_r = o.reduce_amax(x, axis=1)
        ref = golden[f"{k}/int8_rows"]
        eq(o.tensor_quant_cpu(x, amax_r, 8, False, False, _dt(k)), ref)
        if "sparse" not in k:
            eq(o.fake_quant_int(x, amax_r, 8, False, False, x.shape[1], _dt(k)), ref)
            xb = x.reshape(-1, 128)
            eq(o.fake_quant_int(xb, o.reduce_amax(xb, axis=1), 4, False, False, 128, _dt(k)).reshape(x.shape),
               golden[f"{k}/int4_block128"])


def test_fp8_fake_quant(golden):
    for k in _cases(golden):
        x = golden[f"{k}/x"]
        eq(o.fake_quant_fp8(x, o.reduce_amax(x), 1, _dt(k), eager=True), golden[f"{k}/fp8_tensor"])
        eq(o.fake_quant_fp8(x, o.reduce_amax(x, axis=1), x.shape[1], _dt(k), eager=True), golden[f"{k}/fp8_rows"])
        # the CUDA-extension rule (true division) may move the scale by one ulp: outputs stay close
        cu = o.fake_quant_fp8(x, o.reduce_amax(x), 1, _dt(k))
        ref = golden[f"{k}/fp8_tensor"]
        assert np.allclose(cu, ref, rtol=0.07, atol=0, equal_nan=True)
        assert np.mean(cu != ref) < 0.2
        eq(o.fake_quant_fp8(x, None, 1, _dt(k)), golden[f"{k}/fp8_noamax"])


def test_nvfp4_pack_and_qdq(golden):
    n = 0
    for k in _cases(golden):
        if f"{k}/nvfp4_packed" not in golden:
            continue
        n += 1
        x = golden[f"{k}/x"]
        packed, sbits, s2 = o.pack_nvfp4(x)
        eq(packed, golden[f"{k}/nvfp4_packed"])
        eq(sbits, golden[f"{k}/nvfp4_scales"])
        eq(np.float32(s2), golden[f"{k}/nvfp4_wsf2"])
        eq(o.unpack_nvfp4(packed, sbits, s2, _dt(k)), golden[f"{k}/nvfp4_deq"])
    assert n >= 6


def test_nvfp4_dynamic_qdq_equals_qtensor_roundtrip(golden):
    """SURVEY.md 8c: the Triton dynamic formula (IEEE division) == the executed reference's
    NVFP4QTensor quantize->dequantize round trip away from the degenerate corners (A.6)."""
    for k in _cases(golden):
        if f"{k}/nvfp4_deq" not in golden or "ties" in k:
            continue
        x = golden[f"{k}/x"]
        got = o.fake_quant_nvfp4(x, o.reduce_amax(x), _dt(k))
        ref = golden[f"{k}/nvfp4_deq"]
        assert np.mean(got != ref) < 1e-3, np.mean(got != ref)
        if "gauss" in k:
            # the Triton formula keeps -0.0 for negatives that round to zero, the QTensor LUT maps
            # code 8 to +0.0 (nvfp4_tensor.py:27): equal up to the sign of zero
            eqz(got, ref)


def test_fp4_static_scales(golden):
    for k in _cases(golden):
        if f"{k}/fp4_scales_static" not in golden:
            continue
        x = golden[f"{k}/x"]
        bam = o.reduce_block_amax(x, 16)
        eq(o.compute_fp4_scales(bam, o.reduce_amax(x), True, eager=True), golden[f"{k}/fp4_scales_static"])
        eq(o.compute_fp4_scales(bam, o.reduce_amax(x), True, 256.0, eager=True), golden[f"{k}/fp4_scales_static_46"])


def test_nvfp4_static_pack(golden):
    for k in _cases(golden):
        if f"{k}/nvfp4s_packed" not in golden:
            continue
        x = golden[f"{k}/x"]
        bam = o.reduce_block_amax(x, 16)
        packed, sbits, s2 = o.pack_nvfp4(x, o.reduce_amax(x), block_amax=bam)
        eq(sbits, golden[f"{k}/nvfp4s_scales"])
        eq(np.float32(s2), golden[f"{k}/nvfp4s_wsf2"])
        eq(packed, golden[f"{k}/nvfp4s_packed"])


def test_int4_packs(golden):
    n = 0
    for k in _cases(golden):
        if f"{k}/int4cpu_packed" not in golden:
            continue
        n += 1
        x = golden[f"{k}/x"]
        packed, scales = o.pack_int4_blockwise_cpu(x, 128, _dt(k))
        eq(scales, golden[f"{k}/int4cpu_scales"])
        eq(packed, golden[f"{k}/int4cpu_packed"])
        eq(o.pack_int4_export(x, golden[f"{k}/int4exp_scale"], _dt(k), "f32"), golden[f"{k}/int4exp_packed"])
        eq(o.pack_int4_export(x, golden[f"{k}/int4exp_scale_same"], _dt(k), _dt(k)),
           golden[f"{k}/int4exp_packed_same"])
    assert n >= 5


def test_fp8_packs(golden):
    for k in _cases(golden):
        if f"{k}/fp8pack_tensor" not in golden:
            continue
        x = golden[f"{k}/x"]
        d = _dt(k)
        sc = golden[f"{k}/fp8pack_tensor_scale"]
        eq(o.round_to(o.reduce_amax(x) / np.float32(448.0), d), sc)
        eq(o.pack_fp8(x, sc, 1, d, d), golden[f"{k}/fp8pack_tensor"])
        scr = golden[f"{k}/fp8pack_rows_scale"]
        eq(o.pack_fp8(x, scr, x.shape[1], d, d), golden[f"{k}/fp8pack_rows"])
        eq(o.pack_fp8(x, golden[f"{k}/fp8pack_export_scale"], 1, d, "f32", scale_is_0dim=True),
           golden[f"{k}/fp8pack_export"])
        eq(o.pack_fp8(x, golden[f"{k}/fp8pack_export_scale"], 1, d, "f32", scale_is_0dim=False),
           golden[f"{k}/fp8pack_export1"])      # (1,)-shaped fp32 scale: torch promotes the quotient to fp32


def test_histogram(golden):
    n = 0
    for k in _cases(golden):
        if f"{k}/hist1" not in golden:
            continue
        n += 1
        x = golden[f"{k}/x"]
        h = o.HistogramCalibrator(2048)
        h.collect(x)
        eq(h.hist, golden[f"{k}/hist1"])
        h.collect(o.round_to(x * np.float32(1.5), _dt(k)))
        assert h.hist.sum() == golden[f"{k}/hist2"].sum()
        # CPU histc (the only one runnable here) and the CUDA formula the oracle restates may put
        # an element that sits exactly on a bin edge in neighbouring bins: allow +-1 moves
        d = h.hist - golden[f"{k}/hist2"]
        assert np.abs(d).sum() <= 8, np.abs(d).sum()
    assert n == 2


# ---- the reference's own known-answer vectors -------------------------------------------------
def test_e2m1_boundary_vectors():
    """tests/gpu/torch/quantization/test_tensor_quant_cuda.py:236-262."""
    base = np.array([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5, 6], dtype=np.float32)
    tab = np.array([0, 0.5, 1, 1.5, 2, 3, 4, 6], dtype=np.float32)
    for sign in (1.0, -1.0):
        def run(v):
            x = np.concatenate([v, v]).reshape(1, 16).astype(np.float32) * np.float32(sign)
            return o.fake_quant_nvfp4(x, np.abs(x).max(), "f32")[0, :8] * np.float32(sign)
        eqz(run(tab), tab)
        eqz(run(base), np.array([0, 1, 1, 2, 2, 4, 4, 6], dtype=np.float32))
        lo = base.copy(); lo[:-1] -= np.float32(0.1)
        assert np.allclose(run(lo), tab)
        hi = base.copy(); hi[:-1] += np.float32(0.1)
        assert np.allclose(run(hi), np.array([0.5, 1, 1.5, 2, 3, 4, 6, 6], dtype=np.float32))


def test_qtensor_golden_vectors():
    """tests/gpu/torch/quantization/test_qtensor_cuda.py:141-254 (bf16 in, bf16 out)."""
    x8 = np.arange(8, dtype=np.float32).reshape(1, 8)
    # INT4 block 4 (compress + dequantize); cpu and cuda branches agree on this vector
    for pack in (o.pack_int4_blockwise_cpu, o.pack_int4_blockwise_cuda):
        p, s = pack(x8, 4, "bf16")
        got = o.unpack_int4_blockwise(p, s, 4, "bf16").reshape(1, 8)
        assert np.allclose(got, [[0.0, 0.8516, 2.1406, 2.9844, 4, 5, 6, 7]], atol=4e-3)
    # FP8 per tensor / per channel
    x = np.arange(8, dtype=np.float32).reshape(2, 4)
    sc = o.round_bf16(o.reduce_amax(x) / np.float32(448))
    got = o.unpack_fp8(o.pack_fp8(x, sc, 1, "bf16", "bf16"), sc, 1, "bf16")
    eq(got, x)
    scr = o.round_bf16(o.reduce_amax(x, axis=1) / np.float32(448))
    got = o.unpack_fp8(o.pack_fp8(x, scr, 4, "bf16", "bf16"), scr, 4, "bf16")
    assert np.allclose(got, [[0, 0.9609, 1.9219, 3.0], [4, 5, 6, 7]], atol=4e-3)


def test_tiny_amax_zeroes():
    """tests/gpu/torch/quantization/test_tensor_quant_cuda.py:115-119."""
    x = np.array([[0, 1e-9], [-1e-9, 1e-9]], dtype=np.float32)
    eq(o.fake_quant_int(x, np.float32(1e-9), 8, False, True, 1, "f32"), np.zeros_like(x))


def test_nvfp4_pack_block_sizes_32_64():
    """NVFP4QTensor.quantize with block sizes other than 16 (the W4A8_NVFP4_FP8 / NVFP4_MLP_WEIGHT_ONLY presets)."""
    import os

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_nvfp4_blocks.npz"))
    keys = sorted({k.rsplit("/x", 1)[0] for k in g.files if k.endswith("/x")})
    assert len(keys) == 24
    for k in keys:
        bs, d = int(k.split("/")[-1]), k.split("/")[1]
        p, s, s2 = o.pack_nvfp4(g[k + "/x"], block_size=bs)
        assert np.array_equal(p, g[k + "/packed"]) and np.array_equal(s, g[k + "/scale"]) and np.float32(s2) == g[k + "/sf2"], k
        eq(o.unpack_nvfp4(p, s, s2, d), g[k + "/deq"])
