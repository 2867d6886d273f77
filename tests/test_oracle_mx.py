"""The NumPy oracle's MX section must reproduce, bit for bit, what the REAL reference produced:
its C++ element rounding / E8M0 block math (host builds of tensor_quant_mx.h / .cu, oracle/_ref) and
its MXFP8 / MXFP4 QTensor round trips (tests/golden/ref_mx.*.npz, written by oracle/gen_golden.py mx)."""

import hashlib
import json
import os
import sys

import _golden
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle_np as o  # noqa: E402

G = _golden.load("ref_mx")
F32 = np.float32


def f(a):
    return np.asarray(a).view(F32)


def same(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


@pytest.mark.parametrize("fmt", range(9))
def test_convert_to_exmy(fmt):
    x, y = f(G[f"cvt/{fmt}/x"]), f(G[f"cvt/{fmt}/y"])
    assert same(o.convert_to_exmy(x, fmt), y).all()


@pytest.mark.parametrize("fmt", range(9))
@pytest.mark.parametrize("bs", [8, 16, 32])
def test_fake_quant_mx(fmt, bs):
    n = 0
    for dname in ("bf16", "f16", "f32"):
        for kind in ("gauss", "heavy", "ties", "sparse", "ragged"):
            key = f"fq/{fmt}/{bs}/{dname}/{kind}"
            x, y = f(G[key + "/x"]), f(G[key + "/y"])
            got = o.fake_quant_mx(x, bs, fmt, dtype=dname)
            assert same(got, y).all(), key
            n += x.size
    assert n > 0


@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("kind", ["gauss", "heavy", "ties", "sparse", "ragged"])
def test_mxfp8_qtensor(dname, kind):
    key = f"qt/{dname}/{kind}"
    x = f(G[key + "/x"])
    bits, scale = o.pack_mxfp8(x)
    assert (scale == G[key + "/mxfp8/scale"]).all()
    assert (bits == G[key + "/mxfp8/q"]).all()
    assert same(o.unpack_mxfp8(bits, scale, dtype=dname), f(G[key + "/mxfp8/deq"])).all()
    # quantize_with_scale: a given scale reproduces the same bytes
    bits2, _ = o.pack_mxfp8(x, scale_bytes=scale)
    assert (bits2 == bits).all()


@pytest.mark.parametrize("dname", ["bf16", "f16", "f32"])
@pytest.mark.parametrize("kind", ["gauss", "heavy", "ties", "sparse"])
@pytest.mark.parametrize("bs", [32, 16])
def test_mxfp4_qtensor(dname, kind, bs):
    key = f"qt/{dname}/{kind}"
    x = f(G[key + "/x"])
    packed, scale = o.pack_mxfp4(x, bs)
    assert (scale == G[key + f"/mxfp4_{bs}/scale"]).all()
    assert (packed == G[key + f"/mxfp4_{bs}/q"]).all()
    assert same(o.unpack_mxfp4(packed, scale, bs, dtype=dname), f(G[key + f"/mxfp4_{bs}/deq"])).all()


def _digest(a):
    a = np.asarray(a, F32)
    return hashlib.sha256(np.where(np.isnan(a), F32(np.nan), a).astype(F32).tobytes()).hexdigest()


def test_ref_libs_live():
    """The restatement against the reference's element rounding (host build of tensor_quant_mx.h) on a larger random
    set: live where oracle/_ref was built, else against the SHA-256 of what that build returned
    (tests/golden/ref_mx_cvt_sha256.json; NaN payloads made equal).  B200Q_RECORD_GOLDEN=<dir> on a live run writes
    that file to <dir>."""
    import ctypes

    p = os.path.join(ROOT, "oracle", "_ref", "libmxref.so")
    stored = os.path.join(ROOT, "tests", "golden", "ref_mx_cvt_sha256.json")
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.standard_normal(20000).astype(F32) * 4, (rng.standard_normal(5000) * 1e3).astype(F32)])
    if not os.path.exists(p):
        want = json.load(open(stored))
        for fmt in range(9):
            assert _digest(o.convert_to_exmy(x, fmt)) == want[str(fmt)], fmt
        return
    h = ctypes.CDLL(p)
    h.ref_convert_to_exmy_n.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_int]
    digests = {}
    for fmt in range(9):
        y = np.empty_like(x)
        h.ref_convert_to_exmy_n(x.ctypes.data, y.ctypes.data, x.size, fmt)
        assert same(o.convert_to_exmy(x, fmt), y).all()
        digests[str(fmt)] = _digest(y)
    if os.environ.get("B200Q_RECORD_GOLDEN"):
        os.makedirs(os.environ["B200Q_RECORD_GOLDEN"], exist_ok=True)
        with open(os.path.join(os.environ["B200Q_RECORD_GOLDEN"], "ref_mx_cvt_sha256.json"), "w") as fh:
            json.dump(digests, fh, indent=1)
