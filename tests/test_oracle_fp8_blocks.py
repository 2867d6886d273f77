"""FP8 with static 2-D / 1-D block scales: the oracle (eager-rule FP8 fake quant and FP8 pack, applied through the
[A, b1, B, b2] tile view with the tile amax spread over rows) vs the reference run on CPU
(tests/golden/ref_fp8_blocks.*.npz, written by oracle/gen_golden.py fp8_blocks)."""

import os
import sys

import _golden
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle_np as o  # noqa: E402

G = _golden.load("ref_fp8_blocks")
F32 = np.float32


def keys():
    return sorted({k.rsplit("/x", 1)[0] for k in G.files if k.endswith("/x")})


def tile_view(x, b1, b2):
    n, k = x.shape
    xp = np.zeros((-(-n // b1) * b1, -(-k // b2) * b2), dtype=F32)
    xp[:n, :k] = x
    return xp.reshape(xp.shape[0] // b1, b1, xp.shape[1] // b2, b2)


def same(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def case(key):
    _, dname, shape, blk, _ = key.split("/")
    b1, b2 = (int(v) for v in blk.split("x"))
    x = G[key + "/x"]
    return dname, b1, b2, x, tile_view(x, b1, b2)


def test_block_amax_and_fake_quant():
    assert len(keys()) == 12
    for key in keys():
        dname, b1, b2, x, x4 = case(key)
        a, _, b, _ = x4.shape
        amax = np.abs(x4).max(axis=(1, 3))
        assert same(amax.reshape(G[key + "/amax"].shape), G[key + "/amax"]), key
        rows = np.broadcast_to(amax[:, None, :], (a, b1, b)).reshape(-1)
        fq = o.fake_quant_fp8(x4.reshape(-1), rows, b2, dname, eager=True).reshape(a * b1, b * b2)
        assert same(fq[: x.shape[0], : x.shape[1]], G[key + "/fq"]), key


def test_block_pack_and_dequant():
    for key in keys():
        dname, b1, b2, x, x4 = case(key)
        a, _, b, _ = x4.shape
        amax = np.abs(x4).max(axis=(1, 3))
        sc = o.round_to(amax / F32(448.0), dname)
        assert same(sc, G[key + "/scale"]), key
        rows = np.broadcast_to(sc[:, None, :], (a, b1, b)).reshape(-1)
        bits = o.pack_fp8(x4.reshape(-1), rows, b2, dname, dname).reshape(a * b1, b * b2)[: x.shape[0], : x.shape[1]]
        assert np.array_equal(bits, G[key + "/q"]), key
        bp = np.zeros((a * b1, b * b2), dtype=np.uint8)
        bp[: x.shape[0], : x.shape[1]] = bits
        deq = o.unpack_fp8(bp.reshape(-1), rows, b2, dname).reshape(a * b1, b * b2)[: x.shape[0], : x.shape[1]]
        assert same(deq, G[key + "/deq"]), key
        # export: fp32 scales = amax.float() / 448 -> the quotient is NOT rounded to the tensor dtype
        wsf = (amax.astype(F32) / F32(448.0)).astype(F32)
        rows32 = np.broadcast_to(wsf[:, None, :], (a, b1, b)).reshape(-1)
        bits = o.pack_fp8(x4.reshape(-1), rows32, b2, dname, "f32").reshape(a * b1, b * b2)[: x.shape[0], : x.shape[1]]
        assert np.array_equal(bits, G[key + "/q_export"]), key
