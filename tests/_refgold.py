"""Reference results for the GPU tests that run this engine next to the reference's own kernels.

Where the reference's kernels are at hand (``oracle/_ref``, built by ``__graft_entry__.build()`` next to the
reference sources) a test computes the reference side live, as it always did.  Everywhere else it compares with
what those kernels produced on the same seeded inputs, stored in ``tests/golden/<name>/<test function>.<part>.npz``
(split into parts under 1 MB, see ``_golden``):

  * a SHA-256 of the output where the comparison is bit for bit (NaN equals NaN, and -0 equals +0 where the test
    compares zeros by value);
  * where the test counts and bounds mismatches, outputs of up to 64 Ki elements whole, larger ones as a fixed,
    seeded sample of SAMPLE_ROWS rows plus the last row (where a ragged tile ends).  The mismatches found in what is
    stored then count against the test's bound for the whole output, a condition the full comparison implies.

A live run with ``B200Q_RECORD_GOLDEN=<dir>`` in the environment writes ``<dir>/<name>/``.
Entries are keyed by test id and call order, so a test that changes what it compares must be re-recorded.  The
inputs come from torch's seeded CUDA generator and some reference results pass through torch / cuBLAS (the
reference's model forward), so a torch upgrade may call for a re-record even where this engine is unchanged.
"""

from __future__ import annotations

import hashlib
import os

import _golden
import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE_ROWS = 16
WHOLE_ELEMENTS = 1 << 16
_NATIVE = {torch.float32: np.float32, torch.bfloat16: np.uint16, torch.float16: np.uint16}


def digest(t: torch.Tensor, zero_sign: bool = False) -> str:
    t = t.detach().contiguous()
    if t.is_floating_point():
        t = torch.where(torch.isnan(t), torch.full_like(t, float("nan")), t)
        if zero_sign:
            t = torch.where(t == 0, torch.zeros_like(t), t)
    h = hashlib.sha256(f"{tuple(t.shape)} {t.dtype}".encode())
    h.update(t.reshape(-1).view(torch.uint8).cpu().numpy().tobytes())
    return h.hexdigest()


def sample_rows(shape: tuple[int, int], whole: bool = False) -> np.ndarray:
    n_rows = shape[0]
    if whole or n_rows <= SAMPLE_ROWS + 1 or n_rows * shape[1] <= WHOLE_ELEMENTS:
        return np.arange(n_rows)
    rows = np.random.default_rng(0).choice(n_rows - 1, SAMPLE_ROWS, replace=False)
    return np.append(np.sort(rows), n_rows - 1)


def _function(key: str) -> str:
    return key.split("[")[0].split("#")[0]


class Store:
    """The reference results of one test module: live, or read from ``tests/golden/<name>/``."""

    def __init__(self, name: str, live: bool):
        self.name, self.live = name, live
        self.path = os.path.join(GOLDEN, name)
        self.record_dir = os.environ.get("B200Q_RECORD_GOLDEN") if live else None
        self.recorded: dict[str, np.ndarray] = {}
        self.files: dict[str, _golden.Arrays] = {}

    def save(self) -> None:
        by_function: dict[str, dict[str, np.ndarray]] = {}
        for key, value in self.recorded.items():
            by_function.setdefault(_function(key), {})[key] = value
        if self.record_dir and by_function:
            os.makedirs(os.path.join(self.record_dir, self.name), exist_ok=True)
            for fn, entries in by_function.items():
                _golden.save(fn, entries, os.path.join(self.record_dir, self.name))

    def get(self, key: str) -> np.ndarray:
        fn = _function(key)
        if fn not in self.files:
            self.files[fn] = _golden.load(fn, self.path)
        assert key in self.files[fn], f"{key} is not in {self.path}: re-record it where the reference is available"
        return self.files[fn][key]


class RefResults:
    """One test's reference results.  Every call names the reference computation as a callable, which only runs
    where the reference's kernels are present."""

    def __init__(self, store: Store, test_id: str):
        self.store, self.test_id, self.n = store, test_id, 0

    def _key(self) -> str:
        self.n += 1
        return f"{self.test_id}#{self.n}"

    def bits(self, got: torch.Tensor, ref_fn, zero_sign: bool = False) -> torch.Tensor:
        """The reference output to compare ``got`` with bit for bit.  Without the live reference, ``got`` must hash
        to the stored digest; it is then returned, so that the caller's own comparison holds trivially."""
        key = self._key()
        if self.store.live:
            ref = ref_fn()
            if self.store.record_dir:
                self.store.recorded[key] = np.array(digest(ref, zero_sign))
            return ref
        want = str(self.store.get(key))
        assert digest(got, zero_sign) == want, f"{key}: differs from the reference output stored in {self.store.path}"
        return got

    def array(self, ref_fn) -> np.ndarray:
        """A small reference result stored whole (names, counts): ``ref_fn()`` returns it as a NumPy array."""
        key = self._key()
        if self.store.live:
            ref = ref_fn()
            if self.store.record_dir:
                self.store.recorded[key] = ref
            return ref
        return self.store.get(key)

    def rows(self, got: torch.Tensor, ref_fn, whole: bool = False) -> tuple[torch.Tensor, torch.Tensor]:
        """(reference, got) for a mismatch count: the whole outputs when the reference runs live, else the stored
        rows of the reference's output (viewed as [-1, last dim]; all of them with ``whole``, see ``sample_rows``)
        and the same rows of ``got``."""
        key = self._key()
        if self.store.live:
            ref = ref_fn()
            if self.store.record_dir:
                r2 = ref.detach().reshape(-1, ref.shape[-1]) if ref.dim() > 1 else ref.detach().reshape(1, -1)
                idx = torch.from_numpy(sample_rows(tuple(r2.shape), whole)).to(r2.device)
                self.store.recorded[key] = r2[idx].cpu().view(torch.int16 if ref.element_size() == 2 else ref.dtype) \
                    .numpy().view(_NATIVE[ref.dtype])
                self.store.recorded[key + "/dtype"] = np.array(str(ref.dtype))
            return ref, got
        data = self.store.get(key)
        dtype = {str(d): d for d in _NATIVE}[str(self.store.get(key + "/dtype"))]
        ref = torch.from_numpy(data.view(np.int16) if data.dtype == np.uint16 else data).view(dtype).to(got.device)
        g2 = got.reshape(-1, got.shape[-1]) if got.dim() > 1 else got.reshape(1, -1)
        idx = torch.from_numpy(sample_rows(tuple(g2.shape), whole)).to(got.device)
        assert ref.shape == (len(idx), g2.shape[1]), (key, tuple(ref.shape), tuple(g2.shape))
        return ref, g2[idx]
