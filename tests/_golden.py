"""The fixture files under ``tests/golden``: a set of arrays saved as ``<name>.<part>.npz``, split so that no file
goes over 1 MB (each part holds at most PART_BYTES of raw array data).  ``oracle/gen_golden.py`` writes them with
``save``; the tests read them back as one mapping with ``load``."""

from __future__ import annotations

import glob
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PART_BYTES = 900 << 10


class Arrays(dict):
    """name -> array, with the ``files`` listing of ``np.load``'s NpzFile."""

    @property
    def files(self) -> list[str]:
        return list(self)


def save(name: str, arrays: dict, out_dir: str = GOLDEN) -> list[str]:
    for old in glob.glob(os.path.join(out_dir, f"{name}.*.npz")):
        os.remove(old)
    parts, part, size = [], {}, 0
    for key, value in arrays.items():
        value = np.asarray(value)
        if part and size + value.nbytes > PART_BYTES:
            parts.append(part)
            part, size = {}, 0
        part[key] = value
        size += value.nbytes
    parts.append(part)
    paths = []
    for i, p in enumerate(parts):
        paths.append(os.path.join(out_dir, f"{name}.{i}.npz"))
        np.savez_compressed(paths[-1], **p)
    return paths


def load(name: str, in_dir: str = GOLDEN) -> Arrays:
    paths = sorted(glob.glob(os.path.join(in_dir, f"{name}.*.npz")), key=lambda p: int(p.rsplit(".", 2)[1]))
    if not paths:
        raise FileNotFoundError(os.path.join(in_dir, f"{name}.*.npz"))
    out = Arrays()
    for p in paths:
        with np.load(p) as z:
            out.update({k: z[k] for k in z.files})
    return out
