"""Stored outputs of the reference's own compute shaders (tests/golden/refshaders.json, tests/golden/refshaders_libm.npz).

The reference project is not part of this repository.  tests/golden/make_refshaders_golden.py runs its six shaders on the CPU
(oracle/refshaders.py) for every case the tests check and keeps, per output array, a SHA-256 digest of dtype, shape and bytes:
two arrays have the same digest exactly when they are bit-identical.  The tests recompute each case with the oracle or libgsr
and compare digests, so every comparison with the reference stays bit for bit without its sources or its 67 MB asset.
"""
from __future__ import annotations

import functools
import hashlib
import json
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
JSON_PATH = os.path.join(GOLDEN_DIR, "refshaders.json")
LIBM_PATH = os.path.join(GOLDEN_DIR, "refshaders_libm.npz")
LIBM_STEP = 2.0 ** -24   # refshaders_libm.npz holds (libm frame - reference frame) in these steps; the rounding error is <= 3e-8


def digest(a) -> str:
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def bits(a) -> np.ndarray:
    return np.ascontiguousarray(a).view(np.uint32)


def frame_record(fr) -> dict:
    """What the golden file keeps of one oracle.refshaders.ReferenceFrame."""
    vis = np.unique(fr.values)
    rec = {k: digest(getattr(fr, k)) for k in ("keys_unsorted", "values_unsorted", "keys", "values", "bounds", "rgba")}
    rec.update(duplicates=int(fr.duplicates), records=digest(fr.records[vis]), grid_dims=[int(x) for x in fr.grid_dims],
               pick=[int(x) for x in bits(fr.pick)])
    return rec


@functools.lru_cache(maxsize=None)
def _load() -> dict:
    with open(JSON_PATH) as f:
        return json.load(f)


def golden(case: str) -> dict:
    return _load()[case]


def libm_delta() -> np.ndarray:
    """(H, W, 3) int8: the RGB of the reference frame with glibc expf/powf minus the default reference frame, in LIBM_STEP."""
    with np.load(LIBM_PATH) as g:
        return g["delta_rgb"]
