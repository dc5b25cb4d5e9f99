"""Stored outputs of the reference's own code (its CPU routines and its CUDA kernels compiled for sm_100a), so that the
tests compare against them without that code.  tests/golden/make_golden_ref.py ran the reference and wrote, per case, the
digest of every output array; a test computes the digest of this repo's output for the same input and compares.

A digest is exact: equal digests mean the same dtype kind, the same shape and the same elements, as np.array_equal(...,
equal_nan=True) sees them (every NaN counts as one value, -0.0 as 0.0).  Outputs of several MB fit in a few bytes."""
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def digest(a) -> str:
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.asarray(a)
    if a.dtype.kind in "iu":
        a = a.astype(np.int64)
    elif a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a + 0.0).astype(a.dtype)        # one NaN, +0.0 for -0.0
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:16]


def load(name: str):
    with open(os.path.join(GOLD, name)) as f:
        return json.load(f)
