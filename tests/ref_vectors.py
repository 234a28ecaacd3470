"""Stored outputs of the reference's own code (tests/golden/ref_*.npz), for the tests that pin the oracle to it.

tests/golden/make_ref_vectors.py calls the functions compiled from Open3D's headers (oracle/_ref/libo3dref.so, see
oracle/ref_shim) on the same inputs the tests build, and writes what they returned.  An array of at most FULL_LIMIT
elements is stored verbatim; a larger one as its SHA-256 (over dtype, shape and bytes), so the comparison stays
bit-exact, plus a fixed sample of its elements that makes a mismatch readable.  NaNs are compared as NaN, whatever
their payload."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FULL_LIMIT = 1 << 12
SAMPLE = 64


def _canon(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f" and np.isnan(a).any():
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a)
    return a


def digest(a):
    a = _canon(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def pack(out, name, a):
    """Adds array `a` to the dict `out` that make_ref_vectors.py saves."""
    a = _canon(a)
    if a.size <= FULL_LIMIT:
        out[name] = a
        return
    idx = np.sort(np.random.default_rng(a.size).choice(a.size, SAMPLE, replace=False))
    out[name + ".sha256"] = np.array(digest(a))
    out[name + ".index"] = idx
    out[name + ".sample"] = a.reshape(-1)[idx]


class Vectors:
    def __init__(self, module):
        path = os.path.join(GOLDEN, f"ref_{module}.npz")
        with np.load(path) as z:
            self.z = {k: z[k] for k in z.files}

    def __getitem__(self, name):
        return self.z[name]

    def check(self, name, got):
        """Asserts that `got` has the stored array's dtype, shape and bytes."""
        got = _canon(got)
        if name in self.z:
            want = self.z[name]
            assert got.dtype == want.dtype and got.shape == want.shape, (name, got.dtype, got.shape, want.dtype, want.shape)
            bad = got.reshape(-1).view(np.uint8) != want.reshape(-1).view(np.uint8)
            assert not bad.any(), (name, f"{int(bad.sum())} bytes differ")
            return
        if digest(got) == str(self.z[name + ".sha256"]):
            return
        idx, want = self.z[name + ".index"], self.z[name + ".sample"]
        flat = got.reshape(-1)
        differ = None
        if flat.size > idx[-1] and flat.dtype == want.dtype:
            differ = int((_canon(flat[idx]).view(np.uint8) != want.view(np.uint8)).sum())
        raise AssertionError(f"{name}: {got.dtype}{got.shape} differs from the reference; "
                             f"{differ} bytes differ in a {len(idx)}-element sample")
