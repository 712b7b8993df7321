"""Outputs of the reference's own functions, recorded once and replayed, so that the differential tests against the
reference run on any machine.

A test asks for a reference output through a `Recorded` store with a key and a zero-argument function that computes it
with the reference.  When recording (`PNP_RECORD_REFERENCE=1` and the reference tree importable through
oracle/ref_shim.py) the function runs and its result is stored in tests/golden/reference_<name>.json.gz; otherwise the
function is never called and the stored result is used.  The file is gzip-compressed JSON (float64 values round-trip
exactly).  Record with

    PNP_RECORD_REFERENCE=1 python -m pytest tests/<module>.py

What is stored depends on the comparison, so that the fixtures stay small:
  * `value`: small outputs, stored whole and compared as the test compares them;
  * `equal`: a SHA-256 digest (64 bits of it) of the bytes with dtype and shape - bit-exact comparisons stay bit-exact;
  * `close`: for |mine - ref| <= atol on large arrays, a fixed seeded sample of elements (checked element by element)
    and three fixed integer-hash projections sum(x * w) over ALL elements (checked against atol * sum|w|, the bound
    the elementwise tolerance implies, plus the rounding of the sum); `rel` gives the relative L2 distance on the
    sample.
"""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import ref_shim

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_MULT = (2654435761, 2246822519, 3266489917)


def _np(x):
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(x))


def digest(x) -> str:
    a = _np(x)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:16]


def _projections(a):
    """(sum x w_j, sum |x w_j|, sum |w_j|) for the three weight vectors w_j[i] = hash_j(i) in [-0.5, 0.5)."""
    i = np.arange(1, a.size + 1, dtype=np.uint64)
    out = np.empty((3, 3))
    for j, m in enumerate(_MULT):
        w = ((i * np.uint64(m)) % np.uint64(1 << 32)).astype(np.float64) / 2.0 ** 32 - 0.5
        out[:, j] = (w * a).sum(), np.abs(w * a).sum(), np.abs(w).sum()
    return out


def _sample_index(n, k):
    return np.random.RandomState(n % (1 << 31)).randint(0, n, size=min(n, k))


def fingerprint(x, k):
    a = _np(x).astype(np.float64).ravel()
    p = _projections(a)
    return np.concatenate([[a.size], p[0], a[_sample_index(a.size, k)]]).tolist()


class Recorded:
    def __init__(self, name):
        self.path = os.path.join(GOLD, f"reference_{name}.json.gz")
        self.recording = os.environ.get("PNP_RECORD_REFERENCE") == "1"
        if self.recording and not ref_shim.available():
            raise RuntimeError("PNP_RECORD_REFERENCE=1 needs the reference tree (PNP_REFERENCE_ROOT)")
        self.data = {}
        if os.path.exists(self.path):
            with gzip.open(self.path, "rt") as f:
                self.data = json.load(f)

    def _get(self, key, fn, transform):
        if self.recording:
            self.data[key] = transform(fn())
        if key not in self.data:
            pytest.fail(f"{key} is not recorded in {self.path} (record with PNP_RECORD_REFERENCE=1)")
        return np.asarray(self.data[key])

    def value(self, key, fn):
        """The reference output itself (numpy; tensors are converted)."""
        return self._get(key, fn, lambda r: np.asarray(r.detach().cpu() if hasattr(r, "detach") else r).tolist())

    def equal(self, key, mine, fn) -> bool:
        """mine has the same dtype, shape and bits as the reference output."""
        return digest(mine) == str(self._get(key, fn, digest))

    def close(self, key, mine, fn, atol, k=4) -> bool:
        """|mine - ref| <= atol on the sample, and the projections over all elements agree to the same bound."""
        ref = self._get(key, fn, lambda r: fingerprint(r, k))
        m = _np(mine).astype(np.float64).ravel()
        if m.size != int(ref[0]):
            return False
        p = _projections(m)
        tol = atol * p[2] + 2e-12 * p[1]
        return bool(np.all(np.abs(p[0] - ref[1:4]) <= tol)
                    and np.all(np.abs(m[_sample_index(m.size, k)] - ref[4:]) <= atol))

    def rel(self, key, mine, fn, k=256) -> float:
        """Relative L2 distance of mine to the reference output on the stored sample of k elements."""
        ref = self._get(key, fn, lambda r: fingerprint(r, k))
        m = _np(mine).astype(np.float64).ravel()
        assert m.size == int(ref[0])
        s = m[_sample_index(m.size, k)]
        return float(np.linalg.norm(s - ref[4:]) / np.linalg.norm(ref[4:]))

    def save(self):
        if self.recording:
            with open(self.path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
                f.write(json.dumps(self.data, sort_keys=True).encode())


def recorded_fixture(name):
    """A module-scoped fixture yielding `Recorded(name)`, written back at the end of the module when recording."""

    @pytest.fixture(scope="module")
    def fixture():
        r = Recorded(name)
        yield r
        r.save()

    return fixture
