"""What the original implementation computed, for the tests that compare against it.

Where the compiled reference extensions and the reference's own Python are present (oracle/_ref, built by
oracle/build_ref.py), a test computes the reference's outputs live.  Elsewhere it reads what such a live run recorded in
tests/golden/reference/<name>.npz, so the comparison runs from a clean checkout too.  With GF_RECORD_REFERENCE=DIR set, every
live result is also written to DIR/<name>.npz (to be copied into tests/golden/reference/).

Small arrays are stored whole.  A larger one keeps a fixed, seeded sample of its rows (`rows(key)` says which; live it is every
row) and the SHA-256 of the whole array, so that bit-equality checks (`equal`) stay exact.  Floats are hashed with -0.0 folded
into +0.0, as torch.equal compares them.
"""
import atexit
import hashlib
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
SAMPLE_BYTES = 4096            # per stored float array; integer arrays compress well and are stored whole
_RECORD = os.environ.get("GF_RECORD_REFERENCE")
_pending = []


def _np(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.asarray(a)
    return np.ascontiguousarray(a) if a.ndim else a


def digest(a):
    a = _np(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)                    # -0.0 -> +0.0
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


class Reference:
    """Outputs of the reference for one test case: `live` when oracle/_ref is there, else the stored golden."""

    def __init__(self, name, live):
        self.name, self.live, self._a, self._keep = name, bool(live), {}, {}
        if self.live:
            if _RECORD:
                _pending.append(self)
            return
        path = os.path.join(GOLDEN, name + ".npz")
        if not os.path.exists(path):
            pytest.fail(f"{path} missing: record it with GF_RECORD_REFERENCE=DIR where oracle/_ref is built")
        with np.load(path) as z:
            self._a = {k: z[k] for k in z.files}

    def put(self, key, value, rows=None):
        """Record a live reference output (a tensor, array, or list of tuples such as a loop trace).  `rows` picks the rows a
        sampled golden keeps instead of a seeded uniform sample; "digest" keeps only the hash (for `equal` checks)."""
        assert self.live
        self._a[key] = value if isinstance(value, list) else _np(value)
        if rows is not None:
            self._keep[key] = rows

    def __getitem__(self, key):
        v = self._a[key]
        if key + "@trace" in self._a:
            return [tuple(int(x) for x in t) for t in v.tolist()]
        return v

    def __contains__(self, key):
        return key in self._a

    def rows(self, key):
        """Row indices of `self[key]` within the full array (a slice over every row when live or stored whole)."""
        r = self._a.get(key + "@rows")
        return slice(None) if r is None else r

    def equal(self, key, ours):
        """Bitwise equality of `ours` with the reference's full array."""
        if self.live or key + "@sha256" not in self._a:
            return digest(ours) == digest(self._a[key])
        return digest(ours) == str(self._a[key + "@sha256"])

    def save(self, directory):
        out = {}
        for k, v in self._a.items():
            if isinstance(v, list):
                out[k] = np.asarray(v, np.int64).reshape(len(v), 2)
                out[k + "@trace"] = np.zeros(0)
                continue
            out[k + "@sha256"] = np.asarray(digest(v))
            keep = self._keep.get(k)
            if isinstance(keep, str):
                continue
            if keep is not None:
                rows = np.unique(np.asarray(keep, np.int32))
                out[k], out[k + "@rows"] = v[rows], rows
            elif v.dtype.kind == "f" and v.nbytes > SAMPLE_BYTES and v.ndim >= 1:
                n = v.shape[0]
                keep = max(1, min(n, SAMPLE_BYTES * n // v.nbytes))
                rows = np.sort(np.random.RandomState(0).choice(n, keep, replace=False)).astype(np.int32)
                out[k], out[k + "@rows"] = v[rows], rows
            else:
                out[k] = v
        os.makedirs(directory, exist_ok=True)
        np.savez_compressed(os.path.join(directory, self.name + ".npz"), **out)


@atexit.register
def _write_recorded():
    for r in _pending:
        r.save(_RECORD)
