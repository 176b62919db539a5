"""Stored outputs of the original SceneLib2 sources for the tests that compare against them.

A test asks for every reference result through `take(key, fn)`.  Normally the value comes from
tests/golden/ref_<name>.npz, in call order, and every stored value has to be used by the end of the
test.  With SL2_RECORD_REFERENCE=1 and oracle/_ref built from a SceneLib2 checkout (see
oracle/Makefile), `fn` runs the original code and the file is rewritten:

    SL2_RECORD_REFERENCE=1 python -m pytest tests/test_oracle_ref.py

The inputs are not stored: the tests generate them from fixed seeds, as when they were recorded.
Large outputs are kept in part: `cov_sample` keeps a covariance matrix's diagonal, its largest
asymmetry and a fixed, seeded sample of entries; `pick` keeps a seeded sample of an array's entries
(seeded by the case, so that over all cases every entry is compared); `digest` keeps the SHA-256 of
a value the test compares bit for bit.
"""
import hashlib
import os

import numpy as np

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RECORD = os.environ.get("SL2_RECORD_REFERENCE") == "1"
COV_SAMPLE = 64


def cov_index(n):
    """Flat indices (row-major) of the covariance entries kept for an n x n matrix."""
    rng = np.random.default_rng(1000 + n)
    return np.sort(rng.choice(n * n, size=min(n * n, COV_SAMPLE), replace=False))


def pick(a, seed, k):
    """k entries of `a` (flattened), chosen by `seed`; all of them when a has at most k."""
    a = np.asarray(a).reshape(-1)
    if a.size <= k:
        return a
    return a[np.sort(np.random.default_rng(seed).choice(a.size, k, replace=False))]


def digest(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def cov_sample(P):
    P = np.asarray(P)
    return dict(diag=np.diag(P).copy(), entries=P.reshape(-1)[cov_index(P.shape[0])],
                asym=np.abs(P - P.T).max())


def assert_cov_close(P, ref, rtol, d=None):
    """P (full, n x n) against a cov_sample of the reference, relative to sqrt(P_ii P_jj)."""
    n = P.shape[0]
    d = np.sqrt(np.abs(ref["diag"])) + 1e-300 if d is None else d
    i, j = np.divmod(cov_index(n), n)
    assert ref["entries"].shape == i.shape
    assert (np.abs(np.diag(P) - ref["diag"]) <= rtol * d * d).all()
    assert (np.abs(P.reshape(-1)[i * n + j] - ref["entries"]) <= rtol * d[i] * d[j]).all()


def _leaves(v):
    if isinstance(v, dict):
        return v
    if isinstance(v, (tuple, list)):
        return {str(k): x for k, x in enumerate(v)}
    return {"": v}


class Recording:
    def __init__(self, name, oracle=None, strict=True, record=RECORD):
        self.path = os.path.join(G, "ref_%s.npz" % name)
        self.strict = strict
        self.recording = record
        self._rec, self._pos, self._calls = {}, {}, {}
        if self.recording:
            assert oracle is not None and oracle.ref() is not None and oracle.ref_models() is not None, \
                "recording needs oracle/_ref built from the SceneLib2 sources"
            return
        with np.load(self.path) as z:
            data = {k: z[k] for k in z.files}
        for k in sorted({m.split("/")[0] for m in data}):
            self._calls[k] = self._decode(k, data)

    @staticmethod
    def _decode(key, data):
        none = data[key + "/none"]
        kind = str(data[key + "/kind"])
        fields = [m[len(key) + 2:-6] for m in data if m.startswith(key + "/:") and m.endswith(".shape")]
        cols = {}
        for f in fields:
            flat, shapes = data["%s/:%s" % (key, f)], data["%s/:%s.shape" % (key, f)]
            vals, o = [], 0
            for s in shapes:
                size = int(np.prod(s))
                a = flat[o:o + size].reshape(tuple(s))
                vals.append(a.item() if a.ndim == 0 else a)
                o += size
            cols[f] = vals
        out, k = [], 0
        for isnone in none:
            if isnone:
                out.append(None)
                continue
            v = {f: cols[f][k] for f in fields}
            k += 1
            if kind == "tuple":
                v = tuple(v[str(i)] for i in range(len(v)))
            elif kind == "value":
                v = v[""]
            out.append(v)
        return out

    def take(self, key, fn):
        """The reference's value for the next call under `key`: fn() when recording, else the stored one."""
        assert "/" not in key
        if self.recording:
            v = fn()
            self._rec.setdefault(key, []).append(v)
            return v
        i = self._pos.get(key, 0)
        calls = self._calls.get(key, [])
        assert i < len(calls), "%s: no stored reference value #%d for %r" % (self.path, i, key)
        self._pos[key] = i + 1
        return calls[i]

    def close(self):
        if not self.recording:
            if self.strict:
                for k, calls in self._calls.items():
                    assert self._pos.get(k, 0) == len(calls), "%s: %r used %d of %d stored values" % (
                        self.path, k, self._pos.get(k, 0), len(calls))
            return
        out = {}
        for key, calls in self._rec.items():
            real = [v for v in calls if v is not None]
            first = real[0] if real else None
            kind = "dict" if isinstance(first, dict) else "tuple" if isinstance(first, (tuple, list)) else "value"
            out[key + "/none"] = np.array([v is None for v in calls])
            out[key + "/kind"] = np.array(kind)
            leaves = [_leaves(v) for v in real]
            for f in (leaves[0] if leaves else {}):
                arrs = [np.asarray(lv[f]) for lv in leaves]
                out["%s/:%s" % (key, f)] = np.concatenate([a.reshape(-1) for a in arrs])
                out["%s/:%s.shape" % (key, f)] = np.array([a.shape for a in arrs], np.int32).reshape(len(arrs), arrs[0].ndim)
        np.savez_compressed(self.path, **out)
