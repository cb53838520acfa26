"""Stored outputs of the reference's own CUDA kernels (oracle/_ref), so that the GPU tests compare against the reference
on every machine, including one where oracle/_ref cannot be built.

Every comparison has a key: the test's name with its parameters, plus a label.  What is stored per key:
  equal()   the SHA-256 of the reference output (after -0.0 -> 0.0 and one NaN pattern), its shape and dtype: the
            test's output must hash the same, i.e. be bit-identical as torch.equal would say;
  sample()  a fixed, seeded sample of a large floating-point output and its largest magnitude, for comparisons within
            a tolerance.
The stored values are always checked; where oracle/_ref is built, the live reference kernels are compared as well.

Recording (a GPU machine with oracle/_ref built):  PRB_RECORD_REFERENCE=/path/out.npz python -m pytest -m gpu tests
writes every key the run visits; the file goes to tests/golden/reference_gpu.npz.
"""
import atexit
import hashlib
import os
import re

import numpy as np

from oracle import refgpu as R

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_gpu.npz")
RECORD = os.environ.get("PRB_RECORD_REFERENCE")
_golden = None
_recorded = {}


def live():
    """the reference kernels can be run here"""
    return R.available()


def _key(label):
    node = os.environ.get("PYTEST_CURRENT_TEST", "").rsplit(" (", 1)[0].rsplit("/", 1)[-1]
    return re.sub(r"[^A-Za-z0-9_.=+-]", "_", node + "__" + label)


def _np(x):
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(x)


def _canon(a):
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)                 # -0.0 -> 0.0
        a[np.isnan(a)] = np.nan
    return a


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = _canon(_np(a))
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _stored(key, field):
    global _golden
    if _golden is None:
        _golden = dict(np.load(GOLDEN)) if os.path.exists(GOLDEN) else {}
    name = key + "." + field
    assert name in _golden, "no stored reference output %r in %s (record it: see tests/refstore.py)" % (name, GOLDEN)
    return _golden[name]


def _record(key, **fields):
    assert live(), "recording needs oracle/_ref"
    for f, v in fields.items():
        _recorded[key + "." + f] = np.asarray(v)


def equal(label, ours, reference, msg="differs from the reference kernel"):
    """ours == the reference output bit for bit; reference: callable returning the live output"""
    key, a = _key(label), _np(ours)
    if live() or RECORD:
        ref = _np(reference())
        if RECORD:
            _record(key, sha256=digest(ref.astype(a.dtype)), shape=np.array(ref.shape, np.int64))
        assert ref.shape == a.shape and np.array_equal(a, ref), "%s (%s)" % (msg, label)
    if not RECORD:
        assert tuple(_stored(key, "shape")) == a.shape, "%s: shape %s (%s)" % (msg, a.shape, label)
        assert digest(a) == str(_stored(key, "sha256")), "%s: stored reference output (%s)" % (msg, label)


def sample(label, reference, n=8192, seed=0):
    """(flat indices, values, max |value|) of a seeded sample of n elements of a large reference output"""
    key = _key(label)
    if RECORD:
        assert live(), "recording needs oracle/_ref"
        ref = _np(reference())
        idx = np.sort(np.random.default_rng(seed).choice(ref.size, min(n, ref.size), replace=False))
        _record(key, index=idx, value=ref.reshape(-1)[idx], absmax=np.abs(ref).max())
    return _stored_or_recorded(key, "index"), _stored_or_recorded(key, "value"), float(_stored_or_recorded(key, "absmax"))


def _stored_or_recorded(key, field):
    return _recorded[key + "." + field] if RECORD else _stored(key, field)


@atexit.register
def _write():
    if RECORD and _recorded:
        np.savez_compressed(RECORD, **_recorded)
