"""Recorded outputs of the reference's own code (the libraries under oracle/_ref/) for the inputs the tests give it.

oracle/_ref/ can only be built where the reference source tree is present.  Everywhere else the ref_* entry points of the
binding answer from tests/golden/ref_calls.json.gz: what the compiled reference sources returned for exactly the same call,
looked up by a SHA-256 of the entry point's name and all of its arguments.  A call whose arguments were never recorded
raises, so a comparison with the reference runs against the reference's real output or fails; it never passes vacuously.

Scalars and small arrays are stored whole.  A larger array is stored as its fingerprint (dtype, shape, SHA-256 of the bytes)
and comes back as a `Digest`, which supports what the tests do with a reference output they compare against:
`a.tobytes() == d.tobytes()`, `np.array_equal(a, d)`, `len(d)`, `.shape`, `.dtype`, and use as an argument of another
reference call.  Anything else raises; a test that needs more of an output records what it needs with call(..., full=True).

Recording: with the libraries built, run the tests with PLSLAM_REF_RECORD=<file.json.gz>; every live reference call of the
run is added to that file (existing entries kept) when the process exits.
"""
import atexit
import base64
import functools
import gzip
import hashlib
import inspect
import json
import os
import numpy as np
from numpy.lib.format import descr_to_dtype, dtype_to_descr

_HERE = os.path.dirname(os.path.abspath(__file__))
STORE = os.path.join(os.path.dirname(_HERE), "tests", "golden", "ref_calls.json.gz")
FULL_BYTES = 1024         # arrays up to this size are stored whole
_store = None
_recorded = {}
_depth = 0                # > 0 inside a live call: a call made by another one is not recorded on its own


def _descr(dt):
    return json.loads(json.dumps(dtype_to_descr(dt)))


def _dtype(descr):
    return descr_to_dtype(descr if isinstance(descr, str) else [tuple(f) for f in descr])


def fingerprint(a):
    """(dtype descr, shape, SHA-256 of the C-order bytes) of an array or a Digest."""
    if isinstance(a, Digest):
        return a.fp
    a = np.asarray(a)
    return (_descr(a.dtype), list(a.shape), hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())


class _DigestBytes:
    def __init__(self, sha):
        self.sha = sha

    def __eq__(self, other):
        return isinstance(other, (bytes, bytearray)) and hashlib.sha256(other).hexdigest() == self.sha

    def __ne__(self, other):
        return not self == other


class Digest:
    """A recorded reference output array known by its fingerprint only."""

    def __init__(self, fp):
        self.fp = (fp[0], list(fp[1]), fp[2])
        self.dtype, self.shape = _dtype(fp[0]), tuple(fp[1])

    def __len__(self):
        return self.shape[0]

    def tobytes(self):
        return _DigestBytes(self.fp[2])

    def equals(self, other):
        o = np.asarray(other)
        if o.shape != self.shape:
            return False
        if o.dtype != self.dtype:
            cast = o.astype(self.dtype)
            if not np.array_equal(cast, o):
                return False
            o = cast
        return fingerprint(o) == self.fp

    def __array_function__(self, func, types, args, kwargs):
        if func is np.array_equal and len(args) == 2 and not kwargs:
            a, b = args
            return b.equals(a) if isinstance(b, Digest) and not isinstance(a, Digest) else \
                a.equals(b) if not isinstance(b, Digest) else a.fp == b.fp
        raise TypeError(f"a recorded reference output is known by its fingerprint only; {func.__name__} needs the data "
                        "(record it with call(..., full=True))")

    def __repr__(self):
        return f"Digest({self.dtype}, {self.shape}, {self.fp[2][:12]})"


def digest(name, *values):
    """SHA-256 over an entry point's name and argument values (arrays by fingerprint)."""
    h = hashlib.sha256(name.encode())
    for v in values:
        _feed(h, v)
    return h.hexdigest()[:32]


def _feed(h, x):
    if isinstance(x, (np.ndarray, np.generic, Digest)):
        h.update(b"a" + json.dumps(fingerprint(x)).encode())
    elif isinstance(x, (tuple, list)):
        h.update(b"t%d" % len(x))
        for e in x:
            _feed(h, e)
    elif isinstance(x, dict):
        h.update(b"d%d" % len(x))
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    elif x is None or isinstance(x, (bool, int, float, str)):
        h.update(b"s" + repr(x).encode())
    else:
        raise TypeError(f"cannot key a reference call on a {type(x).__name__}")


def _encode(x, full):
    if isinstance(x, (np.ndarray, np.generic)):
        a = np.asarray(x)
        if full or a.nbytes <= FULL_BYTES:
            tag = "g" if isinstance(x, np.generic) else "a"
            return {tag: [_descr(a.dtype), list(a.shape), base64.b64encode(np.ascontiguousarray(a).tobytes()).decode()]}
        return {"h": list(fingerprint(a))}
    if isinstance(x, tuple):
        return {"t": [_encode(e, full) for e in x]}
    if isinstance(x, dict):
        return {"d": [[k, _encode(e, full)] for k, e in x.items()]}
    if isinstance(x, (bool, int, float)):
        return {"p": x}
    raise TypeError(f"cannot record a {type(x).__name__}")


def _decode(e):
    (tag, v), = e.items()
    if tag in ("a", "g"):
        a = np.frombuffer(base64.b64decode(v[2]), _dtype(v[0])).reshape(v[1]).copy()
        return a[()] if tag == "g" else a
    if tag == "h":
        return Digest(v)
    if tag == "t":
        return tuple(_decode(x) for x in v)
    if tag == "d":
        return {k: _decode(x) for k, x in v}
    return v


def _read(path):
    if not os.path.exists(path):
        return {}
    with gzip.open(path, "rt") as f:
        return json.load(f)


def call(name, key_values, live, fn, full=False):
    """fn() when the reference library is built (`live`), else the recorded output of the call keyed by name + key_values.
    full=True: record the output's arrays whole (for a test that computes with them)."""
    global _store, _depth
    key = digest(name, *key_values)
    if live:
        _depth += 1
        try:
            out = fn()
        finally:
            _depth -= 1
        if os.environ.get("PLSLAM_REF_RECORD") and _depth == 0:
            _recorded[key] = _encode(out, full)
        return out
    if _store is None:
        _store = _read(STORE)
    if key not in _store:
        raise LookupError(f"no recorded reference output of {name} for these arguments (key {key}) in {STORE}: build oracle/_ref "
                          "where the reference tree exists and record the call with PLSLAM_REF_RECORD")
    return _decode(_store[key])


def entry(name, live, ref_only=False):
    """Decorator for a binding function that reaches the reference's code: always (`ref_only`) or when called with impl="ref"."""
    def wrap(f):
        sig = inspect.signature(f)

        @functools.wraps(f)
        def g(*args, **kw):
            b = sig.bind(*args, **kw)
            b.apply_defaults()
            if not ref_only and b.arguments.get("impl") != "ref":
                return f(*args, **kw)
            return call(name, [sorted(b.arguments.items())], live(), lambda: f(*args, **kw))
        return g
    return wrap


@atexit.register
def _write():
    path = os.environ.get("PLSLAM_REF_RECORD")
    if not path or not _recorded:
        return
    data = _read(path)
    data.update(_recorded)
    with gzip.GzipFile(path, "wb", mtime=0) as f:
        f.write(json.dumps(data, sort_keys=True, separators=(",", ":")).encode())
