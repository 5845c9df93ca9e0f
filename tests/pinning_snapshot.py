"""A snapshot of the restatement's answers to the questions tests/test_oracle_pinning.py asks the reference.

test_oracle_pinning.py pins the plain-C restatement (oracle/fm_oracle.c) against the reference's own headers compiled
unmodified (oracle/_ref).  That build needs the reference's sources, which the repository does not carry, so where it is
absent the `ref` fixture answers from tests/golden/pinning_port_snapshot.json.gz instead: the RESTATEMENT's answers to
the same calls, recorded by tests/golden/record_pinning_snapshot.py.  Those tests are then a regression check of the
restatement against its own recorded behaviour, not a comparison with the reference; the restatement is compared with
reference-generated data on every machine by tests/test_golden.py (tests/golden/fm_golden.npz).

A test's answers are stored in call order under its node id, with a digest of its whole call sequence (method and
arguments), so a test whose inputs changed fails instead of comparing against answers to other questions.  Answers the
tests compare within a tolerance (`tolerance_compared`) are stored as values; other arrays of more than SMALL elements
are compared bit for bit with `same` and stored as the SHA-256 of their dtype, shape and bytes.
"""
import gzip
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pinning_port_snapshot.json.gz")
SMALL = 64

RECORD_FROM = None          # set by record_pinning_snapshot.py to an oracle: the `ref` fixture then records its answers into RECORDED
RECORDED = {}
_records = None


def tolerance_compared(name, args):
    """calls whose answers test_oracle_pinning.py compares with relerr: predict, and training with the coordinate solvers"""
    from oracle import oracle as O
    return name == "predict" or (name == "train" and args[0].solver in (O.ALS, O.MCMC))


class Digest:
    """an array known by the SHA-256 of its dtype, shape and bytes"""

    def __init__(self, dtype, shape, sha256):
        self.dtype, self.shape, self.sha256 = dtype, tuple(shape), sha256

    @staticmethod
    def of(a):
        a = np.ascontiguousarray(a)
        h = hashlib.sha256()
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
        return h.hexdigest()

    def matches(self, a):
        a = np.asarray(a)
        return a.dtype.str == self.dtype and a.shape == self.shape and Digest.of(a) == self.sha256

    def __repr__(self):
        return "Digest(%s, %s, %s)" % (self.dtype, self.shape, self.sha256[:16])


def same(a, b, equal_nan=False):
    """a equals b element for element; b may be a recorded Digest"""
    if isinstance(b, Digest):
        return b.matches(a)
    return np.array_equal(a, b, equal_nan=equal_nan)


def _canon(x, h):
    """feed an argument into the call-sequence digest"""
    if isinstance(x, np.ndarray):
        h.update(b"A"); h.update(Digest.of(x).encode())
    elif isinstance(x, (list, tuple)):
        h.update(b"L%d" % len(x))
        for e in x:
            _canon(e, h)
    elif isinstance(x, dict):
        h.update(b"D%d" % len(x))
        for k in sorted(x):
            h.update(k.encode()); _canon(x[k], h)
    elif hasattr(x, "_fields_"):                                   # ctypes structure (oracle.Cfg)
        _canon({f[0]: getattr(x, f[0]) for f in x._fields_}, h)
    elif isinstance(x, (bool, np.bool_)):
        h.update(b"B%d" % bool(x))
    elif isinstance(x, (int, np.integer)):
        h.update(b"I%d" % int(x))
    elif isinstance(x, (float, np.floating)):
        h.update(b"F" + float(x).hex().encode())
    elif x is None:
        h.update(b"N")
    else:
        raise TypeError("cannot digest argument of type %s" % type(x))


def _encode(r, values):
    if isinstance(r, np.ndarray):
        if values or r.size <= SMALL:
            return {"array": r.tolist(), "dtype": r.dtype.str, "shape": list(r.shape)}
        return {"digest": Digest.of(r), "dtype": r.dtype.str, "shape": list(r.shape)}
    if isinstance(r, tuple):
        return {"tuple": [_encode(e, values) for e in r]}
    if isinstance(r, list):
        return [_encode(e, values) for e in r]
    if isinstance(r, dict):
        return {"dict": {k: _encode(v, values) for k, v in r.items()}}
    if isinstance(r, (bool, np.bool_)):
        return bool(r)
    if isinstance(r, (int, np.integer)):
        return int(r)
    if isinstance(r, (float, np.floating)):
        return float(r)
    if r is None:
        return None
    raise TypeError("cannot record a result of type %s" % type(r))


def _decode(r):
    if isinstance(r, list):
        return [_decode(e) for e in r]
    if isinstance(r, dict):
        if "array" in r:
            return np.array(r["array"], dtype=np.dtype(r["dtype"])).reshape(r["shape"])
        if "digest" in r:
            return Digest(r["dtype"], r["shape"], r["digest"])
        if "tuple" in r:
            return tuple(_decode(e) for e in r["tuple"])
        return {k: _decode(v) for k, v in r["dict"].items()}
    return r


class _Calls:
    def __init__(self, test_id):
        self.test_id = test_id
        self.h = hashlib.sha256()
        self.n = 0

    def _digest_call(self, name, args, kwargs):
        self.h.update(name.encode())
        _canon(list(args), self.h)
        _canon(dict(kwargs), self.h)
        self.n += 1

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return lambda *args, **kwargs: self._call(name, args, kwargs)


class Recorder(_Calls):
    """forwards every call to a live oracle and keeps its answers for `save`"""

    def __init__(self, oracle, test_id, into):
        super().__init__(test_id)
        self.oracle = oracle
        self.results = []
        into[test_id] = self

    def _call(self, name, args, kwargs):
        self._digest_call(name, args, kwargs)
        r = getattr(self.oracle, name)(*args, **kwargs)
        self.results.append(_encode(r, tolerance_compared(name, args)))
        return r


def save(recorders, path=PATH):
    data = {tid: {"calls": rec.h.hexdigest(), "results": rec.results} for tid, rec in sorted(recorders.items())}
    with gzip.open(path, "wt") as f:
        json.dump(data, f, separators=(",", ":"))


class Replay(_Calls):
    """answers each call with the recorded answer at its position in the test's call sequence"""

    def __init__(self, test_id):
        global _records
        super().__init__(test_id)
        if _records is None:
            with gzip.open(PATH, "rt") as f:
                _records = json.load(f)
        assert test_id in _records, "no recorded answers for %s (tests/golden/record_pinning_snapshot.py)" % test_id
        self.rec = _records[test_id]

    def _call(self, name, args, kwargs):
        self._digest_call(name, args, kwargs)
        assert self.n <= len(self.rec["results"]), "%s makes more calls than were recorded" % self.test_id
        return _decode(self.rec["results"][self.n - 1])

    def finish(self):
        """the test asked exactly the recorded questions"""
        assert self.n == len(self.rec["results"]) and self.h.hexdigest() == self.rec["calls"], (
            "%s asked other questions than were recorded (tests/golden/record_pinning_snapshot.py)" % self.test_id)
