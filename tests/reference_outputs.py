"""What the reference's own code returned in the tests that compare with it, stored so that those comparisons run without it.

The reference pieces (oracle/_ref/, compiled from the original project's sources by `make -C oracle ref`) exist only where those sources
are present.  The tests reach them through Recorded: by default a call returns the stored output of the same call (same test, same
position in it), and once the test has made all its recorded calls, a digest of every input it passed is checked against the digest of
the inputs the reference was given, so a stored answer is never compared with a question that changed.  An array larger than a few
numbers is stored as a 64-bit fingerprint of its bytes (one per field of a record array), which same() compares with what the oracle
computed: the comparisons stay bit for bit and the files stay small.  Arrays that a test reads rather than compares are kept whole:
those of the tests and result keys named in keep=, or every array with keep=ALL.  With CCM_RECORD_REFERENCE=1
(and oracle/_ref built) the reference itself runs and tests/golden/reference/<test module>.npz is rewritten for the tests that ran:

    CCM_RECORD_REFERENCE=1 python -m pytest tests/test_oracle_vs_reference_orb.py
"""
from __future__ import annotations

import atexit
import hashlib
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD = os.environ.get("CCM_RECORD_REFERENCE") == "1"


SMALL = 24        # bytes: arrays up to this size are stored as they are
ALL = "all"


def _fingerprint(a):
    fp = lambda x: hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest()[:8]
    return b"".join(fp(a[f]) for f in a.dtype.names) if a.dtype.names else fp(a)


class Stored:
    """an output of the reference kept as its fingerprint: shape, dtype, len() and fields, compared through same()"""

    def __init__(self, dtype, shape, fp):
        self.dtype, self.shape, self.fp = dtype, tuple(shape), fp

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, field):
        i = self.dtype.names.index(field)
        return Stored(self.dtype[field], self.shape, self.fp[8 * i:8 * i + 8])


def same(a, b):
    """np.array_equal(a, b) where either side may be a Stored output of the reference"""
    if isinstance(a, Stored):
        a, b = b, a
    if isinstance(a, Stored):
        return (a.dtype, a.shape, a.fp) == (b.dtype, b.shape, b.fp)
    if not isinstance(b, Stored):
        return np.array_equal(a, b)
    a = np.asarray(a)
    if a.shape != b.shape or (a.dtype.names or None) != (b.dtype.names or None):
        return False
    if not a.dtype.names and not np.array_equal(a.astype(b.dtype), a):
        return False
    return _fingerprint(np.ascontiguousarray(a, b.dtype)) == b.fp


def _digest(h, x):
    if isinstance(x, Stored):
        h.update(b"a" + x.dtype.str.encode() + repr(x.shape).encode() + x.fp)
    elif isinstance(x, np.ndarray) or isinstance(x, np.generic):
        a = np.ascontiguousarray(x)
        h.update(b"a" + a.dtype.str.encode() + repr(a.shape).encode() + _fingerprint(a))
    elif x is None or isinstance(x, (bool, int, float, str)):
        h.update(b"v" + repr(x).encode())
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d" % len(x))
        for y in x:
            _digest(h, y)
    elif isinstance(x, dict):
        h.update(b"d%d" % len(x))
        for k in sorted(x, key=str):
            _digest(h, str(k)); _digest(h, x[k])
    elif hasattr(x, "__dict__") and not callable(x):
        h.update(b"o" + type(x).__name__.encode())
        _digest(h, {k: v for k, v in vars(x).items() if not callable(v)})
    else:
        h.update(b"?" + type(x).__name__.encode())


def _encode(x, blob, full, keep=()):
    """JSON-able description of a result; array bytes (or fingerprints) are appended to blob"""
    if isinstance(x, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(x)
        off = sum(len(b) for b in blob)
        small = full or a.nbytes <= SMALL
        blob.append(a.tobytes() if small else _fingerprint(a))
        dt = a.dtype.descr if a.dtype.names else a.dtype.str
        return {"a" if small else "h": [dt, list(a.shape), off, len(blob[-1]), isinstance(x, np.generic)]}
    if x is None or isinstance(x, (bool, int, float, str)):
        return {"v": x}
    if isinstance(x, (list, tuple)):
        return {"l" if isinstance(x, list) else "t": [_encode(y, blob, full, keep) for y in x]}
    if isinstance(x, dict):
        return {"d": [[k, _encode(v, blob, full or k in keep)] for k, v in x.items()]}
    raise TypeError(f"cannot store a {type(x).__name__} returned by the reference")


def _decode(e, blob):
    if "h" in e:
        dt, shape, off, n, _ = e["h"]
        dt = np.dtype([tuple(f) for f in dt]) if isinstance(dt, list) else np.dtype(dt)
        return Stored(dt, shape, blob[off:off + n])
    if "a" in e:
        dt, shape, off, n, scalar = e["a"]
        dt = np.dtype([tuple(f) for f in dt]) if isinstance(dt, list) else np.dtype(dt)
        a = np.frombuffer(blob[off:off + n], dt).reshape(shape).copy()
        return a[()] if scalar else a
    if "v" in e:
        return e["v"]
    if "l" in e:
        return [_decode(y, blob) for y in e["l"]]
    if "t" in e:
        return tuple(_decode(y, blob) for y in e["t"])
    return {k: _decode(v, blob) for k, v in e["d"]}


class _Store:
    """the calls of one test module, keyed by test name"""

    def __init__(self, module, keep):
        self.path = os.path.join(GOLDEN, module + ".npz")
        self.keep = keep
        self.tests = {}           # record: name -> {"calls": [[fn, encoded]], "blob": [bytes], "digest": sha}
        self.replay = {}          # replay: name -> {"calls": [...], "blob": bytes, "digest": hex, "pos": int, "h": sha}
        if RECORD:
            atexit.register(self.save)
        elif os.path.exists(self.path):
            with np.load(self.path) as z:
                index = json.loads(bytes(z["index"]).decode())
                for name, t in index.items():
                    self.replay[name] = dict(calls=t["calls"], digest=t["digest"], blob=bytes(z["blob_%d" % t["blob"]]))

    def call(self, fn_name, fn, args, kwargs):
        test = os.environ["PYTEST_CURRENT_TEST"].split("::", 1)[1].rsplit(" ", 1)[0]
        if RECORD:
            t = self.tests.setdefault(test, {"calls": [], "blob": [], "digest": hashlib.sha256()})
            _digest(t["digest"], (fn_name, args, kwargs))
            out = fn(*args, **kwargs)
            full = self.keep == ALL or test.split("[")[0] in self.keep
            t["calls"].append([fn_name, _encode(out, t["blob"], full, () if full else self.keep)])
            return out
        t = self.replay.get(test)
        if t is None:
            pytest.fail(f"no stored reference output for {test} in {self.path}; record it with CCM_RECORD_REFERENCE=1")
        t.setdefault("h", hashlib.sha256())
        pos = t.setdefault("pos", 0)
        if pos >= len(t["calls"]) or t["calls"][pos][0] != fn_name:
            pytest.fail(f"{test}: call {pos} ({fn_name}) is not the one stored in {self.path}; record again with CCM_RECORD_REFERENCE=1")
        _digest(t["h"], (fn_name, args, kwargs))
        t["pos"] = pos + 1
        if t["pos"] == len(t["calls"]):
            t["pos"] = 0
            if t.pop("h").hexdigest() != t["digest"]:
                pytest.fail(f"{test}: the inputs handed to the reference differ from the recorded ones ({self.path})")
        return _decode(t["calls"][pos][1], t["blob"])

    def save(self):
        index, blobs = {}, {}
        if os.path.exists(self.path):
            with np.load(self.path) as z:
                old = json.loads(bytes(z["index"]).decode())
                for name, t in old.items():
                    if name not in self.tests:
                        blobs["blob_%d" % len(index)] = z["blob_%d" % t["blob"]]
                        index[name] = dict(t, blob=len(index))
        for name, t in sorted(self.tests.items()):
            blobs["blob_%d" % len(index)] = np.frombuffer(b"".join(t["blob"]), np.uint8)
            index[name] = {"calls": t["calls"], "digest": t["digest"].hexdigest(), "blob": len(index)}
        os.makedirs(GOLDEN, exist_ok=True)
        np.savez_compressed(self.path, index=np.frombuffer(json.dumps(index, separators=(",", ":")).encode(), np.uint8), **blobs)


class _Object:
    """an object of the reference side whose method calls are recorded as <name>.<method>"""

    def __init__(self, rec, name, factory):
        self._rec, self._name = rec, name
        self.live = factory() if RECORD else None     # the object itself, for a Recorded.call() that post-processes its result

    def __getattr__(self, method):
        f = getattr(self.live, method) if RECORD else None
        return lambda *a, **k: self._rec.store.call(f"{self._name}.{method}", f, a, k)


class Recorded:
    """The oracle module with its reference-side functions (ref_*) recorded or replayed.  live() returns the reference library the
    module's tests use, None where it is not built; only recording needs it."""

    def __init__(self, oracle, module_file, live, keep=()):
        if RECORD and live() is None:
            pytest.fail("CCM_RECORD_REFERENCE=1 needs the reference libraries: make -C oracle ref where the original sources are present")
        self._oracle = oracle
        self.store = _Store(os.path.splitext(os.path.basename(module_file))[0], keep if keep == ALL else set(keep))

    def call(self, name, fn, *args, **kwargs):
        """fn(*args, **kwargs) on the reference side, stored under name"""
        return self.store.call(name, fn, args, kwargs)

    def obj(self, name, factory):
        return _Object(self, name, factory)

    def __getattr__(self, name):
        f = getattr(self._oracle, name)
        if name.startswith("ref_") and callable(f):
            return lambda *a, **k: self.store.call(name, f, a, k)
        return f
