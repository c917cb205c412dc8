"""Stored results of the reference's own compiled hot path, so that tests/test_ref_pin.py pins the oracle to the reference without the
reference's sources (tests/golden/ref_pin.npz).

The tests talk to the reference through ref.Window / ref.CoarseTracker / ref.CoarseInit / ref.make_images / ... (oracle/ref.py).  Under
DMV_REF_RECORD=1 (tests/golden/make_ref_golden.py) those objects are the real ones wrapped by a recorder that logs every call's result per
test; otherwise a replayer hands back the logged results in the same order.  Small results, and those a test marks with whole(), are
stored whole; larger arrays that the tests compare bit for bit (images, Jacobians, per-point states) as a SHA-256 digest of their canonical
bytes; the dense fp64 systems, which the tests compare by relative norm, as a Sketch (norm + fixed random projection)."""
import copy
import hashlib
import json
import os

import numpy as np
import pytest

from helpers import rel as _rel

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin.npz")
WHOLE_SIZE = 64         # arrays up to this many elements are stored whole
SKETCH_SIZE = 1024      # fp64 arrays above this many elements (the dense systems) are stored as a Sketch
SKETCH_ROWS = 64


def _canonical(a):
    """the bytes assert_array_equal compares: -0 == +0, every NaN equal"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind in "fc":
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a + np.zeros((), a.dtype))   # x + 0 maps -0 to +0
    return a


def _sha(a):
    h = hashlib.sha256()
    h.update(str((a.dtype.str, a.shape)).encode())
    h.update(_canonical(a).tobytes())
    return h.hexdigest()[:32]


class Digest:
    """a large array the tests compare bit for bit: shape, dtype and a digest of its canonical bytes"""

    def __init__(self, shape, dtype, sha):
        self.shape, self.dtype, self.sha = tuple(shape), np.dtype(dtype), sha

    def check(self, o, err_msg=""):
        o = np.asarray(o)
        assert o.shape == self.shape, f"{err_msg}: shape {o.shape} != reference {self.shape}"
        assert _sha(o.astype(self.dtype, copy=False)) == self.sha, f"{err_msg}: differs from the reference's result (digest)"


def _projection(n):
    """fixed seeded k x n matrix of +-1/sqrt(k): E |P d|^2 = |d|^2 for every d (relative spread of |P d| about 9 %)"""
    return np.random.default_rng(n).choice([-1.0, 1.0], (SKETCH_ROWS, n)) / np.sqrt(SKETCH_ROWS)


class Sketch:
    """a dense fp64 system the tests compare by relative norm: its norm, a fixed random projection of it (rel() estimates |o - r| from
    that) and whether it is exactly symmetric"""

    def __init__(self, shape, norm, proj, symmetric):
        self.shape, self.norm, self.proj, self.symmetric = tuple(shape), norm, np.asarray(proj, np.float64), bool(symmetric)

    @classmethod
    def of(cls, a):
        a = np.asarray(a, np.float64)
        sym = a.ndim == 2 and a.shape[0] == a.shape[1] and np.array_equal(a, a.T)
        return cls(a.shape, float(np.linalg.norm(a)), _projection(a.size) @ a.reshape(-1), sym)

    def project(self, o):
        o = np.asarray(o, np.float64)
        assert o.shape == self.shape, f"shape {o.shape} != reference {self.shape}"
        return _projection(o.size) @ o.reshape(-1)

    def __add__(self, other):
        return Sketch(self.shape, None, self.proj + other.proj, False)

    def __sub__(self, other):
        return Sketch(self.shape, None, self.proj - other.proj, False)


def rel(a, b):
    """|a - b| / |b| (tests/helpers.py) where b, and possibly a, is a reference result stored whole or as a Sketch"""
    if not isinstance(b, Sketch):
        return _rel(a, b)
    pa = a.proj if isinstance(a, Sketch) else b.project(a)
    return np.linalg.norm(pa - b.proj) / max(b.norm, 1e-300)


def norm(a):
    return a.norm if isinstance(a, Sketch) else np.linalg.norm(a)


def assert_equal(o, r, err_msg=""):
    """np.testing.assert_array_equal(o, r) where r is a reference result, stored whole or as a Digest"""
    if isinstance(r, Digest):
        r.check(o, err_msg)
    else:
        np.testing.assert_array_equal(o, r, err_msg=err_msg)


def assert_symmetric(r):
    assert r.symmetric if isinstance(r, Sketch) else np.array_equal(r, r.T)


# ------------------------------------------------------------------------------------------------------------- encoding of call logs
def _encode(v, key, arrays, whole=()):
    if isinstance(v, dict):
        return {"d": {k: _encode(x, f"{key}.{k}", arrays, ("*",) if k in whole or "*" in whole else ()) for k, x in v.items()}}
    if isinstance(v, (tuple, list)):
        return {"l": [_encode(x, f"{key}.{i}", arrays, whole) for i, x in enumerate(v)]}
    if v is None:
        return {"n": 0}
    a = np.asarray(v)
    if a.dtype == object:
        raise TypeError(f"{key}: cannot store {type(v)}")
    if whole or a.size <= WHOLE_SIZE or (a.dtype == np.float64 and a.size <= SKETCH_SIZE):
        arrays[key] = a
        return {"a": key, "s": int(not isinstance(v, np.ndarray))}
    if a.dtype == np.float64:
        s = Sketch.of(a)
        arrays[key] = s.proj
        return {"k": key, "shape": list(s.shape), "norm": s.norm, "sym": int(s.symmetric)}
    return {"g": _sha(a), "shape": list(a.shape), "dtype": a.dtype.str}


def _decode(t, arrays):
    if "d" in t:
        return {k: _decode(x, arrays) for k, x in t["d"].items()}
    if "l" in t:
        return [_decode(x, arrays) for x in t["l"]]
    if "n" in t:
        return None
    if "a" in t:
        a = arrays[t["a"]]
        return a.item() if t["s"] else a
    if "k" in t:
        return Sketch(t["shape"], t["norm"], arrays[t["k"]], t["sym"])
    return Digest(t["shape"], t["dtype"], t["g"])


def save(logs, path=GOLDEN):
    """one flat buffer per dtype (arrays by offset) and the call logs as JSON"""
    arrays, tree = {}, {}
    for test, calls in logs.items():
        tree[test] = [[name, _encode(v, f"{i}{test}", arrays, keys)] for i, (name, v, keys, _) in enumerate(calls)]
    bufs, index = {}, {}
    for key, a in arrays.items():
        parts = bufs.setdefault(a.dtype.str, [])
        index[key] = [a.dtype.str, sum(p.size for p in parts), list(a.shape)]
        parts.append(np.ascontiguousarray(a).reshape(-1))
    out = {f"buf{i}": np.concatenate(parts) for i, parts in enumerate(bufs.values())}
    names = {dt: f"buf{i}" for i, dt in enumerate(bufs)}
    index = {k: [names[dt], off, shape] for k, (dt, off, shape) in index.items()}
    out["__tree__"] = np.frombuffer(json.dumps({"tree": tree, "index": index}).encode(), np.uint8)
    np.savez_compressed(path, **out)


_LOADED = None


def load(path=GOLDEN):
    global _LOADED
    if _LOADED is None:
        z = np.load(path)
        d = json.loads(bytes(z["__tree__"]).decode())
        bufs = {k: z[k] for k in z.files if k != "__tree__"}
        arrays = {k: bufs[b][off:off + int(np.prod(shape))].reshape(shape) for k, (b, off, shape) in d["index"].items()}
        _LOADED = (d["tree"], arrays)
    return _LOADED


# ------------------------------------------------------------------------------------------------------------- record / replay
_RECORDING = []   # the call log of the test being recorded


def whole(r, *keys):
    """marks the reference result r the test just received (or only these keys of it, a dict) as used beyond a bit-for-bit or relative
    norm comparison: it is stored whole"""
    for e in (_RECORDING[0] if _RECORDING else ()):
        if e[3] == id(r):
            e[2] = keys or ("*",)
    return r


class _Recorder:
    def __init__(self, obj, log, prefix=""):
        self._obj, self._log, self._prefix = obj, log, prefix

    def __getattr__(self, name):
        v = getattr(self._obj, name)
        full = self._prefix + name
        if name == "L":
            return _Recorder(v, self._log, "L.")
        if not callable(v):
            self._log.append([full, v, (), id(v)])
            return v

        def call(*a, **kw):
            r = v(*a, **kw)
            if isinstance(r, (int, float, bool, np.generic, np.ndarray, dict, tuple, list)) or r is None:
                self._log.append([full, copy.deepcopy(r), (), id(r)])
                return r
            return _Recorder(r, self._log)   # a reference object (Window, CoarseTracker, CoarseInit)
        return call


class _Replayer:
    def __init__(self, test, calls, prefix=""):
        self._test, self._calls, self._prefix = test, calls, prefix

    def _next(self, name):
        assert self._calls, f"{self._test}: no stored reference result left for {name} (regenerate with tests/golden/make_ref_golden.py)"
        got, v = self._calls.pop(0)
        assert got == name, f"{self._test}: stored reference call {got}, the test made {name} (regenerate with tests/golden/make_ref_golden.py)"
        return v

    def __getattr__(self, name):
        full = self._prefix + name
        if name == "L":
            return _Replayer(self._test, self._calls, "L.")
        if name in ("levels", "h"):
            return self._next(full)
        if name in ("Window", "CoarseTracker", "CoarseInit"):
            return lambda *a, **kw: self
        return lambda *a, **kw: self._next(full)


def reference(request):
    """what the `ref` fixture of tests/test_ref_pin.py hands to one test: the recording real reference or the replayed one"""
    test = request.node.name
    if os.environ.get("DMV_REF_RECORD") == "1":
        from oracle import ref as real
        if not real.available():
            raise RuntimeError("DMV_REF_RECORD=1 needs the reference build (oracle/_ref/libdso_ref.so)")
        real.lib()
        log = request.config.stash.setdefault(_LOG_KEY, {}).setdefault(test, [])
        del log[:]
        _RECORDING[:] = [log]
        return _Recorder(real, log)
    _RECORDING[:] = []
    tree, arrays = load()
    assert test in tree, f"{test}: no stored reference results (regenerate with tests/golden/make_ref_golden.py)"
    return _Replayer(test, [(n, _decode(t, arrays)) for n, t in tree[test]])


_LOG_KEY = pytest.StashKey[dict]()


def recorded_logs(config):
    return config.stash.get(_LOG_KEY, {})
