"""The reference's own sources (oracle/ref.py) as the tests see them: recorded once, replayed everywhere.

oracle/_ref/libmplref.so compiles only next to the reference's source tree, so a test that compared with it live would skip
on every other machine.  Instead, every call such a test makes on the reference side (constructors, setters, plans, dumps,
TrajSolver solves) is recorded with a digest of its arguments and what it returned, in
tests/golden/reference_calls/<test module>.npz.  By default the classes and functions below replay that recording, in call
order: a call whose name or arguments differ from the recorded one, or a recorded call the test no longer makes, fails the
test (the test changed, or what it feeds the reference changed: record again).  Record with

    MPLB_RECORD_REFERENCE=tests/golden/reference_calls python -m pytest tests/<module>.py

where oracle/_ref/libmplref.so can be built (test_gpu_vs_reference.py also needs a GPU: the library travels with the
tree); the proxies then drive the real library and write <dir>/<test module>.npz (tests of that module that did not run
keep their earlier recording).  Use as `import ref_replay as ref`.

The large dumps (DIGESTED: node tables, pop sequences, maps, LPA* state, spline coefficients) are kept as a Digest of their bytes, in record
and replay mode alike; compare them with `same`."""
import hashlib
import io
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls")
RECORD = os.environ.get("MPLB_RECORD_REFERENCE")

_TAPE = None
_RECORDED = {}  # record mode: module -> {test name: (calls, kinds, results)}

_NODE_TABLE = np.dtype([("key", "i4", 16), ("state", "f8", 13), ("g", "f8"), ("h", "f8"), ("opened", "i4"), ("closed", "i4")])


def _node_table(a):
    """A* node dump -> the fields the tests compare, in key order (the reference returns its hash map's order); entries
    past a key's length (key[15]) are zeroed."""
    key = a["key"].copy()
    pad = np.arange(16)[None, :] >= key[:, 15:16]
    pad[:, 15] = False
    key[pad] = 0
    order = np.lexsort(key[:, ::-1].T)
    out = np.zeros(len(a), dtype=_NODE_TABLE)
    out["key"] = key[order]
    for f in ("state", "g", "h", "opened", "closed"):
        out[f] = a[f][order]
    return out


DIGESTED = {"nodes": _node_table, "pop_keys": None, "get_data": None, "lpa_nodes": None, "lpa_heap": None,
            "lpa_get_linked_nodes": None, "traj_solve": None}


def _array_digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.blake2b(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes(), digest_size=16).hexdigest()


class Digest:
    """Stands for a large array the reference returned: its dtype, shape and a digest of its bytes."""

    def __init__(self, method, hexdigest, dtype, shape):
        self.method, self.hex, self.dtype, self.shape = method, hexdigest, str(dtype), tuple(shape)

    @classmethod
    def of(cls, method, a):
        a = DIGESTED[method](a) if DIGESTED[method] else np.asarray(a)
        return cls(method, _array_digest(a), a.dtype.str, a.shape)

    def matches(self, a):
        """np.array_equal(a, the reference's array), through the digest (records must have the same layout)"""
        a = np.asarray(a)
        if DIGESTED[self.method]:
            a = DIGESTED[self.method](a)
        if a.shape != self.shape:
            return False
        if a.dtype.str != self.dtype:
            if a.dtype.kind == "V":
                return False
            b = a.astype(self.dtype)
            if not np.array_equal(a, b):
                return False
            a = b
        return _array_digest(a) == self.hex

    def __len__(self):
        return self.shape[0]

    def copy(self):
        return self

    def __repr__(self):
        return "Digest(%s %s %s)" % (self.method, self.shape, self.hex)


def same(a, b):
    """np.array_equal where either side may be a Digest."""
    if isinstance(b, Digest):
        return b.matches(a)
    if isinstance(a, Digest):
        return a.matches(b)
    return np.array_equal(a, b)


def _feed(h, x):
    if isinstance(x, _Proxy):
        h.update(b"obj%d" % object.__getattribute__(x, "_id"))
    elif isinstance(x, (list, tuple)):
        h.update(b"[%d" % len(x))
        for y in x:
            _feed(h, y)
        h.update(b"]")
    elif isinstance(x, dict):
        for k in sorted(x):
            h.update(b"k" + k.encode())
            _feed(h, x[k])
    elif isinstance(x, str):
        h.update(b"s" + x.encode())
    elif x is None:
        h.update(b"N")
    else:  # numbers, numpy scalars, records and arrays
        a = np.ascontiguousarray(x)
        h.update(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes())


def _digest(args, kwargs):
    h = hashlib.blake2b(digest_size=8)
    _feed(h, list(args))
    _feed(h, kwargs)
    return h.hexdigest()


def _unwrap(x):
    if isinstance(x, _Proxy):
        return object.__getattribute__(x, "_real")
    if isinstance(x, (list, tuple)):
        return type(x)(_unwrap(y) for y in x)
    if isinstance(x, dict):
        return {k: _unwrap(v) for k, v in x.items()}
    return x


def _load(path, test):
    """-> (calls, kinds, results): the returned arrays of a test are .npy images one after the other in `<test>/blob`"""
    z = np.load(path)
    kinds, blob, off = list(z[test + "/kinds"]), z[test + "/blob"].tobytes(), z[test + "/offsets"]
    parts = [np.load(io.BytesIO(blob[off[k]:off[k + 1]]), allow_pickle=False) for k in range(len(off) - 1)]
    results = []
    for k in kinds:
        n = int(k.split(":")[1])
        results.append(parts[:n])
        parts = parts[n:]
    return list(z[test + "/calls"]), kinds, results


class _Tape:
    def __init__(self, module, test):
        self.module, self.test, self.pos, self.next_id = module, test, 0, 0
        if RECORD:
            self.calls, self.kinds, self.results = [], [], []
            return
        path = os.path.join(GOLD, module + ".npz")
        assert os.path.exists(path), "no recording of the reference's answers: %s" % path
        assert test + "/calls" in np.load(path).files, "%s has no recording for %s" % (path, test)
        self.calls, self.kinds, self.results = _load(path, test)

    def call(self, name, args, kwargs, fn, keep=True):
        key = name + ":" + _digest(args, kwargs)
        method = name.rsplit(".", 1)[-1]
        i = self.pos
        self.pos += 1
        if RECORD:
            r = fn()
            if method in DIGESTED:
                r = Digest.of(method, r)
            if not keep or r is None:
                kind, parts = "none", []
            elif isinstance(r, Digest):
                kind, parts = "digest", [np.array(r.hex), np.array(r.dtype), np.array(r.shape)]
            elif isinstance(r, tuple):
                kind, parts = "tuple", [np.asarray(p) for p in r]
            elif isinstance(r, np.void):
                kind, parts = "record", [np.array([r], dtype=r.dtype)]
            elif isinstance(r, np.ndarray):
                kind, parts = "array", [r]
            else:
                kind, parts = type(r).__name__, [np.asarray(r)]
            self.calls.append(key)
            self.kinds.append("%s:%d" % (kind, len(parts)))
            self.results.append(parts)
            return r
        assert i < len(self.calls), ("call %d (%s) was not recorded" % (i, name), self.test)
        assert self.calls[i] == key, ("call %d differs from the recording" % i, key, self.calls[i], self.test)
        kind, parts = self.kinds[i].split(":")[0], self.results[i]
        if kind == "none":
            return None
        if kind == "digest":
            return Digest(method, str(parts[0]), str(parts[1]), parts[2].tolist())
        if kind == "tuple":
            return tuple(p.copy() for p in parts)
        if kind == "record":
            return parts[0].copy()[0]
        if kind == "array":
            return parts[0].copy()
        return {"int": int, "float": float, "bool": bool}[kind](parts[0])

    def finish(self):
        if not RECORD:
            assert self.pos == len(self.calls), ("the test made %d of the %d recorded calls" % (self.pos, len(self.calls)), self.test)
            return
        mod = _RECORDED.setdefault(self.module, {})
        path = os.path.join(RECORD, self.module + ".npz")
        if not mod and os.path.exists(path):  # keep the tests of this module that are not re-recorded in this run
            for t in {f.rsplit("/", 1)[0] for f in np.load(path).files if f.endswith("/calls")}:
                mod[t] = _load(path, t)
        mod[self.test] = (self.calls, self.kinds, self.results)
        out = {}
        for t, (calls, kinds, results) in mod.items():
            images = []
            for p in (p for parts in results for p in parts):
                buf = io.BytesIO()
                np.save(buf, p, allow_pickle=False)
                images.append(buf.getvalue())
            out[t + "/calls"], out[t + "/kinds"] = np.array(calls), np.array(kinds)
            out[t + "/blob"] = np.frombuffer(b"".join(images), dtype=np.uint8)
            out[t + "/offsets"] = np.cumsum([0] + [len(b) for b in images])
        os.makedirs(RECORD, exist_ok=True)
        np.savez_compressed(path, **out)


@pytest.fixture(autouse=True)
def recorded_reference(request):
    """Autouse in every module that imports it: the test's own tape of reference calls."""
    global _TAPE
    _TAPE = _Tape(request.module.__name__, request.node.name)
    failed = request.session.testsfailed
    yield
    tape, _TAPE = _TAPE, None
    if request.session.testsfailed == failed:  # the test body passed
        tape.finish()


def _tape():
    assert _TAPE is not None, "reference calls are only recorded / replayed inside a test"
    return _TAPE


def _real_ref():
    from oracle import ref
    assert ref.available(), "recording needs oracle/_ref/libmplref.so (built next to the reference's sources)"
    return ref


class _Proxy:
    """Stands for an object of oracle.ref; its methods are recorded / replayed calls."""

    def __init__(self, *args):
        t = _tape()
        object.__setattr__(self, "_id", t.next_id)
        t.next_id += 1
        name = type(self).__name__
        real = t.call(name, args, {}, lambda: getattr(_real_ref(), name)(*_unwrap(args)), keep=False)
        object.__setattr__(self, "_real", real)

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def method(*args, **kwargs):
            real = object.__getattribute__(self, "_real")
            return _tape().call("%d.%s" % (object.__getattribute__(self, "_id"), name), args, kwargs,
                                lambda: getattr(real, name)(*_unwrap(args), **_unwrap(kwargs)))
        return method

    def __setattr__(self, name, value):
        object.__setattr__(self, name, value)
        real = object.__getattribute__(self, "_real")
        if real is not None:  # e.g. _lpa_control, which the real planner's lpa_waypoint reads
            setattr(real, name, _unwrap(value))


class RefMap(_Proxy):
    pass


class RefPlanner(_Proxy):
    pass


def traj_solve(*args, **kwargs):
    return _tape().call("traj_solve", args, kwargs, lambda: _real_ref().traj_solve(*args, **kwargs))


def traj_solve_path(*args, **kwargs):
    return _tape().call("traj_solve_path", args, kwargs, lambda: _real_ref().traj_solve_path(*args, **kwargs))
