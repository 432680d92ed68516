"""What the reference computed, kept with the suite.

Tests that pin the restatements (and through them the CUDA kernels) to the reference's own sources compiled verbatim
(oracle/_ref) need that build only to produce the expected values.  tests/golden/reference.json keeps those values for every
such comparison: a SHA-256 digest of each expected output (outputs are large; equal digests mean bit-identical outputs), and
the few small values that tests feed back into the restatements (a camera centre, a decomposed Sim3) as the values themselves.

    ref.expect(got, live)   got: the restatement's result in the reference's convention; live: None, or a zero-argument
                            callable that computes the same on the reference build.  Asserts got == the stored result and,
                            where live is given, got == live().
    ref.value(live)         a reference-side value used as an input: live() where given (checked against the stored value),
                            otherwise the stored value.

Keys are the test's name, its parameters and the call's position in the test.  To (re)record after changing a case, run the
reference tests where the reference build exists with ORB_SLAM2_B200_RECORD_REFERENCE=1.
"""
import base64
import hashlib
import json
import os

import numpy as np
import pytest

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference.json")
RECORD = os.environ.get("ORB_SLAM2_B200_RECORD_REFERENCE") == "1"
_store = None


def _load():
    global _store
    if _store is None:
        _store = json.load(open(PATH)) if os.path.exists(PATH) else {}
    return _store


def _save():
    with open(PATH, "w") as f:
        json.dump(dict(sorted(_store.items())), f, indent=0, sort_keys=True)
        f.write("\n")


def _canon(x, h):
    """Feeds a canonical byte form of a nested result (tuples / lists / dicts of arrays and scalars) into hash h."""
    if isinstance(x, dict):
        h.update(b"{")
        for k in sorted(x):
            h.update(repr(k).encode()); _canon(x[k], h)
        h.update(b"}")
    elif isinstance(x, (list, tuple)):
        h.update(b"[")
        for v in x:
            _canon(v, h)
        h.update(b"]")
    elif isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x.astype(np.int64) if x.dtype.kind in "biu" else x)     # integers compare by value, as array_equal does
        h.update(f"a{a.dtype.str}{a.shape}".encode()); h.update(a.tobytes())
    elif isinstance(x, (bool, np.bool_)):
        h.update(b"b1" if x else b"b0")
    elif isinstance(x, (int, np.integer)):
        h.update(f"i{int(x)}".encode())
    elif isinstance(x, (float, np.floating)):
        h.update(f"f{float(x)!r}".encode())
    elif x is None:
        h.update(b"n")
    else:
        raise TypeError(type(x))


def digest(x) -> str:
    h = hashlib.sha256()
    _canon(x, h)
    return h.hexdigest()[:32]


def _encode(x):
    if isinstance(x, np.ndarray):
        return {"dtype": x.dtype.str, "shape": list(x.shape), "b64": base64.b64encode(np.ascontiguousarray(x).tobytes()).decode()}
    if isinstance(x, tuple):
        return {"tuple": [_encode(v) for v in x]}
    if isinstance(x, dict):
        return {"dict": {k: _encode(v) for k, v in x.items()}}
    if isinstance(x, (np.bool_, bool)):
        return {"bool": bool(x)}
    if isinstance(x, np.floating):
        return {"dtype": x.dtype.str, "shape": [], "b64": base64.b64encode(x.tobytes()).decode()}
    if isinstance(x, (int, float, np.integer)):
        return x if isinstance(x, (int, float)) else int(x)
    raise TypeError(type(x))


def _decode(x):
    if isinstance(x, dict):
        if "b64" in x:
            a = np.frombuffer(base64.b64decode(x["b64"]), np.dtype(x["dtype"])).reshape(x["shape"]).copy()
            return a[()] if not x["shape"] else a
        if "tuple" in x:
            return tuple(_decode(v) for v in x["tuple"])
        if "dict" in x:
            return {k: _decode(v) for k, v in x["dict"].items()}
        if "bool" in x:
            return x["bool"]
    return x


def _same(a, b):
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(_same(u, v) for u, v in zip(a, b))
    return np.array_equal(a, b)


class Reference:
    def __init__(self, name, params):
        args = ",".join(f"{k}={os.path.basename(v) if isinstance(v, str) else v!r}" for k, v in sorted(params.items()))
        self.prefix = f"{name}[{args}]"
        self.n = 0

    @classmethod
    def of(cls, node):
        """Keyed by the test function (also where another module re-collects it) and its own parameters (not those of
        parametrized fixtures); paths by file name."""
        names = set()
        for m in node.iter_markers("parametrize"):
            a = m.args[0]
            names.update(x.strip() for x in (a.split(",") if isinstance(a, str) else a))
        params = getattr(getattr(node, "callspec", None), "params", {})
        return cls(node.function.__name__, {k: v for k, v in params.items() if k in names})

    def _key(self, kind):
        self.n += 1
        return f"{self.prefix}#{self.n}{kind}"

    def expect(self, got, live=None):
        key, store = self._key(""), _load()
        if live is not None:
            want = live()
            assert _same(got, want), f"{key}: restatement differs from the reference build"
            if RECORD:
                store[key] = digest(want)
                _save()
        assert key in store, f"{key}: no stored reference result (record it where the reference build exists)"
        assert digest(got) == store[key], f"{key}: differs from the stored reference result"

    def value(self, live=None):
        key, store = self._key("=v"), _load()
        if live is not None:
            v = live()
            if RECORD:
                store[key] = _encode(v)
                _save()
            assert key in store and _same(v, _decode(store[key])), f"{key}: stored reference value differs from the reference build"
            return v
        assert key in store, f"{key}: no stored reference value (record it where the reference build exists)"
        return _decode(store[key])


@pytest.fixture
def ref(request):
    return Reference.of(request.node)
