"""Stored results of the compiled reference (oracle/_ref) for the tests that compare with it.

The reference's own sources are not part of this repository, so oracle/_ref can only be built where they are present.
Elsewhere the `ref` fixture is a `Replay` of tests/golden/ref_calls.json.gz: every call a test makes on the reference is
looked up by the test's id and the call's position in that test, the arguments must hash to the recorded ones (so a
changed input, or a draw count handed to `rng_equals` that differs from the recorded one, fails the test), and the
recorded result is returned.  Arrays longer than BIG elements are stored as a SHA-256 of their bytes (`Digest`); compare
them with `helpers.equal_arrays`.

With the reference built and CBS_REF_GOLDEN_RECORD=<path>, the `ref` fixture is a `Recorder` around the real reference
and writes the table to <path> when the session ends (run the tests that use `ref`, then copy the file here).
"""
from __future__ import annotations

import dataclasses
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_calls.json.gz")
BIG = 4096


class Digest:
    """A long array known by its dtype, shape and the SHA-256 of its bytes."""

    def __init__(self, dtype: str, shape, sha: str):
        self.dtype, self.shape, self.sha = dtype, tuple(shape), sha

    def matches(self, a) -> bool:
        a = np.ascontiguousarray(a)
        if a.shape != self.shape:
            return False
        return hashlib.sha256(np.ascontiguousarray(a, dtype=self.dtype).tobytes()).hexdigest() == self.sha

    def __repr__(self):
        return f"Digest({self.dtype}, {self.shape}, {self.sha[:12]})"


class _RngToken:
    """Stands for one reference engine inside a test: its seed and its creation index identify it in fingerprints."""

    def __init__(self, seed: int, index: int, inner=None):
        self.seed, self.index, self.inner = int(seed), index, inner


def _canon(v):
    if isinstance(v, _RngToken):
        return ["rng", v.seed, v.index]
    if isinstance(v, np.ndarray):
        a = np.ascontiguousarray(v)
        return ["nd", a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()]
    if isinstance(v, (bool, np.bool_)):
        return bool(v)
    if isinstance(v, (int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return float(v).hex()
    if isinstance(v, (tuple, list)):
        return [_canon(x) for x in v]
    if dataclasses.is_dataclass(v):
        return [type(v).__name__, {f.name: _canon(getattr(v, f.name)) for f in dataclasses.fields(v)}]
    if v is None or isinstance(v, str):
        return v
    raise TypeError(f"cannot fingerprint {type(v)}")


def _fingerprint(method, args, kwargs) -> str:
    key = json.dumps([method, _canon(list(args)), {k: _canon(kwargs[k]) for k in sorted(kwargs)}], sort_keys=True)
    return hashlib.sha256(key.encode()).hexdigest()


def _encode(v):
    if isinstance(v, np.ndarray):
        a = np.ascontiguousarray(v)
        if a.size > BIG:
            return {"digest": [a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()]}
        vals = [float(x).hex() for x in a.ravel()] if a.dtype.kind == "f" else [int(x) for x in a.ravel()]
        return {"array": [a.dtype.str, list(a.shape), vals]}
    if isinstance(v, dict):
        return {"dict": {k: _encode(x) for k, x in v.items()}}
    if isinstance(v, (tuple, list)):
        return {"tuple": [_encode(x) for x in v]}
    if isinstance(v, (bool, np.bool_)):
        return {"bool": bool(v)}
    if isinstance(v, (int, np.integer)):
        return {"int": int(v)}
    if isinstance(v, (float, np.floating)):
        return {"float": float(v).hex()}
    if v is None:
        return None
    raise TypeError(f"cannot store {type(v)}")


def _decode(e):
    if e is None:
        return None
    (kind, v), = e.items()
    if kind == "array":
        dt, shape, vals = v
        conv = [float.fromhex(x) for x in vals] if np.dtype(dt).kind == "f" else vals
        return np.array(conv, dtype=dt).reshape(shape)
    if kind == "digest":
        return Digest(*v)
    if kind == "dict":
        return {k: _decode(x) for k, x in v.items()}
    if kind == "tuple":
        return tuple(_decode(x) for x in v)
    if kind == "float":
        return float.fromhex(v)
    return v


def _current_test() -> str:
    return os.environ["PYTEST_CURRENT_TEST"].rsplit(" ", 1)[0]


class _Calls:
    """Common part: the per-test call counters and the reference engines handed out in the current test."""

    def __init__(self):
        self.pos, self.rngs = {}, {}

    def _slot(self):
        test = _current_test()
        i = self.pos.get(test, 0)
        self.pos[test] = i + 1
        return test, i

    def _token(self, seed, inner=None):
        test = _current_test()
        k = self.rngs.get(test, 0)
        self.rngs[test] = k + 1
        return _RngToken(seed, k, inner)


class Replay(_Calls):
    def __init__(self, table: dict):
        super().__init__()
        self.table = table

    @staticmethod
    def load() -> "Replay":
        with gzip.open(GOLDEN, "rt") as f:
            return Replay(json.load(f))

    def _calls(self):
        calls = self.table.get(_current_test())
        if calls is None:
            pytest.skip("no stored results of the compiled reference for this test")
        return calls

    def rng(self, seed):
        self._calls()
        return self._token(seed)

    def __getattr__(self, method):
        if method.startswith("_"):
            raise AttributeError(method)
        self._calls()

        def call(*args, **kwargs):
            calls = self._calls()
            test, i = self._slot()
            assert i < len(calls), f"{test}: call {i} ({method}) was never made on the reference"
            rec = calls[i]
            assert rec["m"] == method, f"{test}: call {i} is {method}, the reference was called with {rec['m']}"
            assert rec["in"] == _fingerprint(method, args, kwargs), \
                f"{test}: arguments of call {i} ({method}) differ from those the reference was called with"
            return _decode(rec["out"])
        return call


class Recorder(_Calls):
    def __init__(self, engine, path: str):
        super().__init__()
        self.engine, self.path, self.table = engine, path, {}

    def rng(self, seed):
        return self._token(seed, self.engine.rng(seed))

    def __getattr__(self, method):
        if method.startswith("_"):
            raise AttributeError(method)
        fn = getattr(self.engine, method)

        def call(*args, **kwargs):
            test, i = self._slot()
            unwrap = lambda v: v.inner if isinstance(v, _RngToken) else v  # noqa: E731
            out = fn(*[unwrap(a) for a in args], **{k: unwrap(v) for k, v in kwargs.items()})
            self.table.setdefault(test, []).append({"m": method, "in": _fingerprint(method, args, kwargs),
                                                    "out": _encode(out)})
            return out
        return call

    def save(self):
        with open(self.path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
            f.write(json.dumps(self.table, sort_keys=True).encode())
