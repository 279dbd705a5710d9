"""The unmodified reference's answers to what the tests ask it, recorded once where the reference
is built (oracle/_ref, tests/reflib.py) and replayed everywhere else, so that every comparison
with the reference runs on a plain checkout.

A call of a tests/reflib.py function is keyed by the function's name and its bound arguments.
Arrays, bytes and strings enter the key, and the stored answer, as SHA-256 digests; numbers,
booleans and lists of them are kept as they are.  A replayed answer has the shape of reflib's,
with every array, bytes or str value replaced by a Digest that compares equal to exactly the value
it was recorded from (same dtype, shape and bytes).  An argument computed by the library under
test is part of the key, so a library that computes something else finds no recorded answer.

Record (needs oracle/_ref):  GB200_RECORD_REFERENCE=1 python -m pytest tests"""
import hashlib
import inspect
import json
import os

import numpy as np

import reflib

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_answers.json")


def _sha(data):
    return hashlib.sha256(data).hexdigest()


class Digest:
    """Stands for an array, bytes or str value of the reference without holding it."""

    def __init__(self, kind, sha256, dtype=None, shape=None):
        self.kind, self.sha256, self.dtype, self.shape = kind, sha256, dtype, shape

    @classmethod
    def of(cls, x):
        if isinstance(x, Digest):
            return x
        if isinstance(x, (bytes, bytearray)):
            return cls("bytes", _sha(bytes(x)))
        if isinstance(x, str):
            return cls("str", _sha(x.encode()))
        a = np.ascontiguousarray(x)
        return cls("array", _sha(a.tobytes()), a.dtype.str, list(a.shape))

    def to_json(self):
        return [self.kind, self.sha256] + ([self.dtype, self.shape] if self.kind == "array" else [])

    def __eq__(self, other):
        if self.kind == "array" and not isinstance(other, Digest):
            other = np.asarray(other)
            want = np.dtype(self.dtype)
            if other.dtype != want:  # like np.array_equal: equal values in another integer type are equal
                cast = other.astype(want)
                if not np.array_equal(cast, other):
                    return False
                other = cast
        elif not isinstance(other, (Digest, bytes, bytearray, str)):
            return NotImplemented
        return Digest.of(other).to_json() == self.to_json()

    __hash__ = None

    def __repr__(self):
        return "Digest(%s)" % ", ".join(map(str, self.to_json()))


def sha256(x):
    """SHA-256 (hex) of a bytes or str answer, live or replayed."""
    return Digest.of(x).sha256


def _plain(v):
    """Numbers, booleans and None as JSON takes them; everything else as a digest."""
    if isinstance(v, np.generic):
        v = v.item()
    if v is None or isinstance(v, (bool, int, float)):
        return v
    if isinstance(v, (list, tuple)):
        return [_plain(x) for x in v]
    return {"digest": Digest.of(v).to_json()}


def _unplain(v):
    if isinstance(v, dict):
        kind, sha, *rest = v["digest"]
        return Digest(kind, sha, *rest)
    if isinstance(v, list):
        return [_unplain(x) for x in v]
    return v


def _key(name, args, kwargs):
    bound = inspect.signature(getattr(reflib, name)).bind(*args, **kwargs)
    bound.apply_defaults()

    def arg(v):  # 95 and 95.0 are the same quality
        v = _plain(v)
        return float(v) if isinstance(v, int) and not isinstance(v, bool) else v
    return _sha(json.dumps([name] + [[k, arg(v)] for k, v in bound.arguments.items()]).encode())[:32]


_NOT_ANSWERS = {"available", "lib"}


class Replay:
    """tests/reflib.py's functions, answered from the recorded file."""

    def __init__(self, path=PATH):
        with open(path) as f:
            self._answers = json.load(f)

    def __getattr__(self, name):
        if name.startswith("_") or name in _NOT_ANSWERS or not callable(getattr(reflib, name, None)):
            raise AttributeError(name)

        def call(*args, **kwargs):
            key = _key(name, args, kwargs)
            if key not in self._answers:
                raise AssertionError(
                    f"no recorded answer of the reference for reflib.{name} with these arguments (key {key}): "
                    "either the test asks something new (record it with GB200_RECORD_REFERENCE=1 where "
                    "oracle/_ref is built) or a value the library under test passed on differs from the reference's")
            return _unplain(self._answers[key])
        return call


class Recorder:
    """tests/reflib.py itself (the live reference), remembering every answer it gives."""

    def __init__(self):
        self._answers = {}

    def __getattr__(self, name):
        fn = getattr(reflib, name)
        if name.startswith("_") or name in _NOT_ANSWERS or not callable(fn):
            raise AttributeError(name)

        def call(*args, **kwargs):
            out = fn(*args, **kwargs)
            kept = out[:4] + (None,) if name == "process_rgb" else out  # the last item is a timing
            self._answers[_key(name, args, kwargs)] = _plain(kept)
            return out
        return call

    def save(self, path=PATH):
        """One answer per line, sorted by key (stable diffs when answers are added)."""
        lines = [json.dumps(k) + ": " + json.dumps(v, separators=(",", ":")) for k, v in sorted(self._answers.items())]
        with open(path, "w") as f:
            f.write("{\n" + ",\n".join(lines) + "\n}\n")
