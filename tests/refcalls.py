"""Recorded calls of the reference build (oracle.bind.Ref), so that the tests that compare with the unmodified reference also run
where it cannot be compiled.

RecordingRef wraps the live Ref and keeps every call's result; ReplayRef answers the same calls from tests/golden/ref_calls.npz.
A call is identified by the method name and a digest of its arguments (arrays by dtype, shape and bytes), so the tests drive
either object the same way.  Large results that the tests only ever compare whole (DIGESTED) are kept as a Digest (dtype, shape,
SHA-256 of the bytes); compare them with same().  tests/golden/make_ref_calls.py regenerates the file from a reference build.
"""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_calls.npz")
# per-call output files of the reference, not part of the result
IGNORED_KWARGS = ("dump_path",)
# method -> positions in its result tuple (None: the whole result) that are recorded as a Digest
DIGESTED = {"fft": None, "find_index": (1,), "demod_frame": (0, 1), "eep_deconvolve": None, "uep_deconvolve": None,
            "rs_decode_codewords": (1,)}


class Digest:
    """an array known by dtype, shape and the SHA-256 of its bytes"""

    def __init__(self, dtype, shape, sha256):
        self.dtype, self.shape, self.sha256 = dtype, tuple(shape), sha256

    @classmethod
    def of(cls, a):
        a = np.ascontiguousarray(a)
        return cls(a.dtype.str, a.shape, hashlib.sha256(a.tobytes()).hexdigest())

    def __eq__(self, other):
        return isinstance(other, Digest) and (self.dtype, self.shape, self.sha256) == (other.dtype, other.shape, other.sha256)

    def __repr__(self):
        return f"Digest({self.dtype}, {self.shape}, {self.sha256[:16]}...)"


def same(mine, theirs):
    """bit-for-bit equality (dtype, shape, bytes) of an array with the reference's array or with its Digest"""
    if isinstance(theirs, Digest):
        return Digest.of(mine) == theirs
    a, b = np.ascontiguousarray(mine), np.ascontiguousarray(theirs)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _canon(v):
    if isinstance(v, np.ndarray):
        d = Digest.of(v)
        return ["nd", d.dtype, list(d.shape), d.sha256]
    if isinstance(v, (bool, int, float, str)) or v is None:
        return [type(v).__name__, repr(v)]
    if isinstance(v, np.generic):
        return _canon(v.item())
    if isinstance(v, (list, tuple)):
        return [type(v).__name__] + [_canon(x) for x in v]
    raise TypeError(f"cannot key a reference call on a {type(v).__name__}")


def call_key(name, args, kwargs):
    kw = {k: v for k, v in sorted(kwargs.items()) if k not in IGNORED_KWARGS}
    blob = json.dumps([name, [_canon(a) for a in args], [[k, _canon(v)] for k, v in kw.items()]])
    return name + ":" + hashlib.sha256(blob.encode()).hexdigest()[:24]


def _pack(v, arrays):
    """result -> JSON-able description; arrays go to `arrays` and are referred to by their index"""
    if isinstance(v, Digest):
        return {"digest": [v.dtype, list(v.shape), v.sha256]}
    if isinstance(v, np.ndarray):
        arrays.append(np.ascontiguousarray(v))
        return {"nd": len(arrays) - 1}
    if isinstance(v, np.generic):
        v = v.item()
    if isinstance(v, (bool, int, float, str)) or v is None:
        return {"v": v}
    if isinstance(v, tuple):
        return {"tuple": [_pack(x, arrays) for x in v]}
    if isinstance(v, list):
        return {"list": [_pack(x, arrays) for x in v]}
    if isinstance(v, dict):
        return {"dict": [[k, _pack(x, arrays)] for k, x in v.items()]}
    raise TypeError(f"cannot record a {type(v).__name__}")


def _unpack(d, arrays):
    if "digest" in d:
        return Digest(*d["digest"])
    if "nd" in d:
        return arrays[d["nd"]].copy()
    if "v" in d:
        return d["v"]
    if "tuple" in d:
        return tuple(_unpack(x, arrays) for x in d["tuple"])
    if "list" in d:
        return [_unpack(x, arrays) for x in d["list"]]
    return {k: _unpack(x, arrays) for k, x in d["dict"]}


def _digested(name, out):
    which = DIGESTED.get(name, ())
    if which is None:
        return Digest.of(out)
    if not which:
        return out
    return tuple(Digest.of(x) if i in which else x for i, x in enumerate(out))


class RecordingRef:
    def __init__(self, ref):
        self._ref, self._calls = ref, {}

    def __getattr__(self, name):
        fn = getattr(self._ref, name)

        def call(*args, **kwargs):
            out = fn(*args, **kwargs)
            self._calls[call_key(name, args, kwargs)] = _digested(name, out)
            return out
        return call

    def save(self, path=GOLDEN):
        arrays, index = [], {}
        for k in sorted(self._calls):
            index[k] = _pack(self._calls[k], arrays)
        blob = np.frombuffer(json.dumps(index, sort_keys=True).encode(), np.uint8)
        np.savez_compressed(path, index=blob, **{f"a{i}": a for i, a in enumerate(arrays)})


class ReplayRef:
    def __init__(self, path=GOLDEN):
        with np.load(path) as z:
            self._index = json.loads(z["index"].tobytes().decode())
            self._arrays = [z[f"a{i}"] for i in range(len(z.files) - 1)]

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def call(*args, **kwargs):
            k = call_key(name, args, kwargs)
            if k not in self._index:
                raise KeyError(f"no recorded reference result for ref.{name}() with these arguments ({k}): the inputs differ from the "
                               "ones tests/golden/ref_calls.npz was recorded with (tests/golden/make_ref_calls.py records them again)")
            return _unpack(self._index[k], self._arrays)
        return call
