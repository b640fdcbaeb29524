"""Stored outputs of oracle/_ref for the tests that compare against it.

oracle/_ref is compiled from the original project's sources, which are not part of this repository, so a checkout cannot rebuild it.
`Recorded(name)` stands in for the `oracle.ref` module: every call a test makes through it is replayed from tests/golden/ref/<name>/, one
.npz per test, split below MAX_FILE_BYTES (arrays byte-shuffled and LZMA-compressed: float outputs shrink well below what zlib makes of them).
With NSB_RECORD_REF=1, where oracle/_ref is built, the calls go to the library instead and the file is rewritten when the session ends.

Each stored call keeps a digest of its arguments (arrays, scalars, ctypes structures, and for RefCuda the scene it was created with): a
replay whose arguments differ from the recorded ones fails instead of comparing against the output of another input. Pointers are not
followed and call-backs are not run, so the network parameters behind an inference call-back and the maps behind an NsbFrame pointer
are covered only where the test passes them as `also=` (digested, not given to the call); the model parameters and occupancy grid
of the synthetic scene are pinned by tests/test_golden.py. A call may name a `shrink(outputs) -> outputs` that keeps what the test compares (a seeded sample, the
rows it reads): the test then receives the same shrunk outputs whether they are recorded or replayed. `Recorded.run(what, fn, *args)`
records any function of the reference calls (a chain of calls whose intermediate state is too large to store).
"""
from __future__ import annotations

import atexit
import ctypes as C
import glob
import hashlib
import json
import lzma
import os
import re

import numpy as np
import pytest

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
RECORD = os.environ.get("NSB_RECORD_REF") == "1"
MAX_FILE_BYTES = 900_000


def _feed(h, x):
    if isinstance(x, np.ndarray):
        h.update(f"{x.dtype}{x.shape}".encode())
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (bool, int, float, str, np.generic)) or x is None:
        h.update(repr(x.item() if isinstance(x, np.generic) else x).encode())
    elif isinstance(x, (list, tuple)):
        for y in x:
            _feed(h, y)
    elif isinstance(x, dict):
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    elif isinstance(x, C.Structure):
        for name, typ in x._fields_:
            if typ is C.c_void_p or hasattr(typ, "contents"):
                continue  # addresses change from run to run
            _feed(h, name)
            v = getattr(x, name)
            _feed(h, list(v) if isinstance(v, C.Array) else v)
    elif isinstance(x, C.Array):
        _feed(h, list(x))
    # call-backs and library handles carry no data of their own


def digest(*args, **kwargs) -> str:
    h = hashlib.sha256()
    _feed(h, list(args))
    _feed(h, kwargs)
    return h.hexdigest()[:16]


def sha(t) -> str:
    """SHA-256 of an array's bytes (numpy or torch): what a bit-exact comparison needs of a frame."""
    a = t.contiguous().cpu().numpy() if type(t).__module__ == "torch" else np.ascontiguousarray(t)
    return hashlib.sha256(a.tobytes()).hexdigest()


def frame_digests(out):
    """shrink for a render call whose frame is compared bit for bit: (sha(rgba), sha(depth), info)."""
    fb, depth, info = out
    return sha(fb), sha(depth), info


def _encode(out, arrays, prefix):
    """Outputs -> a JSON structure; arrays go to `arrays` under prefix/i."""
    if isinstance(out, np.ndarray):
        key = f"{prefix}/{len(arrays)}"
        arrays[key] = out
        return {"a": key}
    if type(out).__module__ == "torch":
        key = f"{prefix}/{len(arrays)}"
        arrays[key] = out.cpu().numpy()
        return {"t": key}
    if isinstance(out, tuple):
        return {"s": [_encode(o, arrays, prefix) for o in out]}
    return {"j": json.dumps(out)}


def _decode(spec, arrays):
    if "a" in spec:
        return arrays[spec["a"]]
    if "t" in spec:
        import torch

        return torch.from_numpy(arrays[spec["t"]]).cuda()
    if "s" in spec:
        return tuple(_decode(s, arrays) for s in spec["s"])
    return json.loads(spec["j"])


class _Store:
    def __init__(self, name):
        self.path = os.path.join(GOLDEN_DIR, name)
        self.meta, self.arrays, self.counts, self._loaded, self._rerecorded = {}, {}, {}, False, set()

    def _load(self):
        if not self._loaded:
            for path in sorted(glob.glob(os.path.join(self.path, "*.npz"))):
                with np.load(path) as z:
                    meta = json.loads(str(z["__meta__"]))
                    self.meta.update(meta["calls"])
                    for k, (dtype, shape) in meta["arrays"].items():
                        self.arrays[k] = _unpack(z[k], dtype, shape)
        self._loaded = True

    def key(self, what):
        test = os.environ.get("PYTEST_CURRENT_TEST", "").rsplit(" ", 1)[0].split("::", 1)[-1]
        n = self.counts.get((test, what), 0)
        self.counts[(test, what)] = n + 1
        return f"{test}/{what}/{n}"

    def call(self, what, fn, args, kwargs, shrink=None, also=None, scene=None):
        self._load()
        key = self.key(what)
        d = digest(*args, **kwargs, __also__=also, __scene__=scene)
        if RECORD:
            test = key.split("/", 1)[0]
            if test not in self._rerecorded:  # a test recorded again keeps none of its old calls
                self._rerecorded.add(test)
                for k in [k for k in self.meta if k.split("/", 1)[0] == test]:
                    del self.meta[k]
                for k in [k for k in self.arrays if k.split("/", 1)[0] == test]:
                    del self.arrays[k]
            out = fn(*args, **kwargs)
            if shrink is not None:
                out = shrink(out)
            new = {}
            self.meta[key] = {"inputs": d, "out": _encode(out, new, key)}
            self.arrays.update(new)
            _dirty.add(self)
            return out
        if key not in self.meta:
            pytest.fail(f"{self.path} holds no output for {key}: record it with NSB_RECORD_REF=1 where oracle/_ref is built")
        assert self.meta[key]["inputs"] == d, f"{key}: the inputs differ from the recorded ones (record again with NSB_RECORD_REF=1)"
        return _decode(self.meta[key]["out"], self.arrays)

    def save(self):
        os.makedirs(self.path, exist_ok=True)
        for test in sorted({k.split("/", 1)[0] for k in self.meta}):
            calls = {k: m for k, m in self.meta.items() if k.split("/", 1)[0] == test}
            base = re.sub(r"[^A-Za-z0-9_.-]+", "_", test).strip("_")
            for old in glob.glob(os.path.join(self.path, base + ".npz")) + glob.glob(os.path.join(self.path, base + ".[0-9]*.npz")):
                os.remove(old)
            part, size, parts = {}, 0, []
            for k, m in calls.items():  # a test whose outputs exceed MAX_FILE_BYTES is spread over several files
                packed = {a: _pack(self.arrays[a]) for a in _keys(m["out"])}
                n = sum(v.size for v in packed.values())
                if part and size + n > MAX_FILE_BYTES:
                    parts.append(part)
                    part, size = {}, 0
                part[k] = (m, packed)
                size += n
            parts.append(part)
            for i, part in enumerate(parts):
                meta = {"calls": {k: m for k, (m, _) in part.items()},
                        "arrays": {a: (self.arrays[a].dtype.str, self.arrays[a].shape) for _, pk in part.values() for a in pk}}
                arrays = {a: v for _, pk in part.values() for a, v in pk.items()}
                np.savez(os.path.join(self.path, base + (f".{i}" if i else "") + ".npz"), __meta__=np.array(json.dumps(meta, sort_keys=True)), **arrays)


def _pack(a):
    """Byte-shuffled (all first bytes, then all second bytes, ...) and LZMA-compressed: uint8 [n]."""
    a = np.ascontiguousarray(a)
    raw = a.view(np.uint8).reshape(-1, a.dtype.itemsize).T.tobytes() if a.size else b""
    return np.frombuffer(lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME), np.uint8)


def _unpack(z, dtype, shape):
    dt = np.dtype(dtype)
    raw = np.frombuffer(lzma.decompress(z.tobytes()), np.uint8)
    return raw.reshape(dt.itemsize, -1).T.copy().view(dt).reshape(shape) if raw.size else np.zeros(shape, dt)


def _keys(spec):
    if "a" in spec or "t" in spec:
        yield spec.get("a", spec.get("t"))
    for s in spec.get("s", []):
        yield from _keys(s)


_dirty: set = set()
atexit.register(lambda: [s.save() for s in _dirty])


class _RefCuda:
    """oracle.ref.RefCuda whose calls are recorded or replayed: in replay nothing is created on the GPU."""

    def __init__(self, store, *args):
        from oracle import ref

        self._store, self._rc, self._scene = store, ref.RefCuda(*args) if RECORD else None, digest(*args)

    def __getattr__(self, name):
        real = getattr(self._rc, name) if self._rc is not None else None

        def call(*args, shrink=None, also=None, **kwargs):
            return self._store.call(f"RefCuda.{name}", real, args, kwargs, shrink, also, self._scene)

        return call

    def close(self):
        if self._rc is not None:
            self._rc.close()


class Recorded:
    """Drop-in for the `oracle.ref` module; every function takes the extra keywords `shrink` and `also` (see the module docstring)."""

    def __init__(self, name):
        self._store = _Store(name)

    def RefCuda(self, *args):
        return _RefCuda(self._store, *args)

    def run(self, what, fn, *args, shrink=None, also=None):
        return self._store.call(what, fn, args, {}, shrink, also)

    def __getattr__(self, name):
        from oracle import ref

        attr = getattr(ref, name)
        if not callable(attr) or isinstance(attr, type):
            return attr

        def call(*args, shrink=None, also=None, **kwargs):
            return self._store.call(name, attr, args, kwargs, shrink, also)

        return call
