"""The reference's own decoder (oracle/ref.py) as recorded answers, so that the tests comparing against it run on machines
where the reference is not built.

Every use a test makes of `oracle.ref` -- a constructor, a method call, a property read -- is keyed by a hash of the
instance's earlier uses and of this use's arguments (arrays by dtype, shape and bytes).  The reference's answer is stored
under that key in reference_calls.npz, and replaying looks the key up: a test gets the reference's answer to exactly the
input it passes, and an input that was never recorded is an error, not a skip.  The chirp tables and ifreq() outputs,
which the tests compare byte for byte, are stored as their SHA-256 only (`Digest`) to keep the file small.

To re-record, with oracle/_ref/liblora_ref.so built (new answers are merged into the file's existing ones; the CFO test
needs a GPU because its window is placed by the device's step trace):

    GR_LORA_RECORD_REFERENCE=tests/golden/reference_calls.npz python -m pytest tests/test_ref_pins_oracle.py
    GR_LORA_RECORD_REFERENCE=tests/golden/reference_calls.npz python -m pytest tests/test_gpu_stream.py -k cfo_estimate
"""
from __future__ import annotations

import builtins
import hashlib
import inspect
import io
import json
import os
from pathlib import Path

import numpy as np

STORE = Path(__file__).resolve().parent / "reference_calls.npz"
RECORD_ENV = "GR_LORA_RECORD_REFERENCE"
DIGEST_ONLY = {"downchirp", "upchirp", "downchirp_ifreq", "upchirp_ifreq", "upchirp_ifreq_v", "ifreq"}


class Digest(str):
    """SHA-256 of the bytes of an array the reference returned, stored in place of the array."""


def digest(a) -> Digest:
    return a if isinstance(a, Digest) else Digest(hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())


def _feed(h, v):
    if isinstance(v, np.generic):
        v = v.item()
    if isinstance(v, np.ndarray):
        h.update(f"nd:{v.dtype.str}:{v.shape}:".encode())
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (list, tuple)):
        h.update(b"(")
        for e in v:
            _feed(h, e)
        h.update(b")")
    elif v is None or isinstance(v, (bool, int, float, str, bytes)):
        h.update(f"{type(v).__name__}:{v!r};".encode())
    else:
        raise TypeError(f"cannot key an argument of type {type(v).__name__}")


def _key(prev: str, name: str, args=(), kwargs=None) -> str:
    h = hashlib.sha256(prev.encode() + b"|" + name.encode() + b"|")
    _feed(h, tuple(args))
    _feed(h, tuple(sorted((kwargs or {}).items())))
    return h.hexdigest()[:16]


class _Store:
    def __init__(self, live, out: Path | None):
        self.live, self.out = live, out
        self.calls, self.arrays = {}, {}
        if STORE.exists():
            with np.load(STORE, allow_pickle=False) as z:
                self.calls = json.loads(bytes(z["calls"]).decode())
                self.arrays = {k: z[k] for k in z.files if k != "calls"}

    def _pack(self, v, key, name):
        if isinstance(v, np.generic):
            v = v.item()
        if isinstance(v, np.ndarray):
            if name in DIGEST_ONLY:
                return {"digest": digest(v)}
            aname = f"{key}.{sum(k.startswith(key + '.') for k in self.arrays)}"
            self.arrays[aname] = v
            return {"array": aname}
        if isinstance(v, bytes):
            return {"bytes": v.hex()}
        if isinstance(v, (list, tuple)):
            return {type(v).__name__: [self._pack(e, key, name) for e in v]}
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        raise TypeError(f"cannot record a {type(v).__name__} returned by {name}")

    def _unpack(self, p):
        if not isinstance(p, dict):
            return p
        if "digest" in p:
            return Digest(p["digest"])
        if "array" in p:
            return self.arrays[p["array"]].copy()
        if "bytes" in p:
            return bytes.fromhex(p["bytes"])
        if "tuple" in p:
            return tuple(self._unpack(e) for e in p["tuple"])
        return [self._unpack(e) for e in p["list"]]

    def call(self, key, name, fn):
        if self.live is None:
            if key not in self.calls:
                raise LookupError(f"no recorded answer of the reference for this use of {name} (the input or the order "
                                  f"of calls differs from the recording; re-record with {RECORD_ENV}, see tests/golden/refcalls.py)")
            p = self.calls[key]
            if isinstance(p, dict) and "raises" in p:
                raise getattr(builtins, p["raises"])(p["message"])
            return self._unpack(p)
        for k in [k for k in self.arrays if k.startswith(key + ".")]:
            del self.arrays[k]
        try:
            v = fn()
        except (ValueError, RuntimeError, AssertionError) as exc:
            self.calls[key] = {"raises": type(exc).__name__, "message": str(exc)}
            raise
        self.calls[key] = self._pack(v, key, name)
        return v

    def save(self):
        buf = io.BytesIO()
        np.savez_compressed(buf, calls=np.frombuffer(json.dumps(self.calls, sort_keys=True).encode(), np.uint8),
                            **dict(sorted(self.arrays.items())))
        self.out.write_bytes(buf.getvalue())


class _RecordedDecoder:
    """oracle.ref.RefDecoder, answered from the store."""

    def __init__(self, store, *args, **kwargs):
        self._store, self._prev, self._live = store, _key("RefDecoder", "__init__", args, kwargs), None

        def create():
            self._live = store.live.RefDecoder(*args, **kwargs)
        store.call(self._prev, "RefDecoder", create)

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        from oracle.ref import RefDecoder
        if inspect.isfunction(inspect.getattr_static(RefDecoder, name, None)):
            def method(*args, **kwargs):
                self._prev = _key(self._prev, name, args, kwargs)
                return self._store.call(self._prev, name, lambda: getattr(self._live, name)(*args, **kwargs))
            return method
        self._prev = _key(self._prev, name)
        return self._store.call(self._prev, name, lambda: getattr(self._live, name))


class Reference:
    """Stands in for the module oracle.ref: RefDecoder and its module-level functions."""

    def __init__(self, store):
        self._store = store

    def RefDecoder(self, *args, **kwargs):
        return _RecordedDecoder(self._store, *args, **kwargs)

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def function(*args, **kwargs):
            return self._store.call(_key("oracle.ref", name, args, kwargs), name,
                                    lambda: getattr(self._store.live, name)(*args, **kwargs))
        return function


def open_reference():
    """(Reference, store): replays reference_calls.npz, or, with GR_LORA_RECORD_REFERENCE=<file>, calls the built
    reference and records its answers into <file> when store.save() is called."""
    out = os.environ.get(RECORD_ENV)
    live = None
    if out:
        from oracle import ref as R
        if not R.available():
            raise RuntimeError(f"{RECORD_ENV} is set but the reference is not built (oracle/ref.py)")
        R.lib()
        live = R
    store = _Store(live, Path(out) if out else None)
    return Reference(store), store
