"""The reference's own results for the calls tests/test_ref_pin.py makes, so that the comparison runs without the reference.

oracle/ref_binding.py drives the reference's classes compiled from its sources (oracle/_ref, oracle/build_ref.py); those sources
are not part of this repository.  Every call the tests make through `reference()` is keyed by the name of the test and its position
in the test; tests/golden/ref_pin.npz stores, per call, a digest of the inputs, what the call returned and how it changed the
arrays it was given (as an XOR of the bit patterns, which compresses to almost nothing where nothing changed).  Replaying checks
the digest first: inputs that differ from those the data was made with fail the test instead of comparing against the wrong
results.  File arguments enter the digest by their contents, and a file the reference wrote is written again.

To remake the data where oracle/_ref can be built:  LEXP_MINT_GOLDEN=1 python -m pytest tests/test_ref_pin.py
"""
import hashlib
import json
import lzma
import os

import numpy as np

from oracle.lexp_oracle import COST_FOR_INVALID

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin.npz")
MINT = os.environ.get("LEXP_MINT_GOLDEN") == "1"
_UINT = {4: np.uint32, 8: np.uint64, 2: np.uint16, 1: np.uint8}
DROPPED = -7.25e30          # stands for an element thin() did not keep


def thin(a, keep=1 / 32):
    """A seeded sample of a large result, to keep the stored data small: every non-finite or COST_FOR_INVALID element (masks stay
    whole), a fraction `keep` of the others; the rest read DROPPED.  Pass as `_keep=thin` to a reference call."""
    a = np.array(a, copy=True)
    mask = np.random.default_rng(a.size).random(a.shape) < keep
    mask |= ~np.isfinite(a) | (a == COST_FOR_INVALID)
    a[~mask] = DROPPED
    return a


def kept(a):
    return a != DROPPED


def _digest(name, args, kwargs, extra=""):
    h = hashlib.sha256((name + "|" + extra).encode())

    def feed(a):
        if isinstance(a, (str, os.PathLike)):
            if os.path.isfile(a):
                with open(a, "rb") as f:
                    h.update(b"file:" + f.read())
            else:
                h.update(b"path")                  # where a file goes is not part of the input
            return
        if isinstance(a, (np.ndarray, list, tuple)):
            try:
                x = np.ascontiguousarray(np.asarray(a))
                if x.dtype != object:
                    h.update(f"{x.dtype.str}{x.shape}".encode() + x.tobytes())
                    return
            except ValueError:                     # ragged lists
                pass
        h.update(repr(a).encode())

    for a in args:
        feed(a)
    for k in sorted(kwargs):
        h.update(k.encode())
        feed(kwargs[k])
    return h.hexdigest()[:24]


class _Store:
    def __init__(self):
        self.test, self.n = None, 0
        if MINT:
            self.index, self.arrays = {}, {}
        else:
            with np.load(PATH) as z:
                meta = json.loads(lzma.decompress(z["index"].tobytes()).decode())
                data = np.frombuffer(lzma.decompress(z["data"].tobytes()), np.uint8)
            self.index, self.arrays = meta["calls"], {}
            for k, (off, dt, shape) in meta["arrays"].items():
                n = int(np.prod(shape)) * np.dtype(dt).itemsize
                self.arrays[k] = data[off:off + n].view(np.dtype(dt)).reshape(shape)

    def save(self):
        """One index and one byte string holding every array, each compressed with lzma (several times smaller than zlib here)."""
        parts, where, off = [], {}, 0
        for k, a in self.arrays.items():
            b = np.ascontiguousarray(a)
            where[k] = (off, b.dtype.str, list(b.shape))
            parts.append(b.reshape(-1).view(np.uint8))
            off += b.nbytes
        meta = json.dumps({"calls": self.index, "arrays": where}, sort_keys=True).encode()
        data = np.concatenate(parts).tobytes() if parts else b""
        np.savez(PATH, index=np.frombuffer(lzma.compress(meta, preset=9 | lzma.PRESET_EXTREME), np.uint8),
                 data=np.frombuffer(lzma.compress(data, preset=9 | lzma.PRESET_EXTREME), np.uint8))

    def _enc(self, v, key):
        if isinstance(v, np.ndarray) and v.dtype.kind == "f" and (v == DROPPED).any():
            k = kept(v)                       # thinned: the kept elements and where they are
            self.arrays[key] = v[k]
            self.arrays[key + "m"] = np.packbits(k)
            return {"k": key, "shape": list(v.shape), "dtype": v.dtype.str}
        if isinstance(v, np.ndarray):
            self.arrays[key] = v
            return {"a": key}
        if isinstance(v, tuple):
            return {"t": [self._enc(x, f"{key}.{i}") for i, x in enumerate(v)]}
        if isinstance(v, dict):
            return {"d": {k: self._enc(x, f"{key}.{k}") for k, x in v.items()}}
        if isinstance(v, list) and v and all(isinstance(x, tuple) and len(x) == len(v[0]) for x in v):
            self.arrays[key] = np.asarray(v, np.int32)
            return {"l": key}             # a list of equal-length tuples (rectangles)
        if isinstance(v, np.generic):
            v = v.item()
        if isinstance(v, int) and not isinstance(v, bool):
            return {"i": str(v)}           # uint64 RNG states do not fit a JSON number everywhere
        return {"v": v}                    # float (repr round-trips), bool, None, lists

    def _dec(self, s):
        if "a" in s:
            return self.arrays[s["a"]].copy()
        if "k" in s:
            a = np.full(s["shape"], DROPPED, np.dtype(s["dtype"]))
            n = a.size
            a[np.unpackbits(self.arrays[s["k"] + "m"], count=n).reshape(a.shape).astype(bool)] = self.arrays[s["k"]]
            return a
        if "t" in s:
            return tuple(self._dec(x) for x in s["t"])
        if "d" in s:
            return {k: self._dec(x) for k, x in s["d"].items()}
        if "l" in s:
            return [tuple(int(x) for x in r) for r in self.arrays[s["l"]]]
        if "i" in s:
            return int(s["i"])
        return s["v"]

    def call(self, name, fn, args, kwargs, extra=""):
        if self.test is None:
            raise RuntimeError("reference call outside a test")
        key = f"{self.test}#{self.n}"
        self.n += 1
        reduce = kwargs.pop("_keep", None)
        dig = _digest(name, args, kwargs, extra)
        arrays = [a for a in list(args) + list(kwargs.values()) if isinstance(a, np.ndarray) and a.flags.writeable and a.dtype.itemsize in _UINT]
        if MINT:
            before = [a.copy() for a in arrays]
            out = fn(*args, **kwargs)
            if reduce is not None:
                out = reduce(out)
            changed = {}
            for i, (a, b) in enumerate(zip(arrays, before)):
                if not np.array_equal(a.view(_UINT[a.dtype.itemsize]), b.view(_UINT[b.dtype.itemsize])):
                    changed[str(i)] = self._enc(a.view(_UINT[a.dtype.itemsize]) ^ b.view(_UINT[b.dtype.itemsize]), f"{key}.x{i}")
            for a in args:
                if name == "save_pfm" and isinstance(a, (str, os.PathLike)):
                    with open(a, "rb") as f:
                        changed["file"] = self._enc(np.frombuffer(f.read(), np.uint8).copy(), f"{key}.file")
            self.index[key] = {"name": name, "digest": dig, "out": self._enc(out, f"{key}.o"), "changed": changed}
            return out
        rec = self.index.get(key)
        assert rec is not None and rec["name"] == name, f"{key}: no stored reference result for {name} (remake tests/golden/ref_pin.npz)"
        assert rec["digest"] == dig, f"{key} ({name}): the inputs differ from those the stored reference results were made with"
        for i, s in rec["changed"].items():
            if i == "file":
                path = next(a for a in args if isinstance(a, (str, os.PathLike)))
                with open(path, "wb") as f:
                    f.write(self._dec(s).tobytes())
            else:
                a = arrays[int(i)]
                a.view(_UINT[a.dtype.itemsize])[...] ^= self._dec(s)
        return self._dec(rec["out"])


_store = None


def store():
    global _store
    if _store is None:
        _store = _Store()
    return _store


class _Energy:
    """Stands for ref_binding.RefEnergy: construction is part of every method call's digest."""

    def __init__(self, *args, **kwargs):
        self._extra = _digest("RefEnergy", args, kwargs)
        self._real = None
        if MINT:
            from oracle import ref_binding
            self._real = ref_binding.RefEnergy(*args, **kwargs)

    def close(self):
        if self._real is not None:
            self._real.close()

    def __getattr__(self, name):
        fn = getattr(self._real, name) if self._real is not None else None
        return lambda *a, **k: store().call("RefEnergy." + name, fn, a, k, self._extra)


class _Reference:
    """The module oracle/ref_binding.py as tests/test_ref_pin.py uses it."""
    RefEnergy = _Energy

    def __getattr__(self, name):
        fn = None
        if MINT:
            from oracle import ref_binding
            fn = getattr(ref_binding, name)
        return lambda *a, **k: store().call(name, fn, a, k)


def reference():
    return _Reference()
