"""Compact storage of the layer goldens (reference_layers.npz).

A member with more than MAX_WHOLE elements is stored as four entries: ``<name>#shape``, ``<name>#sha256`` (of the
whole array's canonical bits, see `canonical`), ``<name>#rows`` (SAMPLE_ROWS row indices drawn with a seed derived
from the name) and ``<name>#sample`` (those rows). `Golden` hands such a member back as a `Sampled`. The tests compare
a computed array with it on all of these. The shape and the digest cover every element, and the sampled rows name
the first differing element when they differ. Smaller members are stored whole.
"""
import hashlib
import zlib

import numpy as np

MAX_WHOLE = 2048
SAMPLE_ROWS = 64


def rows_of(a):
    """Rows of an array: its last axis when that is short (a box, a channel group), else its single elements."""
    a = np.asarray(a)
    return a.reshape(-1, a.shape[-1]) if a.ndim and a.shape[-1] <= 16 else a.reshape(-1, 1)


def canonical(a, as_float: bool) -> np.ndarray:
    """What a bit-for-bit comparison compares: float32 with every NaN as one pattern, or int64."""
    a = np.asarray(a)
    if as_float:
        a = a.astype(np.float32)
        return np.ascontiguousarray(np.where(np.isnan(a), np.float32(np.nan), a))
    return np.ascontiguousarray(a.astype(np.int64))


def digest(a) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def shrink(members: dict) -> dict:
    """The entries to store for `members` (name -> array)."""
    out = {}
    for name, a in members.items():
        a = np.asarray(a)
        if a.size <= MAX_WHOLE:
            out[name] = a
            continue
        r = rows_of(a)
        rs = np.random.RandomState(zlib.crc32(name.encode()))
        rows = np.sort(rs.choice(r.shape[0], min(SAMPLE_ROWS, r.shape[0]), replace=False)).astype(np.int32)
        out[name + "#shape"] = np.array(a.shape, np.int64)
        out[name + "#sha256"] = digest(canonical(a, a.dtype.kind == "f"))
        if a.dtype.kind != "f":       # a float result compared with an integer golden is compared as float32
            out[name + "#sha256_f32"] = digest(canonical(a, True))
        out[name + "#rows"] = rows
        out[name + "#sample"] = r[rows]
    return out


class Sampled:
    """A large golden member: shape, digests of the whole array, and a seeded sample of its rows."""

    def __init__(self, shape, sha256, sha256_f32, rows, sample):
        self.shape, self.sha256, self.sha256_f32, self.rows, self.sample = tuple(shape), sha256, sha256_f32, rows, sample

    def check(self, got, what, bits):
        """Assert got equals the stored array; `bits(a, b, what)` compares the sampled rows element by element."""
        got = np.asarray(got)
        assert got.shape == self.shape, (what, got.shape, self.shape)
        bits(rows_of(got)[self.rows], self.sample, f"{what} (sampled rows)")
        as_float = got.dtype.kind == "f" or self.sample.dtype.kind == "f"
        want = self.sha256_f32 if as_float and self.sample.dtype.kind != "f" else self.sha256
        assert np.array_equal(digest(canonical(got, as_float)), want), f"{what}: differs outside the sampled rows"


class Golden:
    """The .npz with every member under its own name (a stored sample comes back as a `Sampled`)."""

    def __init__(self, path):
        self._z = np.load(path)
        self.files = sorted({k.split("#")[0] for k in self._z.files})

    def __contains__(self, name):
        return name in self.files

    def __getitem__(self, name):
        if name in self._z.files:
            return self._z[name]
        if name not in self.files:
            raise KeyError(name)
        z = self._z
        return Sampled(z[name + "#shape"], z[name + "#sha256"],
                       z[name + "#sha256_f32"] if name + "#sha256_f32" in z.files else None,
                       z[name + "#rows"], z[name + "#sample"])
