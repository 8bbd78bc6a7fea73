"""Reference outputs kept under tests/golden/ in reduced form, so that the comparisons with the reference run without it.

An array that a test compares bit for bit is stored as a digest (part of its SHA-256).  An array that a test compares
within a tolerance is stored as its largest magnitude, a fixed sample of SAMPLE entries and a sketch P @ X @ Q with
random +-1 matrices P and Q.  Small arrays are stored whole.  `same` and `abs_err` accept either a whole array or a
`Reduced` one as the reference.  Against a reduced reference `abs_err` returns a lower bound of the largest entrywise
difference, so every check that passes against the whole array also passes against its reduced form.

The reverse does not hold: the reduced check is weaker.  It catches any difference at the sampled entries, and any
non-finite entry.  Elsewhere it only catches a difference once its sketch reaches the tolerance, which for one lone
entry means an error about rows x cols times the tolerance (a 512 x 128 block at 1e-11: about 7e-7 relative).
Errors that spread over many entries (a wrong block, a missing contribution, a stale buffer) move the sketch by far
more than that.  Where oracle/_ref is built, the tests compare with its whole outputs instead."""
import hashlib
import json

import numpy as np

WHOLE = 32  # arrays of at most this many entries are stored as they are
SAMPLE = 8
SKETCH = (4, 2)


def _canonical(a):
    a = np.asarray(a)
    return np.ascontiguousarray(a, np.float64 if a.dtype.kind in "fc" else np.int64)


def digest(a):
    """The first 8 bytes of the SHA-256 of shape and contents: enough to tell any two arrays apart by accident."""
    a = _canonical(a)
    return np.frombuffer(hashlib.sha256(np.asarray(a.shape, np.int64).tobytes() + a.tobytes()).digest()[:8], np.uint8)


def _probes(shape):
    rows = int(shape[0]) if len(shape) else 1
    cols = int(np.prod(shape[1:])) if len(shape) > 1 else 1
    rng = np.random.default_rng([rows, cols, 0x5EED])
    P = rng.choice([-1.0, 1.0], (SKETCH[0], rows))
    Q = rng.choice([-1.0, 1.0], (cols, SKETCH[1] if cols > 1 else 1))
    idx = np.sort(rng.choice(rows * cols, min(SAMPLE, rows * cols), replace=False))
    return P, Q, idx


def _sketch(a, P, Q):
    return P @ np.asarray(a, np.float64).reshape(P.shape[1], Q.shape[0]) @ Q


def reduce_into(out: dict, key: str, a, exact: bool):
    """Store array `a` under `key` in `out` (the arrays of an .npz file)."""
    a = np.asarray(a)
    if a.size <= WHOLE:
        out[key] = a
        return
    out[key + "__shape"] = np.asarray(a.shape, np.int64)
    if exact:
        out[key + "__sha256"] = digest(a)
        return
    P, Q, idx = _probes(a.shape)
    out[key + "__absmax"] = np.float64(np.abs(a).max())
    out[key + "__sample"] = np.asarray(a, np.float64).reshape(-1)[idx]
    out[key + "__sketch"] = _sketch(a, P, Q)


class Reduced:
    def __init__(self, z, key):
        self.key = key
        self.shape = tuple(int(x) for x in z[key + "__shape"])
        self.sha = z[key + "__sha256"] if key + "__sha256" in z.files else None
        if self.sha is None:
            self.absmax = float(z[key + "__absmax"])
            self.sample = z[key + "__sample"]
            self.sketch = z[key + "__sketch"]

    def __len__(self):
        return self.shape[0]

    @property
    def size(self):
        return int(np.prod(self.shape))

    def __repr__(self):
        return f"<reduced reference {self.key} {self.shape}>"


def save(path, arrays: dict):
    """All arrays of one golden file packed into two members (an index and one byte string): a reduced file holds many
    tiny arrays, and an .npz member costs a few hundred bytes of headers."""
    index, blobs, at = {}, [], 0
    for k, a in arrays.items():
        a = np.asarray(a)
        index[k] = [a.dtype.str, list(a.shape), at, a.nbytes]
        blobs.append(a.tobytes())
        at += a.nbytes
    np.savez_compressed(path, index=np.frombuffer(json.dumps(index).encode(), np.uint8),
                        blob=np.frombuffer(b"".join(blobs), np.uint8))


class Packed:
    """A golden file written by `save`, read like an opened .npz."""

    def __init__(self, z):
        self.index = json.loads(bytes(z["index"]).decode())
        self.blob = z["blob"]
        self.files = list(self.index)

    def __getitem__(self, k):
        dtype, shape, at, n = self.index[k]
        return np.frombuffer(self.blob[at:at + n].tobytes(), np.dtype(dtype)).reshape(shape)


def open_golden(path):
    z = np.load(path, allow_pickle=False)
    return Packed(z) if set(z.files) == {"index", "blob"} else z


def load(z, key):
    """The reference array `key` of the opened .npz `z`: an ndarray, or a `Reduced` one."""
    if key in z.files:
        return z[key]
    return Reduced(z, key)


def same(have, want) -> bool:
    if isinstance(want, Reduced):
        if want.sha is None:
            raise TypeError(f"{want.key} is stored for comparisons within a tolerance")
        return tuple(np.shape(have)) == want.shape and np.array_equal(digest(have), want.sha)
    return np.array_equal(have, want)


def absmax(want) -> float:
    return want.absmax if isinstance(want, Reduced) else float(np.abs(want).max())


def abs_err(have, want) -> float:
    """max |have - want| (a lower bound of it for a reduced `want`; inf if the shapes differ or `have` holds a NaN or
    an infinity)."""
    if tuple(np.shape(have)) != tuple(want.shape):
        return float("inf")
    if not np.all(np.isfinite(have)):  # the reference has none; the sample and the sketch could miss or hide one
        return float("inf")
    if not isinstance(want, Reduced):
        return float(np.abs(np.asarray(have) - want).max()) if want.size else 0.0
    P, Q, idx = _probes(want.shape)
    sampled = float(np.abs(np.asarray(have, np.float64).reshape(-1)[idx] - want.sample).max())
    # every entry of P @ D @ Q sums |D| over rows x cols terms with weight 1
    sketched = float(np.abs(_sketch(have, P, Q) - want.sketch).max()) / (P.shape[1] * Q.shape[0])
    return max(sampled, sketched)


def rel_err(have, want) -> float:
    return abs_err(have, want) / max(absmax(want), 1e-300)
