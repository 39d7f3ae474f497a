"""Calls into the reference build (oracle/_ref/*.so), recorded once and replayed where that build is absent.

The reference libraries are compiled from the original project's sources, which only some build machines hold.  A test
reaches them through the `reference` fixture (tests/conftest.py):

    r = reference.new(ref.RefMapper, prm, laser)      # an object of the reference build
    ok, pose = r.process(ranges[i], odom[i], t)       # its methods
    cells = reference.call("lines", fn, segs)         # any other computation on the reference build

Where the reference build is present every call goes to it.  Elsewhere each call is answered from
tests/golden/reference/<test module>.pkl.xz, in the order the test made it, after checking that the test passed the same
arguments as when it was recorded (so a changed workload fails instead of comparing against stale numbers).  Arrays
above 64 KB are stored as a SHA-256 digest of their bytes; `same()` and `same_bits()` compare against either form.

Record (where the reference build is present):  B2S_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"
and, for the GPU tests that use the fixture, the same with -m gpu on a machine with a GPU."""
import ctypes
import dataclasses
import hashlib
import lzma
import os
import pickle

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
_INLINE_BYTES = 65536  # arrays larger than this are kept as a digest only


@dataclasses.dataclass(frozen=True)
class Digest:
    """An array result too large to store: its dtype, shape and the SHA-256 of its bytes."""
    dtype: str
    shape: tuple
    sha256: str


@dataclasses.dataclass(frozen=True)
class Opaque:
    """A result that cannot be stored (a ctypes vtable, say); it can only be passed back to the reference."""
    type_name: str


def _sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def same(ours, theirs, equal_nan=False) -> bool:
    """np.array_equal, where `theirs` may be a recorded Digest: then the bytes must match."""
    if isinstance(theirs, Digest):
        a = np.asarray(ours)
        if a.shape != theirs.shape:
            return False
        if a.dtype.str != theirs.dtype:
            b = a.astype(theirs.dtype)
            if not np.array_equal(b, a):
                return False
            a = b
        return _sha(a) == theirs.sha256
    return np.array_equal(ours, theirs, equal_nan=equal_nan)


def same_bits(ours, theirs) -> bool:
    """Equal dtype, shape and bytes (float bit patterns included), where `theirs` may be a recorded Digest."""
    a = np.asarray(ours)
    if isinstance(theirs, Digest):
        return a.dtype.str == theirs.dtype and same(a, theirs)
    b = np.asarray(theirs)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _key(x):
    """A stable description of an argument (arrays by content digest)."""
    if isinstance(x, _Proxy):
        return ("proxy", x._label)
    if isinstance(x, Opaque):
        return ("opaque", x.type_name)
    if isinstance(x, np.ndarray):
        return ("nd", x.dtype.str, x.shape, _sha(x))
    if isinstance(x, np.generic):
        return ("np", x.dtype.str, repr(x.item()))
    if x is None or isinstance(x, (bool, int, float, str, bytes)):
        return repr(x)
    if isinstance(x, (tuple, list)):
        return tuple(_key(v) for v in x)
    if isinstance(x, dict):
        return tuple(sorted((k, _key(v)) for k, v in x.items()))
    if dataclasses.is_dataclass(x):
        return (type(x).__name__,) + tuple(_key(getattr(x, f.name)) for f in dataclasses.fields(x))
    if isinstance(x, ctypes.Structure):
        if any(issubclass(f[1], (ctypes._Pointer, ctypes._CFuncPtr, ctypes.c_void_p)) for f in x._fields_):
            return ("opaque", type(x).__name__)  # addresses differ from run to run
        return (type(x).__name__,) + tuple(_key(getattr(x, f[0])) for f in x._fields_)
    if isinstance(x, ctypes.Array):
        return tuple(_key(v) for v in x)
    return ("opaque", type(x).__name__)


def _args_digest(args, kw) -> str:
    return hashlib.sha256(repr((_key(tuple(args)), _key(kw))).encode()).hexdigest()[:16]


def _store(x):
    """What is kept of a result."""
    if isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        if a.nbytes > _INLINE_BYTES:
            return Digest(a.dtype.str, a.shape, _sha(a))
        return a.copy()
    if x is None or isinstance(x, (bool, int, float, str, bytes, np.generic)):
        return x
    if isinstance(x, tuple):
        return tuple(_store(v) for v in x)
    if isinstance(x, list):
        return [_store(v) for v in x]
    if isinstance(x, dict):
        return {k: _store(v) for k, v in x.items()}
    return Opaque(type(x).__name__)


class _Proxy:
    """A reference-build object: live (calls go to `_obj`) or replayed (`_obj` is None)."""

    def __init__(self, session, label, obj):
        self._session, self._label, self._obj = session, label, obj

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        target = None if self._obj is None else getattr(self._obj, name)
        return lambda *a, **kw: self._session._do(f"{self._label}.{name}", target, a, kw)


class Session:
    """The reference calls of one test."""

    def __init__(self, module: str, test: str, live: bool, record: bool):
        self.path = os.path.join(GOLDEN, module + ".pkl.xz")
        self.test, self.live, self.record = test, live, record
        self.calls, self._n, self._depth = [], {}, 0
        if not live:
            if not os.path.exists(self.path):
                raise RuntimeError(f"no recorded reference calls in {self.path}; record them where oracle/_ref/ is built")
            with lzma.open(self.path, "rb") as f:
                book = pickle.load(f)
            if test not in book:
                raise RuntimeError(f"{self.path} has no recording for {test}; record it where oracle/_ref/ is built")
            self.calls = book[test]
        self._next = 0

    def new(self, cls, *args, **kw) -> _Proxy:
        k = self._n[cls.__name__] = self._n.get(cls.__name__, -1) + 1
        label = f"{cls.__name__}#{k}"
        obj = self._do(label + ".new", cls if self.live else None, args, kw, keep=False)
        return _Proxy(self, label, obj)

    def call(self, name: str, fn, *args, **kw):
        return self._do(name, fn, args, kw)

    def _do(self, label, fn, args, kw, keep=True):
        if self._depth:  # inside a recorded call: only the outermost one is recorded
            return fn(*args, **kw)
        digest = _args_digest(args, kw)
        if self.live:
            self._depth += 1
            try:
                out = fn(*args, **kw)
            finally:
                self._depth -= 1
            if self.record:
                self.calls.append((label, digest, _store(out) if keep else None))
            return out
        assert self._next < len(self.calls), f"{self.test}: more reference calls than were recorded ({label})"
        want_label, want_digest, out = self.calls[self._next]
        self._next += 1
        assert (label, digest) == (want_label, want_digest), \
            f"{self.test}: call {self._next} is {label} {digest}, the recording has {want_label} {want_digest}"
        return out

    def finish(self):
        if not self.live:
            assert self._next == len(self.calls), f"{self.test}: {len(self.calls) - self._next} recorded calls not made"
        elif self.record:
            book = {}
            if os.path.exists(self.path):
                with lzma.open(self.path, "rb") as f:
                    book = pickle.load(f)
            book[self.test] = self.calls
            os.makedirs(GOLDEN, exist_ok=True)
            with lzma.open(self.path, "wb", preset=9) as f:
                pickle.dump(book, f, protocol=4)
