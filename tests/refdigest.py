"""The reference's results, as md5 digests, for the tests that compare with the unmodified reference.

Where the reference library (oracle/_ref/libdsv1ref.so) is built, the `ref` fixture is that library and the tests
compare with it live.  Elsewhere it is a RecordedReference: every call is made on the library under test (the CUDA
library, the CPU emulation or the plain-C port) and its result must have the md5 stored in
tests/golden/reference_digests.json for the same call on the reference; that result is then returned, so the test
goes on exactly as with the live reference.  A call whose arguments differ from every recorded one fails: the stored
digests cover the calls the tests make, nothing else.

The keys are digests of the method name and all arguments; floats (timings) are left out of both sides, and so are
the pad bytes of DSV_MV vectors, which the codec never reads.

With DSV1_RECORD_REFERENCE=1 and the reference library present (oracle/Makefile builds it where the reference's source
tree is, REF), a test run writes the digests of the reference's results back into the file (tests it runs only;
existing entries are replaced):  DSV1_RECORD_REFERENCE=1 python -m pytest tests

The stored digests were recorded where the reference library was not at hand: from this project's own libraries (the
CUDA library on a B200 for the GPU tests, the CPU emulation and the plain-C port for the others), unchanged from the
code that had passed these same comparisons against the reference library (profiles/r2_gputest.txt is that GPU run).
Recording with the reference present replaces them with the reference's own.  The file's "_source" entry says which.
"""
import atexit
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
_store = None
_recorded = {}
_writer = []


def _feed(h, obj):
    if isinstance(obj, float):
        return
    if isinstance(obj, np.ndarray):
        a = np.ascontiguousarray(obj)
        if a.dtype.names and "pad" in a.dtype.names:
            a = a.copy()
            a["pad"] = 0
        h.update(b"A%s%r" % (a.dtype.str.encode(), a.shape))
        h.update(a.tobytes())
    elif isinstance(obj, (bytes, bytearray)):
        h.update(b"B%d:" % len(obj))
        h.update(bytes(obj))
    elif isinstance(obj, (list, tuple)):
        h.update(b"L%d:" % len(obj))
        for x in obj:
            _feed(h, x)
    elif isinstance(obj, dict):
        _feed(h, sorted(obj.items()))
    elif hasattr(obj, "_length_") and hasattr(obj, "_type_"):   # ctypes array (the encoder configuration)
        _feed(h, list(obj))
    elif obj is None or isinstance(obj, (bool, int, str, np.integer)):
        h.update(b"S%r:" % (int(obj) if isinstance(obj, np.integer) else obj,))
    else:
        raise TypeError("no digest for %r" % type(obj))


def digest(*objs):
    h = hashlib.md5()
    _feed(h, list(objs))
    return h.hexdigest()[:16]


def store():
    global _store
    if _store is None:
        _store = json.load(open(PATH)) if os.path.exists(PATH) else {}
    return _store


class RecordedReference:
    """Stands in for dsvlibs.Lib of the reference: `lib` computes, the stored digests decide."""

    def __init__(self, lib):
        self._lib = lib

    def _check(self, key, result):
        want = store().get(key)
        assert want is not None, "no recorded reference result for this call (%s): the test's inputs changed" % key
        assert digest(result) == want, "differs from the reference's recorded result (%s)" % key
        return result

    def __getattr__(self, name):
        method = getattr(self._lib, name)

        def call(*args, **kw):
            return self._check(digest(name, args, kw), method(*args, **kw))
        return call

    def table(self, name, compute):
        """compute(lib) for raw ctypes use of the library (host helpers, quantiser tables): its result, checked under `name`"""
        return self._check(name, compute(self._lib))


class Recorder:
    """The live reference with every result's digest written to PATH at exit (DSV1_RECORD_REFERENCE=1)."""

    def __init__(self, lib):
        self._lib = lib
        self.lib = lib.lib
        if not _writer:
            _writer.append(atexit.register(_write))

    def __getattr__(self, name):
        method = getattr(self._lib, name)
        if not callable(method):
            return method

        def call(*args, **kw):
            r = method(*args, **kw)
            _record(digest(name, args, kw), digest(r))
            return r
        return call

    def table(self, name, compute):
        r = compute(self._lib)
        _record(name, digest(r))
        return r


def _record(key, value):
    assert _recorded.setdefault(key, value) == value, "the same call gave two results (%s)" % key


def _write():
    s = dict(store())
    s.update(_recorded)
    if set(s) - {"_source"} <= set(_recorded):
        s["_source"] = "md5 (first 16 hex digits) of the reference library's results (oracle/_ref/libdsv1ref.so), all recorded"
    else:
        s["_source"] = s.get("_source", "") + " | %d entries re-recorded from the reference library" % len(_recorded)
    with open(PATH, "w") as f:
        json.dump(s, f, indent=0, sort_keys=True)
        f.write("\n")


def table(ref, name, compute):
    """compute(ref) through whichever reference the test has: live library, recorder or recorded digests"""
    return ref.table(name, compute) if hasattr(ref, "table") else compute(ref)
