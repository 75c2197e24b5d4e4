"""Stored answers of the unmodified reference (oracle/_ref/libxsmm_ref.so) for the tests that compare against it.

The reference is only built where its source tree is available. So that the comparisons also run everywhere else, the
answers it gave on the tests' seeded inputs are kept in tests/golden/ref/<test module>.npz:

  same(fn, got)       fn() computes the reference's answer; asserts that `got` equals it bit for bit
  sampled(fn, got)    -> (want, got): the reference's answer and `got`, for a tolerance comparison by the caller
  value(fn)           -> the reference's answer itself (small results: return codes, statistics)

fn() returns a numpy array (any shape; None where the reference declines the case). With the reference library present
fn() runs and its result is used as is. Without it the stored answer is used: `same` compares a 64-bit digest of the
canonical bytes, `sampled` returns a fixed, seeded sample of SAMPLE elements of both arrays (the whole arrays when they
are small). Answers are keyed by test id and call order, so a test must ask in a deterministic order; the answers of one
test are stored as one byte string with a table of (offset, length, dtype) per call.

To re-record (where the reference is built), run the tests with LIBXSMM_B200_RECORD_REF=<directory>: the answers
are merged into <directory>/<test module>.npz at exit; copy those files to tests/golden/ref/."""
import atexit
import hashlib
import os
import zlib

import numpy as np

from oracle_ffi import ref_lib

STORE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
RECORD = os.environ.get("LIBXSMM_B200_RECORD_REF")
SAMPLE = 128
LIVE = ref_lib is not None
_stores, _recorded, _calls = {}, {}, {}


def _key():
    cur = os.environ["PYTEST_CURRENT_TEST"].rsplit(" (", 1)[0]
    module = os.path.basename(cur.split("::", 1)[0])[:-3]
    test = cur.split("::", 1)[1]
    n = _calls.get((module, test), 0)
    _calls[(module, test)] = n + 1
    return module, (test, n)


def _load(path):
    tests = {}
    if os.path.exists(path):
        with np.load(path) as z:
            for name in z.files:
                if name.endswith(":data"):
                    test = name[:-5]
                    data, table = z[name].tobytes(), z[test + ":table"]
                    tests[test] = [np.frombuffer(data[int(o):int(o) + int(n)], dtype=np.dtype(str(t))) for o, n, t in table]
    return tests


def _stored(module, key):
    if module not in _stores:
        _stores[module] = _load(os.path.join(STORE, module + ".npz"))
    test, n = key
    answers = _stores[module].get(test, [])
    assert n < len(answers), "no stored reference answer for %s::%s call %d (record with LIBXSMM_B200_RECORD_REF)" % (module, test, n)
    return answers[n]


def _record(module, key, arr):
    if RECORD:
        if not _recorded:
            atexit.register(_flush)
        test, n = key
        answers = _recorded.setdefault(module, {}).setdefault(test, [])
        assert n == len(answers)
        answers.append(np.ascontiguousarray(arr).ravel())


def _flush():
    os.makedirs(RECORD, exist_ok=True)
    for module, new in _recorded.items():
        path = os.path.join(RECORD, module + ".npz")
        tests = _load(path)
        tests.update(new)
        out = {}
        for test, answers in tests.items():
            sizes = [a.nbytes for a in answers]
            offsets = np.cumsum([0] + sizes[:-1])
            out[test + ":data"] = np.frombuffer(b"".join(a.tobytes() for a in answers), dtype=np.uint8)
            out[test + ":table"] = np.array([(str(o), str(n), a.dtype.str) for o, n, a in zip(offsets, sizes, answers)])
        np.savez_compressed(path, **out)


def _canonical(a):
    """bytes of `a` with every floating-point NaN replaced by one bit pattern (the payload is not part of the contract)"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.array(np.nan, dtype=a.dtype), a)
    return a.view(np.uint8).tobytes()


def _digest(a):
    return np.frombuffer(hashlib.blake2b(_canonical(a), digest_size=8).digest(), dtype=np.uint8)


def _positions(key, size):
    if size <= SAMPLE:
        return slice(None)
    rng = np.random.default_rng(zlib.crc32(("%s#%d" % key).encode()))
    return np.sort(rng.choice(size, SAMPLE, replace=False))


def value(fn):
    module, key = _key()
    if not LIVE:
        return _stored(module, key)
    v = np.asarray(fn())
    _record(module, key, v)
    return v


def same(fn, got, msg=None):
    module, key = _key()
    got = np.asarray(got)
    if not LIVE:
        assert np.array_equal(_digest(got), _stored(module, key)), (msg, "differs from the stored reference answer")
        return
    want = np.asarray(fn())
    _record(module, key, _digest(want))
    assert want.shape == got.shape and _canonical(want) == _canonical(got), msg


def sampled(fn, got):
    module, key = _key()
    got = np.asarray(got).ravel()
    if not LIVE:
        want = _stored(module, key)
        return (None if want.size == 0 else want), got[_positions(key, got.size)]
    want = fn()
    if want is None:
        _record(module, key, np.zeros(0))
        return None, got
    want = np.asarray(want).ravel()
    _record(module, key, want[_positions(key, want.size)])
    return want, got
