"""Stored outputs of the reference's own code, so that the tests comparing the oracle with it run without the reference.

The tests of tests/test_ref_pins.py, tests/test_ref_sources.py and tests/test_oracle_8pt.py compare the oracle with the
reference's unmodified sources (oracle/_ref, which can only be built where those sources are).  Every reference call of
those tests goes through a RefStore, keyed by test name and call number:
  * oracle/_ref built: the reference is called, and its result must equal the stored one;
  * oracle/_ref absent: the stored result stands in for the call, so the comparison with the oracle still runs;
  * PLB_RECORD_REFERENCE=1 with oracle/_ref built: the store is rewritten from the reference's results (run the whole
    test module).
The inputs of these tests are generated from fixed seeds, so the n-th call of a test always sees the same input.
Where a test only asks for bitwise equality (REF.same), the store keeps one SHA-256 over all results of the test instead
of the results themselves: without the reference, the oracle's results must hash to it.
One file per test function: tests/golden/<store>/<test function>.pkl.xz."""
import hashlib
import lzma
import os
import pickle

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def same(a, b):
    """Bitwise equality of nested results (NaN equal to NaN)."""
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, (tuple, list)):
        return isinstance(b, (tuple, list)) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind in "fc" or b.dtype.kind in "fc":
        return bool(np.array_equal(a, b, equal_nan=True))
    return bool(np.array_equal(a, b))


def canonical(a):
    """Bytes that are equal exactly when `same` holds (NaN, and -0.0 / 0.0, each in one form; bools and ints alike)."""
    if isinstance(a, dict):
        return b"D%d" % len(a) + b"".join(canonical(k) + canonical(a[k]) for k in sorted(a))
    if isinstance(a, (tuple, list)):
        return b"L%d" % len(a) + b"".join(canonical(x) for x in a)
    if isinstance(a, str):
        return b"S" + a.encode()
    a = np.asarray(a)
    if a.dtype.kind in "fc":
        a = np.asarray(a, dtype=np.complex128 if a.dtype.kind == "c" else np.float64) + 0.0
        a = np.where(np.isnan(a), np.nan, a)
    else:
        a = a.astype(np.int64)
    return b"A" + a.dtype.str.encode() + repr(a.shape).encode() + np.ascontiguousarray(a).tobytes()


class RefStore:
    def __init__(self, name, live):
        self.dir = os.path.join(HERE, name)
        self.live = bool(live)
        self.record = self.live and os.environ.get("PLB_RECORD_REFERENCE") == "1"
        self.files = {}  # test function -> {key: result}
        self.data, self.test, self.calls, self.stored, self.hash = None, None, 0, True, None

    def begin(self, node, stored=True):
        """Start a test (a pytest item).  stored=False: a test that runs only where the reference is; nothing is kept."""
        self.test, self.calls, self.stored, self.hash = node.name, 0, stored, hashlib.sha256()
        func = node.originalname
        if func not in self.files:
            path = os.path.join(self.dir, func + ".pkl.xz")
            if self.record or not stored or not os.path.exists(path):  # nothing stored: a test without reference calls
                self.files[func] = {}
            else:
                with lzma.open(path, "rb") as f:
                    self.files[func] = pickle.load(f)
        self.data = self.files[func]

    def __call__(self, call):
        """The result of `call()` (a call into the reference), or its stored value where the reference is absent."""
        key = f"{self.test}#{self.calls}"
        self.calls += 1
        if not self.live:
            if key not in self.data:
                raise KeyError(f"no stored reference result for {key}: regenerate with PLB_RECORD_REFERENCE=1")
            return self.data[key]
        value = call()
        if self.record and self.stored:
            self.data[key] = value
        elif self.stored:
            assert key in self.data and same(value, self.data[key]), f"the reference's result for {key} differs from the stored one"
        return value

    def same(self, call, ours):
        """Bitwise equality of `ours` with the result of `call()` (a call into the reference).  Without the reference it is
        decided by end(), which compares the hash of all of the test's results with the stored one."""
        if not self.live:
            self.hash.update(canonical(ours))
            return True
        ref = call()
        self.hash.update(canonical(ref))
        return same(ref, ours)

    def end(self):
        """Finish a test: the hash of its REF.same results must be the stored one (recorded with PLB_RECORD_REFERENCE=1)."""
        key, digest = f"{self.test}#sha256", self.hash.hexdigest()
        if self.hash.digest() == hashlib.sha256().digest() or not self.stored:
            return  # no REF.same in this test
        if self.record:
            self.data[key] = digest
        else:
            assert self.data.get(key) == digest, f"{self.test}: results differ from the reference's (hash of all results)"

    def save(self):
        if not self.record:
            return
        os.makedirs(self.dir, exist_ok=True)
        for func, data in self.files.items():
            if data:
                with lzma.open(os.path.join(self.dir, func + ".pkl.xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as f:
                    pickle.dump(data, f, protocol=4)
