"""Stored digests of what the reference's own code returned in the tests that pin the oracle on it bit for bit.

Those tests compare the oracle's restatements with the reference's own loops compiled from the reference tree
(oracle/_ref/libkkref.so, see oracle/Makefile).  That library can only be built where the reference tree is present, so each
such test also hashes the arrays it compared and checks the hash against tests/golden/reference_digests.json: where the
library is absent, the comparison with the reference still runs against its recorded results.  A digest covers dtype,
shape and values, with -0.0 read as 0.0 and every NaN as one NaN (the equality np.array_equal tests).  To record the
digests again, build oracle/_ref and run the tests with B200SP_RECORD_REFERENCE_DIGESTS=1: every test then asserts its
live comparison first and stores the digest of arrays equal to the reference's output."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
RECORD = os.environ.get("B200SP_RECORD_REFERENCE_DIGESTS") == "1"
_stored = None


def digest(arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.array(a, order="C")  # a copy in logical (C) order
        if a.dtype.kind == "f":
            a += a.dtype.type(0)  # -0.0 -> 0.0
            a[np.isnan(a)] = np.nan
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()[:32]


def _load():
    global _stored
    if _stored is None:
        with open(PATH) as f:
            _stored = json.load(f)
    return _stored


class Case:
    """The arrays one test case compared with the reference, in the order it compared them."""

    def __init__(self, live, *key):
        self.live = live  # the reference's library is loaded and the test compared with it directly
        self.key = "/".join(str(k) for k in key)
        self.arrays = []

    def add(self, *arrays):
        self.arrays.extend(arrays)

    def check(self):
        d = digest(self.arrays)
        if RECORD:
            assert self.live, f"{self.key}: recording needs oracle/_ref/libkkref.so"
            stored = _load()
            stored[self.key] = d
            with open(PATH, "w") as f:
                json.dump(stored, f, indent=0, sort_keys=True)
                f.write("\n")
            return
        want = _load().get(self.key)
        assert want is not None, f"{self.key}: no recorded digest of the reference's output"
        assert d == want, f"{self.key}: the output differs from the reference's recorded output"
