"""Recorded outputs for the tests that compare with the reference (libsdr itself).

A build of the reference (oracle/_ref/ref_harness, compiled by oracle/Makefile from libsdr's sources) is
not part of this repository, so those tests also check their outputs on the same seeded inputs against
SHA-256 digests recorded when the outputs matched the reference's: tests/golden/reference_digests.json maps
a case name to the digest of every output array of the case.  tests/golden/gen_reference_digests.py records
them and says where each came from.
"""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
RECORD = None        # gen_reference_digests.py sets a dict here: check() then records instead of comparing
_table = None


def digest(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def check(case, **arrays):
    """Every array equals, bit for bit (dtype and shape included), the reference's recorded output."""
    global _table
    got = {k: digest(v) for k, v in arrays.items()}
    if RECORD is not None:
        RECORD[case] = got
        return
    if _table is None:
        with open(PATH) as f:
            _table = json.load(f)
    assert case in _table, "no recorded reference outputs for " + case
    want = _table[case]
    assert sorted(got) == sorted(want), (case, sorted(got), sorted(want))
    bad = sorted(k for k in want if got[k] != want[k])
    assert not bad, "%s: %s differ from the reference's recorded outputs" % (case, ", ".join(bad))
