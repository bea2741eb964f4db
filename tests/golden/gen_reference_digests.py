#!/usr/bin/env python
"""Records tests/golden/reference_digests.json, the reference's outputs that tests/recorded.py checks.

    python tests/golden/gen_reference_digests.py

Runs the tests that compare with the reference with recording switched on.  It needs oracle/_ref/ref_harness
(the reference's build, oracle/Makefile), so that every recorded output has just been compared with the
reference's own, and it writes nothing unless all of those tests pass.

The committed file was recorded from the oracle and the product without the reference's build, at a revision
where these same tests, with the same code and inputs, had last passed against it bit for bit.  The bracket_*
cases are the exception: they record the int16 oracle's outputs on the float bracket's inputs, which were
only bracketed, not compared bit for bit, against the reference.
"""
import json
import os
import sys

import pytest

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROOT = os.path.dirname(TESTS)
SELECTION = ["test_oracle_vs_live_reference.py", "test_float_oracle_bracketed_by_reference.py",
             "test_cpp_host.py::test_wav_nodes_vs_live_reference"]


def main():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_harness")):
        sys.exit("oracle/_ref/ref_harness is not built: only outputs compared with the reference's may be recorded")
    sys.path.insert(0, TESTS)
    import recorded
    recorded.RECORD = {}
    if pytest.main(["-q", "-p", "no:cacheprovider"] + [os.path.join(TESTS, s) for s in SELECTION]) != 0:
        sys.exit("a comparison failed: nothing recorded")
    with open(recorded.PATH, "w") as f:
        json.dump(recorded.RECORD, f, indent=1, sort_keys=True)
        f.write("\n")
    print("recorded %d cases in %s" % (len(recorded.RECORD), recorded.PATH))


if __name__ == "__main__":
    main()
