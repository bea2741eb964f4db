"""The bit-exact integer arithmetic of IQBaseBand<int16_t> / <int8_t> is written once, in
libsdr_b200/csrc/iqbb_int_common.cuh, for the single-channel and the channel-bank kernels.  A second copy of the NCO
product or of a small device helper could drift from the first and break bit-exactness for only some shapes, tap counts
or channel counts."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "libsdr_b200", "csrc")

NCO_PRODUCT = r"\(uint32_t\)\w+\.x \* \(uint32_t\)\w+ - \(uint32_t\)\w+\.y \* \(uint32_t\)\w+"
HELPERS = {"unpack16": "void", "pad32": "int", "warp_sum": "float", "cp_async_commit": "void"}


def _sources():
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh", ".cc", ".h")):
            yield name, open(os.path.join(CSRC, name), encoding="utf-8").read()


def test_integer_nco_product_is_written_once():
    hits = [(name, m.group(0)) for name, text in _sources() for m in re.finditer(NCO_PRODUCT, text)]
    assert len(hits) == 1, hits
    assert hits[0][0] == "iqbb_int_common.cuh", hits


def test_shared_device_helpers_are_defined_once():
    for helper, ret in HELPERS.items():
        definition = re.compile(r"\b%s\s+%s\s*\(" % (ret, helper))
        where = [name for name, text in _sources() for _ in definition.finditer(text)]
        assert len(where) == 1, (helper, where)
