"""Stored digests of what the reference side returned in the tests that compare with the compiled reference
(oracle/_ref), so that each of those comparisons also runs where oracle/_ref is not built.

A test hands expect() the arrays of the code under test and, where oracle/_ref is built, the same arrays from the
reference: they must be equal, and their SHA-256 must be the one stored in tests/golden/reference_pins_v1.json.
With SDR_RECORD_PINS=<file> set, expect() records the digests into <file> instead, with the side they were checked
against: the compiled reference where oracle/_ref is built, else the oracle (oracle/sdr_oracle.c)."""
import atexit
import hashlib
import json
import os

import numpy as np

import _oracle as O

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins_v1.json")
_RECORD = os.environ.get("SDR_RECORD_PINS")
if _RECORD and not os.path.exists(PATH):
    PINS = {}
else:
    with open(PATH) as f:
        PINS = json.load(f)["pins"]
_recorded = {}


def digest(arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s;" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def expect(key, got, ref=None):
    """got, ref: lists of arrays (ref None where oracle/_ref is not built)."""
    if ref is not None:
        assert len(got) == len(ref), key
        for i, (a, b) in enumerate(zip(got, ref)):
            a, b = np.asarray(a), np.asarray(b)
            assert a.shape == b.shape and a.tobytes() == b.astype(a.dtype).tobytes(), \
                "%s: item %d differs from the compiled reference" % (key, i)
    if _RECORD:
        _recorded[key] = {"sha256": digest(got), "from": "compiled reference" if O.ref("radiodiags") else "oracle"}
        return
    assert key in PINS, "no stored pin for %s" % key
    assert digest(got) == PINS[key], "%s differs from what the compiled reference returned" % key


@atexit.register
def _write():
    if _RECORD and _recorded:
        old = {}
        if os.path.exists(_RECORD):
            with open(_RECORD) as f:
                old = json.load(f)
        old.update(_recorded)
        with open(_RECORD, "w") as f:
            json.dump(old, f, indent=1, sort_keys=True)
