"""Digests of what the UNMODIFIED reference code (oracle/_ref, compiled from the reference sources by oracle/Makefile)
returns on the seeded inputs of the tests that compare with it, stored in reference_digests.json by
tests/golden/make_golden_digests.py.  The tests compare their own outputs with these digests, so the comparison with the
reference runs where its sources are not available.  Integer arrays are hashed by value (as int64) with their shape, so
equal digests mean the arrays are np.array_equal."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_digests.json")
_table: dict = {}


def digest(x) -> str:
    h = hashlib.sha256()
    if isinstance(x, np.ndarray):
        a = x.astype("<i8") if x.dtype.kind in "biu" else x.astype("<f8") if x.dtype.kind == "f" else x
        h.update(repr(a.shape).encode())
        h.update(a.dtype.str.encode())
        h.update(np.ascontiguousarray(a).tobytes())
    else:
        h.update(json.dumps(x).encode())
    return h.hexdigest()[:24]


def digests(fields: dict) -> dict:
    return {k: digest(v) for k, v in fields.items()}


def variant_fields(w: dict, images_to_int8) -> dict:
    """oracle.variant_encode output -> the compared fields (images as the encoder's int32 and as the stored int8)."""
    return dict(keys=list(w["keys"]), positions=w["positions"], depths=w["depths"], freqs=w["freqs"], region_of=w["region_of"],
                images=w["images"], images_i8=images_to_int8(w["images"]))


def reads_fields(reads, pos_end, n_bad) -> dict:
    f = {k: getattr(reads, k) for k in ("pos", "seq_off", "cigar_off", "flags", "mapq", "seq", "qual", "cigar")}
    return dict(f, pos_end=pos_end, n_bad=n_bad)


def expect(case: str, fields: dict) -> None:
    """Every field given must equal the reference's output for `case`."""
    if not _table:
        with open(PATH) as f:
            _table.update(json.load(f))
    want = _table[case]
    assert fields and set(fields) <= set(want), (case, sorted(fields), sorted(want))
    bad = [k for k, v in digests(fields).items() if v != want[k]]
    assert not bad, "%s: differs from the reference output in %s" % (case, bad)
