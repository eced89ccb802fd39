"""Writes tests/golden/wire_format_golden.npz: the bytes the REFERENCE's serialize() (pairhmm/interface/PairHMMHostInterface.cpp,
compiled into oracle/_ref/libhostif_ref.so by oracle/Makefile) writes for the cases of tests/test_wire_format_ref.py, reads and
haplotypes, as uint8 arrays named <case>/reads and <case>/haps.
    python tests/golden/make_wire_golden.py            # from the reference's own writer (needs oracle/_ref)
    python tests/golden/make_wire_golden.py --writer   # from acc_genomics_b200.batch's writer

The committed file was written with --writer, because the reference's sources are not part of this repository.  Those bytes are
the reference's: tests/test_wire_format_ref.py had checked this writer byte for byte against the reference's serialize() on
exactly these cases (DESIGN.md section 6), and neither the writer nor the case generator changed after that check.  Regenerate
with --writer only from a tree whose writer has passed that live check.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import test_wire_format_ref as T  # noqa: E402
from acc_genomics_b200 import batch as B  # noqa: E402


def main():
    ref = None
    if "--writer" not in sys.argv:
        ref = T.load_reference()
        assert ref is not None, "oracle/_ref/libhostif_ref.so is not built (needs the reference's sources)"
    out = {}
    for case in sorted(T.CASES):
        b = T.CASES[case]()
        rs, hs = T.ref_serialize(ref, b)["ptr"] if ref is not None else (B.serialize_reads(b), B.serialize_haps(b))
        out[f"{case}/reads"] = np.frombuffer(rs, dtype=np.uint8)
        out[f"{case}/haps"] = np.frombuffer(hs, dtype=np.uint8)
        print(f"{case}: {len(rs)} + {len(hs)} bytes")
    path = os.path.join(HERE, "wire_format_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
